"""CPU restatement of the VB-PCA plate with known per-entry observation weights, mode B.

TEST INFRASTRUCTURE ONLY, like plate_oracle.py: the checker of ``PlateEngine(..., weights=S)``.

Model: x_nd ~ N(w_d . z_n + mu_d, 1 / (tau s_nd)) for every entry with x_nd not NaN and s_nd > 0 (with per-dimension noise
1 / (tau_d s_nd)).  The per-row noise precision of the masked plate, Lambda_n = tau diag(mask_n), becomes tau diag(s_n): the
reference's generic operators take an arbitrary per-row Constant precision (nodes/node.py:203-227), so the Z, W and Mu updates
are those of PlateOracle with the effective mask E() replaced by S (zero where x is missing).  What S does NOT replace is the
count of observations:

  Beta   qa = a0 + nE / 2 with nE the NUMBER of observed entries of positive weight; qb = b0 + resid2 / 2 with the weighted
         resid2 = sum_nd s_nd <(x_nd - w_d z_n - mu_d)^2>
  bound  X term  -nE/2 ln 2pi + nE/2 (ln qa - ln qb) - tau resid2 / 2 + 1/2 sum_{s_nd > 0} ln s_nd
         (the last term is the data constant of the precisions tau s_nd; ln<tau> as the unweighted model)

With S = the 0/1 mask both classes reduce to PlateOracle / DiagNoiseOracle exactly (test_oracle_weights.py checks it).
"""
import numpy as np

from oracle.noise_oracle import DiagNoiseOracle
from oracle.plate_oracle import LN2PI, PlateOracle


def effective_weights(X, weights):
    """(S, C): S the weights with zeros where x is missing, C the 0/1 mask of the observed entries of positive weight."""
    O = ~np.isnan(np.asarray(X, dtype=np.float64))
    S = np.where(O, np.asarray(weights, dtype=np.float64), 0.0)
    return S, (S > 0)


class _Weighted(object):
    """What the weighted classes share: S in place of the mask, the count C kept apart, the data constant of the bound."""

    def _set_weights(self, weights):
        self.S, self.C = effective_weights(self.X, weights)

    def E(self):
        return self.S

    def lns(self):
        """1/2 sum over the observed entries of positive weight of ln s_nd."""
        return 0.5 * float(np.sum(np.log(self.S[self.C])))


class WeightedPlateOracle(_Weighted, PlateOracle):
    """PlateOracle (mode B, scalar noise) with per-entry weights."""

    def __init__(self, X, q, weights, **kw):
        if kw.pop("mode", "B") != "B":
            raise ValueError("observation weights are a mode-B model")
        super().__init__(X, q, mode="B", **kw)
        self._set_weights(weights)
        self.qa = self.a0 + 0.5 * self.C.sum()

    def elbo_terms(self):
        t = super().elbo_terms()
        nE = float(self.C.sum())
        t["X"] = float(-0.5 * nE * LN2PI + 0.5 * nE * (np.log(self.qa) - np.log(self.qb)) - 0.5 * self.tau * self._resid2()
                       + self.lns())
        return t


class WeightedDiagNoiseOracle(_Weighted, DiagNoiseOracle):
    """DiagNoiseOracle (per-dimension noise) with per-entry weights."""

    def __init__(self, X, q, weights, a0=1e-3, b0=1e-3, **kw):
        super().__init__(X, q, a0=a0, b0=b0, **kw)
        self._set_weights(weights)
        self.qa = self.a0 + 0.5 * self.C.sum(0)

    def elbo_terms(self):
        t = super().elbo_terms()
        cnt = self.C.sum(0).astype(np.float64)
        qa, qb = self.qa, self.qb
        t["X"] = float(np.sum(-0.5 * cnt * LN2PI + 0.5 * cnt * (np.log(qa) - np.log(qb)) - 0.5 * (qa / qb) * self.resid_d())
                       + self.lns())
        return t


def synth_weighted(N, D, q, missing, tau, decades=3.0, seed=0):
    """(X, S, W): data whose entries have known precisions tau * s_nd, s log-uniform over `decades` decades (geometric mean
    1), with Bernoulli(missing) erasures; W the true loading matrix."""
    rng = np.random.RandomState(seed)
    W, Z, mu = rng.randn(D, q), rng.randn(N, q), rng.randn(D)
    S = 10.0 ** rng.uniform(-0.5 * decades, 0.5 * decades, size=(N, D))
    X = Z @ W.T + mu[None, :] + rng.randn(N, D) / np.sqrt(tau * S)
    if missing > 0:
        X[rng.rand(N, D) < missing] = np.nan
    return X, S, W
