"""CPU restatement of the VB-PCA plate with a row-wise W posterior, mode B.

TEST INFRASTRUCTURE ONLY, like plate_oracle.py: the checker of ``PlateEngine(..., w_posterior="rows")``.

Model: the likelihood of the plate classes it mixes into (PlateOracle, DiagNoiseOracle and their weighted forms) with
q(W) = prod_d N(w_d | wbar_d, Sigma_d) -- one full q x q covariance per data dimension (Ilin & Raiko 2010) in place of the
q column nodes of the reference's ``hstack`` (diagonal covariances).  With the statistics T1_d = sum_n e_nd <z_n z_n^T>,
Ast_d = sum_n e_nd x_nd zbar_n, Bst_d = sum_n e_nd zbar_n (e the mask, or the weights):

  W      Lambda_d = diag(<alpha>) + tau_d T1_d,  eta_d = tau_d (Ast_d - mu_d Bst_d),  Sigma_d = Lambda_d^-1,  wbar_d = Sigma_d eta_d
  G      G_d = wbar_d wbar_d^T + Sigma_d  (the Z step and the residual read it; nothing else changes)
  Wvar   diag Sigma_d (the ARD update and the prior part of the W bound read it, as before)
  bound  W: sum_i [-D/2 ln 2pi + 1/2 ln det(alpha_i I_D) - alpha_i/2 sum_d <w_di^2>]          (prior part, unchanged)
            - sum_d [-q/2 ln 2pi - 1/2 qld_d - q/2],  qld_d = 0.5 / ln prod diag chol(Lambda_d)   (entropy of D row nodes)
         with the reference's q_ln_det quirk (gaussian.py:120) applied per row node, as PlateOracle applies it per column node.

q = 1: every update equals the column oracle's.  The bound's W entropy groups the quirk by node, so it equals the column
oracle's only when the nodes coincide too (D = 1); test_oracle_wrows.py checks both.
"""
import numpy as np

from oracle.noise_oracle import DiagNoiseOracle
from oracle.plate_oracle import LN2PI, PlateOracle
from oracle.weights_oracle import WeightedDiagNoiseOracle, WeightedPlateOracle


class _WRows(object):
    """What the row-wise classes share: the W step, G, the W bound term and the Wcov state key."""

    STATE_KEYS = PlateOracle.STATE_KEYS + ("Wcov",)

    @property
    def Wcov(self):
        if getattr(self, "_Wcov", None) is None:
            self._Wcov = np.einsum("di,ij->dij", self.Wvar, np.eye(self.q))
        return self._Wcov

    @Wcov.setter
    def Wcov(self, v):
        self._Wcov = np.array(v, dtype=np.float64)

    def taus(self):
        return np.broadcast_to(np.asarray(self.tau, dtype=np.float64), (self.D,))

    def update_W(self):
        q, E = self.q, self.E()
        T1 = (E.T @ self.M2().reshape(self.N, q * q)).reshape(self.D, q, q)
        T2 = (E * (self.Xe() - self.mu[None, :])).T @ self.Zbar
        tau = self.taus()
        Lam = np.diag(self.alpha())[None] + tau[:, None, None] * T1
        eta = tau[:, None] * T2
        np.linalg.cholesky(Lam)                  # raises LinAlgError on a row that is not positive definite
        S = np.linalg.inv(Lam)
        S = 0.5 * (S + np.transpose(S, (0, 2, 1)))
        self.Wcov = S
        self.Wbar = np.einsum("dij,dj->di", S, eta)
        self.Wvar = np.diagonal(S, axis1=1, axis2=2).copy()

    def Wld(self):
        """ln prod diag chol(Lambda_d) = -1/2 ln det Sigma_d per row."""
        return -0.5 * np.linalg.slogdet(self.Wcov)[1]

    def G(self):
        return self.Wbar[:, :, None] * self.Wbar[:, None, :] + self.Wcov

    def elbo_terms(self):
        t = super().elbo_terms()
        D, q = self.D, self.q
        al = self.alpha()
        lndet_al = D * (np.log(self.al_qa) - np.log(self.al_qb)) if self.ard else np.full(q, D * np.log(self.alpha0))
        ww = np.sum(self.Wbar ** 2, 0) + np.sum(self.Wvar, 0)
        prior = np.sum(-0.5 * D * LN2PI + 0.5 * lndet_al - 0.5 * al * ww)
        qld = 0.5 / self.Wld()
        t["W"] = float(prior - np.sum(-0.5 * q * LN2PI - 0.5 * qld - 0.5 * q))
        return t

    def load_state(self, st):
        st = dict(st)
        wcov = st.pop("Wcov", None)
        super().load_state(st)
        if wcov is not None:
            self.Wcov = wcov
            self.Wvar = np.diagonal(self.Wcov, axis1=1, axis2=2).copy()
        elif "Wvar" in st:
            self._Wcov = None

    def state(self):
        out = super().state()
        out["Wcov"] = self.Wcov.copy()
        return out


class WRowsPlateOracle(_WRows, PlateOracle):
    """PlateOracle (mode B, scalar noise) with the row-wise W posterior."""

    def __init__(self, X, q, **kw):
        if kw.pop("mode", "B") != "B":
            raise ValueError("the row-wise W posterior is a mode-B model")
        super().__init__(X, q, mode="B", **kw)


class WRowsDiagNoiseOracle(_WRows, DiagNoiseOracle):
    """DiagNoiseOracle (per-dimension noise) with the row-wise W posterior."""


class WRowsWeightedPlateOracle(_WRows, WeightedPlateOracle):
    """WeightedPlateOracle with the row-wise W posterior."""


class WRowsWeightedDiagNoiseOracle(_WRows, WeightedDiagNoiseOracle):
    """WeightedDiagNoiseOracle with the row-wise W posterior."""


def synth_correlated(N, D, q, missing, seed=0, noise_prec=20.0, rho=0.8, spread=10.0):
    """Data whose W_true has correlated columns of spread scales: W = G C^T diag(s), with C the Cholesky factor of the
    AR(1) correlation rho^|i-j| and column scales s log-spaced over `spread`; returns (X, W_true)."""
    rng = np.random.RandomState(seed)
    idx = np.arange(q)
    C = np.linalg.cholesky(rho ** np.abs(idx[:, None] - idx[None, :]))
    s = np.logspace(0.0, -np.log10(spread), q)
    W = (rng.randn(D, q) @ C.T) * s[None, :]
    Z = rng.randn(N, q)
    mu = rng.randn(D)
    X = Z @ W.T + mu[None, :] + rng.randn(N, D) / np.sqrt(noise_prec)
    if missing > 0:
        X[rng.rand(N, D) < missing] = np.nan
    return X, W
