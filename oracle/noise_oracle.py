"""CPU restatement of the VB-PCA plate with per-dimension noise precisions (factor analysis), mode B.

TEST INFRASTRUCTURE ONLY, like plate_oracle.py: the checker of ``PlateEngine(..., noise="diagonal")``.

Model: x_nd ~ N(w_d . z_n + mu_d, 1 / tau_d) for the observed entries, tau_d ~ Gamma(a0_d, b0_d) with one Gamma
posterior per data dimension -- the reference's ``DiagonalGamma`` (nodes/nodes_todo.py:159-204: update 187-190, bound
198-203) as the noise node of the masked plate.  Everything else is PlateOracle's mode B with Lambda_n = diag(tau * O_n):

  Z     qprec_n = P0 + sum_d O_nd tau_d G_d,  eta_n = h0 + sum_d O_nd tau_d (x_nd - mu_d) wbar_d
  W     prec_di = alpha_i + tau_d T1_d[ii],   wbar_di = tau_d m2 / prec_di
  Mu    prec_d  = alpha_mu + tau_d cnt_d,     mu_d = tau_d (colx_d - wbar_d . Bst_d) / prec_d
  Beta  qa_d = a0_d + cnt_d / 2 (constant),   qb_d = b0_d + r_d / 2,  r_d = sum_n O_nd <(x_nd - w_d z_n - mu_d)^2>
  bound X: sum_d [-cnt_d/2 ln 2pi + cnt_d/2 (ln qa_d - ln qb_d) - tau_d r_d / 2]  (ln<tau>, as the scalar model);
        Beta: the sum over d of the Gamma bound.  W, Mu, Z, Alpha: unchanged.

With every qb_d equal to qb and shared priors the updates reduce to PlateOracle's (test_oracle_noise_diag.py checks it).
"""
import numpy as np

from oracle.plate_oracle import PlateOracle


class DiagNoiseOracle(PlateOracle):
    """PlateOracle (mode B) with qa, qb, a0, b0 of shape (D,)."""

    def __init__(self, X, q, a0=1e-3, b0=1e-3, **kw):
        if kw.pop("mode", "B") != "B":
            raise ValueError("per-dimension noise is a mode-B model")
        super().__init__(X, q, mode="B", **kw)
        D = self.D
        self.a0 = np.broadcast_to(np.asarray(a0, dtype=np.float64), (D,)).copy()
        self.b0 = np.broadcast_to(np.asarray(b0, dtype=np.float64), (D,)).copy()
        self.qa = self.a0 + 0.5 * self.O.sum(0)
        self.qb = np.full(D, 0.5)

    # update_W and update_Mu of PlateOracle broadcast tau over d already; the Z step needs tau inside the row sums
    def update_Z(self, lo=0, hi=None):
        hi = self.N if hi is None else hi
        q = self.q
        Et = self.E()[lo:hi] * self.tau[None, :]                 # O_nd tau_d
        Gf = self.G().reshape(self.D, q * q)
        L = self.P0[None] + (Et @ Gf).reshape(-1, q, q)
        eta = (self.P0 @ self.m0)[None, :] + (Et * (self.Xe()[lo:hi] - self.mu[None, :])) @ self.Wbar
        U = np.linalg.cholesky(L)
        Sig = np.linalg.inv(L)
        Sig = 0.5 * (Sig + np.transpose(Sig, (0, 2, 1)))
        self.Sig[lo:hi] = Sig
        self.Zbar[lo:hi] = np.einsum("nij,nj->ni", Sig, eta)
        self.qldZ[lo:hi] = 0.5 / np.sum(np.log(np.diagonal(U, axis1=1, axis2=2)), axis=1)

    def resid_d(self):
        """r_d = sum_n O_nd <(x_nd - w_d z_n - mu_d)^2>, shape (D,)."""
        E, q = self.E(), self.q
        m = self.Zbar @ self.Wbar.T + self.mu[None, :]
        trGM = self.M2().reshape(self.N, q * q) @ self.G().reshape(self.D, q * q).T
        wz = self.Zbar @ self.Wbar.T
        per = (self.Xe() - m) ** 2 + trGM - wz ** 2 + self.muvar[None, :]
        return np.sum(E * per, axis=0)

    def update_Beta(self):
        self.qb = self.b0 + 0.5 * self.resid_d()

    def elbo_terms(self):
        # the W, Mu, Z and Alpha terms do not involve the noise: PlateOracle's, evaluated with a placeholder scalar Gamma
        qa, qb, a0, b0 = self.qa, self.qb, self.a0, self.b0
        self.qa, self.qb, self.a0, self.b0 = 1.0, 1.0, 1.0, 1.0
        try:
            t = super().elbo_terms()
        finally:
            self.qa, self.qb, self.a0, self.b0 = qa, qb, a0, b0
        cnt = self.O.sum(0).astype(np.float64)
        LN2PI = np.log(2.0 * np.pi)
        t["X"] = float(np.sum(-0.5 * cnt * LN2PI + 0.5 * cnt * (np.log(qa) - np.log(qb)) - 0.5 * (qa / qb) * self.resid_d()))
        t["Beta"] = float(np.sum(self._gamma_llb(a0, b0, qa, qb)))
        return t

    def load_state(self, st):
        st = dict(st)
        qb = st.pop("qb", None)
        super().load_state(st)
        if qb is not None:
            self.qb = np.broadcast_to(np.asarray(qb, dtype=np.float64), (self.D,)).copy()

    def state(self):
        out = super().state()
        out["qb"] = self.qb.copy()
        return out


def synth_fa(N, D, q, missing, tau, seed=0):
    """Factor-analysis data: x_nd = w_d . z_n + mu_d + noise of precision tau_d, with Bernoulli(missing) erasures."""
    rng = np.random.RandomState(seed)
    W, Z, mu = rng.randn(D, q), rng.randn(N, q), rng.randn(D)
    X = Z @ W.T + mu[None, :] + rng.randn(N, D) / np.sqrt(np.asarray(tau, dtype=np.float64))[None, :]
    if missing > 0:
        X[rng.rand(N, D) < missing] = np.nan
    return X
