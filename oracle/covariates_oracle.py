"""CPU restatement of the VB-PCA plate with known per-row covariates (fixed effects), mode B.

TEST INFRASTRUCTURE ONLY, like plate_oracle.py: the checker of ``PlateEngine(..., covariates=C)``.

Model: x_nd ~ N(w_d . z_n + b_d . c_n + mu_d, 1/tau) (1/tau_d with per-dimension noise; 1/(tau s_nd) with weights) for the
observed entries, with c_n (k,) known, z_n ~ N(m0, P0^-1) free (q,), and the effects B (D, k) a Gaussian node of the same
kind as W: with column posteriors, q(W, B) is the product of the q + k column nodes of [W | B] (prior precision alpha_i,
shared alpha0 or one ARD Gamma per column, B's columns included); with the row-wise posterior, q(w_d, b_d) is one joint
(q + k)-dimensional Gaussian per data dimension.  The mixin keeps the loadings as one (D, q + k) array [W | B] and the latent
rows as [zbar_n | c_n]; the known columns have no variance (Sig_n has zero blocks beyond the free q x q one).

  Z     A_n = P0 + sum_d e_nd tau_d E[w_d w_d^T]
        e_n = P0 m0 + sum_d e_nd tau_d [(x_nd - mu_d - bbar_d . c_n) wbar_d - Cov(w_d, b_d) c_n]
            (the last two terms are -E[w_d b_d^T] c_n + (x_nd - mu_d) wbar_d; Cov(w_d, b_d) = 0 with column posteriors)
        Sigma_n = A_n^-1, zbar_n = Sigma_n e_n
  W, B  the base class's update on the second moments <[z;c][z;c]^T>_n = [[<zz^T>_n, zbar_n c_n^T], [c_n zbar_n^T,
        c_n c_n^T]] (the mixin keeps Sig's known blocks at zero, so M2() is exactly these): Gauss-Seidel over the columns of
        [W | B] (columns) or one joint solve per row (rows)
  Mu, tau  the base class's, on the same moments: their residual is x_nd - w_d . z_n - b_d . c_n - mu_d
  bound Z: the KL terms of the q free dimensions only (written here);  W: the base class's prior / entropy terms of every
        column node (or row node) of [W | B], so B's KL is that of W's columns;  X, Beta, Alpha: the base class's.
  test_oracle_covariates.py restates the column-mode W / B step, Mu and the residual from the model (x - w z - b c - mu,
  <(b_d . c_n)^2> = c_n^T E[b_d b_d^T] c_n) and checks the mixin against them.

With every c_n = 0 the free part equals the covariate-free model, and B stays at its prior: bbar = 0, Bvar = 1 / alpha
(test_oracle_covariates.py checks it, and checks the direct Z step against conditioning a q + k Gaussian on its known tail).
"""
import numpy as np

from oracle.noise_oracle import DiagNoiseOracle
from oracle.plate_oracle import LN2PI, PlateOracle
from oracle.weights_oracle import WeightedDiagNoiseOracle, WeightedPlateOracle
from oracle.wrows_oracle import (WRowsDiagNoiseOracle, WRowsPlateOracle, WRowsWeightedDiagNoiseOracle,
                                 WRowsWeightedPlateOracle)


class _Covariates(object):
    """The mixin: construct as Base(X, q, covariates=C, ...) with q the number of free latent dimensions."""

    def __init__(self, X, q, covariates, P0=None, m0=None, **kw):
        C = np.asarray(covariates, dtype=np.float64)
        qz, k = int(q), int(C.shape[1])
        super().__init__(X, qz + k, **kw)
        self.qz, self.k, self.cov_c = qz, k, C
        self.P0z = np.eye(qz) if P0 is None else np.asarray(P0, dtype=np.float64).reshape(qz, qz)
        self.m0z = np.zeros(qz) if m0 is None else np.asarray(m0, dtype=np.float64).reshape(qz)
        # the base class's prior is read by nothing but update_Z / the Z bound, which the mixin replaces
        self.P0 = np.zeros((qz + k, qz + k))
        self.P0[:qz, :qz] = self.P0z
        self.m0 = np.zeros(qz + k)
        self.Zbar[:, qz:] = C
        self.Sig[:, qz:, :] = 0.0
        self.Sig[:, :, qz:] = 0.0

    def taus(self):
        return np.broadcast_to(np.asarray(self.tau, dtype=np.float64), (self.D,))

    def update_Z(self, lo=0, hi=None):
        hi = self.N if hi is None else hi
        qz = self.qz
        Et = self.E()[lo:hi] * self.taus()[None, :]             # e_nd tau_d
        Gw = self.G()                                            # E[w'_d w'_d^T], w' = [w ; b]
        Eww = Gw[:, :qz, :qz].reshape(self.D, qz * qz)
        covwb = Gw[:, :qz, qz:] - self.Wbar[:, :qz, None] * self.Wbar[:, None, qz:]    # Cov(w_d, b_d) (D, q, k)
        c = self.cov_c[lo:hi]
        A = self.P0z[None] + (Et @ Eww).reshape(-1, qz, qz)
        r = self.Xe()[lo:hi] - self.mu[None, :] - c @ self.Wbar[:, qz:].T                # x - mu - bbar . c
        e = (self.P0z @ self.m0z)[None, :] + (Et * r) @ self.Wbar[:, :qz]
        e -= np.einsum("nd,dik,nk->ni", Et, covwb, c)
        U = np.linalg.cholesky(A)
        S = np.linalg.inv(A)
        S = 0.5 * (S + np.transpose(S, (0, 2, 1)))
        self.Sig[lo:hi, :qz, :qz] = S
        self.Zbar[lo:hi, :qz] = np.einsum("nij,nj->ni", S, e)
        self.qldZ[lo:hi] = 0.5 / np.sum(np.log(np.diagonal(U, axis1=1, axis2=2)), axis=1)

    def elbo_terms(self):
        t = super().elbo_terms()
        qz = self.qz
        Z, S = self.Zbar[:, :qz], self.Sig[:, :qz, :qz]
        M2 = Z[:, :, None] * Z[:, None, :] + S
        P0, m0 = self.P0z, self.m0z
        quad = np.einsum("ij,nji->n", P0, M2) + m0 @ P0 @ m0 - 2.0 * (Z @ (P0 @ m0))
        t["Z"] = float(np.sum(-0.5 * qz * LN2PI + 0.5 * np.linalg.slogdet(P0)[1] - 0.5 * quad
                              - (-0.5 * qz * LN2PI - 0.5 * self.qldZ - 0.5 * qz)))
        return t

    # ---- state in the engine's layout: Zbar (N, q), Sig (N, q, q), Wbar / Wvar (D, q), Bbar / Bvar (D, k)
    def user_state(self):
        qz = self.qz
        st = self.state()
        out = {"Zbar": st["Zbar"][:, :qz], "Sig": st["Sig"][:, :qz, :qz], "Wbar": st["Wbar"][:, :qz],
               "Bbar": st["Wbar"][:, qz:], "Wvar": st["Wvar"][:, :qz], "Bvar": st["Wvar"][:, qz:]}
        for key in ("mu", "muvar", "qb", "al_qb", "Wcov"):
            if key in st:
                out[key] = st[key]
        return {key: np.array(v, copy=True) for key, v in out.items()}

    def load_user_state(self, st):
        st = dict(st)
        qz = self.qz
        for a, b in (("Wbar", "Bbar"), ("Wvar", "Bvar")):
            if a in st or b in st:
                cur = np.array(getattr(self, a), copy=True)
                if a in st:
                    cur[:, :qz] = st[a]
                if b in st:
                    cur[:, qz:] = st.pop(b)
                st[a] = cur
        if "Zbar" in st:
            st["Zbar"] = np.concatenate([np.asarray(st["Zbar"], dtype=np.float64), self.cov_c], 1)
        if "Sig" in st:
            S = np.zeros((self.N, self.q, self.q))
            S[:, :qz, :qz] = st["Sig"]
            st["Sig"] = S
        self.load_state(st)


class CovPlateOracle(_Covariates, PlateOracle):
    """PlateOracle (mode B, scalar noise) with known covariates."""

    def __init__(self, X, q, covariates, **kw):
        if kw.pop("mode", "B") != "B":
            raise ValueError("covariates are a mode-B model")
        super().__init__(X, q, covariates, mode="B", **kw)


class CovDiagNoiseOracle(_Covariates, DiagNoiseOracle):
    """DiagNoiseOracle with known covariates."""


class CovWeightedPlateOracle(_Covariates, WeightedPlateOracle):
    """WeightedPlateOracle with known covariates: construct as (X, q, covariates, weights=S, ...)."""


class CovWeightedDiagNoiseOracle(_Covariates, WeightedDiagNoiseOracle):
    """WeightedDiagNoiseOracle with known covariates."""


class CovWRowsPlateOracle(_Covariates, WRowsPlateOracle):
    """Row-wise W posterior: one joint Gaussian over [w_d ; b_d] per data dimension."""


class CovWRowsDiagNoiseOracle(_Covariates, WRowsDiagNoiseOracle):
    pass


class CovWRowsWeightedPlateOracle(_Covariates, WRowsWeightedPlateOracle):
    pass


class CovWRowsWeightedDiagNoiseOracle(_Covariates, WRowsWeightedDiagNoiseOracle):
    pass


def cov_oracle_class(diag=False, weighted=False, rows=False):
    """The oracle class of one combination of the modes that compose with covariates."""
    return {(False, False, False): CovPlateOracle, (True, False, False): CovDiagNoiseOracle,
            (False, True, False): CovWeightedPlateOracle, (True, True, False): CovWeightedDiagNoiseOracle,
            (False, False, True): CovWRowsPlateOracle, (True, False, True): CovWRowsDiagNoiseOracle,
            (False, True, True): CovWRowsWeightedPlateOracle, (True, True, True): CovWRowsWeightedDiagNoiseOracle}[
        (bool(diag), bool(weighted), bool(rows))]


def synth_covariates(N, D, q, k, missing, tau=20.0, seed=0, cscale=1.0):
    """(X, C, W, B, mu): x_nd = w_d z_n + b_d c_n + mu_d + N(0, 1/tau), c_n ~ cscale * N(0, 1), b_d ~ N(0, 1) / cscale,
    Bernoulli(missing) erasures."""
    rng = np.random.RandomState(seed)
    W, Z, mu = rng.randn(D, q), rng.randn(N, q), rng.randn(D)
    B = rng.randn(D, k) / cscale
    C = cscale * rng.randn(N, k)
    X =Z @ W.T + C @ B.T + mu[None, :] + rng.randn(N, D) / np.sqrt(tau)
    if missing > 0:
        X[rng.rand(N, D) < missing] = np.nan
    return X, C, W, B, mu
