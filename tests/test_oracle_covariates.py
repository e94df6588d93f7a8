"""CPU tests of the covariate oracle (oracle/covariates_oracle.py), the checker of PlateEngine(..., covariates=C): the direct
Z step against conditioning the (q + k)-dimensional Gaussian of the augmented plate on its known tail, zero covariates
against the covariate-free model, a monotone bound, and recovery of B, W and tau from synthetic data (whose tolerances the
GPU full-size test reuses)."""
import numpy as np
import pytest

from helpers import tensor_rel
from oracle.covariates_oracle import cov_oracle_class, synth_covariates
from oracle.noise_oracle import DiagNoiseOracle
from oracle.plate_oracle import LN2PI, PlateOracle
from oracle.weights_oracle import WeightedPlateOracle

# recovery tolerances, from test_recovers_B_W_tau at N = 4000, D = 40, q = 3, k = 2 (tau = 20, 20 % missing), which measures
# 0.037, 0.0044 and 0.32 degrees, with a margin of 2.5-4.5x.  The B error is mostly the sample correlation of Z and C
# (~ 1/sqrt(N)), so at the full size of the GPU test the estimates are only tighter
REC_B = 0.1            # ||B_hat - B||_F / ||B||_F
REC_TAU = 0.02         # |tau_hat / tau - 1|
REC_ANGLE = 1.0        # largest principal angle between span(W_hat) and span(W), degrees

COMBOS = [(d, w, r) for d in (False, True) for w in (False, True) for r in (False, True)]


def make(X, q, C, diag, weighted, rows, S=None, **kw):
    cls = cov_oracle_class(diag, weighted, rows)
    if diag:
        kw.setdefault("a0", 0.2)
    if weighted:
        kw["weights"] = S
    return cls(X, q, C, **kw)


def init_state(N, D, q, k, seed=0, diag=False):
    rng = np.random.RandomState(seed)
    return {"Wbar": rng.randn(D, q), "Bbar": rng.randn(D, k), "Wvar": rng.rand(D, q) + 0.5, "Bvar": rng.rand(D, k) + 0.5,
            "mu": rng.randn(D) * 0.1, "muvar": np.ones(D), "Zbar": rng.randn(N, q),
            "Sig": np.tile(np.eye(q), (N, 1, 1)) * (rng.rand(N, 1, 1) + 0.5), "qb": (rng.rand(D) + 0.3) if diag else 0.7,
            "al_qb": rng.rand(q + k) + 0.5}


def load(o, st):
    o.load_user_state(st)
    if o.ard:
        o.al_qb = st["al_qb"].copy()


def augmented_update_Z(o, lo=0, hi=None):
    """The Z step of the augmented plate: K1 at q' = q + k with P0' = blockdiag(P0, 0), h0' = [h0 ; 0], then the Gaussian
    conditioned on its known tail: A = qprec'_zz, e = eta'_z - qprec'_zc c."""
    hi = o.N if hi is None else hi
    qz, q = o.qz, o.q
    Et = o.E()[lo:hi] * o.taus()[None, :]
    P0a = np.zeros((q, q))
    P0a[:qz, :qz] = o.P0z
    h0a = np.concatenate([o.P0z @ o.m0z, np.zeros(o.k)])
    L = P0a[None] + (Et @ o.G().reshape(o.D, q * q)).reshape(-1, q, q)
    eta = h0a[None] + (Et * (o.Xe()[lo:hi] - o.mu[None, :])) @ o.Wbar
    A = L[:, :qz, :qz]
    e = eta[:, :qz] - np.einsum("nik,nk->ni", L[:, :qz, qz:], o.cov_c[lo:hi])
    U = np.linalg.cholesky(A)
    S = np.linalg.inv(A)
    S = 0.5 * (S + np.transpose(S, (0, 2, 1)))
    o.Sig[lo:hi, :qz, :qz] = S
    o.Zbar[lo:hi, :qz] = np.einsum("nij,nj->ni", S, e)
    o.qldZ[lo:hi] = 0.5 / np.sum(np.log(np.diagonal(U, axis1=1, axis2=2)), axis=1)


def augmented_Z_bound(o):
    """The Z term of the bound as the engine takes it: the base formula at q' with P0', and -k folded into ln det P0."""
    q, k = o.q, o.k
    P0a = np.zeros((q, q))
    P0a[:o.qz, :o.qz] = o.P0z
    m0a = np.concatenate([o.m0z, np.zeros(k)])
    M2 = o.M2()
    quad = np.einsum("ij,nji->n", P0a, M2) + m0a @ P0a @ m0a - 2.0 * (o.Zbar @ (P0a @ m0a))
    lndet = np.linalg.slogdet(o.P0z)[1] - k
    return float(np.sum(-0.5 * q * LN2PI + 0.5 * lndet - 0.5 * quad - (-0.5 * q * LN2PI - 0.5 * o.qldZ - 0.5 * q)))


def _data(N, D, q, k, seed, weighted):
    X, C, _, _, _ = synth_covariates(N, D, q, k, 0.25, tau=10.0, seed=seed)
    S = 10.0 ** np.random.RandomState(seed + 1).uniform(-1, 1, size=(N, D)) if weighted else None
    return X, C, S


@pytest.mark.parametrize("diag,weighted,rows", COMBOS)
@pytest.mark.parametrize("ard", [False, True])
def test_direct_equals_augmented(diag, weighted, rows, ard):
    N, D, q, k = 150, 13, 3, 2
    X, C, S = _data(N, D, q, k, 5, weighted)
    st = init_state(N, D, q, k, seed=1, diag=diag)
    a = make(X, q, C, diag, weighted, rows, S, ard=ard)
    b = make(X, q, C, diag, weighted, rows, S, ard=ard)
    load(a, st)
    load(b, st)
    b.update_Z = lambda lo=0, hi=None: augmented_update_Z(b, lo, hi)
    for it in range(4):
        ea, eb = a.iterate(), b.iterate()
        assert abs(ea - eb) <= 1e-12 * abs(ea), (it, ea, eb)
        assert abs(a.elbo_terms()["Z"] - augmented_Z_bound(a)) <= 1e-12 * abs(ea)
        sa, sb = a.user_state(), b.user_state()
        for key in sa:
            assert tensor_rel(sa[key], sb[key]) < 1e-12, (it, key, tensor_rel(sa[key], sb[key]))
    # the known tail stays exact
    assert np.array_equal(a.Zbar[:, q:], C) and not np.any(a.Sig[:, q:, :]) and not np.any(a.Sig[:, :, q:])


@pytest.mark.parametrize("base,diag,weighted", [(PlateOracle, False, False), (DiagNoiseOracle, True, False),
                                                (WeightedPlateOracle, False, True)])
def test_zero_covariates(base, diag, weighted):
    """c_n = 0: Z, W, Mu and tau are those of the covariate-free model, B stays at its prior (bbar = 0, Bvar = 1/alpha0),
    and the bound differs by B's prior / entropy terms in closed form."""
    N, D, q, k = 120, 11, 3, 2
    X, _, S = _data(N, D, q, k, 7, weighted)
    st = init_state(N, D, q, k, seed=2, diag=diag)
    st["Bbar"][:] = 0.0
    kw = {"a0": 0.2} if diag else {}
    o = make(X, q, np.zeros((N, k)), diag, weighted, False, S)
    r = base(X, q, S, **kw) if weighted else base(X, q, **kw)
    load(o, st)
    free = {key: v for key, v in st.items() if key not in ("Bbar", "Bvar", "al_qb")}
    r.load_state(free)
    al = o.alpha0
    for it in range(4):
        eo, er = o.iterate(), r.iterate()
        us = o.user_state()
        for key in ("Zbar", "Sig", "Wbar", "Wvar", "mu", "muvar"):
            assert tensor_rel(us[key], getattr(r, key)) < 1e-12, (it, key)
        assert tensor_rel(np.asarray(o.tau), np.asarray(r.tau)) < 1e-12
        assert not np.any(us["Bbar"]) and np.allclose(us["Bvar"], 1.0 / al, rtol=1e-15, atol=0)
        # B's columns: prior - entropy, with Bvar = 1/alpha0 in every entry
        qld = 0.5 / (0.5 * D * np.log(al))
        extra = k * (0.5 * D * np.log(al) - 0.5 * D + 0.5 * qld + 0.5 * D)
        assert abs((eo - er) - extra) <= 1e-10 * abs(er), (it, eo - er, extra)


@pytest.mark.parametrize("diag,weighted,rows", [(False, False, False), (True, True, False), (False, False, True),
                                                (True, False, True)])
def test_bound_is_non_decreasing(diag, weighted, rows):
    N, D, q, k = 300, 16, 3, 2
    X, C, S = _data(N, D, q, k, 9, weighted)
    o = make(X, q, C, diag, weighted, rows, S, ard=True)
    load(o, init_state(N, D, q, k, seed=3, diag=diag))
    b = np.array([o.iterate() for _ in range(40)])
    assert np.all(np.isfinite(b))
    # (from sweep 5 on, as the other oracles' tests: the reference's q_ln_det quirk makes the first sweeps' bound no ELBO)
    d = np.diff(b[5:])
    assert np.all(d >= -1e-9 * np.abs(b[6:])), d.min()


def principal_angle_deg(A, B):
    qa, _ = np.linalg.qr(A)
    qb, _ = np.linalg.qr(B)
    s = np.linalg.svd(qa.T @ qb, compute_uv=False)
    return float(np.degrees(np.arccos(np.clip(s.min(), -1.0, 1.0))))


def recovery_errors(Bhat, tau_hat, What, B, tau, W):
    return (float(np.linalg.norm(Bhat - B) / np.linalg.norm(B)), float(abs(tau_hat / tau - 1.0)), principal_angle_deg(What, W))


def test_recovers_B_W_tau():
    N, D, q, k, tau = 4000, 40, 3, 2, 20.0
    X, C, W, B, mu = synth_covariates(N, D, q, k, 0.2, tau=tau, seed=21)
    o = make(X, q, C, False, False, False)
    rng = np.random.RandomState(0)
    load(o, {"Wbar": rng.randn(D, q), "Bbar": np.zeros((D, k)), "Zbar": rng.randn(N, q), "qb": 0.5})
    for _ in range(150):
        o.iterate()
    us = o.user_state()
    eb, et, ea = recovery_errors(us["Bbar"], o.tau, us["Wbar"], B, tau, W)
    assert eb < REC_B and et < REC_TAU and ea < REC_ANGLE, (eb, et, ea)


def test_W_B_Mu_residual_from_the_model():
    """The W / B step (columns), Mu and the residual, restated from the model x_nd = w_d z_n + b_d c_n + mu_d + noise with the
    known c_n, against the mixin's base-class updates at q' on the augmented moments."""
    N, D, q, k = 140, 9, 3, 2
    X, C, _ = _data(N, D, q, k, 13, False)
    o = make(X, q, C, False, False, False)
    load(o, init_state(N, D, q, k, seed=6))
    o.iterate()
    O = o.O.astype(np.float64)
    Xe = np.where(o.O, X, 0.0)
    tau, al = o.tau, o.alpha()
    Z, S = o.Zbar[:, :q].copy(), o.Sig[:, :q, :q].copy()
    Ezz = Z[:, :, None] * Z[:, None, :] + S
    W, Wv = o.Wbar[:, :q].copy(), o.Wvar[:, :q].copy()
    B, Bv = o.Wbar[:, q:].copy(), o.Wvar[:, q:].copy()
    mu, muvar = o.mu.copy(), o.muvar.copy()
    # residual: <(x - w z - b c - mu)^2> = (x - wbar zbar - bbar c - mu)^2 + zbar^T Cov(w) zbar + tr(E[ww^T] Sig)
    #                                      + c^T Cov(b) c + muvar   (Cov(w, b) = 0 with column posteriors)
    m = Z @ W.T + C @ B.T + mu[None, :]
    EwwT = W[:, :, None] * W[:, None, :] + np.einsum("di,ij->dij", Wv, np.eye(q))
    per = ((Xe - m) ** 2 + (Z ** 2) @ Wv.T + np.einsum("dij,nji->nd", EwwT, S) + (C ** 2) @ Bv.T + muvar[None, :])
    assert abs(np.sum(O * per) - o._resid2()) <= 1e-12 * np.sum(O * per)
    # W columns, then B columns, Gauss-Seidel in that order
    R = O * (Xe - mu[None, :])
    for i in range(q):
        prec = al[i] + tau * (O.T @ Ezz[:, i, i])
        m2 = tau * (R.T @ Z[:, i])
        for j in range(q):
            if j != i:
                m2 -= tau * (O.T @ Ezz[:, i, j]) * W[:, j]
        m2 -= tau * np.einsum("nd,n,nj,dj->d", O, Z[:, i], C, B)
        W[:, i], Wv[:, i] = m2 / prec, 1.0 / prec
    for j in range(k):
        prec = al[q + j] + tau * (O.T @ C[:, j] ** 2)
        m2 = tau * (R.T @ C[:, j]) - tau * np.einsum("nd,n,ni,di->d", O, C[:, j], Z, W)
        for l in range(k):
            if l != j:
                m2 -= tau * (O.T @ (C[:, j] * C[:, l])) * B[:, l]
        B[:, j], Bv[:, j] = m2 / prec, 1.0 / prec
    o.update_W()
    us = o.user_state()
    for key, ref in (("Wbar", W), ("Wvar", Wv), ("Bbar", B), ("Bvar", Bv)):
        assert tensor_rel(us[key], ref) < 1e-12, (key, tensor_rel(us[key], ref))
    # Mu: prec = alpha_mu + tau sum_n O, mu = tau sum_n O (x - wbar zbar - bbar c) / prec
    prec = o.alpha_mu + tau * O.sum(0)
    mu_ref = tau * np.sum(O * (Xe - Z @ W.T - C @ B.T), 0) / prec
    o.update_Mu()
    assert tensor_rel(o.mu, mu_ref) < 1e-12 and tensor_rel(o.muvar, 1.0 / prec) < 1e-15
