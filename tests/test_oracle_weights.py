"""CPU tests of the weighted plate oracle (oracle/weights_oracle.py), the checker of PlateEngine(..., weights=S): its reduction
to the unweighted oracles, its Z / W / Mu updates against a per-row restatement of the reference's generic operators with
Lambda_n = tau diag(s_n), zero weights as missing entries, and a monotone bound."""
import numpy as np

from oracle.noise_oracle import DiagNoiseOracle
from oracle.plate_oracle import PlateOracle, synth_pca
from oracle.weights_oracle import WeightedDiagNoiseOracle, WeightedPlateOracle, synth_weighted


def init_state(N, D, q, seed=0, diag=False):
    rng = np.random.RandomState(seed)
    return {"Wbar": rng.randn(D, q), "Wvar": rng.rand(D, q) + 0.5, "mu": rng.randn(D) * 0.1, "muvar": np.ones(D),
            "Zbar": rng.randn(N, q), "Sig": np.tile(np.eye(q), (N, 1, 1)) * (rng.rand(N, 1, 1) + 0.5),
            "qb": (rng.rand(D) + 0.3) if diag else 0.7}


def test_mask_weights_reproduce_unweighted_oracles():
    N, D, q = 60, 7, 3
    X = synth_pca(N, D, q, 0.3, seed=3)
    mask = (~np.isnan(X)).astype(np.float64)
    for ard in (False, True):
        for diag in (False, True):
            init = init_state(N, D, q, seed=1, diag=diag)
            if diag:
                a, b = DiagNoiseOracle(X, q, a0=0.2, ard=ard), WeightedDiagNoiseOracle(X, q, mask, a0=0.2, ard=ard)
            else:
                a, b = PlateOracle(X, q, ard=ard), WeightedPlateOracle(X, q, mask, ard=ard)
            a.load_state(init)
            b.load_state(init)
            np.testing.assert_array_equal(a.qa, b.qa)
            for _ in range(3):
                assert a.iterate() == b.iterate()
            for k in ("Wbar", "Wvar", "mu", "muvar", "Zbar", "Sig", "qb"):
                np.testing.assert_array_equal(getattr(a, k), getattr(b, k))


def _rowwise_reference(X, S, st, tau, alpha, alpha_mu, P0, m0):
    """The reference's generic operators, one row / one data dimension at a time, with the Constant per-row precision
    Lambda_n = tau diag(s_n) (zero where x is missing) -- dense matrix algebra, no shared code with the oracle."""
    N, D = X.shape
    q = st["Wbar"].shape[1]
    Xz = np.where(np.isnan(X), 0.0, X)
    Sz = np.where(np.isnan(X), 0.0, S)
    W, Wv, mu = st["Wbar"], st["Wvar"], st["mu"]
    # Z_n (node.py:203-227 + gaussian.py:117-123): m1 = sum_d Lambda_dd <w_d w_d^T>, m2 = <W>^T Lambda (x_n - mu)
    Zbar, Sig = np.zeros((N, q)), np.zeros((N, q, q))
    for n in range(N):
        Lam = tau * np.diag(Sz[n])
        m1 = np.zeros((q, q))
        for d in range(D):
            m1 += Lam[d, d] * (np.outer(W[d], W[d]) + np.diag(Wv[d]))
        prec = P0 + m1
        Sig[n] = np.linalg.inv(prec)
        Zbar[n] = Sig[n] @ (P0 @ m0 + W.T @ Lam @ (Xz[n] - mu))
    # W columns, Gauss-Seidel (nodes_todo.py:43-62): row d of column i from the rows' precisions Lambda_n[d, d]
    M2 = Zbar[:, :, None] * Zbar[:, None, :] + Sig
    Wn, Wvn = W.copy(), Wv.copy()
    for i in range(q):
        for d in range(D):
            lam = tau * Sz[:, d]
            prec = alpha[i] + np.sum(lam * M2[:, i, i])
            m2 = np.sum(lam * (Xz[:, d] - mu[d]) * Zbar[:, i])
            for j in range(q):
                if j != i:
                    m2 -= np.sum(lam * M2[:, i, j]) * Wn[d, j]
            Wn[d, i] = m2 / prec
            Wvn[d, i] = 1.0 / prec
    # Mu (node.py:95-110): precision alpha_mu + sum_n Lambda_n[d, d], mean from the residuals x - W z
    mun = np.zeros(D)
    for d in range(D):
        lam = tau * Sz[:, d]
        prec = alpha_mu + lam.sum()
        mun[d] = np.sum(lam * (Xz[:, d] - Zbar @ Wn[d])) / prec
    return {"Zbar": Zbar, "Sig": Sig, "Wbar": Wn, "Wvar": Wvn, "mu": mun}


def test_updates_match_rowwise_generic_operators():
    N, D, q = 40, 6, 3
    X, S, _ = synth_weighted(N, D, q, 0.25, tau=5.0, seed=4)
    S[np.random.RandomState(5).rand(N, D) < 0.1] = 0.0           # some zero weights on observed entries
    rng = np.random.RandomState(6)
    A = rng.randn(q, q)
    P0, m0 = A @ A.T + q * np.eye(q), rng.randn(q)
    o = WeightedPlateOracle(X, q, S, alpha0=0.3, alpha_mu=0.2, P0=P0, m0=m0)
    init = init_state(N, D, q, seed=2)
    o.load_state(init)
    tau = o.tau
    ref = _rowwise_reference(X, S, init, tau, o.alpha(), o.alpha_mu, P0, m0)
    o.update_Z()
    o.update_W()
    o.update_Mu()
    for k in ("Zbar", "Sig", "Wbar", "Wvar", "mu"):
        err = np.max(np.abs(getattr(o, k) - ref[k])) / np.max(np.abs(ref[k]))
        assert err < 1e-12, (k, err)


def test_zero_weight_is_missing():
    N, D, q = 50, 8, 2
    X, S, _ = synth_weighted(N, D, q, 0.2, tau=10.0, seed=7)
    zero = np.random.RandomState(8).rand(N, D) < 0.15
    S[zero] = 0.0
    Xn = X.copy()
    Xn[zero] = np.nan
    for cls, kw in ((WeightedPlateOracle, {}), (WeightedDiagNoiseOracle, {"a0": 0.5})):
        init = init_state(N, D, q, seed=3, diag=cls is WeightedDiagNoiseOracle)
        a, b = cls(X, q, S, **kw), cls(Xn, q, S, **kw)
        a.load_state(init)
        b.load_state(init)
        for _ in range(3):
            la, lb = a.iterate(), b.iterate()
            assert abs(la - lb) <= 1e-12 * abs(lb)
        for k in ("Wbar", "mu", "Zbar", "Sig", "qb"):
            np.testing.assert_allclose(getattr(a, k), getattr(b, k), rtol=1e-12, atol=1e-12)


def test_bound_non_decreasing():
    N, D, q = 300, 10, 3
    X, S, _ = synth_weighted(N, D, q, 0.2, tau=20.0, seed=9)
    for cls in (WeightedPlateOracle, WeightedDiagNoiseOracle):
        o = cls(X, q, S, ard=True)
        o.load_state(init_state(N, D, q, seed=4, diag=cls is WeightedDiagNoiseOracle))
        b = o.learn(30)
        assert np.all(np.isfinite(b))
        d = np.diff(b[5:])
        assert np.all(d >= -1e-9 * np.abs(np.array(b[6:]))), d.min()
