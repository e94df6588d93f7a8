"""CPU checks of the per-dimension noise oracle (oracle/noise_oracle.py): it reduces to the scalar-noise oracle when every
tau_d is the same, it agrees with a row-by-row dense restatement of the model, and it recovers heteroscedastic noise."""
import numpy as np
import pytest

from oracle.noise_oracle import DiagNoiseOracle, synth_fa
from oracle.plate_oracle import PlateOracle, synth_pca


def rand_state(N, D, q, seed=0):
    rng = np.random.RandomState(seed)
    return {"Wbar": rng.randn(D, q), "Wvar": rng.rand(D, q) + 0.5, "mu": rng.randn(D) * 0.1, "muvar": rng.rand(D) + 0.5,
            "Zbar": rng.randn(N, q), "Sig": np.tile(np.eye(q), (N, 1, 1)) * (rng.rand(N, 1, 1) + 0.5)}


def rel(a, b):
    return np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(np.max(np.abs(np.asarray(b))), 1e-300)


@pytest.mark.parametrize("ard", [False, True])
def test_equal_precisions_reduce_to_the_scalar_oracle(ard):
    N, D, q = 300, 17, 4
    X = synth_pca(N, D, q, 0.25, seed=3)
    X[5] = np.nan                                                     # an all-missing row
    st = rand_state(N, D, q, seed=1)
    s = PlateOracle(X, q, mode="B", ard=ard)
    d = DiagNoiseOracle(X, q, ard=ard)
    s.load_state(dict(st, qb=0.8))
    d.load_state(dict(st, qb=d.qa * 0.8 / s.qa))                      # tau_d = tau for every d
    np.testing.assert_allclose(d.tau, s.tau, rtol=1e-15)
    assert abs(d.resid_d().sum() - s._resid2()) <= 1e-12 * abs(s._resid2())
    for step in ("update_W", "update_Z", "update_Mu"):
        getattr(s, step)()
        getattr(d, step)()
        for k in ("Wbar", "Wvar", "Zbar", "Sig", "mu", "muvar"):
            assert rel(getattr(d, k), getattr(s, k)) <= 1e-14, (step, k)


def test_matches_a_row_by_row_restatement():
    """Lambda_n = diag(tau * O_n), written out one row / one data dimension at a time."""
    N, D, q = 60, 7, 3
    rng = np.random.RandomState(4)
    tau = np.exp(rng.uniform(0, np.log(1e3), D))
    X = synth_fa(N, D, q, 0.3, tau, seed=5)
    X[7] = np.nan
    st = rand_state(N, D, q, seed=6)
    o = DiagNoiseOracle(X, q, a0=rng.rand(D) + 0.1, b0=rng.rand(D) + 0.1)
    o.load_state(dict(st, qb=rng.rand(D) + 0.2))
    O = ~np.isnan(X)
    Xz = np.where(O, X, 0.0)
    t = o.tau.copy()
    G = [np.outer(o.Wbar[d], o.Wbar[d]) + np.diag(o.Wvar[d]) for d in range(D)]
    M2 = [np.outer(o.Zbar[n], o.Zbar[n]) + o.Sig[n] for n in range(N)]

    # r_d: sum over the observed entries of <(x - w.z - mu)^2> = (x - wbar.zbar - mu)^2 + tr(G_d M2_n) - (wbar.zbar)^2 + muvar
    r = np.zeros(D)
    for n in range(N):
        for d in range(D):
            if O[n, d]:
                wz = o.Wbar[d] @ o.Zbar[n]
                r[d] += (Xz[n, d] - wz - o.mu[d]) ** 2 + np.trace(G[d] @ M2[n]) - wz ** 2 + o.muvar[d]
    assert rel(o.resid_d(), r) <= 1e-12

    # Z: one row at a time
    Zref, Sref = np.zeros((N, q)), np.zeros((N, q, q))
    for n in range(N):
        lam = t * O[n]
        L = np.eye(q) + sum(lam[d] * G[d] for d in range(D))
        eta = o.Wbar.T @ (lam * (Xz[n] - o.mu))
        Sref[n] = np.linalg.inv(L)
        Zref[n] = Sref[n] @ eta
    o.update_Z()
    assert rel(o.Zbar, Zref) <= 1e-12 and rel(o.Sig, Sref) <= 1e-12

    # W: one data dimension at a time, columns in Gauss-Seidel order
    M2 = [np.outer(o.Zbar[n], o.Zbar[n]) + o.Sig[n] for n in range(N)]
    W = o.Wbar.copy()
    Wv = np.zeros((D, q))
    for d in range(D):
        rows = np.nonzero(O[:, d])[0]
        T = sum(M2[n] for n in rows)
        for i in range(q):
            prec = o.alpha()[i] + t[d] * T[i, i]
            m2 = t[d] * sum((Xz[n, d] - o.mu[d]) * o.Zbar[n, i] for n in rows)
            m2 -= t[d] * sum(T[i, j] * W[d, j] for j in range(q) if j != i)
            W[d, i], Wv[d, i] = m2 / prec, 1.0 / prec
    o.update_W()
    assert rel(o.Wbar, W) <= 1e-12 and rel(o.Wvar, Wv) <= 1e-12

    # Mu
    mu, muv = np.zeros(D), np.zeros(D)
    for d in range(D):
        rows = np.nonzero(O[:, d])[0]
        prec = o.alpha_mu + t[d] * rows.size
        mu[d] = t[d] * sum(Xz[n, d] - o.Wbar[d] @ o.Zbar[n] for n in rows) / prec
        muv[d] = 1.0 / prec
    o.update_Mu()
    assert rel(o.mu, mu) <= 1e-12 and rel(o.muvar, muv) <= 1e-12


def test_recovers_heteroscedastic_noise():
    """tau_d log-uniform in [1, 1e3], 100 sweeps from a random state.  The sampling error of a variance from ~4500 entries is
    about sqrt(2 / 4500) = 2 %, and most tau_d come out within a few per cent; a few do not.  On this data the column with
    tau = 150 settles 27 % low and stays there over 400 sweeps; started from the generating W, Z and tau it drifts the same way
    (25 % low after 100 sweeps), so this is where the mean-field posterior settles and not a lack of
    convergence.  The test pins what the model does: 85 % of the columns within 10 %, every column within 35 %."""
    N, D, q = 5000, 20, 3
    rng = np.random.RandomState(11)
    tau = np.exp(rng.uniform(0, np.log(1e3), D))
    X = synth_fa(N, D, q, 0.1, tau, seed=12)
    o = DiagNoiseOracle(X, q)
    o.load_state(dict(rand_state(N, D, q, seed=13), qb=1.0))
    bounds = o.learn(100)
    assert np.all(np.isfinite(bounds))
    assert np.all(np.diff(bounds[10:]) > -1e-6 * np.abs(bounds[10:-1]))
    err = np.abs(o.tau / tau - 1.0)
    assert np.mean(err < 0.10) >= 0.85 and np.max(err) < 0.35, err
