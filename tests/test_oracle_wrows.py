"""CPU tests of the row-wise W posterior oracle (oracle/wrows_oracle.py), the checker of PlateEngine(..., w_posterior="rows"):
its reduction to the column oracle at q = 1, the Gauss-Seidel fixed point of the column update, the variance inequality of an
SPD inverse, a per-row restatement of the W step from explicitly summed statistics, and a monotone bound."""
import numpy as np
import pytest

from helpers import tensor_rel
from oracle.noise_oracle import DiagNoiseOracle
from oracle.plate_oracle import PlateOracle
from oracle.weights_oracle import WeightedDiagNoiseOracle, WeightedPlateOracle, synth_weighted
from oracle.wrows_oracle import (WRowsDiagNoiseOracle, WRowsPlateOracle, WRowsWeightedDiagNoiseOracle,
                                 WRowsWeightedPlateOracle, synth_correlated)

# (rows class, columns class, weighted, per-dimension noise)
CLASSES = [(WRowsPlateOracle, PlateOracle, False, False), (WRowsDiagNoiseOracle, DiagNoiseOracle, False, True),
           (WRowsWeightedPlateOracle, WeightedPlateOracle, True, False),
           (WRowsWeightedDiagNoiseOracle, WeightedDiagNoiseOracle, True, True)]


def init_state(N, D, q, seed=0, diag=False):
    rng = np.random.RandomState(seed)
    return {"Wbar": rng.randn(D, q), "Wvar": rng.rand(D, q) + 0.5, "mu": rng.randn(D) * 0.1, "muvar": np.ones(D),
            "Zbar": rng.randn(N, q), "Sig": np.tile(np.eye(q), (N, 1, 1)) * (rng.rand(N, 1, 1) + 0.5),
            "qb": (rng.rand(D) + 0.3) if diag else 0.7, "al_qb": rng.rand(q) + 0.5}


def make(cls, X, q, S, weighted, diag, ard=False):
    kw = {"ard": ard}
    if diag:
        kw["a0"] = 0.2
    return cls(X, q, S, **kw) if weighted else cls(X, q, **kw)


def data(N, D, q, seed):
    X, S, _ = synth_weighted(N, D, q, 0.25, tau=10.0, seed=seed)
    return X, S


def load(o, init):
    o.load_state(init)
    if o.ard:
        o.al_qb = init["al_qb"].copy()


@pytest.mark.parametrize("rows_cls,cols_cls,weighted,diag", CLASSES)
@pytest.mark.parametrize("ard", [False, True])
def test_q1_equals_columns(rows_cls, cols_cls, weighted, diag, ard):
    """q = 1: one W column is D scalar rows, so every update and state agrees; the bound's W entropy groups the reference's
    q_ln_det quirk by node (one node of D entries against D nodes of one), so it agrees term by term once that grouping is
    undone, and outright at D = 1."""
    for N, D in ((80, 9), (40, 1)):
        X, S = data(N, D, 1, seed=D)
        init = init_state(N, D, 1, seed=2, diag=diag)
        a, b = make(cols_cls, X, 1, S, weighted, diag, ard), make(rows_cls, X, 1, S, weighted, diag, ard)
        load(a, init)
        load(b, init)
        for _ in range(4):
            a.update_W()
            b.update_W()
            for k in ("Wbar", "Wvar"):
                np.testing.assert_allclose(getattr(b, k), getattr(a, k), rtol=1e-13, atol=0)
            np.testing.assert_allclose(b.Wcov[:, 0, 0], a.Wvar[:, 0], rtol=1e-13)
            for step in ("update_Z", "update_Alpha", "update_Mu", "update_Beta"):
                getattr(a, step)()
                getattr(b, step)()
            for k in ("Wbar", "Wvar", "mu", "muvar", "Zbar", "Sig", "qb", "al_qb"):
                assert tensor_rel(getattr(b, k), getattr(a, k)) <= 1e-12, k
            ta, tb = a.elbo_terms(), b.elbo_terms()
            for k in ta:
                if k != "W":
                    assert tb[k] == ta[k] or abs(tb[k] - ta[k]) <= 1e-12 * abs(ta[k]), (k, tb[k], ta[k])
            # the column node's q_ln_det is 0.5 / sum_d ln sqrt(prec_d), the row nodes' sum_d 0.5 / ln sqrt(prec_d)
            lnc = 0.5 * np.log(1.0 / a.Wvar[:, 0])
            undo = 0.5 * np.sum(0.5 / lnc) - 0.5 * (0.5 / np.sum(lnc))
            assert abs(tb["W"] - undo - ta["W"]) <= 1e-11 * abs(ta["W"]), (tb["W"], undo, ta["W"])
            if D == 1:
                assert abs(tb["W"] - ta["W"]) <= 1e-12 * abs(ta["W"])


@pytest.mark.parametrize("rows_cls,cols_cls,weighted,diag", CLASSES)
def test_gauss_seidel_fixed_point(rows_cls, cols_cls, weighted, diag):
    """With Z, mu and tau held, repeated column passes converge to the row solve's wbar."""
    N, D, q = 150, 12, 4
    X, S = data(N, D, q, seed=5)
    init = init_state(N, D, q, seed=3, diag=diag)
    a, b = make(cols_cls, X, q, S, weighted, diag, True), make(rows_cls, X, q, S, weighted, diag, True)
    load(a, init)
    load(b, init)
    b.update_W()
    for it in range(100000):
        old = a.Wbar.copy()
        a.update_W()
        if np.max(np.abs(a.Wbar - old)) <= 1e-14 * np.max(np.abs(a.Wbar)):
            break
    assert it < 99999
    assert np.max(np.abs(a.Wbar - b.Wbar)) <= 1e-11 * np.max(np.abs(b.Wbar))


@pytest.mark.parametrize("rows_cls,cols_cls,weighted,diag", CLASSES)
def test_row_variances_bound_column_variances(rows_cls, cols_cls, weighted, diag):
    """(Lambda^-1)_ii >= 1 / Lambda_ii for SPD Lambda: the rows' Wvar is at least the columns' 1 / prec on the same state."""
    N, D, q = 120, 10, 6
    X, _ = synth_correlated(N, D, q, 0.3, seed=4)
    S = np.random.RandomState(4).rand(N, D) + 0.5
    init = init_state(N, D, q, seed=6, diag=diag)
    a, b = make(cols_cls, X, q, S, weighted, diag), make(rows_cls, X, q, S, weighted, diag)
    load(a, init)
    load(b, init)
    a.update_W()
    b.update_W()
    assert np.all(b.Wvar >= a.Wvar * (1.0 - 1e-13))
    assert np.any(b.Wvar > a.Wvar * 1.01)


def _restated_w_step(X, E, Zbar, Sig, mu, tau, alpha):
    """The W step from statistics summed by explicit loops over rows and data dimensions; each block solved on its own."""
    N, D = X.shape
    q = Zbar.shape[1]
    Wbar, Wcov = np.zeros((D, q)), np.zeros((D, q, q))
    for d in range(D):
        T1, Ast, Bst = np.zeros((q, q)), np.zeros(q), np.zeros(q)
        for n in range(N):
            if np.isnan(X[n, d]) or E[n, d] == 0.0:
                continue
            T1 += E[n, d] * (np.outer(Zbar[n], Zbar[n]) + Sig[n])
            Ast += E[n, d] * X[n, d] * Zbar[n]
            Bst += E[n, d] * Zbar[n]
        Lam = np.diag(alpha) + tau[d] * T1
        Wcov[d] = np.linalg.solve(Lam, np.eye(q))
        Wbar[d] = np.linalg.solve(Lam, tau[d] * (Ast - mu[d] * Bst))
    return Wbar, Wcov


@pytest.mark.parametrize("rows_cls,cols_cls,weighted,diag", CLASSES)
@pytest.mark.parametrize("ard", [False, True])
def test_w_step_restated(rows_cls, cols_cls, weighted, diag, ard):
    N, D, q = 70, 8, 5
    X, S = data(N, D, q, seed=7)
    init = init_state(N, D, q, seed=8, diag=diag)
    o = make(rows_cls, X, q, S, weighted, diag, ard)
    load(o, init)
    o.update_Z()
    E = S if weighted else np.ones_like(X)
    tau = np.broadcast_to(np.asarray(o.tau, dtype=np.float64), (D,))
    W, C = _restated_w_step(X, E, o.Zbar, o.Sig, o.mu, tau, o.alpha())
    o.update_W()
    np.testing.assert_allclose(o.Wbar, W, rtol=1e-11, atol=1e-12 * np.max(np.abs(W)))
    np.testing.assert_allclose(o.Wcov, C, rtol=1e-11, atol=1e-12 * np.max(np.abs(C)))
    np.testing.assert_array_equal(o.Wvar, np.diagonal(o.Wcov, axis1=1, axis2=2))
    np.testing.assert_allclose(o.Wld(), 0.5 * np.linalg.slogdet(np.linalg.inv(C))[1], rtol=1e-12)
    st = o.state()
    assert st["Wcov"].shape == (D, q, q)


@pytest.mark.parametrize("rows_cls,cols_cls,weighted,diag", CLASSES)
def test_bound_non_decreasing(rows_cls, cols_cls, weighted, diag):
    N, D, q = 300, 10, 3
    X, S = data(N, D, q, seed=9)
    o = make(rows_cls, X, q, S, weighted, diag, True)
    load(o, init_state(N, D, q, seed=4, diag=diag))
    b = o.learn(30)
    assert np.all(np.isfinite(b))
    d = np.diff(b[5:])
    assert np.all(d >= -1e-9 * np.abs(np.array(b[6:]))), d.min()
