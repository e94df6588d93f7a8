"""Shared helpers for the parity tests (test infrastructure)."""
import os

import numpy as np

from oracle.plate_oracle import PlateOracle

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

STATE_KEYS = ("Wbar", "Wvar", "mu", "muvar", "Zbar", "Sig", "Xhat", "V", "qb")


def load_golden(name):
    return dict(np.load(os.path.join(GOLDEN, name), allow_pickle=False))


def golden_state(g, prefix):
    st = {k: g[prefix + k] for k in STATE_KEYS}
    if prefix + "al_qb" in g:
        st["al_qb"] = g[prefix + "al_qb"]
    return st


def tensor_rel(a, b):
    """Tensor-wise relative error max|a-b| / max|b| (SURVEY 8d)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    den = max(float(np.max(np.abs(b))), 1e-300)
    return float(np.max(np.abs(a - b))) / den


def refined_inverse(A, steps=3):
    """Inverses of a batch of float64 SPD matrices [.., q, q] in extended precision (np.longdouble): a float64 inverse of the
    equilibrated matrix, refined by Newton steps X <- X + X (I - A X) in long double.  The equilibration keeps the start
    inside Newton's region of convergence for matrices whose diagonal spans many orders of magnitude."""
    A = np.asarray(A, dtype=np.float64)
    q = A.shape[-1]
    d = 1.0 / np.sqrt(np.diagonal(A, axis1=-2, axis2=-1).astype(np.longdouble))
    Al = d[..., :, None] * A.astype(np.longdouble) * d[..., None, :]
    X = np.linalg.inv(Al.astype(np.float64)).astype(np.longdouble)
    eye = np.eye(q, dtype=np.longdouble)
    for _ in range(steps):
        X = X + X @ (eye - Al @ X)
    return d[..., :, None] * X * d[..., None, :]


def half_logdet_ld(A):
    """ln prod diag chol(A) = 0.5 ln det A of a batch of float64 SPD matrices, by a Cholesky factorisation in long double."""
    L = np.array(A, dtype=np.longdouble)
    q = L.shape[-1]
    out = np.zeros(L.shape[:-2], dtype=np.longdouble)
    for k in range(q):
        piv = np.sqrt(L[..., k, k])
        out += np.log(piv)
        col = L[..., k + 1:, k] / piv[..., None]
        L[..., k + 1:, k + 1:] -= col[..., :, None] * col[..., None, :]
        L[..., k + 1:, k] = col
    return out


def oracle_from_golden(g, mode="A"):
    o = PlateOracle(g["X"], int(g["q"]), mode=mode, ard=bool(int(g.get("ard", 0))))
    o.load_state(golden_state(g, "init_"))
    return o


def numpy_stats(X, Zbar, Sig, q):
    """The packed statistics buffer (pyvb_b200._layout.StatLayout) of a row block, in numpy -- the quantity
    that is all-reduced.  X may hold NaN (= not observed)."""
    from pyvb_b200._layout import StatLayout, SC_SXX, SC_NE, SC_NROWS
    from oracle.plate_oracle import pack_sym
    N, D = X.shape
    L = StatLayout(D, q)
    O = (~np.isnan(X)).astype(np.float64)
    X0 = np.where(np.isnan(X), 0.0, X)
    M2 = pack_sym(Zbar[:, :, None] * Zbar[:, None, :] + Sig)
    out = np.zeros(L.len)
    v = L.views(out)
    v["T1"][:] = O.T @ M2
    v["Bst"][:] = O.T @ Zbar
    v["Ast"][:] = X0.T @ Zbar
    v["cnt"][:] = O.sum(0)
    v["colx"][:] = X0.sum(0)
    v["S"][:] = M2.sum(0)
    v["zsum"][:] = Zbar.sum(0)
    v["scal"][SC_SXX] = (X0 ** 2).sum()
    v["scal"][SC_NE] = O.sum()
    v["scal"][SC_NROWS] = N
    return out


def w_update_from_stats(stats, D, q, Wbar, mu, tau, alpha):
    """Gauss-Seidel W-column update written against the stats buffer (what wupdate_kernel computes)."""
    from pyvb_b200._layout import StatLayout
    L = StatLayout(D, q)
    v = L.views(stats)
    ii, jj = np.tril_indices(q)
    T1 = np.zeros((D, q, q))
    T1[:, ii, jj] = v["T1"]
    T1[:, jj, ii] = v["T1"]
    W = Wbar.copy()
    Wvar = np.zeros_like(W)
    for i in range(q):
        prec = (alpha[i] if np.ndim(alpha) else alpha) + tau * T1[:, i, i]
        m2 = v["Ast"][:, i] - mu * v["Bst"][:, i]
        for j in range(q):
            if j != i:
                m2 = m2 - T1[:, i, j] * W[:, j]
        W[:, i] = tau * m2 / prec
        Wvar[:, i] = 1.0 / prec
    return W, Wvar
