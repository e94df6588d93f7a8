"""CPU: the Gauss-Jordan formulation of the batched q x q solve (oracle/gj_oracle.py = the arithmetic of kernels_k2g.cu) against
the reference's route, scipy cho_factor / cho_solve(., I) / dot (nodes/gaussian.py:117-123), and against an inverse refined in
extended precision: elimination without pivoting must not cost accuracy on SPD input."""
import numpy as np
import pytest
from scipy.linalg import cho_factor, cho_solve

from helpers import refined_inverse, tensor_rel
from oracle.gj_oracle import gj_solve


def _case(N, q, seed, cond):
    rng = np.random.RandomState(seed)
    B = rng.randn(N, q, q)
    A = B @ B.transpose(0, 2, 1)
    s = np.logspace(0, np.log10(cond), q)
    Qm = np.linalg.qr(rng.randn(q, q))[0]
    return 0.02 * A + (Qm * s) @ Qm.T, rng.randn(N, q) * 3.0


@pytest.mark.parametrize("q", [4, 16, 32])
@pytest.mark.parametrize("cond", [1e2, 1e4, 1e6])
def test_gauss_jordan_is_as_accurate_as_the_cholesky_route(q, cond):
    A, eta = _case(60, q, seed=q, cond=cond)
    X = refined_inverse(A)
    ref = np.stack([cho_solve(cho_factor(a), np.eye(q)) for a in A])
    Sg, z, ld = gj_solve(A, eta)
    e_ref, e_gj = tensor_rel(ref, X), tensor_rel(Sg, X)
    assert e_gj < 4 * e_ref + 1e-15, (e_gj, e_ref)
    assert tensor_rel(Sg, ref) < 50 * cond * 1.2e-16
    assert tensor_rel(z, np.einsum("nij,nj->ni", ref, eta)) < 50 * cond * 1.2e-16
    chol_ld = np.array([np.log(np.prod(np.diag(cho_factor(a)[0]))) for a in A])     # gaussian.py:120
    assert tensor_rel(ld, chol_ld) < (1e-12 if cond <= 1e4 else 1e-10)     # (a sum of logarithms of both signs)


def test_gauss_jordan_flags_an_indefinite_matrix():
    A, eta = _case(5, 8, seed=1, cond=10.0)
    A[3] -= 50.0 * np.eye(8)
    _, _, ld = gj_solve(A, eta)
    assert np.isnan(ld[3]) and np.all(np.isfinite(ld[[0, 1, 2, 4]]))
