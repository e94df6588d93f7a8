"""CPU: the blocked symmetric sweep of the batched q x q solve (oracle/sweep_oracle.py = kernels_k2s.cu restated lane by lane on
the packed row: the batched scalar LDL^T elimination of the 8 x 8 pivot tiles, the DMMA fragments of the panel products and of the
trailing update, the in-place intermediates) against the reference's route, scipy cho_factor / cho_solve(., I) / dot
(nodes/gaussian.py:117-123), and against an inverse refined in extended precision.

The inverse of a pivot tile is only applied in factored form (W = old L^-T, M_IJ -= W D^-1 W^T: block Cholesky), so blocking must
not cost accuracy: over 4 seeds of the adversarial spectrum below (a randomly rotated log-spaced spectrum makes the leading 8 x 8
block as badly conditioned as it gets) the error stays within 1.7 x of the Cholesky route at cond 1e6 for q = 16, 32, 64.  (The first
version, with the explicit inverse of the pivot tile, was 22 x / 3,000 x worse at q = 32 / 16.)"""
import numpy as np
import pytest
from scipy.linalg import cho_factor, cho_solve

from helpers import refined_inverse, tensor_rel
from oracle.sweep_oracle import sweep_solve
from oracle.tsweep_oracle import tsweep_solve


def _case(N, q, seed, cond):
    rng = np.random.RandomState(seed)
    B = rng.randn(N, q, q)
    A = B @ B.transpose(0, 2, 1)
    s = np.logspace(0, np.log10(cond), q)
    Qm = np.linalg.qr(rng.randn(q, q))[0]
    return 0.02 * A + (Qm * s) @ Qm.T, rng.randn(N, q) * 3.0


@pytest.mark.parametrize("layout", ["packed", "tiles"])
@pytest.mark.parametrize("q", [8, 16, 32, 64])
@pytest.mark.parametrize("cond", [1e2, 1e4, 1e6])
def test_blocked_sweep_is_as_accurate_as_the_cholesky_route(q, cond, layout):
    A, eta = _case(9, q, seed=q, cond=cond)                      # (9: the last group is ragged)
    X = refined_inverse(A)
    ref = np.stack([cho_solve(cho_factor(a), np.eye(q)) for a in A])
    Sg, z, ld, M2 = (sweep_solve if layout == "packed" else tsweep_solve)(A, eta, mpw=(1 if layout == "packed" else 2) if q == 64 else 4)
    e_ref, e_s = tensor_rel(ref, X), tensor_rel(Sg, X)
    assert e_s < 4 * e_ref + 1e-15, (e_s, e_ref)
    assert tensor_rel(Sg, ref) < 50 * cond * 1.2e-16
    zr = np.einsum("nij,nj->ni", ref, eta)
    assert tensor_rel(z, zr) < 50 * cond * 1.2e-16
    assert tensor_rel(M2, ref + zr[:, :, None] * zr[:, None, :]) < 50 * cond * 1.2e-16
    chol_ld = np.array([np.log(np.prod(np.diag(cho_factor(a)[0]))) for a in A])     # gaussian.py:120
    assert tensor_rel(ld, chol_ld) < (1e-12 if cond <= 1e4 else 1e-10)


def test_blocked_sweep_flags_an_indefinite_matrix():
    A, eta = _case(5, 16, seed=1, cond=10.0)
    A[3] -= 50.0 * np.eye(16)
    _, _, ld, _ = sweep_solve(A, eta)
    assert np.isnan(ld[3]) and np.all(np.isfinite(ld[[0, 1, 2, 4]]))
