"""K2 alone through the C-ABI (pyvb_zsolve_f64): batched q x q Cholesky / inverse / solve in place on MZ rows,
against numpy/LAPACK -- the arithmetic of Gaussian.update, /root/reference/src/pyvb/nodes/gaussian.py:117-123
(cho_factor, cho_solve(., I), dot(qcov, .), q_ln_det from prod(diag(chol))).  One kernel per q: thread per matrix
(q = 8), Gauss-Jordan in registers (q = 16, 32), blocked symmetric sweep (q = 64)."""
import numpy as np
import pytest

from helpers import tensor_rel

pytestmark = pytest.mark.gpu


def _case(N, q, seed, cond):
    rng = np.random.RandomState(seed)
    B = rng.randn(N, q, q)
    A = B @ B.transpose(0, 2, 1)
    # spread the spectrum: cond(A) ~ cond
    s = np.logspace(0, np.log10(cond), q)
    Qm = np.linalg.qr(rng.randn(q, q))[0]
    A = 0.02 * A + (Qm * s) @ Qm.T
    eta = rng.randn(N, q) * 3.0
    return A, eta


def _run(q, A, eta, want_sig=True):
    import torch
    from pyvb_b200 import _cabi
    lib = _cabi.lib()
    N = A.shape[0]
    ii, jj = np.tril_indices(q)
    P = q * (q + 1) // 2
    ld, zoff = int(lib.pyvb_mz_pitch(q)), int(lib.pyvb_gw_woff(q))
    MZ = np.zeros((N, ld))
    MZ[:, :P] = A[:, ii, jj]
    MZ[:, zoff:zoff + q] = eta
    dev = torch.device("cuda", 0)
    mz = torch.as_tensor(MZ, device=dev)
    sig = torch.zeros(N, P, dtype=torch.float64, device=dev)
    logdet = torch.zeros(N, dtype=torch.float64, device=dev)
    gl = torch.zeros(144, dtype=torch.float64, device=dev)
    nz = int(lib.pyvb_zsums_len(N, q))
    nblk = int(lib.pyvb_zsums_blocks(N, q))
    zs = torch.full((max(nz, 1),), float("nan"), dtype=torch.float64, device=dev)
    _cabi.check(lib.pyvb_zsolve_f64(N, q, mz.data_ptr(), ld, sig.data_ptr() if want_sig else 0,
                                    logdet.data_ptr(), gl.data_ptr(), zs.data_ptr() if nz else 0,
                                    torch.cuda.current_stream(dev).cuda_stream), "zsolve")
    torch.cuda.synchronize()
    kw = int(lib.pyvb_zsums_kw(q))
    return (mz.cpu().numpy(), sig.cpu().numpy(), logdet.cpu().numpy(), gl.cpu().numpy(),
            zs.cpu().numpy()[:nblk * kw] if nblk else None, zoff)


@pytest.mark.parametrize("q,N", [(8, 1000), (16, 1), (16, 4099), (32, 2500), (32, 3), (64, 700), (64, 1)])
def test_zsolve_matches_lapack(q, N):
    A, eta = _case(N, q, seed=q + N, cond=1e4)
    out, sig, logdet, gl, zs, zoff = _run(q, A, eta)
    ii, jj = np.tril_indices(q)
    P = q * (q + 1) // 2
    Sg = np.linalg.inv(A)
    z = np.einsum("nij,nj->ni", Sg, eta)
    M2 = Sg + z[:, :, None] * z[:, None, :]
    assert tensor_rel(out[:, zoff:zoff + q], z) < 1e-10
    assert tensor_rel(out[:, :P], M2[:, ii, jj]) < 1e-10
    assert tensor_rel(sig, Sg[:, ii, jj]) < 1e-10
    assert tensor_rel(logdet, 0.5 * np.linalg.slogdet(A)[1]) < 1e-12
    assert float(gl[11]) == 0.0
    if zs is not None:
        kw = 2 * (zoff + q) + 4                         # [column sums | 4 scalars | column maxima of |.|]
        part = zs.reshape(-1, kw)
        tot = part[:, :zoff + q + 4].sum(0)
        mx = part[:, zoff + q + 4:].max(0)              # (bounds on) the column maxima
        true = np.abs(out).max(0)
        cols = list(range(P)) + list(range(zoff, zoff + q))
        assert np.all(mx[cols] >= true[cols] * (1 - 1e-12))
        if q == 8:                                      # thread per matrix
            assert np.allclose(mx[cols], true[cols], rtol=2e-6)        # high-word maxima, rounded up
        else:                                           # PSD bound sqrt(max <z_i z_i> max <z_j z_j>): tight on the diagonal
            di = [i * (i + 1) // 2 + i for i in range(q)]
            assert np.allclose(mx[di], true[di], rtol=1e-12)
        assert tensor_rel(tot[:P], out[:, :P].sum(0)) < 1e-12
        assert tensor_rel(tot[zoff:zoff + q], out[:, zoff:zoff + q].sum(0)) < 1e-12
        assert tot[zoff + q + 2] == N
        assert abs(tot[zoff + q + 1] - logdet.sum()) <= 1e-12 * abs(logdet.sum())


@pytest.mark.parametrize("q", [8, 16, 32, 64])
def test_zsolve_flags_non_pd(q):
    N = 64
    A, eta = _case(N, q, seed=5, cond=10.0)
    A[17] -= 50.0 * np.eye(q)           # indefinite
    out, sig, logdet, gl, zs, zoff = _run(q, A, eta, want_sig=False)
    assert float(gl[11]) == 1.0
