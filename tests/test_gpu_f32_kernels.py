"""FP32 variant (precision="f32"), stage by stage, against float64 references through the C-ABI.

A Z step of the FP32 variant is K1-f32 (tcgen05 contraction into float rows [eta | qprec packed | pad], kernels_f32.cu),
then the batched solve IN PLACE on those float rows with FP64 arithmetic inside (K2a zsolve_tpm_kernel<16, true>,
kernels_k2t.cu; K2b zsolve_blocked_kernel<32|64, true>, kernels_k2.cu), which also writes the three-way bf16 split of the
finished rows (MP: the only input the statistics read of the rows) and, at q = 16 / 32, per-CTA column-sum partials.
The statistics K3-f32 (pyvb_stats_f32) multiply bf16 operands with FP32 accumulation per row chunk.  test_gpu_f32.py checks
K1-f32 and whole sweeps tensor-wise; here every stage is checked per entry, per row and per data dimension, with bounds
derived from its arithmetic (u32 = 2^-24, u64 = 2^-53):

  K2 rows      |out - ref| <= u32 |ref| + C_SOLVE cond u64 max|row|: one float32 rounding of the FP64 result plus the
               FP64 solve error (C_SOLVE = 2q covers the forward error of a Cholesky inverse, ~q cond u64 ||Sigma||, and
               that of the LAPACK reference); ref = float64 LAPACK on the float32 inputs as stored, widened
  K2 Sig       tensor-wise 1e-10 up to cond 1e4, 1e-8 at cond 1e6 (FP64 inverse, error ~ cond u64)
  K2 logdet    tensor-wise 1e-12 up to cond 1e4, 1e-10 at cond 1e6 (ln det moves by tr(A^-1 dA) <= q cond u64)
  planes       h + m + l == the stored float row exactly, and bit-identical to torch's round-to-nearest split
  partials     column sums of the FP64 values before their float32 rounding: (u32 + 2 N u64) sum|v| against the stored rows
  K3-f32 (i)   C_ACC k u32 sum_n |a_n b_n| against the same bf16 operands in float64, k = FP32 additions per accumulator and
               row chunk (3 products per row for T1 / Bst, 5 for Ast), C_ACC = 2 (the tensor cores may truncate a sum)
  K3-f32 (ii)  (i) + the representation error against the original float64 data and rows: x_h + x_m keeps 16 bits
               (2^-16 |x|), the rows are rounded once to float32 (u32) and x_m z_l is not formed (u32 |x z|)

Every check prints its worst error over its bound."""
import numpy as np
import pytest

from helpers import numpy_stats, tensor_rel, w_update_from_stats
from oracle.plate_oracle import synth_pca

pytestmark = pytest.mark.gpu

U32, U64 = 2.0 ** -24, 2.0 ** -53
C_ACC = 2.0
SENT = -768.0            # sentinel of the unwritten entries: exact in bf16, float32 and float64
NPOOL = 64               # K2 inputs: data dimensions = distinct SPD matrices (one observed dimension per row)
CONDS = (1e2, 1e4, 1e6)  # matrix d of the pool has condition number ~ CONDS[d % 3]
SIG_TOL = {1e2: 1e-10, 1e4: 1e-10, 1e6: 1e-8}
LOGDET_TOL = {1e2: 1e-12, 1e4: 1e-12, 1e6: 1e-10}


def _lib():
    from pyvb_b200 import _cabi
    return _cabi, _cabi.lib()


def _dev():
    import torch
    return torch.device("cuda", 0)


def _stream():
    import torch
    return torch.cuda.current_stream(_dev()).cuda_stream


def _split3(v):
    """Three-way bf16 split of a float32 tensor with torch's round-to-nearest conversions, in float32."""
    import torch
    h = v.to(torch.bfloat16)
    r = v - h.float()
    m = r.to(torch.bfloat16)
    return h, m, (r - m.float()).to(torch.bfloat16)


def _bits(t):
    """Integer view of a tensor (bitwise comparison that also holds for -0.0 / NaN patterns)."""
    import torch
    return t.contiguous().view({8: torch.int64, 4: torch.int32, 2: torch.int16}[t.element_size()])


def _report(what, err, bound):
    ratio = float(np.max(err / bound)) if np.size(err) else 0.0
    print("%-48s worst err / bound = %.3g" % (what, ratio))
    assert ratio <= 1.0, (what, ratio)


# --------------------------------------------------------------------------------------------- K2 inputs through K1-f32
def _k2_inputs(N, q, seed, nonpd_row=None):
    """Z-step operands whose K1-f32 output rows are SPD matrices of chosen condition: row n observes one data dimension
    d(n) of a pool of NPOOL, G_d (the packed columns of GT) is the SPD matrix d, x_nd W[:, d] its eta (W random, x random
    per row, so every row differs); P0 = 0, h0 = 0, tau = 1.  With nonpd_row, that row alone gets an indefinite matrix."""
    import torch
    dev = torch.device("cuda", 0)
    _, lib = _lib()
    rng = np.random.RandomState(seed)
    P, ncp, poff = q * (q + 1) // 2, int(lib.pyvb_f32_pitch(q)), int(lib.pyvb_f32_poff(q))
    ii, jj = np.tril_indices(q)
    G = np.zeros((ncp, NPOOL))
    for d in range(NPOOL):
        B = rng.randn(q, q)
        Qm = np.linalg.qr(rng.randn(q, q))[0]
        A = 0.02 * B @ B.T + (Qm * np.logspace(0, np.log10(CONDS[d % 3]), q)) @ Qm.T
        if d == NPOOL - 1:
            A = A - 50.0 * np.eye(q) if nonpd_row is not None else A
        G[poff:poff + P, d] = A[ii, jj]
    dsel = rng.randint(0, NPOOL - 1, size=N)
    if nonpd_row is not None:
        dsel[nonpd_row] = NPOOL - 1
    x = rng.randn(N).astype(np.float32)
    xs = _split3(torch.as_tensor(x, device=dev))
    planes = torch.zeros(3, N, NPOOL, dtype=torch.bfloat16, device=dev)
    rows, cols = torch.arange(N, device=dev), torch.as_tensor(dsel, device=dev)
    planes[0, rows, cols] = 1.0
    planes[1, rows, cols] = xs[0]
    planes[2, rows, cols] = xs[1]
    GT = torch.stack(_split3(torch.as_tensor(G, dtype=torch.float32, device=dev))).contiguous()
    WT = torch.stack(_split3(torch.as_tensor(3.0 * rng.randn(q, NPOOL), dtype=torch.float32, device=dev))).contiguous()
    gl = torch.zeros(144, dtype=torch.float64, device=dev)
    gl[2] = 1.0
    return {"q": q, "N": N, "planes": planes, "GT": GT, "WT": WT, "gl": gl, "dsel": dsel,
            "P0": torch.zeros(q, q, dtype=torch.float64, device=dev), "h0": torch.zeros(q, dtype=torch.float64, device=dev)}


def _k1_rows(inp):
    """The rows K1-f32 leaves for the batched solve (the same launch pyvb_zstep_f32 makes first)."""
    import torch
    cabi, lib = _lib()
    q, N = inp["q"], inp["N"]
    MZ = torch.full((N, int(lib.pyvb_f32_pitch(q))), SENT, dtype=torch.float32, device=_dev())
    cabi.check(lib.pyvb_zstep_k1_f32(N, NPOOL, q, inp["planes"].data_ptr(), inp["GT"].data_ptr(), inp["WT"].data_ptr(),
                                     inp["P0"].data_ptr(), inp["h0"].data_ptr(), inp["gl"].data_ptr(), MZ.data_ptr(),
                                     _stream()), "zstep_k1_f32")
    return MZ


def _outputs(q, nalloc):
    import torch
    _, lib = _lib()
    dev, ncp, P = _dev(), int(lib.pyvb_f32_pitch(q)), q * (q + 1) // 2
    return {"MZ": torch.full((nalloc, ncp), SENT, dtype=torch.float32, device=dev),
            "MP": torch.full((3, nalloc, ncp), SENT, dtype=torch.bfloat16, device=dev),
            "Sig": torch.full((nalloc, P), SENT, dtype=torch.float64, device=dev),
            "logdet": torch.full((nalloc,), SENT, dtype=torch.float64, device=dev)}


def _zstep(inp, out, lo, hi, zsums=None):
    """pyvb_zstep_f32 on rows [lo, hi) of arrays of nalloc rows, pointers offset as PlateEngine.update_Z does."""
    cabi, lib = _lib()
    q, nalloc = inp["q"], inp["N"]
    ncp, P = int(lib.pyvb_f32_pitch(q)), q * (q + 1) // 2
    cabi.check(lib.pyvb_zstep_f32(hi - lo, nalloc, NPOOL, q, inp["planes"].data_ptr() + lo * NPOOL * 2,
                                  inp["GT"].data_ptr(), inp["WT"].data_ptr(), inp["P0"].data_ptr(), inp["h0"].data_ptr(),
                                  inp["gl"].data_ptr(), out["MZ"].data_ptr() + lo * ncp * 4,
                                  out["MP"].data_ptr() + lo * ncp * 2, out["Sig"].data_ptr() + lo * P * 8,
                                  out["logdet"].data_ptr() + lo * 8, 0 if zsums is None else zsums.data_ptr(),
                                  _stream()), "zstep_f32")


def _check_planes(MZ, MP, q, rows, what):
    """MP holds the three-way bf16 split of the stored float rows: exact in float64, bit-identical to the CPU split, and
    nothing written past the q + P used columns."""
    import torch
    used = q + q * (q + 1) // 2
    v = MZ[rows, :used]
    assert torch.equal(MP[:, rows, :used].double().sum(0), v.double()), what
    for p, ref in enumerate(_split3(v)):
        assert torch.equal(_bits(MP[p, rows, :used]), _bits(ref)), (what, "plane", p)
    assert bool((MP[:, rows, used:].float() == SENT).all()), what


# ------------------------------------------------------------------------------------------------------------- (a), (b), (d)
K2_CASES = [(16, N) for N in (1, 31, 33, 4099, 50_001)] + \
           [(32, N) for N in (1, 31, 33, 2999, 7_001)] + \
           [(64, N) for N in (1, 31, 33, 2999, 4_001)]
# K2a: 32 rows per warp, 5 warps per CTA, at most 148 CTAs (23,680 rows per pass of the grid-stride loop); K2b: one row per
# warp, 10 warps x 296 CTAs at q = 32 (2,960 rows), 11 warps x 148 CTAs at q = 64 (1,628 rows).  The last N of each q
# takes more than one pass; 4099 / 2999 are not multiples of 32 / 10 / 11.


@pytest.mark.parametrize("q,N", K2_CASES)
def test_k2_f32_rows_match_lapack(q, N):
    """The batched solve on FP32 rows against float64 LAPACK on the same float32 inputs, per entry and per row; the bf16
    planes of the finished rows; the column-sum partials (q = 16, 32)."""
    import torch
    _, lib = _lib()
    P, ncp, zoff, poff = q * (q + 1) // 2, int(lib.pyvb_f32_pitch(q)), int(lib.pyvb_f32_zoff(q)), int(lib.pyvb_f32_poff(q))
    assert lib.pyvb_f32_supported(NPOOL, q) == 1
    inp = _k2_inputs(N, q, seed=1000 * q + N)
    rows_in = _k1_rows(inp).double().cpu().numpy()
    out = _outputs(q, N)
    nz = int(lib.pyvb_zsums_len_f32(N, q))
    assert (nz > 0) == (q != 64)
    zs = torch.full((max(nz, 1),), float("nan"), dtype=torch.float64, device=_dev())
    _zstep(inp, out, 0, N, zs if nz else None)
    torch.cuda.synchronize()

    ii, jj = np.tril_indices(q)
    A = np.zeros((N, q, q))
    A[:, ii, jj] = rows_in[:, poff:poff + P]
    A[:, jj, ii] = rows_in[:, poff:poff + P]
    eta = rows_in[:, zoff:zoff + q]
    ev = np.linalg.eigvalsh(A)
    assert ev[:, 0].min() > 0
    cond = ev[:, -1] / ev[:, 0]
    Sg = np.linalg.inv(A)
    z = np.einsum("nij,nj->ni", Sg, eta)
    ref = np.zeros((N, ncp))
    ref[:, zoff:zoff + q] = z
    ref[:, poff:poff + P] = (Sg + z[:, :, None] * z[:, None, :])[:, ii, jj]
    got = out["MZ"].double().cpu().numpy()
    c_solve = 2.0 * q
    # |out - ref| <= u32 |ref| + solve term, reported as the part beyond the float32 rounding over the solve term (the
    # rounding alone comes within 2^-24 of its bound)
    excess = np.maximum(np.abs(got - ref) - U32 * np.abs(ref), 0.0)
    solve = c_solve * cond[:, None] * U64 * np.abs(ref).max(1, keepdims=True)
    _report("K2 q=%d N=%d rows (C_SOLVE=%g)" % (q, N, c_solve), excess[:, :q + P], np.broadcast_to(solve, excess.shape)[:, :q + P])
    assert np.all(got[:, q + P:] == 0.0)                          # K1's zero padding is left as it is

    sig, logdet = out["Sig"].cpu().numpy(), out["logdet"].cpu().numpy()
    ld_ref = 0.5 * np.linalg.slogdet(A)[1]
    cls = inp["dsel"] % 3
    for k, c in enumerate(CONDS):
        sel = cls == k
        if not sel.any():
            continue
        assert cond[sel].max() < 2 * c
        e_sig, e_ld = tensor_rel(sig[sel], Sg[sel][:, ii, jj]), tensor_rel(logdet[sel], ld_ref[sel])
        _report("K2 q=%d N=%d Sig, cond %.0e" % (q, N, c), e_sig, SIG_TOL[c])
        _report("K2 q=%d N=%d logdet, cond %.0e" % (q, N, c), e_ld, LOGDET_TOL[c])
    assert float(inp["gl"][11]) == 0.0

    _check_planes(out["MZ"], out["MP"], q, slice(0, N), "K2 q=%d N=%d planes" % (q, N))

    if nz:                                                        # (d) the column-sum partials
        kw = int(lib.pyvb_zsums_kw(q))
        pp = int(lib.pyvb_gw_woff(q))
        assert nz % kw == 0
        tot = zs.cpu().numpy().reshape(nz // kw, kw)[:, :pp + q + 4].sum(0)
        stored = out["MZ"].double().cpu().numpy()
        for name, cols, src in (("<zz^T>", slice(0, P), slice(poff, poff + P)), ("zbar", slice(pp, pp + q), slice(zoff, zoff + q))):
            s = stored[:, src]
            bnd = (U32 * (1 + 2.0 ** -10) + 2 * N * U64) * np.abs(s).sum(0) + 1e-300
            _report("K2 q=%d N=%d partials %s" % (q, N, name), np.abs(tot[cols] - s.sum(0)), bnd)
        for name, off, v in (("sum 0.5/logdet", 0, 0.5 / logdet), ("sum logdet", 1, logdet)):
            _report("K2 q=%d N=%d partials %s" % (q, N, name), abs(tot[pp + q + off] - v.sum()),
                    2 * N * U64 * np.abs(v).sum())
        assert tot[pp + q + 2] == N and tot[pp + q + 3] == 0.0


@pytest.mark.parametrize("q", [16, 32, 64])
def test_k2_f32_flags_non_pd(q):
    import torch
    N = 64
    inp = _k2_inputs(N, q, seed=5, nonpd_row=17)
    out = _outputs(q, N)
    _zstep(inp, out, 0, N)
    torch.cuda.synchronize()
    assert float(inp["gl"][11]) == 1.0
    assert not np.isfinite(float(out["logdet"][17]))


# ------------------------------------------------------------------------------------------------------------------- (c)
@pytest.mark.parametrize("q", [16, 32, 64])
def test_zstep_f32_row_ranges(q):
    """pyvb_zstep_f32 on [lo, hi) of arrays of nalloc rows writes exactly those rows, in every array and every bf16
    plane, bit-identical to a full-range call, and leaves every other row alone."""
    import torch
    nalloc = 700
    inp = _k2_inputs(nalloc, q, seed=77 + q)
    full = _outputs(q, nalloc)
    _zstep(inp, full, 0, nalloc)
    torch.cuda.synchronize()
    _check_planes(full["MZ"], full["MP"], q, slice(0, nalloc), "full range q=%d" % q)
    for lo, hi in [(0, 300), (128, 450), (37, 611), (333, 700)]:
        got = _outputs(q, nalloc)
        _zstep(inp, got, lo, hi)
        torch.cuda.synchronize()
        outside = torch.ones(nalloc, dtype=torch.bool, device=_dev())
        outside[lo:hi] = False
        for name in ("MZ", "MP", "Sig", "logdet"):
            g, f = got[name], full[name]
            if name == "MP":
                for p in range(3):
                    assert torch.equal(_bits(g[p, lo:hi]), _bits(f[p, lo:hi])), (q, lo, hi, "MP plane", p)
                    assert bool((g[p][outside].float() == SENT).all()), (q, lo, hi, "MP plane written outside", p)
            else:
                assert torch.equal(_bits(g[lo:hi]), _bits(f[lo:hi])), (q, lo, hi, name)
                assert bool((g[outside] == SENT).all()), (q, lo, hi, name + " written outside the range")
        _check_planes(got["MZ"], got["MP"], q, slice(lo, hi), "range [%d, %d) q=%d" % (lo, hi, q))
    assert float(inp["gl"][11]) == 0.0


# ------------------------------------------------------------------------------------------------------------------- (e)
STATS_CASES = [(16, 32, 1, True), (16, 96, 63, False), (16, 256, 65, True), (16, 1056, 6161, False),
               (16, 32, 100_000, True), (32, 32, 65, False), (32, 96, 6161, True), (32, 256, 1, False),
               (32, 1056, 63, True), (32, 256, 20_000, False)]
# D = 32 / 96 / 256 / 1056: less than one 128-wide d tile, a partial tile, whole tiles, several tiles and a partial one;
# N = 6161 and 20,000 take several row chunks, the last one partial


@pytest.mark.parametrize("q,D,N,dead_col", STATS_CASES)
def test_stats_f32_matches_float64(q, D, N, dead_col):
    """K3-f32 per data dimension: T1 / Bst / Ast against (i) the same bf16 operands accumulated in float64 and (ii) the
    float64 statistics of the original data and rows; the entries taken from xcache and the K2 partials exactly."""
    import torch
    from pyvb_b200._layout import ALGO_F32, SC_LOGDETZ, SC_NE, SC_NROWS, SC_QLDZ, SC_SXX, StatLayout
    cabi, lib = _lib()
    dev, st = _dev(), _stream()
    P, ncp = q * (q + 1) // 2, int(lib.pyvb_f32_pitch(q))
    X = synth_pca(N, D, q, 0.3, seed=N + D + q)
    if N >= 2:
        X[0, :] = np.nan                                          # an all-missing row
        X[1, :] = 1.5                                             # a fully observed row (but for the dead column)
    if dead_col:
        X[:, D - 2] = np.nan                                      # a data dimension nobody observes: cnt = 0
    rng = np.random.RandomState(q + D)
    Zbar = rng.randn(N, q)
    L0 = np.tril(0.3 * rng.randn(q, q)) + np.eye(q)
    Sig = np.broadcast_to(L0 @ L0.T, (N, q, q)) * rng.uniform(0.1, 1.0, size=(N, 1, 1))
    ii, jj = np.tril_indices(q)
    M2 = (Sig + Zbar[:, :, None] * Zbar[:, None, :])[:, ii, jj]
    rows = np.zeros((N, ncp), dtype=np.float32)
    rows[:, :q], rows[:, q:q + P] = Zbar, M2
    rows_t = torch.as_tensor(rows, device=dev)
    MP = torch.stack(_split3(rows_t)).contiguous()
    Xd = torch.as_tensor(X, device=dev)
    planes = torch.zeros(3, N, D, dtype=torch.bfloat16, device=dev)
    cabi.check(lib.pyvb_prepare_x_f32(N, D, Xd.data_ptr(), D, planes.data_ptr(), st), "prepare_x_f32")

    O = ~np.isnan(X)
    X0 = np.where(O, X, 0.0)
    xcache = torch.as_tensor(np.concatenate([O.sum(0), X0.sum(0), [(X0 ** 2).sum(), O.sum()]]).astype(np.float64),
                             device=dev)
    kw, pp = int(lib.pyvb_zsums_kw(q)), int(lib.pyvb_gw_woff(q))
    nz = int(lib.pyvb_zsums_len_f32(N, q))
    logdet = rng.uniform(1.0, 3.0, size=N)
    zs = np.zeros(nz)
    zs[:P] = rows[:, q:q + P].astype(np.float64).sum(0)
    zs[pp:pp + q] = rows[:, :q].astype(np.float64).sum(0)
    zs[pp + q:pp + q + 3] = (0.5 / logdet).sum(), logdet.sum(), N
    zsums = torch.as_tensor(zs, device=dev)
    L = StatLayout(D, q)
    ws_bytes = int(lib.pyvb_stats_workspace_bytes(N, D, q, ALGO_F32))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    stats = torch.full((L.len,), float("nan"), dtype=torch.float64, device=dev)
    cabi.check(lib.pyvb_stats_f32(N, N, D, q, planes.data_ptr(), MP.data_ptr(), stats.data_ptr(), ws.data_ptr(), ws_bytes,
                                  xcache.data_ptr(), zsums.data_ptr(), None, st), "stats_f32")
    torch.cuda.synchronize()
    got = L.views(stats.cpu().numpy())

    # entries that do not come from the tensor cores: exact
    xc = xcache.cpu().numpy()
    assert np.array_equal(got["cnt"], xc[:D]) and np.array_equal(got["colx"], xc[D:2 * D])
    assert got["scal"][SC_SXX] == xc[2 * D] and got["scal"][SC_NE] == xc[2 * D + 1]
    assert np.array_equal(got["S"], zs[:P]) and np.array_equal(got["zsum"], zs[pp:pp + q])
    assert (got["scal"][SC_QLDZ], got["scal"][SC_LOGDETZ], got["scal"][SC_NROWS]) == tuple(zs[pp + q:pp + q + 3])
    others = [k for k in range(len(got["scal"])) if k not in (SC_SXX, SC_NE, SC_QLDZ, SC_LOGDETZ, SC_NROWS)]
    assert np.all(got["scal"][others] == 0.0)
    if dead_col:
        assert got["cnt"][D - 2] == 0.0
        for k in ("T1", "Bst", "Ast"):
            assert np.all(got[k][D - 2] == 0.0), k

    # (i) the same bf16 operands, summed in float64 (on the device: the products are exact, the sums FP64)
    nch = ws_bytes // (L.len * 8)                                 # the workspace holds one partial per row chunk
    rpc = -(-N // nch)
    rpc = max(32, -(-rpc // 32) * 32)                             # rows per chunk, as launch_stats_f32 sets them
    f64 = torch.float64
    Om, xh, xm = (planes[p].to(f64) for p in range(3))
    Bh, Bm, Bl = (MP[p, :, :q + P].to(f64) for p in range(3))
    B, absB = Bh + Bm + Bl, Bh.abs() + Bm.abs() + Bl.abs()
    T_i, absT = (Om.t() @ B).cpu().numpy(), (Om.t() @ absB).cpu().numpy()
    A_i = (xh.t() @ B[:, :q] + xm.t() @ (Bh + Bm)[:, :q]).cpu().numpy()
    absA = (xh.abs().t() @ absB[:, :q] + xm.abs().t() @ (Bh.abs() + Bm.abs())[:, :q]).cpu().numpy()
    kT, kA = 3 * rpc, 5 * rpc
    fp64 = (N + nch) * U64
    bT = (C_ACC * kT * U32 + fp64) * absT + 1e-300
    bA = (C_ACC * kA * U32 + fp64) * absA + 1e-300
    tag = "K3 q=%d D=%d N=%d (%d chunks of %d rows)" % (q, D, N, nch, rpc)
    _report(tag + " (i) T1", np.abs(got["T1"] - T_i[:, q:]), bT[:, q:])
    _report(tag + " (i) Bst", np.abs(got["Bst"] - T_i[:, :q]), bT[:, :q])
    _report(tag + " (i) Ast", np.abs(got["Ast"] - A_i), bA)

    # (ii) helpers.numpy_stats on the original float64 data and rows
    ref = L.views(numpy_stats(X, Zbar, Sig, q))
    absM = O.T.astype(np.float64) @ np.abs(np.concatenate([Zbar, M2], 1))
    absXZ = np.abs(X0).T @ np.abs(Zbar)
    rep = U32 * (1 + 2.0 ** -10)
    _report(tag + " (ii) T1", np.abs(got["T1"] - ref["T1"]), bT[:, q:] + rep * absM[:, q:])
    _report(tag + " (ii) Bst", np.abs(got["Bst"] - ref["Bst"]), bT[:, :q] + rep * absM[:, :q])
    _report(tag + " (ii) Ast", np.abs(got["Ast"] - ref["Ast"]), bA + (2.0 ** -16 + 2 * rep) * (1 + 2.0 ** -8) * absXZ)


def test_stats_f32_rejects_q64():
    """pyvb_zstep_f32 runs q = 64, but K2 leaves no column-sum partials there, and the FP32 statistics have no other
    source for the sums over the rows: PYVB_EINVAL, not a wrong answer."""
    import torch
    from pyvb_b200._layout import ALGO_F32, StatLayout
    _, lib = _lib()
    N, D, q = 65, 32, 64
    dev = _dev()
    assert lib.pyvb_f32_supported(D, q) == 1 and lib.pyvb_zsums_len_f32(N, q) == 0
    ncp = int(lib.pyvb_f32_pitch(q))
    planes = torch.zeros(3, N, D, dtype=torch.bfloat16, device=dev)
    MP = torch.zeros(3, N, ncp, dtype=torch.bfloat16, device=dev)
    ws_bytes = int(lib.pyvb_stats_workspace_bytes(N, D, q, ALGO_F32))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    stats = torch.zeros(StatLayout(D, q).len, dtype=torch.float64, device=dev)
    xcache = torch.zeros(2 * D + 2, dtype=torch.float64, device=dev)
    zsums = torch.zeros(int(lib.pyvb_zsums_kw(q)), dtype=torch.float64, device=dev)
    rc = lib.pyvb_stats_f32(N, N, D, q, planes.data_ptr(), MP.data_ptr(), stats.data_ptr(), ws.data_ptr(), ws_bytes,
                            xcache.data_ptr(), zsums.data_ptr(), None, _stream())
    assert rc == -1                                               # PYVB_EINVAL


# ------------------------------------------------------------------------------------------------------------------- (f)
@pytest.mark.parametrize("q,k", [(16, 100), (16, 300), (32, 100), (32, 300)])
def test_engine_f32_range_sweep(q, k):
    """update_Z(0, k); update_Z(k, N) on an FP32 engine against update_Z(): the same rows, planes, Sig and log-dets bit
    for bit, the same T1 / Bst / Ast bit for bit, the row sums (rebuilt by _zsums_from_state instead of K2's partials)
    within the bound of the partials; then the W update against its numpy definition."""
    import torch
    from pyvb_b200 import PlateEngine
    from pyvb_b200._layout import SC_LOGDETZ, SC_NROWS, SC_QLDZ, StatLayout
    N, D = 700, 64
    X = synth_pca(N, D, q, 0.25, seed=q + k)
    X[1, :] = np.nan
    rng = np.random.RandomState(11)
    init = {"Wbar": rng.randn(D, q), "Wvar": np.ones((D, q)), "mu": 0.1 * rng.randn(D), "muvar": np.ones(D),
            "Zbar": rng.randn(N, q), "Sig": np.tile(np.eye(q), (N, 1, 1)), "qb": 0.5}
    e_full = PlateEngine(X, q, mode="B", device="cuda:0", precision="f32")
    e_rng = PlateEngine(X, q, mode="B", device="cuda:0", precision="f32")
    e_full.set_state(init)
    e_rng.set_state(init)
    e_full.update_Z()
    e_rng.update_Z(0, k)
    e_rng.update_Z(k, N)
    torch.cuda.synchronize()
    for name in ("MZ", "MP", "Sig", "logdet"):
        assert torch.equal(_bits(getattr(e_rng, name)), _bits(getattr(e_full, name))), (q, k, name)

    L = StatLayout(D, q)
    e_full._ensure_stats()                                        # the row sums from K2's partials
    s_full = e_full.stats.cpu().numpy().copy()
    e_rng._ensure_stats()                                         # the row sums rebuilt from the state
    s_rng = e_rng.stats.cpu().numpy().copy()
    e_full._zsums_from_state()
    e_full._stats_fresh = False
    e_full._ensure_stats()
    s_rebuilt = e_full.stats.cpu().numpy().copy()
    v_full = L.views(s_full)
    rows = e_full.MZ.double().cpu().numpy()
    logdet = e_full.logdet.cpu().numpy()
    with np.errstate(divide="ignore"):
        qld = 0.5 / logdet
    P = q * (q + 1) // 2
    for s, what in ((s_rng, "range sweep"), (s_rebuilt, "_zsums_from_state")):
        v = L.views(s)
        for key in ("T1", "Bst", "Ast", "cnt", "colx"):
            assert np.array_equal(v[key], v_full[key]), (what, key)
        tag = "engine q=%d k=%d %s" % (q, k, what)
        for key, src in (("S", rows[:, q:q + P]), ("zsum", rows[:, :q])):
            bnd = (U32 * (1 + 2.0 ** -10) + 2 * N * U64) * np.abs(src).sum(0)
            _report(tag + " " + key, np.abs(v[key] - v_full[key]), bnd)
        for sc, src in ((SC_QLDZ, qld), (SC_LOGDETZ, logdet)):
            if not np.isfinite(v_full["scal"][sc]):             # 0.5 / logdet of the all-missing row (logdet 0) is inf
                assert v["scal"][sc] == v_full["scal"][sc], (tag, sc)
                continue
            _report(tag + " scal %d" % sc, abs(v["scal"][sc] - v_full["scal"][sc]), 2 * N * U64 * np.abs(src).sum())
        assert v["scal"][SC_NROWS] == N

    sm = e_rng.get_state_small()
    Wref, Wvref = w_update_from_stats(s_rng, D, q, sm["Wbar"], sm["mu"], sm["tau"], sm["alpha"])
    e_rng.update_W()
    assert tensor_rel(e_rng.Wbar.cpu().numpy(), Wref) < 1e-10
    assert tensor_rel(e_rng.Wvar.cpu().numpy(), Wvref) < 1e-10
    e_rng.check()


# ------------------------------------------------------------------------------------------------------------------- (g)
@pytest.mark.parametrize("q", [16, 32, 64])
def test_k1_f32_row_edges(q):
    """K1-f32 per row: an all-missing row is exactly [h0 | P0 packed | 0]; rows past N in the partial last 128-row tile
    are not written."""
    import torch
    cabi, lib = _lib()
    dev, st = _dev(), _stream()
    N, nbuf, D = 200, 256, 64
    P, ncp, zoff, poff = q * (q + 1) // 2, int(lib.pyvb_f32_pitch(q)), int(lib.pyvb_f32_zoff(q)), int(lib.pyvb_f32_poff(q))
    X = synth_pca(N, D, q, 0.2, seed=q)
    X[3, :] = np.nan
    X[N - 1, :] = np.nan                                          # the last row, in the partial tile
    rng = np.random.RandomState(q)
    B = rng.randn(q, q)
    P0 = (B @ B.T + q * np.eye(q)).astype(np.float32).astype(np.float64)    # float32-exact: K1 keeps P0 / h0 as float
    h0 = rng.randn(q).astype(np.float32).astype(np.float64)
    Wbar, Wvar, mu = (torch.as_tensor(a, device=dev) for a in (rng.randn(D, q), rng.rand(D, q) + 0.1, rng.randn(D)))
    Xd = torch.as_tensor(X, device=dev)
    planes = torch.zeros(3, N, D, dtype=torch.bfloat16, device=dev)
    cabi.check(lib.pyvb_prepare_x_f32(N, D, Xd.data_ptr(), D, planes.data_ptr(), st), "prepare_x_f32")
    GT = torch.zeros(3, ncp, D, dtype=torch.bfloat16, device=dev)
    WT = torch.zeros(3, q, D, dtype=torch.bfloat16, device=dev)
    cabi.check(lib.pyvb_pack_gw_f32(D, q, Wbar.data_ptr(), Wvar.data_ptr(), mu.data_ptr(), GT.data_ptr(), WT.data_ptr(), st),
               "pack_gw_f32")
    P0_t, h0_t = torch.as_tensor(P0, device=dev), torch.as_tensor(h0, device=dev)
    gl = torch.zeros(144, dtype=torch.float64, device=dev)
    gl[2] = 2.5
    MZ = torch.full((nbuf, ncp), SENT, dtype=torch.float32, device=dev)
    cabi.check(lib.pyvb_zstep_k1_f32(N, D, q, planes.data_ptr(), GT.data_ptr(), WT.data_ptr(), P0_t.data_ptr(),
                                     h0_t.data_ptr(), gl.data_ptr(), MZ.data_ptr(), st), "zstep_k1_f32")
    torch.cuda.synchronize()
    out = MZ.double().cpu().numpy()
    ii, jj = np.tril_indices(q)
    prior = np.zeros(ncp)
    prior[zoff:zoff + q], prior[poff:poff + P] = h0, P0[ii, jj]
    for r in (3, N - 1):
        assert np.array_equal(out[r], prior), r
    assert np.all(out[N:] == SENT)
    assert np.all(np.isfinite(out[:N])) and np.all(out[:N, q + P:] == 0.0)
