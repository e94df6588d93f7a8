"""K1 and K3 on the FP64 tensor cores (kernels_dmma.cu) through the C-ABI, per entry, against references more precise than
the kernels:

  K1   zstep_dmma_kernel<Q, ETA, WT>   [S.O | S.O.(X - mu)] @ Gw  ->  [qprec packed | 0 | eta] in every MZ row
  K3   stats_dmma_kernel<Q, XO, WT>    [S.O | S.O.X]^T @ [<zz^T> | zbar]  ->  T1, Bst, Ast per row chunk in ws[chunk][stat layout]
       (+ the column sums, the per-row scalars and the fixed-order second stage behind pyvb_stats_f64)

Variants: plain and weighted (WT) at q = 8, 16, 32, 64; the eta-only K1 (ETA, inside pyvb_zstep_i8_f64) and the Ast-only K3
(XO, inside pyvb_stats_i8_f64) at q = 16, 32, 64; the generic statistics at the D that the DMMA path does not take.

1. Exact cases.  Integer X, mu = k/4, wbar = k/8, Wvar = k/64 > 0, weights k/8 in [0, 2], tau a power of two, dyadic P0 / h0,
   integer MZ columns and power-of-two log-dets: every product and every partial sum is a multiple of a dyadic grid below 2^53
   grid units (asserted), so every summation order gives the same float64 result and the kernels must match a plain numpy
   float64 reference BIT FOR BIT -- at N around a row tile, around one and two grid passes of the persistent K1, around K3's
   pipeline step and row chunk, at shapes that leave an empty trailing chunk and at a partial last data-dimension tile.  Every
   case also needs more than 24 significant bits (asserted): an FP32 accumulation cannot pass.
2. Rounding cases.  Real data with G columns spread over 1e+-8, one X feature scaled by 1e6, MZ rows spread over 1e+-6 and
   entries that cancel.  Per entry |got - ref| <= gamma_{k+2} sum|terms| against a long-double reference of the float64 inputs
   (k = D + 1 terms for K1: the D products and P0 / h0 of the fma epilogue; k = N for K3).
3. Reads and writes.  Guard rows and a NaN sentinel with its own payload around every output; K1 must leave [0, P) = qprec,
   [P, Pp) = +0.0, [Pp, Pp + q) = eta and nothing else; a second call with X / S read through a padded pitch full of NaN and
   +-1e300, rows past N of 1e300, NaN weights on unobserved entries, a NaN MZ pad / pitch tail / guard rows and NaN-filled ws and
   stats must give the same bits.  K3's per-chunk partials in ws are checked against the Python restatement of its chunking.
4. The checkers are shown to pass on numpy restatements of the kernels and to fail on a dropped row, a row counted twice, an
   ignored weight, an entry off by 10 x its bound and a write into the pitch tail (CPU).

The tile and grid geometry is parsed from the ZC / SC specialisations of kernels_dmma.cu; a CPU test pins it to the table the
sizes were chosen from, so a retuned configuration fails loudly instead of moving the boundaries away from the tested sizes."""
import functools
import os
import re
from math import gcd

import numpy as np
import pytest

from pyvb_b200._layout import (ALGO_DMMA, ALGO_DMMA_K1, ALGO_GENERIC, GL_I8BAD, GL_LEN, GL_TAU, SC_LOGDETZ, SC_NE, SC_NROWS,
                               SC_QLDZ, SC_SXX, StatLayout)

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "pyvb_b200", "csrc")
U = 2.0 ** -53
NSM = 148
SENT = np.array([0x7FF80000DEADBEEF], dtype=np.uint64).view(np.float64)[0]   # a quiet NaN with its own payload
GUARD = 3                                                                    # sentinel rows before and after every output
XPAD = 16                                                                    # extra pitch of the poisoned X / S
Q4 = (8, 16, 32, 64)
Q3 = (16, 32, 64)


# ============================================================================================== geometry (kernels_dmma.cu)
def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


@functools.lru_cache(maxsize=None)
def _spec(struct):
    """{q: {WM, WN, RGW, KC, ST, OCC, NCT}} of the `template <> struct ZC<q>` / `SC<q>` specialisations."""
    out = {}
    for q, body in re.findall(r"template <> struct %s<(\d+)>\s*\{\s*static constexpr int ([^;]*);" % struct,
                              _src("kernels_dmma.cu")):
        out[int(q)] = {k.strip(): int(v) for k, v in (kv.split("=") for kv in body.split(","))}
    assert sorted(out) == list(Q4), (struct, out)
    return out


@functools.lru_cache(maxsize=None)
def _variant_consts():
    """The constants ZT / STT override for the ETA, WT and XO variants."""
    s = _src("kernels_dmma.cu")
    m = re.search(r"ST = ETA \? \(Q <= 16 \? (\d+) : (\d+)\) : \(\(WT && Q == 8\) \? (\d+) : C::ST\), OCC = ETA \? (\d+) :", s)
    kc_eta = re.search(r"KC = ETA \? (\d+) : C::KC", s)
    kc_xo = re.search(r"KC = XO \? (\d+) : C::KC", s)
    assert m and kc_eta and kc_xo, "ZT / STT no longer have the expected form"
    return {"st_eta16": int(m.group(1)), "st_eta64": int(m.group(2)), "st_wt8": int(m.group(3)), "occ_eta": int(m.group(4)),
            "kc_eta": int(kc_eta.group(1)), "kc_xo": int(kc_xo.group(1))}


def k1_geom(q, kind):
    """Rows per row tile R, rows per grid pass, K chunk and pipeline stages of the K1 kernel of (q, kind)."""
    c, v = _spec("ZC")[q], _variant_consts()
    if kind == "eta":
        wm, kc, occ, nct = c["WM"] * c["WN"], v["kc_eta"], v["occ_eta"], 1
        st = v["st_eta16"] if q <= 16 else v["st_eta64"]
    else:
        wm, kc, occ, nct = c["WM"], c["KC"], c["OCC"], c["NCT"]
        st = v["st_wt8"] if (kind == "wt" and q == 8) else c["ST"]
    R = wm * c["RGW"] * 8
    assert (NSM * occ) % nct == 0
    return {"R": R, "pass": NSM * occ // nct * R, "KC": kc, "ST": st}


def k3_geom(q, xo=False):
    """Rows per pipeline step KC, data dimensions per CTA DT and column tiles NCT of the K3 kernel of q."""
    c, v = _spec("SC")[q], _variant_consts()
    wm = c["WM"] * c["WN"] if xo else c["WM"]
    return {"KC": v["kc_xo"] if xo else c["KC"], "DT": wm * c["RGW"] * 8, "NCT": 1 if xo else c["NCT"]}


def stats_dmma_nchunks(N, D, q):
    """Restatement of stats_dmma_nchunks (kernels_dmma.cu)."""
    kc, dt, nct = 16, 128, 1
    if q >= 32:
        kc, dt = 8, 32
    if q == 64:
        nct = _spec("SC")[64]["NCT"]
    ndt = -(-D // dt) * nct
    step = NSM // gcd(NSM, ndt)
    by_rows = -(-N // (64 * kc))
    k = max(1, (4 * NSM) // (step * ndt))
    c = k * step
    if c > by_rows:
        c = (by_rows // step) * step
    if c < 1:
        c = by_rows if by_rows >= 1 else 1
    return min(c, 1024)


I8_CL, I8_BM, I8_BKB, I8_CT = 2, 128, 64, 32      # kernels_i8.cu (pinned by test_geometry_matches_the_kernel_source)


def stats_i8_nchunks(N, D, q):
    """Restatement of stats_i8_nchunks (kernels_i8.cu): the row chunks of the XO kernel inside pyvb_stats_i8_f64."""
    ncl = NSM // I8_CL
    ncols = (q * (q + 1) // 2 + q + 31) & ~31
    per = ((-(-D // I8_BM) + I8_CL - 1) // I8_CL) * (ncols // I8_CT)
    step = ncl // gcd(ncl, per)
    by_rows = max(1, N // (32 * I8_BKB))
    c = max(1, -(-(6 * ncl) // (per * step))) * step
    if c > by_rows:
        c = (by_rows // step) * step if by_rows >= step else by_rows
    c = max(c, -(-N // (1 << 23)))
    return min(c, 1024)


def chunk_rows(N, nch, kc):
    """Rows per chunk of launch_stats_q: ceil(N / nch) rounded up to the pipeline step."""
    rpc = -(-(-(-N // nch)) // kc) * kc
    return max(rpc, kc)


def empty_chunks(N, D, q):
    nch = stats_dmma_nchunks(N, D, q)
    return nch - -(-N // chunk_rows(N, nch, k3_geom(q)["KC"]))


# shapes whose last row chunk is empty (two at q = 32, D = 48), and the largest XO case
EMPTY = {8: (75783, 256), 16: (75783, 256), 32: (37892, 256), 64: (37892, 48)}
XO_LARGE = (37892, 256)


def _layout(q):
    P = q * (q + 1) // 2
    PP = (P + 7) & ~7
    return P, PP, PP + q + 4          # P, Pp (the zbar / eta offset), the MZ and Gw pitch (pyvb_mz_pitch)


def _packed(q):
    ii, jj = np.tril_indices(q)       # p(i, j) = i (i + 1) / 2 + j, i >= j
    return ii, jj


def _diag_cols(q):
    return np.array([i * (i + 1) // 2 + i for i in range(q)])


# ============================================================================================== inputs and references
def _observed(rng, N, D, frac=0.3):
    """About 30 % missing; all-missing and fully observed rows at the start, the end and inside the block."""
    O = rng.rand(N, D) >= frac
    if N >= 8:
        for r in (0, N // 2, N - 1):
            O[r] = False
        for r in (1, N // 2 + 1, N - 2):
            O[r] = True
    return O


def _bits_equal(a, b):
    a, b = np.ascontiguousarray(a, dtype=np.float64), np.ascontiguousarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


def _is_sent(a):
    return _bits_equal(a, np.full(np.shape(a), SENT))


def _fp32_inexact(a):
    """Some entry needs more than 24 significant bits."""
    a = np.asarray(a, dtype=np.float64)
    return bool(np.any(a.astype(np.float32).astype(np.float64) != a))


def _assert_exact_grid(abs_sum, grid, what):
    """Precondition of the exact cases: every partial sum is a multiple of `grid` below 2^53 grid units."""
    assert float(np.max(abs_sum)) / grid < 2.0 ** 53, (what, float(np.max(abs_sum)) / grid)


def k1_exact_inputs(kind, q, N, D, seed):
    rng = np.random.RandomState(seed)
    O = _observed(rng, N, D)
    X = np.where(O, rng.randint(-4096, 4097, (N, D)).astype(np.float64), np.nan)
    mu = rng.randint(-256, 257, D) / 4.0
    Wb = rng.randint(-8192, 8193, (D, q)) / 8.0
    Wv = rng.randint(1, 1025, (D, q)) / 64.0
    ii, jj = _packed(q)
    G = Wb[:, ii] * Wb[:, jj] + np.where(ii == jj, Wv[:, ii], 0.0)
    S = rng.randint(0, 17, (N, D)) / 8.0 if kind == "wt" else None
    P0 = rng.randint(-64, 65, (q, q)) / 16.0
    P0 = P0 + P0.T + 8.0 * q * np.eye(q)
    return {"X": X, "O": O, "S": S, "mu": mu, "Wb": Wb, "Wv": Wv, "G": G, "tau": 2.0 ** rng.randint(-2, 3), "P0": P0,
            "h0": rng.randint(-64, 65, q) / 16.0}


def k1_reference(inp, dtype=np.float64):
    """qprec = P0 + tau (S.O) @ G and eta = h0 + tau (S.O.(X - mu)) @ wbar in `dtype`, and sum |terms| of each entry."""
    O, S, X = inp["O"], inp["S"], inp["X"]
    w = np.ones_like(X) if S is None else S
    Ao = np.where(O, w, 0.0).astype(dtype)
    Ax = np.where(O, w.astype(dtype) * (np.where(O, X, 0.0).astype(dtype) - inp["mu"].astype(dtype)), 0.0)
    ii, jj = _packed(len(inp["h0"]))
    tau = dtype(inp["tau"])
    p0 = inp["P0"][ii, jj].astype(dtype)
    h0 = inp["h0"].astype(dtype)
    return {"qprec": p0 + tau * (Ao @ inp["G"].astype(dtype)), "eta": h0 + tau * (Ax @ inp["Wb"].astype(dtype)),
            "qabs": np.abs(p0) + tau * (np.abs(Ao) @ np.abs(inp["G"]).astype(dtype)),
            "eabs": np.abs(h0) + tau * (np.abs(Ax) @ np.abs(inp["Wb"]).astype(dtype))}


def k1_exact_reference(inp):
    ref = k1_reference(inp)
    grid = inp["tau"] / 512.0              # G: 1/64, weights 1/8 (qprec); x - mu: 1/4, weights 1/8, wbar 1/8 (eta)
    _assert_exact_grid(ref["qabs"], grid, "qprec")
    _assert_exact_grid(ref["eabs"], grid, "eta")
    return ref


def k3_exact_inputs(kind, q, N, D, seed):
    rng = np.random.RandomState(seed)
    O = _observed(rng, N, D)
    P = q * (q + 1) // 2
    M = rng.randint(-1024, 1025, (N, P)).astype(np.float64)
    M[:, _diag_cols(q)] = rng.randint(1, 1025, (N, q))
    return {"X": np.where(O, rng.randint(-1024, 1025, (N, D)).astype(np.float64), np.nan), "O": O,
            "S": rng.randint(0, 17, (N, D)) / 8.0 if kind == "wt" else None, "M": M,
            "Z": rng.randint(-1024, 1025, (N, q)).astype(np.float64), "ld": 2.0 ** rng.randint(-3, 4, N)}


def k3_reference(inp, dtype=np.float64, rows=None):
    """The statistics buffer of rows `rows` (default all) in `dtype`, and sum |terms| of every entry (same layout)."""
    X, O, S, M, Z, ld = inp["X"], inp["O"], inp["S"], inp["M"], inp["Z"], inp["ld"]
    if rows is not None:
        X, O, M, Z, ld = X[rows], O[rows], M[rows], Z[rows], ld[rows]
        S = None if S is None else S[rows]
    N, D = X.shape
    q = Z.shape[1]
    L = StatLayout(D, q)
    w = np.ones_like(X) if S is None else S
    Ao = np.where(O, w, 0.0).astype(dtype)
    x0 = np.where(O, X, 0.0).astype(dtype)
    Ax = Ao * x0
    Md, Zd, ldd = M.astype(dtype), Z.astype(dtype), ld.astype(dtype)
    out, ab = np.zeros(L.len, dtype=dtype), np.zeros(L.len, dtype=dtype)
    v, a = L.views(out), L.views(ab)
    v["T1"][:], a["T1"][:] = Ao.T @ Md, Ao.T @ np.abs(Md)
    v["Bst"][:], a["Bst"][:] = Ao.T @ Zd, Ao.T @ np.abs(Zd)
    v["Ast"][:], a["Ast"][:] = Ax.T @ Zd, np.abs(Ax).T @ np.abs(Zd)
    v["cnt"][:], a["cnt"][:] = Ao.sum(0), Ao.sum(0)
    v["colx"][:], a["colx"][:] = Ax.sum(0), np.abs(Ax).sum(0)
    v["S"][:], a["S"][:] = Md.sum(0), np.abs(Md).sum(0)
    v["zsum"][:], a["zsum"][:] = Zd.sum(0), np.abs(Zd).sum(0)
    v["scal"][SC_SXX] = a["scal"][SC_SXX] = (Ax * x0).sum()
    v["scal"][SC_NE] = a["scal"][SC_NE] = float(np.count_nonzero(O & (w > 0)))
    v["scal"][SC_NROWS] = a["scal"][SC_NROWS] = N
    v["scal"][SC_QLDZ] = a["scal"][SC_QLDZ] = (dtype(0.5) / ldd).sum()
    v["scal"][SC_LOGDETZ] = a["scal"][SC_LOGDETZ] = ldd.sum()
    return out, ab


def k3_exact_reference(inp):
    ref, ab = k3_reference(inp)
    _assert_exact_grid(ab, 1.0 / 16.0, "statistics")        # weights 1/8, 0.5 / logdet >= 2^-4, everything else integer
    return ref


def xcache_of(stats, D, q):
    v = StatLayout(D, q).views(stats)
    return np.concatenate([v["cnt"], v["colx"], [v["scal"][SC_SXX], v["scal"][SC_NE]]])


# ============================================================================================== checkers
def gamma(n):
    return n * U / (1.0 - n * U)


def _ratios(got, ref, bound):
    """Per-entry |got - ref| / bound (0 where equal; NaN -> inf: a NaN is a failure, not a pass)."""
    err = np.abs(np.asarray(got, dtype=np.longdouble) - ref).astype(np.float64)
    b = np.asarray(bound, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(err == 0.0, 0.0, err / b)
    r[np.isnan(r)] = np.inf
    return r


def k1_round_ratios(got, ref, D):
    """Worst |got - ref| / (gamma_{k+2} sum|terms|) of qprec and eta, k = D + 1 (the D products and P0 / h0 of the fma)."""
    g = gamma(D + 3)
    out = {}
    for key, ab in (("qprec", "qabs"), ("eta", "eabs")):
        if key in got:
            out[key] = float(_ratios(got[key], ref[key], g * ref[ab]).max())
    return out


K3_NAMES = ("T1", "Bst", "Ast", "cnt", "colx", "S", "zsum")
K3_SCAL = {"SXX": SC_SXX, "NE": SC_NE, "NROWS": SC_NROWS, "QLDZ": SC_QLDZ, "LOGDETZ": SC_LOGDETZ}


def k3_round_ratios(got, ref, ab, N, D, q, names=K3_NAMES + tuple(K3_SCAL)):
    """Worst |got - ref| / (gamma_{k+2} sum|terms|) of every statistic (k = N; N D for SXX); NE and NROWS must be exact."""
    L = StatLayout(D, q)
    vg, vr, va = L.views(np.asarray(got)), L.views(ref), L.views(ab)
    out = {}
    for k in names:
        if k in K3_SCAL:
            i = K3_SCAL[k]
            if k in ("NE", "NROWS"):
                out[k] = 0.0 if vg["scal"][i] == vr["scal"][i] else np.inf
            else:
                g = gamma(N * D + 2) if k == "SXX" else gamma(N + 2)
                out[k] = float(_ratios(vg["scal"][i:i + 1], vr["scal"][i:i + 1], g * va["scal"][i:i + 1]).max())
        else:
            out[k] = float(_ratios(vg[k], vr[k], gamma(N + 2) * va[k]).max())
    others = np.setdiff1d(np.arange(16), list(K3_SCAL.values()))
    out["other scalars 0"] = 0.0 if not np.any(vg["scal"][others]) else np.inf
    return out


def k3_exact_mismatches(got, ref, D, q):
    """Names of the statistics (and scalar slots) that are not bit-identical to the exact reference."""
    L = StatLayout(D, q)
    vg, vr = L.views(np.asarray(got)), L.views(ref)
    bad = [k for k in K3_NAMES if not _bits_equal(vg[k], vr[k])]
    bad += ["scal[%d]" % i for i in range(16) if not _bits_equal(vg["scal"][i:i + 1], vr["scal"][i:i + 1])]
    return bad


def k1_write_failures(mz, N, q, ref, kind, eta_only=False):
    """What a K1 call left in MZ [GUARD + N + GUARD][pitch] (filled with SENT before the call) that it should not have:
    rows [0, N) must be [qprec | +0.0 | eta | untouched tail] (eta_only: [untouched | eta | untouched tail]), guard rows untouched.
    ref: exact qprec / eta."""
    P, PP, ld = _layout(q)
    rows = mz[GUARD:GUARD + N]
    bad = []
    if not (_is_sent(mz[:GUARD]) and _is_sent(mz[GUARD + N:])):
        bad.append("guard rows written")
    if eta_only:
        if not _is_sent(rows[:, :PP]):
            bad.append("[0, Pp) written")
    else:
        if not _bits_equal(rows[:, :P], ref["qprec"]):
            bad.append("[0, P) != qprec")
        if kind != "eta" and not _bits_equal(rows[:, P:PP], np.zeros((N, PP - P))):
            bad.append("[P, Pp) != +0.0")
    if not _bits_equal(rows[:, PP:PP + q], ref["eta"]):
        bad.append("[Pp, Pp + q) != eta")
    if not _is_sent(rows[:, PP + q:]):
        bad.append("pitch tail written")
    return bad


# ============================================================================================== device calls
@pytest.fixture(scope="module")
def dev():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pyvb_b200 import _cabi
    return _cabi


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to("cuda")


def _stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def _host(t):
    import torch
    torch.cuda.synchronize()
    return t.cpu().numpy()


def _data_buffer(A, N, poison, fill_unobserved=None, O=None):
    """[N + GUARD][ld] host copy of A [N][D]: ld = D (clean) or D + XPAD with the pad columns NaN / +-1e300 and rows past N of
    1e300 (poison).  fill_unobserved: the value of the entries whose x is NaN (weights)."""
    N, D = A.shape
    ld = D + (XPAD if poison else 0)
    B = np.zeros((N + GUARD, ld))
    B[:N, :D] = A
    if fill_unobserved is not None:
        B[:N, :D][~O] = fill_unobserved[~O] if np.ndim(fill_unobserved) else fill_unobserved
    if poison:
        B[:N, D::2] = SENT
        B[:N, D + 1::4] = 1e300
        B[:N, D + 3::4] = -1e300
        B[N:] = 1e300
    return B, ld


def _mz_buffer(q, N, M, Z, poison):
    """MZ [GUARD + N + GUARD][pitch]: rows [GUARD, GUARD + N) = [M | pad | Z | tail]; pad, tail, guard rows 0 or SENT."""
    P, PP, ld = _layout(q)
    B = np.full((N + 2 * GUARD, ld), SENT if poison else 0.0)
    B[GUARD:GUARD + N, :P] = M
    B[GUARD:GUARD + N, PP:PP + q] = Z
    return B


def run_k1(cabi, kind, inp, poison, k1_only=1):
    """One K1 call (k1_only: the pyvb_zstep_i8_f64 mode for kind "eta") on MZ rows full of SENT with guard rows; returns the host
    copies of MZ, Sig, logdet and gl (MZ / Sig / logdet with their guard rows)."""
    import torch
    lib = cabi.lib()
    X, O, S = inp["X"], inp["O"], inp["S"]
    N, D = X.shape
    q = len(inp["h0"])
    P, PP, ld = _layout(q)
    assert ld == lib.pyvb_mz_pitch(q) == lib.pyvb_gw_pitch(q) and PP == lib.pyvb_gw_woff(q)
    Gw = np.zeros((D, ld))
    Gw[:, :P], Gw[:, PP:PP + q], Gw[:, PP + q] = inp["G"], inp["Wb"], inp["mu"]
    Xb, ldx = _data_buffer(X, N, poison)
    x, gw, p0, h0 = _t(Xb), _t(Gw), _t(inp["P0"]), _t(inp["h0"])
    gl = np.zeros(GL_LEN)
    gl[GL_TAU] = inp["tau"]
    gld = _t(gl)
    mz = _t(np.full((N + 2 * GUARD, ld), SENT))
    sg = _t(np.full((N + 2 * GUARD, P), SENT))
    lg = _t(np.full(N + 2 * GUARD, SENT))
    mzp, st = mz.data_ptr() + GUARD * ld * 8, _stream()
    if kind == "plain":
        rc = lib.pyvb_zstep_f64(N, D, q, x.data_ptr(), ldx, gw.data_ptr(), ld, p0.data_ptr(), h0.data_ptr(), gld.data_ptr(),
                                mzp + PP * 8, ld, mzp, ld, sg.data_ptr() + GUARD * P * 8, lg.data_ptr() + GUARD * 8, None,
                                ALGO_DMMA_K1, st)
    elif kind == "wt":
        # the weights of unobserved entries are never read: finite values in the clean call, NaN in the poisoned one
        Sb, lds = _data_buffer(S, N, poison, fill_unobserved=SENT if poison else 2.0 - S, O=O)
        s = _t(Sb)
        rc = lib.pyvb_zstep_w_f64(N, D, q, x.data_ptr(), ldx, s.data_ptr(), lds, gw.data_ptr(), ld, p0.data_ptr(),
                                  h0.data_ptr(), gld.data_ptr(), mzp + PP * 8, ld, mzp, ld, sg.data_ptr() + GUARD * P * 8,
                                  lg.data_ptr() + GUARD * 8, None, ALGO_DMMA_K1, st)
    else:
        assert lib.pyvb_i8_supported(D, q)
        mask = torch.zeros(int(lib.pyvb_i8_mask_bytes(N, D)), dtype=torch.uint8, device="cuda")
        cabi.check(lib.pyvb_prepare_mask_i8(N, D, x.data_ptr(), ldx, mask.data_ptr(), st), "prepare_mask_i8")
        gi = torch.zeros(int(lib.pyvb_i8_digits_bytes(D, q)), dtype=torch.uint8, device="cuda")
        gs = torch.zeros(int(lib.pyvb_i8_ncols(q)), dtype=torch.float64, device="cuda")
        wb, wv = _t(inp["Wb"]), _t(inp["Wv"])
        rc = lib.pyvb_zstep_i8_f64(N, D, q, x.data_ptr(), ldx, mask.data_ptr(), wb.data_ptr(), wv.data_ptr(), gw.data_ptr(),
                                   ld, p0.data_ptr(), h0.data_ptr(), gld.data_ptr(), mzp, ld, gi.data_ptr(), gs.data_ptr(),
                                   sg.data_ptr() + GUARD * P * 8, lg.data_ptr() + GUARD * 8, None, k1_only, st)
    cabi.check(rc, "K1 %s" % kind)
    return {"MZ": _host(mz), "Sig": _host(sg), "logdet": _host(lg), "gl": _host(gld), "gl_in": gl}


def run_k3(cabi, kind, inp, poison, xcache=None, xvalid=0, algo=ALGO_DMMA):
    """One statistics call; returns the stats (guards stripped), whether the stats guards and the bytes behind the workspace
    are untouched, the workspace (as doubles), xcache and (XO) the INT8 guard counters."""
    import torch
    lib = cabi.lib()
    X, O, S, M, Z = inp["X"], inp["O"], inp["S"], inp["M"], inp["Z"]
    N, D = X.shape
    q = Z.shape[1]
    P, PP, ld = _layout(q)
    L = StatLayout(D, q)
    Xb, ldx = _data_buffer(X, N, poison)
    x = _t(Xb)
    mz = _t(_mz_buffer(q, N, M, Z, poison))
    mzp = mz.data_ptr() + GUARD * ld * 8
    lg = _t(inp["ld"])
    fill = SENT if poison else 0.0
    stats = _t(np.full(L.len + 2 * GUARD, fill))
    sp = stats.data_ptr() + GUARD * 8
    xc = _t(np.full(2 * D + 2, fill) if xcache is None else xcache)
    st = _stream()
    out = {}
    if kind == "xo":
        wsb = int(lib.pyvb_stats_i8_workspace_bytes(N, D, q))
        ws = _t(np.full(wsb // 8 + 64, fill))
        maskt = torch.zeros(int(lib.pyvb_stats_i8_maskt_bytes(N, D)), dtype=torch.uint8, device="cuda")
        cabi.check(lib.pyvb_prepare_maskt_i8(N, D, x.data_ptr(), ldx, maskt.data_ptr(), st), "prepare_maskt_i8")
        zi = torch.zeros(int(lib.pyvb_stats_i8_digits_bytes(N, q)), dtype=torch.uint8, device="cuda")
        scr = torch.zeros(int(lib.pyvb_stats_i8_scratch_len(q)), dtype=torch.float64, device="cuda")
        rc = lib.pyvb_stats_i8_f64(N, D, q, x.data_ptr(), ldx, maskt.data_ptr(), mzp, ld, lg.data_ptr(), zi.data_ptr(),
                                   scr.data_ptr(), sp, ws.data_ptr(), wsb, xc.data_ptr(), None, None, st)
        go = int(lib.pyvb_stats_i8_guard_offset(q))
        out["i8_guard"] = _host(scr)[go:go + 2]
    else:
        wsb = int(lib.pyvb_stats_workspace_bytes(N, D, q, algo))
        ws = _t(np.full(wsb // 8 + 64, fill))
        if kind == "wt":
            Sb, lds = _data_buffer(S, N, poison, fill_unobserved=SENT if poison else 2.0 - S, O=O)
            s = _t(Sb)
            rc = lib.pyvb_stats_w_f64(N, D, q, x.data_ptr(), ldx, s.data_ptr(), lds, mzp + PP * 8, ld, mzp, ld, lg.data_ptr(),
                                      sp, ws.data_ptr(), wsb, xc.data_ptr(), xvalid, None, 0, None, algo, st)
        else:
            rc = lib.pyvb_stats_f64(N, D, q, x.data_ptr(), ldx, None, None, None, mzp + PP * 8, ld, mzp, ld, lg.data_ptr(),
                                    sp, ws.data_ptr(), wsb, xc.data_ptr(), xvalid, None, 0, None, algo, st)
    cabi.check(rc, "K3 %s" % kind)
    sh, wh = _host(stats), _host(ws)
    gv = np.full(GUARD, fill)
    out.update({"stats": sh[GUARD:GUARD + L.len], "guards": _bits_equal(sh[:GUARD], gv) and _bits_equal(sh[-GUARD:], gv),
                "ws": wh[:wsb // 8], "behind_ws": _bits_equal(wh[wsb // 8:], np.full(64, fill)), "xcache": _host(xc)})
    return out


def _fail_msg(fails):
    return "; ".join("%s: %s" % f for f in fails)


# ============================================================================================== 1 + 3. exact cases, K1
K1_SIZES = ("1", "R-1", "R", "R+1", "pass-1", "pass", "pass+1", "2pass+3")
K1_DMIN = {"plain": 16, "wt": 16, "eta": 64}     # one tile has fewer K chunks than pipeline stages (asserted below)


def k1_size(label, g):
    R, npass = g["R"], g["pass"]
    return {"1": 1, "R-1": R - 1, "R": R, "R+1": R + 1, "pass-1": npass - 1, "pass": npass, "pass+1": npass + 1,
            "2pass+3": 2 * npass + 3}[label]


K1_CASES = ([(kind, q, n, K1_DMIN[kind]) for kind in ("plain", "wt") for q in Q4 for n in K1_SIZES] +
            [("eta", q, n, K1_DMIN["eta"]) for q in Q3 for n in K1_SIZES] +
            [(kind, q, "pass+1", 128) for kind in ("plain", "wt", "eta") for q in (Q3 if kind == "eta" else Q4)] +
            [(kind, q, "R+1", 1024) for kind in ("plain", "wt", "eta") for q in (Q3 if kind == "eta" else Q4)])


@pytest.mark.gpu
@pytest.mark.parametrize("kind,q,size,D", K1_CASES)
def test_k1_exact(dev, kind, q, size, D):
    """Bit-exact qprec / eta rows at a row-tile or grid-pass boundary; the writes; a second call through poisoned inputs."""
    g = k1_geom(q, kind)
    N = k1_size(size, g)
    inp = k1_exact_inputs(kind, q, N, D, seed=1000 * q + N + D)
    ref = k1_exact_reference(inp)
    assert _fp32_inexact(ref["qprec"]) and _fp32_inexact(ref["eta"])
    P, PP, ld = _layout(q)
    tag = "K1 %s q=%d N=%d D=%d (R=%d, pass=%d)" % (kind, q, N, D, g["R"], g["pass"])
    fails = []
    a = run_k1(dev, kind, inp, poison=False)
    fails += [(tag, f) for f in k1_write_failures(a["MZ"], N, q, ref, kind)]
    if not (_is_sent(a["Sig"]) and _is_sent(a["logdet"])):
        fails.append((tag, "Sig / logdet written"))
    gl_expect = a["gl_in"].copy()
    if kind == "eta":
        gl_expect[GL_I8BAD] = 0.0
    if not _bits_equal(a["gl"], gl_expect):
        fails.append((tag, "gl changed (INT8 guard counter %r)" % a["gl"][GL_I8BAD]))
    # poisoned reads (padded pitch, rows past N, NaN weights where x is NaN) and a repeated call: the same bits
    b = run_k1(dev, kind, inp, poison=True, k1_only=3 if kind == "eta" else 1)
    if kind == "eta":         # the eta kernel alone: nothing but the eta columns
        fails += [(tag + " eta alone", f) for f in k1_write_failures(b["MZ"], N, q, ref, kind, eta_only=True)]
    elif not _bits_equal(a["MZ"], b["MZ"]):
        fails.append((tag, "poisoned / repeated call not bit-identical"))
    print("%s: %s" % (tag, "ok" if not fails else _fail_msg(fails)))
    assert not fails, _fail_msg(fails)


# ============================================================================================== 1 + 3. exact cases, K3
K3_SIZES = ("KC-1", "KC+1", "64KC-1", "64KC+1", "chunks")


def k3_shape(kind, q, label):
    g = k3_geom(q, kind == "xo")
    KC, Dp = g["KC"], g["DT"] + 16                         # D = DT + 16: a partial last data-dimension tile
    if label == "large":
        return XO_LARGE if kind == "xo" else EMPTY[q]
    return {"KC-1": KC - 1, "KC+1": KC + 1, "64KC-1": 64 * KC - 1, "64KC+1": 64 * KC + 1, "chunks": 9000}[label], Dp


K3_CASES = ([(kind, q, n) for kind in ("plain", "wt", "xo") for q in (Q3 if kind == "xo" else Q4)
             for n in K3_SIZES + ("large",)] +
            [(kind, 32, "D1024") for kind in ("plain", "wt", "xo")])


def _chunk_partial_failures(inp, ws, kind, nch, kc, names):
    """ws[chunk][stat layout]: the T1 / Bst / Ast partials of every chunk k (rows [k rpc, (k + 1) rpc)) bit-identical to the exact
    sums of those rows -- empty chunks included, which must hold zeros."""
    N, D = inp["X"].shape
    q = inp["Z"].shape[1]
    L = StatLayout(D, q)
    rpc = chunk_rows(N, nch, kc)
    bad = []
    for k in range(nch):
        rows = np.arange(k * rpc, min(N, (k + 1) * rpc))
        ref = L.views(k3_reference(inp, rows=rows)[0])
        got = L.views(ws[k * L.len:(k + 1) * L.len])
        for name in names:
            if not _bits_equal(got[name], ref[name]):
                bad.append("chunk %d/%d (%d rows) %s" % (k, nch, len(rows), name))
    return bad


@pytest.mark.gpu
@pytest.mark.parametrize("kind,q,size", K3_CASES)
def test_k3_exact(dev, kind, q, size):
    """The whole statistics buffer bit-exact around a pipeline step, a row chunk, across many chunks (with an empty trailing one
    where the chunking leaves one) and a partial last d tile; xcache; per-chunk partials; poisoned reads; repeated calls."""
    N, D = (5000, 1024) if size == "D1024" else k3_shape(kind, q, size)
    xo = kind == "xo"
    g = k3_geom(q, xo)
    nch = stats_i8_nchunks(N, D, q) if xo else stats_dmma_nchunks(N, D, q)
    if size == "large" and not xo:
        assert empty_chunks(N, D, q) >= 1, "the shape no longer leaves an empty chunk"
    inp = k3_exact_inputs(kind, q, N, D, seed=100 * q + N + D)
    ref = k3_exact_reference(inp)
    assert _fp32_inexact(ref)
    tag = "K3 %s q=%d N=%d D=%d (KC=%d, DT=%d, %d chunks of %d rows)" % (kind, q, N, D, g["KC"], g["DT"], nch,
                                                                       chunk_rows(N, nch, g["KC"]))
    fails = []
    xc_ref = xcache_of(ref, D, q)
    a = run_k3(dev, kind, inp, poison=False, xcache=xc_ref if xo else None)
    fails += [(tag, "%s not exact" % m) for m in k3_exact_mismatches(a["stats"], ref, D, q)]
    if not _bits_equal(a["xcache"], xc_ref):
        fails.append((tag, "xcache"))
    if xo and np.any(a["i8_guard"]):
        fails.append((tag, "INT8 accuracy guard fired: %r" % a["i8_guard"]))
    # poisoned: padded X / S pitch, rows past N, NaN weights where x is NaN, NaN MZ pad / tail / guard rows, NaN ws and stats
    b = run_k3(dev, kind, inp, poison=True, xcache=xc_ref if xo else None)
    if not _bits_equal(a["stats"], b["stats"]):
        fails.append((tag, "poisoned call differs: %s" % k3_exact_mismatches(b["stats"], ref, D, q)))
    if not (a["guards"] and b["guards"] and a["behind_ws"] and b["behind_ws"]):
        fails.append((tag, "write outside stats / the workspace"))
    if xo and np.any(b["i8_guard"]):
        fails.append((tag, "INT8 accuracy guard fired (poisoned): %r" % b["i8_guard"]))
    fails += [(tag, f) for f in _chunk_partial_failures(inp, b["ws"], kind, nch, g["KC"],
                                                        ("Ast",) if xo else ("T1", "Bst", "Ast"))]
    if not xo:                # the cached X-only sums: the same bytes
        c = run_k3(dev, kind, inp, poison=False, xcache=a["xcache"], xvalid=1)
        if not _bits_equal(c["stats"], a["stats"]):
            fails.append((tag, "xcache_valid = 1 differs"))
    print("%s: %s" % (tag, "ok" if not fails else _fail_msg(fails[:8])))
    assert not fails, _fail_msg(fails[:20])


@pytest.mark.gpu
@pytest.mark.parametrize("wt", [False, True])
@pytest.mark.parametrize("q", Q4)
@pytest.mark.parametrize("D", [1, 17, 37])
@pytest.mark.parametrize("N", [1, 300, 16500])
def test_generic_stats_exact(dev, N, D, q, wt):
    """The generic statistics (where algo=auto sends D % 16 != 0) bit-exact, 1 ... 64 row chunks; poisoned reads."""
    kind = "wt" if wt else "plain"
    lib = dev.lib()
    assert not lib.pyvb_algo_supported(ALGO_DMMA, D, q)
    inp = k3_exact_inputs(kind, q, N, D, seed=7 * N + D + q)
    ref = k3_exact_reference(inp)
    a = run_k3(dev, kind, inp, poison=False, algo=ALGO_GENERIC)
    b = run_k3(dev, kind, inp, poison=True, algo=ALGO_GENERIC)
    bad = k3_exact_mismatches(a["stats"], ref, D, q)
    assert not bad, bad
    assert _bits_equal(a["xcache"], xcache_of(ref, D, q))
    assert _bits_equal(a["stats"], b["stats"]) and a["guards"] and b["guards"] and a["behind_ws"] and b["behind_ws"]


# ============================================================================================== 2. rounding cases
ROUND_N = 1300          # crosses row tiles at every q and the first grid pass at q = 64 (1184 rows)


def k1_round_inputs(kind, q, N, D, seed):
    rng = np.random.RandomState(seed)
    O = _observed(rng, N, D)
    O[:, :2] = True                                           # features 0, 1 and 4, 5: cancelling pairs, always observed
    O[:, 4:6] = True
    X = rng.randn(N, D)
    X[:, 3] *= 1e6                                            # one feature on another scale
    mu = rng.randn(D)
    X[:, 5] = X[:, 4] - mu[4] + mu[5]                         # (x5 - mu5) ~ (x4 - mu4) ...
    X = np.where(O, X, np.nan)
    P = q * (q + 1) // 2
    G = rng.randn(D, P) * 10.0 ** rng.uniform(-8, 8, P)[None, :]      # G columns spread over 1e+-8
    G[1] = -G[0] * (1 + 2.0 ** -30)                                   # ... qprec: d = 0 and 1 cancel
    Wb = rng.randn(D, q) * 10.0 ** rng.uniform(-8, 8, q)[None, :]
    Wb[5] = -Wb[4]                                                    # ... eta: d = 4 and 5 cancel
    S = rng.uniform(0.0, 2.0, (N, D)) if kind == "wt" else None
    if S is not None:
        S[:, 5] = S[:, 4]
    B = rng.randn(q, q)
    return {"X": X, "O": O, "S": S, "mu": mu, "Wb": Wb, "Wv": np.ones((D, q)), "G": G, "tau": 0.7312, "P0": B @ B.T + q * np.eye(q),
            "h0": rng.randn(q)}


K1_ROUND = [(kind, q) for kind in ("plain", "wt") for q in Q4] + [("eta", q) for q in Q3]


def _k1_round_D(kind, q):
    return 128 if kind == "eta" else (64 if q == 64 else 144)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,q", K1_ROUND)
def test_k1_rounding(dev, kind, q):
    """Real data, spread and cancelling columns: every qprec / eta entry within gamma_{D+3} sum|terms| of long double."""
    D = _k1_round_D(kind, q)
    inp = k1_round_inputs(kind, q, ROUND_N, D, seed=q + len(kind))
    ref = k1_reference(inp, np.longdouble)
    r = run_k1(dev, kind, inp, poison=False, k1_only=3)          # (eta: the DMMA eta kernel alone)
    P, PP, ld = _layout(q)
    rows = r["MZ"][GUARD:GUARD + ROUND_N]
    got = {"eta": rows[:, PP:PP + q]}
    if kind != "eta":
        got["qprec"] = rows[:, :P]
    ratios = k1_round_ratios(got, ref, D)
    print("K1 %s q=%d N=%d D=%d worst err / bound: %s" % (kind, q, ROUND_N, D, ratios))
    assert all(v <= 1.0 for v in ratios.values()), ratios


def k3_round_inputs(kind, q, N, D, seed):
    rng = np.random.RandomState(seed)
    O = _observed(rng, N, D)
    P = q * (q + 1) // 2
    scale = 10.0 ** rng.uniform(-6, 6, N)                           # MZ rows spread over 1e+-6
    M = rng.randn(N, P) * scale[:, None]
    M[:, _diag_cols(q)] = np.abs(M[:, _diag_cols(q)])
    Z = rng.randn(N, q) * np.sqrt(scale)[:, None]
    for r in range(2, N - 2, 97):                                   # cancelling row pairs, observed alike
        M[r + 1], Z[r + 1], O[r + 1] = -M[r] * (1 + 2.0 ** -30), -Z[r] * (1 + 2.0 ** -30), O[r]
        M[r + 1, _diag_cols(q)] = M[r, _diag_cols(q)]
    X = rng.randn(N, D)
    X[:, 2] *= 1e6
    return {"X": np.where(O, X, np.nan), "O": O, "S": rng.uniform(0.0, 2.0, (N, D)) if kind == "wt" else None, "M": M, "Z": Z,
            "ld": rng.uniform(0.5, 3.0, N)}


K3_ROUND = [(kind, q) for kind in ("plain", "wt") for q in Q4] + [("xo", q) for q in Q3]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,q", K3_ROUND)
def test_k3_rounding(dev, kind, q):
    """Real data, rows spread over 1e+-6, a feature at 1e6, cancelling rows: every statistic within gamma_{N+2} sum|terms| of
    long double (XO: Ast; the INT8 sums' rounding is test_gpu_i8.py's)."""
    xo = kind == "xo"
    D = k3_geom(q, xo)["DT"] + 16
    inp = k3_round_inputs(kind, q, ROUND_N, D, seed=3 * q + len(kind))
    ref, ab = k3_reference(inp, np.longdouble)
    xc = xcache_of(k3_reference(inp)[0], D, q) if xo else None
    r = run_k3(dev, kind, inp, poison=False, xcache=xc)
    names = ("Ast", "S", "zsum", "QLDZ", "LOGDETZ", "NROWS") if xo else K3_NAMES + tuple(K3_SCAL)
    ratios = k3_round_ratios(r["stats"], ref, ab, ROUND_N, D, q, names)
    print("K3 %s q=%d N=%d D=%d worst err / bound: %s" % (kind, q, ROUND_N, D, ratios))
    assert all(v <= 1.0 for v in ratios.values()), ratios
    assert _bits_equal(xcache_of(r["stats"], D, q), r["xcache"])
    if xo:
        assert not np.any(r["i8_guard"]), r["i8_guard"]


# ============================================================================================== CPU: geometry
def test_geometry_matches_the_kernel_source():
    """The tile / pass / chunk geometry the sizes above were chosen from, recomputed from kernels_dmma.cu and kernels_i8.cu."""
    for kind in ("plain", "wt"):
        assert {q: (k1_geom(q, kind)["R"], k1_geom(q, kind)["pass"]) for q in Q4} == \
            {8: (128, 37888), 16: (64, 18944), 32: (32, 4736), 64: (32, 1184)}, kind
    assert {q: (k1_geom(q, "eta")["R"], k1_geom(q, "eta")["pass"]) for q in Q3} == \
        {16: (64, 18944), 32: (128, 37888), 64: (128, 37888)}
    assert _spec("ZC")[64]["NCT"] == 4 and k1_geom(8, "wt")["ST"] == 2 and k1_geom(8, "plain")["ST"] == 3
    for kind in ("plain", "wt", "eta"):                          # the smallest D: fewer K chunks than pipeline stages
        for q in (Q3 if kind == "eta" else Q4):
            g = k1_geom(q, kind)
            assert K1_DMIN[kind] // g["KC"] < g["ST"], (kind, q, g)
    assert {q: (k3_geom(q)["KC"], k3_geom(q)["DT"]) for q in Q4} == {8: (16, 128), 16: (16, 128), 32: (8, 32), 64: (8, 32)}
    assert {q: (k3_geom(q, True)["KC"], k3_geom(q, True)["DT"]) for q in Q3} == {16: (16, 128), 32: (16, 128), 64: (16, 128)}
    assert k3_geom(64)["NCT"] == 4
    s = _src("kernels_dmma.cu")                                  # stats_dmma_nchunks hard-codes (kc, dt) per q
    assert "if (q >= 32) { kc = 8; dt = 32; }" in s and "int kc = 16, dt = 128, nct = 1;" in s
    # the empty trailing chunks (74 chunks of 1040 rows at q = 8, 16; two empty ones at q = 32, D = 48)
    assert [(stats_dmma_nchunks(*EMPTY[q], q), chunk_rows(EMPTY[q][0], stats_dmma_nchunks(*EMPTY[q], q), k3_geom(q)["KC"]),
             empty_chunks(*EMPTY[q], q)) for q in Q4] == [(74, 1040, 1), (74, 1040, 1), (74, 520, 1), (74, 520, 1)]
    assert empty_chunks(75783, 48, 32) == 2
    for kind in ("plain", "wt", "xo"):
        for q in (Q3 if kind == "xo" else Q4):
            g = k3_geom(q, kind == "xo")
            N, D = k3_shape(kind, q, "KC-1")
            assert D % g["DT"] == 16 and D % 16 == 0
    # the INT8 constants of stats_i8_nchunks
    i8 = _src("kernels_i8.cu")
    assert re.search(r"constexpr int BM = %d, BKB = %d, ST = \d+, CT = %d;" % (I8_BM, I8_BKB, I8_CT), i8)
    assert re.search(r"constexpr int I8_CL = %d;" % I8_CL, i8)
    assert stats_i8_nchunks(*XO_LARGE, 16) > 1 and stats_i8_nchunks(9000, 144, 32) > 1


# ============================================================================================== CPU: the checkers have teeth
def _np_k3(inp, nch, kc, drop=None, twice=None, ignore_weight=None):
    """numpy restatement of the statistics: float64 partial sums per chunk (the kernels' chunking) added in order, with an
    optional fault: a row left out, a row counted twice, one weight taken as 1."""
    N, D = inp["X"].shape
    q = inp["Z"].shape[1]
    inp = dict(inp)
    if ignore_weight is not None:
        S = inp["S"].copy()
        S[ignore_weight] = 1.0
        inp["S"] = S
    rows = np.array([r for r in range(N) if r != drop] + ([twice] if twice is not None else []))
    rpc = chunk_rows(N, nch, kc)
    total = np.zeros(StatLayout(D, q).len)
    for k in range(nch):
        total += k3_reference(inp, rows=rows[(rows >= k * rpc) & (rows < (k + 1) * rpc)])[0]
    return total


def test_checkers_have_teeth():
    """The exact, rounding and write checks pass on numpy restatements of the kernels and fail on a dropped row, a row counted
    twice, an ignored weight, an entry off by 10 x its bound and a write into the pitch tail."""
    # K3, exact: the chunked restatement is bit-identical to the plain reference; every fault is seen
    for kind, q, N, D in (("plain", 8, 300, 144), ("wt", 16, 300, 144), ("wt", 32, 200, 48)):
        inp = k3_exact_inputs(kind, q, N, D, seed=5)
        ref = k3_exact_reference(inp)
        kc = k3_geom(q)["KC"]
        nch = 5
        assert k3_exact_mismatches(_np_k3(inp, nch, kc), ref, D, q) == []
        assert "T1" in k3_exact_mismatches(_np_k3(inp, nch, kc, drop=N // 3), ref, D, q)
        assert "Ast" in k3_exact_mismatches(_np_k3(inp, nch, kc, twice=N - 3), ref, D, q)
        if kind == "wt":
            o = np.argwhere(inp["O"] & (inp["S"] != 1.0))[7]
            bad = k3_exact_mismatches(_np_k3(inp, nch, kc, ignore_weight=tuple(o)), ref, D, q)
            assert "T1" in bad and "cnt" in bad, bad
        # K3, rounding: float64 chunked sums pass the long-double bounds; the faults, and one entry off by 10 x, do not
        rin = k3_round_inputs(kind, q, N, D, seed=6)
        rref, rab = k3_reference(rin, np.longdouble)
        ok = k3_round_ratios(_np_k3(rin, nch, kc), rref, rab, N, D, q)
        assert max(ok.values()) <= 1.0, ok
        assert max(ok[k] for k in ("T1", "Ast")) > 0.0           # the bounds are not so loose that float64 sits at 0
        assert k3_round_ratios(_np_k3(rin, nch, kc, drop=N // 3), rref, rab, N, D, q)["T1"] > 1.0
        assert k3_round_ratios(_np_k3(rin, nch, kc, twice=1), rref, rab, N, D, q)["Ast"] > 1.0
        if kind == "wt":
            o = tuple(np.argwhere(rin["O"])[11])
            assert k3_round_ratios(_np_k3(rin, nch, kc, ignore_weight=o), rref, rab, N, D, q)["cnt"] > 1.0
        got = _np_k3(rin, nch, kc)
        L = StatLayout(D, q)
        for name, idx in (("T1", (3, 1)), ("Ast", (D - 1, q - 1)), ("S", (2,)), ("colx", (D // 2,))):
            bad = got.copy()
            b = L.views(bad)[name]
            bnd = gamma(N + 2) * np.asarray(L.views(rab)[name], dtype=np.float64)
            b[idx] += 10.0 * bnd[idx]
            assert k3_round_ratios(bad, rref, rab, N, D, q)[name] > 5.0, name
        bad = got.copy()
        L.views(bad)["scal"][SC_QLDZ] *= 1 + 1e-9
        assert k3_round_ratios(bad, rref, rab, N, D, q)["QLDZ"] > 1.0
    # K1: float64 restatement (fma epilogue) passes; one entry off by 10 x its bound, an ignored weight fail
    for kind, q, D in (("plain", 16, 144), ("wt", 8, 144), ("wt", 64, 64)):
        N = 40
        rin = k1_round_inputs(kind, q, N, D, seed=9)
        ref = k1_reference(rin, np.longdouble)
        got = {k: np.asarray(v, dtype=np.float64) for k, v in k1_reference(rin).items()}
        ok = k1_round_ratios(got, ref, D)
        assert max(ok.values()) <= 1.0, ok
        for key, ab, idx in (("qprec", "qabs", (N // 2, 1)), ("eta", "eabs", (N - 1, q - 1))):
            bad = dict(got)
            bad[key] = got[key].copy()
            bad[key][idx] += 10.0 * gamma(D + 3) * float(ref[ab][idx])
            assert k1_round_ratios(bad, ref, D)[key] > 5.0, key
        if kind == "wt":
            r2 = dict(rin)
            r2["S"] = rin["S"].copy()
            o = tuple(np.argwhere(rin["O"][:, 6:])[3] + [0, 6])
            r2["S"][o] = 1.0
            got2 = {k: np.asarray(v, dtype=np.float64) for k, v in k1_reference(r2).items()}
            assert max(k1_round_ratios(got2, ref, D).values()) > 1.0
    # K1 writes: the rows as the kernel leaves them pass; a write into the pitch tail, the pad or a guard row fails
    for q in Q4:
        inp = k1_exact_inputs("plain", q, 12, 16, seed=q)
        ref = k1_exact_reference(inp)
        P, PP, ld = _layout(q)
        mz = np.full((12 + 2 * GUARD, ld), SENT)
        mz[GUARD:GUARD + 12, :P], mz[GUARD:GUARD + 12, P:PP], mz[GUARD:GUARD + 12, PP:PP + q] = ref["qprec"], 0.0, ref["eta"]
        assert k1_write_failures(mz, 12, q, ref, "plain") == []
        for r, c, what in ((GUARD + 5, PP + q, "pitch tail written"), (GUARD + 11, ld - 1, "pitch tail written"),
                           (GUARD - 1, 0, "guard rows written"), (GUARD + 12, PP, "guard rows written")):
            bad = mz.copy()
            bad[r, c] = 0.0
            assert what in k1_write_failures(bad, 12, q, ref, "plain"), (q, r, c)
        if PP > P:
            bad = mz.copy()
            bad[GUARD + 3, P] = -0.0
            assert "[P, Pp) != +0.0" in k1_write_failures(bad, 12, q, ref, "plain")
        bad = mz.copy()
        bad[GUARD + 3, 0] = np.nextafter(bad[GUARD + 3, 0], np.inf)
        assert "[0, P) != qprec" in k1_write_failures(bad, 12, q, ref, "plain")
