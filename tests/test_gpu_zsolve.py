"""K2 in FP64 alone through the C-ABI (pyvb_zsolve_f64): the batched q x q SPD inverse / solve IN PLACE on the MZ rows,
[qprec packed | pad | eta] -> [<zz^T> packed | pad | zbar], plus Sigma, ln prod diag chol and the per-CTA partials -- the
arithmetic of Gaussian.update, /root/reference/src/pyvb/nodes/gaussian.py:117-123 (cho_factor, cho_solve(., I), dot(qcov, .),
q_ln_det).  One kernel per q: thread per matrix (q = 8, kernels_k2t.cu), Gauss-Jordan in registers (q = 16, 32, kernels_k2g.cu),
blocked symmetric sweep (q = 64, kernels_k2s.cu).

Inputs: a pool of SPD matrices A_k = D_k H_k D_k (cond(H_k) 1e2 ... 1e8, diag(D_k) spread up to 1e+-4), whose inverse S_k and
half log-determinant are computed once in long double from the float64 matrix as stored.  Row n solves 2^s A_k (s in [-20, 20])
with its own eta_n: the power-of-two scale is exact, so S_n = 2^-s S_k and the log-determinant moves by q s ln2 / 2, and
zeta_n = S_n eta_n costs O(q^2) in long double.  Rows of every condition, spread and scale are interleaved (every warp group
mixes them), so a row of small scale cannot hide behind a large one: every bound is per row.

Per-row bounds (u = 2^-53, kappa = the float64 condition number of the equilibrated matrix, c = 2):
  Sigma    |Sigma_ij - S_ij| <= c q kappa u sqrt(S_ii S_jj)
  zbar     |z_i - zeta_i| <= c q kappa u sqrt(S_ii) sum_j sqrt(S_jj) |eta_j| + u |zeta_i|
  <zz^T>   what the two imply for zeta_i zeta_j + S_ij, plus the rounding of the fused multiply-add that forms it
  logdet   |ld - lambda| <= c q kappa u + 4 u |lambda|
  LAPACK   the tight check: the largest scaled error |Sigma_ij - S_ij| / sqrt(S_ii S_jj) of a row is at most 8 x that of scipy's
           cho_factor / cho_solve on the same float64 matrix, plus q u (the restatements in oracle/ stay within 1.7 x of it)
The partials, the writes (guard rows, pad and pitch tail, optional outputs, repeated calls) and non-PD rows are checked per
kernel at every boundary of its grid: N = 1, around a warp group, around one CTA's rows and around one and two grid passes.
Every check prints its worst error over its bound."""
import functools

import numpy as np
import pytest
from scipy.linalg import cho_factor, cho_solve

from helpers import half_logdet_ld, refined_inverse

U = 2.0 ** -53
C_SOLVE = 2.0
LAPACK_FAC = 8.0
CONDS = (1e2, 1e4, 1e6, 1e8)     # pool entry k: cond(H_k) ~ CONDS[k % 4]
SPREADS = (0, 2, 4)              # ... diag(D_k) = 10^uniform(-e, e), e = SPREADS[(k // 4) % 3]
NPOOL = 96
SMAX = 20                        # row scales 2^s, |s| <= SMAX
GROUP = {8: 32, 16: 8, 32: 2, 64: 2}   # matrices per warp group: a lane / 4 lanes / 16 lanes / half a warp per matrix
GUARD = 40                       # sentinel rows before and after every output
SENT = -768.0
CHUNK = 256                      # rows per block of the long-double checks
ROW_CHECKS = ("Sigma", "zbar", "<zz^T>", "logdet", "LAPACK")


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


def _sym(A):
    """The symmetric matrix of the lower triangle (what the kernels read of a packed row)."""
    return np.tril(A) + np.swapaxes(np.tril(A, -1), -1, -2)


def _scaled_err(Sp, ref, q):
    """Per row: max_ij |Sp_ij - ref_ij| / sqrt(ref_ii ref_jj) over the packed lower triangle (Sp [n, P], ref [n, q, q])."""
    ii, jj = np.tril_indices(q)
    d = np.sqrt(np.diagonal(ref, axis1=-2, axis2=-1))
    return (np.abs(Sp - ref[:, ii, jj]) / (d[:, ii] * d[:, jj])).astype(np.float64).max(1)


@functools.lru_cache(maxsize=None)
def _pool(q, npool=NPOOL):
    """SPD matrices A_k = D_k H_k D_k (float64, symmetric) with long-double references, and per entry the scaled error of
    LAPACK's route on 2^p A_k, p = 0, 1 (on 2^s A_k it is that of p = s mod 2: every operation but the square roots of the
    Cholesky factorisation commutes exactly with a power-of-two scale)."""
    assert np.finfo(np.longdouble).eps < 1e-18, "the references need an 80-bit (or wider) long double"
    A = np.empty((npool, q, q))
    for k in range(npool):
        H = _case(1, q, 1000 * q + k, CONDS[k % 4])[0][0]
        e = SPREADS[(k // 4) % 3]
        d = 10.0 ** np.random.RandomState(k).uniform(-e, e, q)
        A[k] = _sym(d[:, None] * H * d[None, :])
    S = refined_inverse(A)
    dg = np.sqrt(np.diagonal(A, axis1=1, axis2=2))
    lap = np.empty((npool, 2))
    ii, jj = np.tril_indices(q)
    for k in range(npool):
        for p in (0, 1):
            Ap = A[k] * 2.0 ** p
            Sl = cho_solve(cho_factor(Ap), np.eye(q))
            lap[k, p] = _scaled_err(Sl[None, ii, jj], S[k:k + 1] / np.longdouble(2.0 ** p), q)[0]
    return {"A": A, "S": S, "hld": half_logdet_ld(A), "lap": lap,
            "kappa": np.linalg.cond(A / (dg[:, :, None] * dg[:, None, :])),
            "cond": np.array([CONDS[k % 4] for k in range(npool)]),
            "spread": np.array([SPREADS[(k // 4) % 3] for k in range(npool)])}


def _rows(q, N, seed, npool=NPOOL):
    """Row n: pool entry k(n) (consecutive rows step through all four conditions), scale 2^s(n), eta_n."""
    rng = np.random.RandomState(seed)
    k = (7 * np.arange(N) + rng.randint(npool)) % npool
    s = rng.randint(-SMAX, SMAX + 1, size=N)
    return k, s, rng.randn(N, q) * 3.0


def _inputs(q, pool, k, s):
    ii, jj = np.tril_indices(q)
    return np.ldexp(pool["A"][k][:, ii, jj], s[:, None])


def _refs(q, pool, k, s, eta):
    """Long-double references and per-entry bounds of rows (k, s, eta)."""
    ii, jj = np.tril_indices(q)
    sc = np.exp2(-s.astype(np.float64)).astype(np.longdouble)
    S = pool["S"][k] * sc[:, None, None]
    dS = np.sqrt(np.diagonal(S, axis1=1, axis2=2))
    e = eta.astype(np.longdouble)
    zeta = np.einsum("nij,nj->ni", S, e)
    Sp = S[:, ii, jj]
    kap = C_SOLVE * q * pool["kappa"][k] * U
    bS = (kap[:, None] * dS[:, ii] * dS[:, jj]).astype(np.float64)
    bz = (kap[:, None] * dS * (dS * np.abs(e)).sum(1)[:, None] + U * np.abs(zeta)).astype(np.float64)
    zi, zj = np.abs(zeta[:, ii]).astype(np.float64), np.abs(zeta[:, jj]).astype(np.float64)
    bM = (1 + 2 * U) * (bS + bz[:, ii] * (zj + bz[:, jj]) + zi * bz[:, jj]) + U * (zi * zj + np.abs(Sp).astype(np.float64))
    lam = pool["hld"][k] + q * s * np.log(np.longdouble(2)) / 2
    bld = kap + 4 * U * np.abs(lam).astype(np.float64)
    return {"S": S, "Sp": Sp, "zeta": zeta, "M": Sp + zeta[:, ii] * zeta[:, jj], "lam": lam,
            "bS": bS, "bz": bz, "bM": bM, "bld": bld, "blap": LAPACK_FAC * pool["lap"][k, s & 1] + q * U}


def _row_ratios(q, pool, k, s, eta, sig, z, m2, ld):
    """Per row, the worst error over its bound of each row check; sig, m2 packed [N, P], z [N, q], ld [N]."""
    N = len(k)
    out = {c: np.zeros(N) for c in ROW_CHECKS}
    for a in range(0, N, CHUNK):
        b = min(N, a + CHUNK)
        r = _refs(q, pool, k[a:b], s[a:b], eta[a:b])
        eS = _scaled_err(sig[a:b], r["S"], q)
        out["Sigma"][a:b] = (np.abs(sig[a:b] - r["Sp"]).astype(np.float64) / r["bS"]).max(1)
        out["zbar"][a:b] = (np.abs(z[a:b] - r["zeta"]).astype(np.float64) / r["bz"]).max(1)
        out["<zz^T>"][a:b] = (np.abs(m2[a:b] - r["M"]).astype(np.float64) / r["bM"]).max(1)
        out["logdet"][a:b] = np.abs(ld[a:b] - r["lam"]).astype(np.float64) / r["bld"]
        out["LAPACK"][a:b] = eS / r["blap"]
    for c in ROW_CHECKS:                             # a NaN is a failure, not a pass
        out[c][np.isnan(out[c])] = np.inf
    return out


def _report(what, ratio, fails):
    print("%-60s worst err / bound = %.3g" % (what, ratio))
    if not ratio <= 1.0:
        fails.append((what, ratio))


def _report_rows(tag, pool, k, s, ratios, fails):
    """One line per (condition, spread) of the pool entries: the worst ratio of every row check."""
    for cond in CONDS:
        for e in SPREADS:
            sel = (pool["cond"][k] == cond) & (pool["spread"][k] == e)
            if not sel.any():
                continue
            worst = {c: float(ratios[c][sel].max()) for c in ROW_CHECKS}
            print("%s cond %.0e spread 1e+-%d: %s" % (tag, cond, e, "  ".join("%s %.3g" % kv for kv in worst.items())))
            for c, v in worst.items():
                if not v <= 1.0:
                    n = np.flatnonzero(sel)[np.argmax(ratios[c][sel])]
                    fails.append(("%s cond %.0e spread %d %s (row %d, k %d, s %d)" % (tag, cond, e, c, n, k[n], s[n]), v))


def _partial_ratios(q, out, ld, part):
    """K2's per-CTA partials [column sums (PP + q) | sum 0.5/logdet, sum logdet, rows, 0 | bounds on the column maxima (PP + q)]
    of the output rows out [N, >= PP + q] and their log-dets: dict name -> worst err / bound (<= 1 passes)."""
    N, nblk = len(ld), part.shape[0]
    P = q * (q + 1) // 2
    PP = (P + 7) & ~7
    OROW = PP + q
    cols = np.r_[0:P, PP:OROW]                       # the packed and zbar columns (the pad is passed through)
    v = out[:, cols]
    tot = part[:, :OROW + 4].astype(np.longdouble).sum(0)
    r = {}
    r["column sums"] = float(np.max(np.abs(tot[cols] - v.astype(np.longdouble).sum(0)).astype(np.float64) /
                                    ((N + nblk) * U * np.abs(v).sum(0) + 1e-300)))
    for name, slot, x in (("sum 0.5/logdet", 0, 0.5 / ld), ("sum logdet", 1, ld)):
        err = abs(float(tot[OROW + slot] - x.astype(np.longdouble).sum()))
        r[name] = err / ((N + nblk + 1) * U * np.abs(x).sum() + 1e-300)
    r["rows == N"] = 0.0 if tot[OROW + 2] == N else np.inf
    r["slot 3 == 0"] = 0.0 if np.all(part[:, OROW + 3] == 0.0) else np.inf
    mx = part[:, OROW + 4:].max(0)[cols]
    true = np.abs(v).max(0)
    r["maxima >= max|column|"] = 0.0 if np.all(mx >= true) else np.inf
    if q == 8:                                       # high words of |v|, rounded up by one unit
        r["maxima tight (2^-20)"] = float(np.max((mx - true) / (2.0 ** -20 * true + 1e-300)))
    else:                                            # sqrt(max <z_i z_i> max <z_j z_j>): exact on the diagonal, max|z_i| exact
        tight = [i * (i + 1) // 2 + i for i in range(q)] + list(range(P, P + q))
        r["maxima tight (1e-12)"] = float(np.max((mx[tight] - true[tight]) / (1e-12 * true[tight] + 1e-300)))
    for key in r:
        if np.isnan(r[key]):
            r[key] = np.inf
    return r


def _lib():
    from pyvb_b200 import _cabi
    return _cabi, _cabi.lib()


def _geometry(q):
    """(rows per CTA, rows per grid pass) of the K2 kernel of q, from the number of partials it writes."""
    _, lib = _lib()
    n = 1
    while lib.pyvb_zsums_blocks(n, q) < 2:
        n += 1
    rpc = n - 1
    assert lib.pyvb_zsums_blocks(148 * rpc, q) == 148 and lib.pyvb_zsums_blocks(148 * rpc + 1, q) == 148
    return rpc, 148 * rpc


# N at the boundaries of a kernel's grid, from (matrices per warp group, rows per CTA, rows per grid pass); N = 1 is a
# plain integer case of every q (CASES)
SIZES = {"group-1": lambda g, rpc, npass: g - 1, "group+1": lambda g, rpc, npass: g + 1,
         "rpc-1": lambda g, rpc, npass: rpc - 1, "rpc+1": lambda g, rpc, npass: rpc + 1,
         "npass-1": lambda g, rpc, npass: npass - 1, "npass+1": lambda g, rpc, npass: npass + 1,
         "2npass+3": lambda g, rpc, npass: 2 * npass + 3}


def _size(q, n):
    return n if isinstance(n, int) else SIZES[n](GROUP[q], *_geometry(q))


def _call(q, Ap, eta, sig=True, zs=True):
    """One pyvb_zsolve_f64 call on the rows [Ap | pad | eta | tail] (pad and pitch tail hold SENT) with GUARD rows of SENT before
    and after MZ, Sigma and logdet and behind the partials; returns the whole buffers, guards included."""
    import torch
    _cabi, lib = _lib()
    N = Ap.shape[0]
    P = q * (q + 1) // 2
    ld, zoff = int(lib.pyvb_mz_pitch(q)), int(lib.pyvb_gw_woff(q))
    MZ = np.full((N + 2 * GUARD, ld), SENT)
    MZ[GUARD:GUARD + N, :P] = Ap
    MZ[GUARD:GUARD + N, zoff:zoff + q] = eta
    dev = torch.device("cuda", 0)
    f64 = torch.float64
    mz = torch.as_tensor(MZ, device=dev)
    sg = torch.full((N + 2 * GUARD, P), SENT, dtype=f64, device=dev)
    lg = torch.full((N + 2 * GUARD,), SENT, dtype=f64, device=dev)
    gl = torch.zeros(144, dtype=f64, device=dev)
    nz = int(lib.pyvb_zsums_len(N, q))
    zsb = torch.full((nz + GUARD,), SENT, dtype=f64, device=dev)
    _cabi.check(lib.pyvb_zsolve_f64(N, q, mz.data_ptr() + GUARD * ld * 8, ld, sg.data_ptr() + GUARD * P * 8 if sig else 0,
                                    lg.data_ptr() + GUARD * 8, gl.data_ptr(), zsb.data_ptr() if zs else 0,
                                    torch.cuda.current_stream(dev).cuda_stream), "zsolve")
    torch.cuda.synchronize()
    return {"MZ": mz.cpu().numpy(), "Sig": sg.cpu().numpy(), "logdet": lg.cpu().numpy(), "gl": gl.cpu().numpy(),
            "zs": zsb.cpu().numpy(), "nz": nz}


def _same(a, b):
    return a.shape == b.shape and np.array_equal(np.ascontiguousarray(a).view(np.int64), np.ascontiguousarray(b).view(np.int64))


def _is_sent(a):
    return _same(a, np.full(a.shape, SENT))


CASES = ([(8, 1000), (16, 1), (16, 4099), (32, 2500), (32, 3), (64, 700), (64, 1), (8, 1), (32, 1)] +
         [(q, n) for q in (8, 16, 32, 64) for n in SIZES])


@pytest.mark.gpu
@pytest.mark.parametrize("q,N", CASES)
def test_zsolve_matches_lapack(q, N):
    """Every output row against the long-double references (per-row bounds and no worse than LAPACK), and the partials."""
    N = _size(q, N)
    pool = _pool(q)
    k, s, eta = _rows(q, N, seed=7919 * q + N)
    r = _call(q, _inputs(q, pool, k, s), eta)
    P = q * (q + 1) // 2
    zoff = (P + 7) & ~7
    out = r["MZ"][GUARD:GUARD + N]
    sig, ld = r["Sig"][GUARD:GUARD + N], r["logdet"][GUARD:GUARD + N]
    fails = []
    _report("K2 q=%d N=%d gl[NONPD] == 0" % (q, N), 0.0 if r["gl"][11] == 0.0 else np.inf, fails)
    ratios = _row_ratios(q, pool, k, s, eta, sig, out[:, zoff:zoff + q], out[:, :P], ld)
    _report_rows("K2 q=%d N=%d" % (q, N), pool, k, s, ratios, fails)
    _, lib = _lib()
    nblk = int(lib.pyvb_zsums_blocks(N, q))
    part = r["zs"][:r["nz"]].reshape(nblk, int(lib.pyvb_zsums_kw(q)))
    for name, v in _partial_ratios(q, out, ld, part).items():
        _report("K2 q=%d N=%d partials: %s" % (q, N, name), v, fails)
    assert not fails, fails


@pytest.mark.gpu
@pytest.mark.parametrize("q,N", CASES)
def test_zsolve_writes_nothing_else(q, N):
    """No write outside the N rows and their used columns (guard rows, the pad [P, PP) and the pitch tail past PP + q keep what was
    there); Sigma = NULL and / or zsums = NULL change nothing else; a second call is bit-identical, partials included."""
    N = _size(q, N)
    pool = _pool(q)
    k, s, eta = _rows(q, N, seed=7919 * q + N)
    Ap = _inputs(q, pool, k, s)
    full = _call(q, Ap, eta)
    P = q * (q + 1) // 2
    zoff = (P + 7) & ~7
    rows = slice(GUARD, GUARD + N)
    fails = []

    def check(what, ok):
        _report("K2 q=%d N=%d %s" % (q, N, what), 0.0 if ok else np.inf, fails)

    check("MZ guard rows", _is_sent(full["MZ"][:GUARD]) and _is_sent(full["MZ"][GUARD + N:]))
    check("MZ pad [P, PP) passed through", _is_sent(full["MZ"][rows, P:zoff]))
    check("MZ pitch tail passed through", _is_sent(full["MZ"][rows, zoff + q:]))
    check("Sigma guard rows", _is_sent(full["Sig"][:GUARD]) and _is_sent(full["Sig"][GUARD + N:]))
    check("logdet guard rows", _is_sent(full["logdet"][:GUARD]) and _is_sent(full["logdet"][GUARD + N:]))
    check("nothing behind the partials", _is_sent(full["zs"][full["nz"]:]))
    check("gl: only NONPD, and 0", not np.any(full["gl"]))
    again = _call(q, Ap, eta)
    check("second call bit-identical", all(_same(full[key], again[key]) for key in ("MZ", "Sig", "logdet", "zs", "gl")))
    nosig = _call(q, Ap, eta, sig=False)
    check("Sigma = NULL: the rest bit-identical", all(_same(full[key], nosig[key]) for key in ("MZ", "logdet", "zs")) and
          _is_sent(nosig["Sig"]))
    nozs = _call(q, Ap, eta, zs=False)
    check("zsums = NULL: the rest bit-identical", all(_same(full[key], nozs[key]) for key in ("MZ", "Sig", "logdet")) and
          _is_sent(nozs["zs"]))
    neither = _call(q, Ap, eta, sig=False, zs=False)
    check("both NULL: MZ, logdet bit-identical", _same(full["MZ"], neither["MZ"]) and _same(full["logdet"], neither["logdet"]))
    assert not fails, fails


def _bad_rows(q, rpc, npass):
    """Non-PD matrices by row: indefinite, a NaN entry, a PSD matrix with an all-zero row and column (its pivot is exactly 0 in
    every kernel: an elimination leaves a zero row zero) -- in row 0, beside valid rows of one warp group, in the second grid
    pass and in the last row."""
    g = GROUP[q]
    indef = _case(1, q, seed=5, cond=10.0)[0][0] - 50.0 * np.eye(q)     # (the earlier test's non-PD row)
    H = _case(2, q, seed=6, cond=1e4)[0]
    nan1, nan2, zero1, zero2 = H[0].copy(), H[1].copy(), H[0].copy(), H[1].copy()
    nan1[q - 1, 1] = nan1[1, q - 1] = np.nan
    nan2[q // 2, q // 2] = np.nan
    zero1[3, :] = zero1[:, 3] = 0.0
    zero2[q - 1, :] = zero2[:, q - 1] = 0.0
    N = npass + 2 * g + 5
    return N, {0: indef, g + 1: nan1, 17: zero1, npass + 1: nan2, npass + g + 1: zero2, N - 1: indef}


@pytest.mark.gpu
@pytest.mark.parametrize("q", [8, 16, 32, 64])
def test_zsolve_flags_non_pd(q):
    """Several non-PD rows in one call: counted exactly, a non-finite log-det each, and every other row bit-identical to the same
    call with valid matrices in their place."""
    rpc, npass = _geometry(q)
    N, bad = _bad_rows(q, rpc, npass)
    pool = _pool(q)
    k, s, eta = _rows(q, N, seed=31 * q)
    Ap = _inputs(q, pool, k, s)
    ref = _call(q, Ap, eta)
    ii, jj = np.tril_indices(q)
    Abad = Ap.copy()
    for n, A in bad.items():
        Abad[n] = A[ii, jj]
    got = _call(q, Abad, eta)
    idx = np.array(sorted(bad))
    keep = np.setdiff1d(np.arange(N), idx) + GUARD
    fails = []
    _report("K2 q=%d N=%d gl[NONPD] == %d" % (q, N, len(bad)), 0.0 if got["gl"][11] == len(bad) else np.inf, fails)
    _report("K2 q=%d N=%d logdet of the bad rows not finite" % (q, N),
            0.0 if not np.any(np.isfinite(got["logdet"][idx + GUARD])) else np.inf, fails)
    for key in ("MZ", "Sig", "logdet"):
        _report("K2 q=%d N=%d other rows' %s bit-identical" % (q, N, key), 0.0 if _same(got[key][keep], ref[key][keep]) else np.inf,
                fails)
    _report("K2 q=%d N=%d guard rows" % (q, N), 0.0 if all(_is_sent(got[key][:GUARD]) and _is_sent(got[key][GUARD + N:])
                                                          for key in ("MZ", "Sig", "logdet")) else np.inf, fails)
    assert not fails, fails


# --------------------------------------------------------------------------------------------- the checks have teeth (CPU)
def _lapack_route(A, eta):
    """The reference's route: cho_factor, cho_solve(., I), dot(qcov, eta), ln prod diag chol (as a sum of logarithms)."""
    Sg, z, ld = [], [], []
    for a, e in zip(A, eta):
        c = cho_factor(a)
        S = cho_solve(c, np.eye(a.shape[0]))
        Sg.append(S)
        z.append(S @ e)
        ld.append(np.sum(np.log(np.diag(c[0]))))
    return np.array(Sg), np.array(z), np.array(ld)


def _np_partials(q, out, ld, nblk):
    """Partials of rows out [N, PP + q] in nblk contiguous blocks, in the layout of the kernels (exact column maxima)."""
    P = q * (q + 1) // 2
    OROW = (P + 7 & ~7) + q
    part = np.zeros((nblk, 2 * OROW + 4))
    for b, r in enumerate(np.array_split(np.arange(len(ld)), nblk)):
        part[b, :OROW] = out[r].sum(0)
        part[b, OROW:OROW + 3] = (0.5 / ld[r]).sum(), ld[r].sum(), len(r)
        part[b, OROW + 4:] = np.abs(out[r]).max(0)
    return part


def test_zsolve_checks_have_teeth():
    """The row and partial checks above pass on the numpy restatements of the kernels (oracle/gj_oracle.py, oracle/tsweep_oracle.py)
    and on scipy's route, and fail on a result with one entry off by 10 x its bound, or one row's Sigma scaled by 1 + 1e-9."""
    from oracle.gj_oracle import gj_solve
    from oracle.tsweep_oracle import tsweep_solve
    solvers = {8: _lapack_route, 16: gj_solve, 32: _lapack_route, 64: lambda A, e: tsweep_solve(A, e, mpw=2)[:3]}
    for q, N in ((8, 40), (16, 40), (32, 16), (64, 6)):
        npool = 24 if q < 64 else 12
        pool = _pool(q, npool)
        k, s, eta = _rows(q, N, seed=q, npool=npool)
        A = _sym(np.ldexp(pool["A"][k], s[:, None, None]))
        Sg, z, ld = solvers[q](A, eta)
        ii, jj = np.tril_indices(q)
        sig = Sg[:, ii, jj]
        m2 = (Sg + z[:, :, None] * z[:, None, :])[:, ii, jj]
        ratios = _row_ratios(q, pool, k, s, eta, sig, z, m2, ld)
        for c in ROW_CHECKS:
            assert ratios[c].max() <= 1.0, (q, c, ratios[c].max())
        r = _refs(q, pool, k, s, eta)
        n = N // 2
        for name, arr, bnd, idx in (("Sigma", sig, r["bS"], (n, 1)), ("zbar", z, r["bz"], (n, q - 1)),
                                    ("<zz^T>", m2, r["bM"], (n, 2)), ("logdet", ld, r["bld"], (n,))):
            bad = arr.copy()
            bad[idx] += 10.0 * bnd[idx]
            args = {"sig": sig, "z": z, "m2": m2, "ld": ld}
            args[{"Sigma": "sig", "zbar": "z", "<zz^T>": "m2", "logdet": "ld"}[name]] = bad
            got = _row_ratios(q, pool, k, s, eta, **args)[name]
            assert got[n] > 5.0 and np.all(np.delete(got, n) <= 1.0), (q, name, got[n])
        n2 = int(np.flatnonzero(pool["cond"][k] == 1e2)[0])
        bad = sig.copy()
        bad[n2] *= 1.0 + 1e-9
        got = _row_ratios(q, pool, k, s, eta, bad, z, m2, ld)
        assert got["Sigma"][n2] > 1.0 and got["LAPACK"][n2] > 1.0, (q, got["Sigma"][n2], got["LAPACK"][n2])

        # partials: exact block sums / maxima pass; a column sum off by 10 x its bound, or a maximum below the column's, fail
        zoff = (q * (q + 1) // 2 + 7) & ~7
        out = np.zeros((N, zoff + q))
        out[:, :q * (q + 1) // 2], out[:, zoff:] = m2, z
        part = _np_partials(q, out, ld, 3)
        assert all(v <= 1.0 for v in _partial_ratios(q, out, ld, part).values())
        bad = part.copy()
        bad[1, 0] += 10.0 * (N + 3) * U * np.abs(out[:, 0]).sum()
        assert _partial_ratios(q, out, ld, bad)["column sums"] > 1.0
        bad = part.copy()
        bad[:, zoff + q + 4 + zoff] = np.abs(out[:, zoff]).max() * (1 - 1e-15)
        assert _partial_ratios(q, out, ld, bad)["maxima >= max|column|"] > 1.0
        bad = part.copy()
        bad[:, zoff + q + 2] += 1.0
        assert _partial_ratios(q, out, ld, bad)["rows == N"] > 1.0
