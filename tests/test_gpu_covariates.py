"""GPU tests of known row covariates (PlateEngine(..., covariates=C)): sweep-by-sweep parity with the covariate oracle on the
INT8, DMMA and sparse paths with every noise model, weights, ARD and both W posteriors; the condition / finish kernels' writes,
determinism and row ranges; the INT8 statistics against the DMMA ones; an unnormalised covariate; the forced INT8 guard; the
error contract; two GPUs; and a full-size fit."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import tensor_rel
from oracle.covariates_oracle import cov_oracle_class, synth_covariates
from test_gpu_sparse import _free_port, densify
from test_oracle_covariates import REC_ANGLE, REC_B, REC_TAU, principal_angle_deg

pytestmark = pytest.mark.gpu
TOL = 1e-9
KEYS = ("Zbar", "Sig", "Wbar", "Wvar", "Bbar", "Bvar", "mu", "qb")


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pyvb_b200 import PlateEngine
    return PlateEngine


def rand_init(N, D, q, k, seed=0, diag=False, rows=False, bscale=0.5):
    rng = np.random.RandomState(seed)
    st = {"Wbar": rng.randn(D, q), "Bbar": rng.randn(D, k) * bscale, "Wvar": rng.rand(D, q) + 0.5, "Bvar": rng.rand(D, k) + 0.5,
          "mu": rng.randn(D) * 0.1, "muvar": np.ones(D), "Zbar": rng.randn(N, q),
          "Sig": np.tile(np.eye(q), (N, 1, 1)) * (rng.rand(N, 1, 1) + 0.5), "qb": (rng.rand(D) + 0.3) if diag else 0.7,
          "al_qb": rng.rand(q + k) + 0.5}
    if rows:
        B = rng.randn(D, q + k, q + k) * (0.3 / np.sqrt(q + k))
        st["Wcov"] = B @ np.transpose(B, (0, 2, 1)) + np.einsum("di,ij->dij", rng.rand(D, q + k) + 0.5, np.eye(q + k))
        del st["Wvar"], st["Bvar"]
    return st


def to_sparse(X):
    import scipy.sparse as sp
    O = ~np.isnan(X)
    r, c = np.nonzero(O)
    return sp.csr_matrix((X[r, c], (r, c)), shape=X.shape)


def case_data(N, D, q, k, dens, weighted, seed, cscale=1.0):
    X, C, _, _, _ = synth_covariates(N, D, q, k, 0.2 if dens is None else 1.0 - dens, tau=10.0, seed=seed, cscale=cscale)
    X[3] = np.nan                                            # an all-missing row
    Wd = None
    if weighted:
        Wd = np.where(np.isnan(X), 0.0, 10.0 ** np.random.RandomState(seed + 1).uniform(-1, 1, size=X.shape))
    if dens is None:
        return X, X, Wd, Wd
    A = to_sparse(X)
    Wt = None
    if weighted:
        import scipy.sparse as sp
        Wt = sp.csr_matrix((Wd[A.nonzero()], A.nonzero()), shape=X.shape)
    return A, X, Wt, Wd


def user_keys(st):
    return [key for key in KEYS + ("Wcov", "al_qb") if key in st]


def run_parity(eng, N, D, q, k, algo, dens, weighted, diag, ard, rows, sweeps=3, cscale=1.0, expect_i8=None):
    from pyvb_b200._layout import GL_ELBO_W
    A, X, Wt, Wd = case_data(N, D, q, k, dens, weighted, seed=N + D + q, cscale=cscale)
    C = synth_covariates(N, D, q, k, 0.0, seed=N + D + q, cscale=cscale)[1]
    init = rand_init(N, D, q, k, seed=1, diag=diag, rows=rows, bscale=0.5 / cscale)
    # P0 = 2 I: the all-missing row 3 then has a finite bound term (the reference's q_ln_det = .5 / ln prod diag chol is
    # infinite for a row whose precision is the identity)
    kw = {"a0": np.random.RandomState(D).rand(D) + 0.01} if diag else {}
    kw["P0"] = 2.0 * np.eye(q)
    o = cov_oracle_class(diag, weighted, rows)(X, q, C, ard=ard, weights=Wd, **kw) if weighted else \
        cov_oracle_class(diag, weighted, rows)(X, q, C, ard=ard, **kw)
    o.load_user_state(init)
    if ard:
        o.al_qb = init["al_qb"].copy()
    e = eng(A, q, algo=algo, ard=ard, weights=Wt, noise="diagonal" if diag else "scalar",
            w_posterior="rows" if rows else "columns", covariates=C, **kw)
    if expect_i8 is not None:
        assert bool(e.use_i8) == expect_i8
    e.set_state(init)
    e.fall = []                                              # INT8 guard fall-backs of each sweep's Z step
    for it in range(sweeps):
        before = e.i8_fallbacks()[0]
        ref, got = o.iterate(), e.iterate()
        e.fall.append(e.i8_fallbacks()[0] - before)
        assert np.isfinite(ref) and abs(got - ref) <= TOL * abs(ref), (it, got, ref)
        ew, ow = float(e.gl[GL_ELBO_W].item()), o.elbo_terms()["W"]
        assert abs(ew - ow) <= TOL * abs(ow), (it, ew, ow)
        st, us = e.get_state(), o.user_state()
        for key in user_keys(us):
            if key == "al_qb" and not ard:
                continue
            assert tensor_rel(st[key], us[key]) < TOL, (it, key, tensor_rel(st[key], us[key]))
    e.check()
    return e, o


# (N, D, q, k, algo, sparse density or None, weighted, per-dimension noise, ARD, rows): INT8 at q' = 16, 32, 64, DMMA at
# q' = 8 .. 64, generic at q' = 7, 13, 23 (explicit and chosen by "auto"), sparse at q' = 8, 16, 32; every noise model,
# weights, ARD and both W posteriors; N leaves partial tiles
CASES = [(701, 128, 12, 4, "auto", None, False, False, False, False), (603, 128, 28, 4, "auto", None, False, True, True, False),
         (501, 128, 60, 4, "auto", None, False, False, True, True), (517, 64, 6, 2, "dmma", None, True, True, True, False),
         (611, 128, 13, 3, "dmma", None, True, False, False, True), (409, 64, 31, 1, "dmma", None, False, False, True, False),
         (333, 64, 56, 8, "dmma", None, False, True, False, False), (403, 45, 5, 3, "auto", 0.6, False, True, False, False),
         (411, 100, 14, 2, "auto", 0.3, True, False, True, True), (505, 200, 29, 3, "auto", 0.2, False, False, False, False),
         (301, 40, 5, 2, "generic", None, True, True, True, False), (257, 70, 10, 3, "auto", None, False, False, False, False),
         (180, 48, 20, 3, "generic", None, False, True, False, False), (150, 64, 9, 7, "generic", None, True, False, True, False)]


@pytest.mark.parametrize("N,D,q,k,algo,dens,weighted,diag,ard,rows", CASES)
def test_sweeps_match_oracle(eng, N, D, q, k, algo, dens, weighted, diag, ard, rows):
    expect = (algo == "auto" and dens is None and not weighted and q + k in (16, 32, 64)) or None
    run_parity(eng, N, D, q, k, algo, dens, weighted, diag, ard, rows, expect_i8=expect)


def test_unnormalised_covariate(eng):
    """A covariate of scale 1e4 (effects of scale 1e-4): the INT8 path stays 1e-9-accurate per row; guard fall-backs are
    allowed (their count is printed)."""
    e, o = run_parity(eng, 1200, 128, 12, 4, "auto", None, False, False, False, False, sweeps=3, cscale=1e4, expect_i8=True)
    st, us = e.get_state(), o.user_state()
    rel = np.abs(st["Zbar"] - us["Zbar"]).max(1) / np.maximum(np.abs(us["Zbar"]).max(1), 1e-300)
    assert rel.max() < TOL, rel.max()
    print("INT8 guard fall-backs with a 1e4 covariate, per sweep:", e.fall)
    assert 0 in e.fall                                       # at least one sweep's Z step ran on INT8 and was accepted


def _sweep_bytes(e, sweeps):
    el = [e.iterate() for _ in range(sweeps)]
    st = e.get_state()
    return np.array(el).tobytes(), {key: np.asarray(st[key]).tobytes() for key in user_keys(st)}


@pytest.mark.parametrize("algo,dens,rows", [("auto", None, False), ("dmma", None, True), ("auto", 0.3, False),
                                           ("generic", None, False)])
def test_bit_identical_ranges_and_round_trip(eng, algo, dens, rows):
    N, D, q, k = 1500, 128, 13, 3
    A, _, _, _ = case_data(N, D, q, k, dens, False, seed=11)
    C = synth_covariates(N, D, q, k, 0.0, seed=11)[1]
    init = rand_init(N, D, q, k, seed=5, rows=rows)
    wp = "rows" if rows else "columns"
    runs = []
    for _ in range(2):
        e = eng(A, q, algo=algo, ard=True, covariates=C, w_posterior=wp)
        e.set_state(init)
        runs.append(_sweep_bytes(e, 3))
    assert runs[0] == runs[1]
    st = e.get_state()
    e2 = eng(A, q, algo=algo, ard=True, covariates=C, w_posterior=wp)
    e2.set_state(st)
    st2 = e2.get_state()
    for key in user_keys(st):
        assert np.asarray(st[key]).tobytes() == np.asarray(st2[key]).tobytes(), key
    small = e.get_state_small()
    assert small["Wbar"].shape == (D, q) and small["Bbar"].shape == (D, k)
    row = e.get_row(7)
    assert np.array_equal(row["Zbar"], st["Zbar"][7]) and np.array_equal(row["Sig"], st["Sig"][7])
    out = []
    for split in (None, 640):                               # 640: a multiple of the INT8 mask tile (128)
        e = eng(A, q, algo=algo, covariates=C, w_posterior=wp)
        e.set_state(init)
        e.iterate()
        e.update_W()
        if split is None:
            e.update_Z()
        else:
            e.update_Z(0, split)
            e.update_Z(split, N)
        out.append((e.MZ.cpu().numpy().tobytes(), e.Sig.cpu().numpy().tobytes(), e.logdet.cpu().numpy().tobytes()))
    assert out[0] == out[1]


@pytest.mark.parametrize("qt,k", [(8, 1), (16, 4), (32, 5), (64, 4), (64, 33)])
def test_condition_and_finish_write_only_the_tail(eng, qt, k):
    """condition / finish on poisoned rows: every byte outside the last k packed rows and eta' / zbar' stays; the written
    entries are the definition (condition: eta_z - qprec_zc c in order, 0, I, c; finish: c_i c_j, c), bit for bit; a second
    call is bit-identical."""
    from pyvb_b200 import _cabi
    lib = _cabi.lib()
    N = 1000
    pitch = int(lib.pyvb_mz_pitch(qt))
    woff = int(lib.pyvb_gw_woff(qt))
    qf = qt - k
    p0, pt = qf * (qf + 1) // 2, qt * (qt + 1) // 2
    rng = np.random.RandomState(qt + k)
    MZh = rng.randn(N + 2, pitch)
    MZh[:, pt:woff] = np.nan                                 # pad
    MZh[:, woff + qt:] = 1e300                               # pitch tail
    Ch = rng.randn(N, k) * 10.0 ** rng.uniform(-3, 3, size=(N, k))
    dev = torch.device("cuda", torch.cuda.current_device())
    MZ = torch.as_tensor(MZh, device=dev)
    C = torch.as_tensor(Ch, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    _cabi.check(lib.pyvb_zknown_condition_f64(N, qt, k, C.data_ptr(), k, MZ.data_ptr() + pitch * 8, pitch, st), "cond")
    got = MZ.cpu().numpy()
    ref = MZh.copy()
    ii, jj = np.tril_indices(qt)
    for n in range(N):
        r, c = ref[n + 1], Ch[n]
        e = r[woff:woff + qf].copy()
        for j in range(k):
            e = e - r[(qf + j) * (qf + j + 1) // 2 + np.arange(qf)] * c[j]
        r[woff:woff + qf] = e
        r[p0:pt] = (ii[p0:] == jj[p0:]).astype(np.float64)
        r[woff + qf:woff + qt] = c
    # fma chains and the numpy restatement round differently only in eta_z: compare it to 1e-12, everything else exactly
    mask = np.ones(pitch, bool)
    mask[woff:woff + qf] = False
    assert np.array_equal(got[:, mask], ref[:, mask], equal_nan=True)
    assert tensor_rel(got[:, woff:woff + qf], ref[:, woff:woff + qf]) < 1e-12
    MZ2 = torch.as_tensor(MZh, device=dev)
    _cabi.check(lib.pyvb_zknown_condition_f64(N, qt, k, C.data_ptr(), k, MZ2.data_ptr() + pitch * 8, pitch, st), "cond")
    assert MZ2.cpu().numpy().tobytes() == got.tobytes()
    _cabi.check(lib.pyvb_zknown_finish_f64(N, qt, k, C.data_ptr(), k, MZ.data_ptr() + pitch * 8, pitch, st), "finish")
    fin = MZ.cpu().numpy()
    ref2 = got.copy()
    for n in range(N):
        c = Ch[n]
        cc = jj[p0:] >= qf
        ref2[n + 1, p0:pt][cc] = c[ii[p0:][cc] - qf] * c[jj[p0:][cc] - qf]
        ref2[n + 1, woff + qf:woff + qt] = c
    assert np.array_equal(fin, ref2, equal_nan=True)


def test_i8_statistics_match_dmma(eng):
    """With covariates, the INT8 statistics (rebuilt column maxima) agree with the DMMA statistics to 1e-11."""
    N, D, q, k = 3001, 128, 12, 4
    X, _, _, _ = case_data(N, D, q, k, None, False, seed=3)
    C = synth_covariates(N, D, q, k, 0.0, seed=3)[1] * 30.0
    init = rand_init(N, D, q, k, seed=2)
    P0 = 2.0 * np.eye(q)                                     # (a finite bound term for the all-missing row 3)
    a, b = eng(X, q, covariates=C, P0=P0), eng(X, q, algo="dmma", covariates=C, P0=P0)
    assert a.use_i8 and a.use_i8_stats and not b.use_i8
    for e in (a, b):
        e.set_state(init)
        e.iterate()
        e.update_W()
        e.update_Z()
    b.MZ.copy_(a.MZ)
    b.logdet.copy_(a.logdet)
    for e in (a, b):
        e._stats_fresh = False
        e._ensure_stats()
    sa, sb = a.stats.cpu().numpy(), b.stats.cpu().numpy()
    assert tensor_rel(sa, sb) < 1e-11, tensor_rel(sa, sb)
    assert a.i8_fallbacks()[1] == 0


_FORCED = r"""
import sys, numpy as np, torch
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
from pyvb_b200 import PlateEngine
from test_gpu_covariates import case_data, rand_init
from oracle.covariates_oracle import synth_covariates
N, D, q, k = 900, 128, 12, 4
X = case_data(N, D, q, k, None, False, seed=8)[0]
C = synth_covariates(N, D, q, k, 0.0, seed=8)[1]
ei, ed = PlateEngine(X, q, algo="i8", covariates=C), PlateEngine(X, q, algo="dmma", covariates=C)
st = rand_init(N, D, q, k, seed=3)
for s in range(3):
    for e in (ei, ed):
        e.set_state(st)
        e.update_Z()
    assert torch.equal(ei.MZ, ed.MZ) and torch.equal(ei.logdet, ed.logdet) and torch.equal(ei.Sig, ed.Sig), s
    ed.iterate()
    st = ed.get_state()
assert ei.i8_fallbacks()[0] == 3, ei.i8_fallbacks()
print("forced ok")
"""


def test_forced_guard_reproduces_dmma(tmp_path):
    """PYVB_I8_GUARD=force (read once per process, hence the subprocess): every INT8 Z step falls back to K1-DMMA ->
    condition -> K2 and leaves the DMMA path's rows bit for bit."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "forced.py"
    script.write_text(_FORCED)
    env = dict(os.environ, PYVB_I8_GUARD="force")
    r = subprocess.run([sys.executable, str(script), root], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "forced ok" in r.stdout, r.stdout + r.stderr


def test_errors(eng):
    N, D, q = 64, 64, 12
    X, C, _, _, _ = synth_covariates(N, D, q, 4, 0.2, seed=1)
    with pytest.raises(ValueError, match="mode='B'"):
        eng(X, q, mode="A", covariates=C)
    with pytest.raises(ValueError, match="precision='f64'"):
        eng(X, q, precision="f32", covariates=C)
    with pytest.raises(ValueError, match="<= 64"):
        eng(X, 62, covariates=C)
    with pytest.raises(ValueError, match="shape"):
        eng(X, q, covariates=C[:, 0])
    with pytest.raises(ValueError, match="one row per row"):
        eng(X, q, covariates=C[:10])
    bad = C.copy()
    bad[5, 1] = np.nan
    with pytest.raises(ValueError, match="finite"):
        eng(X, q, covariates=bad)
    for e in (eng(X, 3, covariates=C), eng(X[:, :40], q, covariates=C), eng(X, q, algo="generic", covariates=C)):
        # q' = 7, D % 16 != 0, explicit: the generic path
        assert not e.use_i8 and (e.algo == 1 or not e.lib.pyvb_algo_supported(2, e.D, e.q))
    with pytest.raises(ValueError, match="q in"):
        eng(to_sparse(X), 3, covariates=C)                   # sparse at q' = 7
    e = eng(X, q, covariates=C)
    with pytest.raises(NotImplementedError):
        e.set_X(torch.as_tensor(X, device=e.device))
    with pytest.raises(NotImplementedError):
        e.iterate_from_host(torch.as_tensor(X))
    with pytest.raises(ValueError, match="Bbar"):
        eng(X, 16).set_state({"Bbar": np.zeros((D, 4))})


def test_full_size_fit(eng):
    """C2 shape (1M x 256, 20 % missing, q = 12, k = 4: q' = 16 on INT8), 50 sweeps from init_random: B, tau and the W
    subspace recovered within the oracle-derived tolerances, a finite bound non-decreasing over sweeps 10-50, no guard
    fall-back."""
    N, D, q, k, tau = 1_000_000, 256, 12, 4, 4.0
    dev = torch.device("cuda", torch.cuda.current_device())
    g = torch.Generator(device=dev)
    g.manual_seed(31)
    f64 = torch.float64
    W = torch.randn(D, q, generator=g, device=dev, dtype=f64)
    B = torch.randn(D, k, generator=g, device=dev, dtype=f64)
    mu = torch.randn(D, generator=g, device=dev, dtype=f64)
    C = torch.randn(N, k, generator=g, device=dev, dtype=f64)
    X = torch.empty(N, D, dtype=f64, device=dev)
    for lo in range(0, N, 1 << 17):
        n = min(1 << 17, N - lo)
        Z = torch.randn(n, q, generator=g, device=dev, dtype=f64)
        x = Z @ W.T + C[lo:lo + n] @ B.T + mu + torch.randn(n, D, generator=g, device=dev, dtype=f64) / tau ** 0.5
        x[torch.rand(n, D, generator=g, device=dev) < 0.2] = float("nan")
        X[lo:lo + n] = x
    e = eng(X, q, covariates=C)
    assert e.use_i8
    e.init_random(seed=3)
    b = e.run(50).cpu().numpy()
    e.check()
    assert np.all(np.isfinite(b))
    assert np.all(np.diff(b[9:]) >= -1e-9 * np.abs(b[10:])), np.diff(b[9:]).min()
    assert e.i8_fallbacks() == (0, 0)
    st = e.get_state_small()
    Bt, Wt = B.cpu().numpy(), W.cpu().numpy()
    eb = float(np.linalg.norm(st["Bbar"] - Bt) / np.linalg.norm(Bt))
    et = abs(float(st["tau"]) / tau - 1.0)
    ea = principal_angle_deg(st["Wbar"], Wt)
    print("full-size recovery: B %.3g, tau %.3g, W angle %.3g deg" % (eb, et, ea))
    assert eb < REC_B and et < REC_TAU and ea < REC_ANGLE, (eb, et, ea)


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist
    from pyvb_b200 import PlateEngine
    from pyvb_b200.dist import shard_rows
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    N, D, q, k = 3001, 128, 12, 4
    X, C, _, _, _ = synth_covariates(N, D, q, k, 0.2, seed=3)
    init = rand_init(N, D, q, k, seed=1)
    lo, hi = shard_rows(N, world, rank)
    e = PlateEngine(X[lo:hi], q, device=dev, distributed=True, row_offset=lo, covariates=C[lo:hi])
    loc = dict(init)
    for key in ("Zbar", "Sig"):
        loc[key] = loc[key][lo:hi]
    e.set_state(loc)
    elbo = [e.iterate() for _ in range(4)]
    st = e.get_state_small()
    e.check()
    np.savez(os.path.join(out_dir, "r%d.npz" % rank), elbo=np.array(elbo), Wbar=st["Wbar"], Bbar=st["Bbar"], qb=st["qb"])
    e.close()
    dist.destroy_process_group()


def test_two_gpu_sharded(tmp_path):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    N, D, q, k = 3001, 128, 12, 4
    X, C, _, _, _ = synth_covariates(N, D, q, k, 0.2, seed=3)
    o = cov_oracle_class()(X, q, C)
    o.load_user_state(rand_init(N, D, q, k, seed=1))
    ref = np.array([o.iterate() for _ in range(4)])
    a, b = (np.load(os.path.join(str(tmp_path), "r%d.npz" % r)) for r in range(2))
    for key in ("elbo", "Wbar", "Bbar", "qb"):
        assert np.asarray(a[key]).tobytes() == np.asarray(b[key]).tobytes(), key
    assert np.max(np.abs(a["elbo"] - ref) / np.abs(ref)) < TOL
    assert tensor_rel(a["Bbar"], o.user_state()["Bbar"]) < TOL
