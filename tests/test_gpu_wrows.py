"""GPU tests of the row-wise W posterior (PlateEngine(..., w_posterior="rows")): sweep-by-sweep parity with the rows oracle on the
INT8, DMMA, generic and sparse paths, the Gauss-Seidel fixed point of the column update on the device, the default path
unchanged, determinism, row ranges and the state round trip, the error contract, a row-sharded run on two GPUs and a full-size
run."""
import os

import numpy as np
import pytest
import torch

from helpers import tensor_rel
from oracle.wrows_oracle import (WRowsDiagNoiseOracle, WRowsPlateOracle, WRowsWeightedDiagNoiseOracle,
                                 WRowsWeightedPlateOracle)
from oracle.weights_oracle import synth_weighted
from test_gpu_sparse import _free_port, densify, sparse_pca
from test_gpu_weights import sparse_weights, weights_like

pytestmark = pytest.mark.gpu
TOL = 1e-9


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pyvb_b200 import PlateEngine
    return PlateEngine


def rand_init(N, D, q, seed=0, diag=False, S=None):
    """A random state with a full SPD Wcov per row; qb puts tau near the data's (as test_gpu_weights.rand_init)."""
    rng = np.random.RandomState(seed)
    qb = (rng.rand(D) + 0.3) if diag else 0.7
    if S is not None:
        qb = 0.1 * (1.0 + 0.5 * (np.asarray(S) > 0).sum(0 if diag else None))
    B = rng.randn(D, q, q) * (0.3 / np.sqrt(q))
    Wcov = B @ np.transpose(B, (0, 2, 1)) + np.einsum("di,ij->dij", rng.rand(D, q) + 0.5, np.eye(q))
    return {"Wbar": rng.randn(D, q), "Wcov": Wcov, "mu": rng.randn(D) * 0.1, "muvar": np.ones(D),
            "Zbar": rng.randn(N, q), "Sig": np.tile(np.eye(q), (N, 1, 1)) * (rng.rand(N, 1, 1) + 0.5),
            "qb": qb, "al_qb": rng.rand(q) + 0.5}


def same_bound(got, ref):
    return (not np.isfinite(got)) if not np.isfinite(ref) else abs(got - ref) <= TOL * abs(ref)


def data(N, D, q, dens, weighted, seed):
    """(input for the engine, dense X with NaN, weights for the engine or None, dense weights or None)."""
    if dens is None:
        X, _, _ = synth_weighted(N, D, q, 0.2, tau=10.0, seed=seed)
        S = weights_like(N, D, seed + 1) if weighted else None
        return X, X, S, S
    A = sparse_pca(N, D, q, dens, seed=seed)
    X = densify(A)
    if not weighted:
        return A, X, None, None
    Wd = np.where(np.isnan(X), 0.0, weights_like(N, D, seed + 1))
    return A, X, sparse_weights(A, Wd), Wd


def oracle(X, q, Wd, diag, ard, kw):
    if Wd is None:
        return (WRowsDiagNoiseOracle if diag else WRowsPlateOracle)(X, q, ard=ard, **kw)
    return (WRowsWeightedDiagNoiseOracle if diag else WRowsWeightedPlateOracle)(X, q, Wd, ard=ard, **kw)


# (N, D, q, algo, sparse density or None, weighted, per-dimension noise, ARD): at every q each path (INT8 from q = 16 on,
# DMMA, generic, CSR), each noise model, ARD on and off and weights on and off appear at least once
CASES = [(700, 64, 8, "auto", None, False, False, False), (500, 64, 8, "dmma", None, True, True, True),
         (300, 40, 8, "generic", None, True, False, True), (400, 45, 8, "auto", 0.6, False, True, False),
         (700, 128, 16, "auto", None, False, False, True), (600, 128, 16, "dmma", None, True, True, False),
         (200, 48, 16, "generic", None, False, True, True), (600, 300, 16, "auto", 0.1, True, False, False),
         (600, 128, 32, "auto", None, False, True, True), (600, 128, 32, "dmma", None, True, False, False),
         (150, 40, 32, "generic", None, True, True, False), (500, 200, 32, "auto", 0.2, False, False, True),
         (500, 128, 64, "auto", None, False, True, False), (500, 64, 64, "dmma", None, False, False, True),
         (200, 70, 64, "generic", None, True, False, True), (300, 150, 64, "auto", 0.5, True, True, False)]


@pytest.mark.parametrize("N,D,q,algo,dens,weighted,diag,ard", CASES)
def test_sweeps_match_oracle(eng, N, D, q, algo, dens, weighted, diag, ard):
    from pyvb_b200._layout import GL_ELBO_W
    A, X, Wt, Wd = data(N, D, q, dens, weighted, seed=N + D + q)
    init = rand_init(N, D, q, seed=1, diag=diag, S=Wd)
    kw = {"a0": np.random.RandomState(D).rand(D) + 0.01} if diag else {}
    o = oracle(X, q, Wd, diag, ard, kw)
    o.load_state(init)
    if ard:
        o.al_qb = init["al_qb"].copy()
    e = eng(A, q, algo=algo, ard=ard, weights=Wt, noise="diagonal" if diag else "scalar", w_posterior="rows", **kw)
    if algo == "auto" and dens is None and not weighted and q >= 16:
        assert e.use_i8
    e.set_state(init)
    for it in range(3):
        ref, got = o.iterate(), e.iterate()
        assert same_bound(got, ref), (it, got, ref)
        ew, ow = float(e.gl[GL_ELBO_W].item()), o.elbo_terms()["W"]
        assert abs(ew - ow) <= TOL * abs(ow), (it, ew, ow)
    e.check()
    st = e.get_state()
    for k in ("Wbar", "Wvar", "Wcov", "mu", "muvar", "Zbar", "Sig", "qb", "tau"):
        assert tensor_rel(st[k], getattr(o, k)) < TOL, (k, tensor_rel(st[k], getattr(o, k)))
    if ard:
        assert tensor_rel(st["al_qb"], o.al_qb) < TOL


@pytest.mark.parametrize("N,D,q,algo", [(800, 128, 16, "auto"), (600, 64, 32, "generic"), (400, 64, 64, "dmma")])
def test_column_passes_converge_to_the_row_solve(eng, N, D, q, algo):
    """On frozen statistics, repeated Gauss-Seidel column updates (wupdate_kernel) reach the row solve's wbar (K2)."""
    X = synth_weighted(N, D, q, 0.2, tau=10.0, seed=q)[0]
    init = rand_init(N, D, q, seed=2)
    del init["Wcov"]
    init["Wvar"] = np.random.RandomState(3).rand(D, q) + 0.5
    c, r = eng(X, q, algo=algo, ard=True), eng(X, q, algo=algo, ard=True, w_posterior="rows")
    c.set_state(init)
    r.set_state(init)
    r.update_W()
    wr = r.Wbar.cpu().numpy()
    for it in range(20000):
        old = c.Wbar.clone()
        c.update_W()
        if float((c.Wbar - old).abs().max()) <= 1e-14 * float(c.Wbar.abs().max()):
            break
    assert it < 19999
    assert tensor_rel(c.Wbar.cpu().numpy(), wr) < 1e-10, tensor_rel(c.Wbar.cpu().numpy(), wr)


def _bytes(e, sweeps):
    el = [e.iterate() for _ in range(sweeps)]
    st = e.get_state()
    keys = [k for k in ("Wbar", "Wvar", "Wcov", "mu", "muvar", "Zbar", "Sig", "qb", "al_qb") if k in st]
    return np.array(el).tobytes(), {k: np.asarray(st[k]).tobytes() for k in keys}


@pytest.mark.parametrize("algo,dens", [("auto", None), ("generic", None), ("auto", 0.2)])
def test_default_is_columns(eng, algo, dens):
    N, D, q = 900, 128, 16
    A = data(N, D, q, dens, False, seed=3)[0]
    init = rand_init(N, D, q, seed=2)
    del init["Wcov"]
    init["Wvar"] = np.random.RandomState(4).rand(D, q) + 0.5
    out = []
    for kw in ({}, {"w_posterior": "columns"}):
        e = eng(A, q, algo=algo, ard=True, **kw)
        e.set_state(init)
        out.append(_bytes(e, 3))
    assert out[0] == out[1]


@pytest.mark.parametrize("algo,dens,weighted", [("auto", None, False), ("dmma", None, True), ("generic", None, False),
                                                ("auto", 0.05, True)])
def test_runs_are_bit_identical_ranges_compose_and_state_round_trips(eng, algo, dens, weighted):
    N, D, q = 1500, 128, 16
    A, _, Wt, Wd = data(N, D, q, dens, weighted, seed=11)
    init = rand_init(N, D, q, seed=5, S=Wd)
    runs = []
    for _ in range(2):
        e = eng(A, q, algo=algo, ard=True, weights=Wt, w_posterior="rows")
        e.set_state(init)
        runs.append(_bytes(e, 3))
    assert runs[0] == runs[1]
    st = e.get_state()
    e2 = eng(A, q, algo=algo, ard=True, weights=Wt, w_posterior="rows")
    e2.set_state(st)
    st2 = e2.get_state()
    for k in ("Wbar", "Wvar", "Wcov", "mu", "muvar", "Zbar", "Sig", "qb", "al_qb"):
        assert np.asarray(st[k]).tobytes() == np.asarray(st2[k]).tobytes(), k
    out = []
    for split in (None, 640):
        e = eng(A, q, algo=algo, weights=Wt, w_posterior="rows")
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


def test_iterate_from_host(eng):
    """The streamed sweep (dense, scalar noise, unweighted; the data uploaded in chunks) gives the resident sweep's result."""
    N, D, q = 5003, 128, 32
    X = synth_weighted(N, D, q, 0.25, tau=10.0, seed=12)[0]
    init = rand_init(N, D, q, seed=6)
    a, b = eng(X, q, w_posterior="rows"), eng(X, q, w_posterior="rows")
    Xh = torch.as_tensor(X).pin_memory()
    for e in (a, b):
        e.set_state(init)
    b._ensure_stats()
    b.X.fill_(0.0)
    for it in range(3):
        ra = a.iterate()
        rb = float(b.trace[b.iterate_from_host(Xh, nchunks=5)].item())
        assert abs(ra - rb) <= 1e-12 * abs(ra), (it, ra, rb)
    sa, sb = a.get_state(), b.get_state()
    for k in ("Wbar", "Wcov", "mu", "Zbar", "Sig"):
        assert tensor_rel(sb[k], sa[k]) < 1e-12, k


def test_errors(eng):
    N, D = 64, 64
    X = synth_weighted(N, D, 16, 0.2, tau=10.0, seed=1)[0]
    with pytest.raises(ValueError, match="mode='B'"):
        eng(X, 16, mode="A", w_posterior="rows")
    with pytest.raises(ValueError, match="precision='f64'"):
        eng(X, 16, precision="f32", w_posterior="rows")
    for q in (4, 12, 48):
        with pytest.raises(ValueError, match="q in"):
            eng(X, q, w_posterior="rows")
    with pytest.raises(ValueError, match="w_posterior"):
        eng(X, 16, w_posterior="full")
    e = eng(X, 16, w_posterior="rows")
    for lo, hi in ((0, 8), (4, 16), (3, 3)):
        with pytest.raises(ValueError, match="column range"):
            e.update_W(lo, hi)
    e.update_W(0, 16)
    e.update_Alpha(0, 8)
    c = eng(X, 16)
    with pytest.raises(ValueError, match="Wcov"):
        c.set_state({"Wcov": np.tile(np.eye(16), (D, 1, 1))})
    bad = np.tile(np.eye(16), (D, 1, 1))
    bad[3, 0, 0] = -1.0
    with pytest.raises(ValueError, match="positive definite"):
        e.set_state({"Wcov": bad})


def test_nonpd_row_is_reported(eng):
    """A W row whose precision is not positive definite is counted and raised by check(), naming Z or W."""
    N, D, q = 256, 64, 16
    X = synth_weighted(N, D, q, 0.2, tau=10.0, seed=2)[0]
    e = eng(X, q, w_posterior="rows")
    e.set_state(rand_init(N, D, q, seed=3))
    e.gl[16:16 + q] = -1e12                                 # <alpha> < 0: Lambda_d = diag(alpha) + tau T1_d is indefinite
    e.update_W()
    with pytest.raises(np.linalg.LinAlgError, match="Z or W"):
        e.check()


def test_full_size_fit(eng):
    """Config-2 shape (1M x 256, q = 16, 20 % missing, default INT8 path), 30 sweeps from init_random."""
    N, D, q = 1_000_000, 256, 16
    dev = torch.device("cuda", torch.cuda.current_device())
    g = torch.Generator(device=dev)
    g.manual_seed(29)
    W = torch.randn(D, q, generator=g, device=dev, dtype=torch.float64)
    mu = torch.randn(D, generator=g, device=dev, dtype=torch.float64)
    X = torch.empty(N, D, dtype=torch.float64, device=dev)
    for lo in range(0, N, 1 << 17):
        n = min(1 << 17, N - lo)
        Z = torch.randn(n, q, generator=g, device=dev, dtype=torch.float64)
        x = Z @ W.T + mu + 0.5 * torch.randn(n, D, generator=g, device=dev, dtype=torch.float64)
        x[torch.rand(n, D, generator=g, device=dev) < 0.2] = float("nan")
        X[lo:lo + n] = x
    e = eng(X, q, w_posterior="rows")
    assert e.use_i8
    e.init_random(seed=3)
    b = e.run(30).cpu().numpy()
    from pyvb_b200._layout import GL_NONPD
    assert float(e.gl[GL_NONPD].item()) == 0.0
    e.check()
    assert np.all(np.isfinite(b))
    assert np.all(np.diff(b[5:]) >= -1e-9 * np.abs(b[6:]))
    assert np.all(np.isfinite(e.Wcov.cpu().numpy()))


def _worker(rank, world, port, shape, out_dir):
    import torch.distributed as dist
    from pyvb_b200 import PlateEngine
    from pyvb_b200.dist import shard_rows
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    N, D, q, diag = shape
    X = synth_weighted(N, D, q, 0.2, tau=10.0, seed=3)[0]
    init = rand_init(N, D, q, seed=1, diag=diag)
    lo, hi = shard_rows(N, world, rank)
    e = PlateEngine(X[lo:hi], q, device=dev, distributed=True, row_offset=lo, noise="diagonal" if diag else "scalar",
                    w_posterior="rows")
    loc = dict(init)
    for k in ("Zbar", "Sig"):
        loc[k] = loc[k][lo:hi]
    e.set_state(loc)
    elbo = [e.iterate() for _ in range(4)]
    st = e.get_state_small()
    e.check()
    np.savez(os.path.join(out_dir, "r%d.npz" % rank), elbo=np.array(elbo), Wbar=st["Wbar"], Wcov=st["Wcov"],
             qb=st["qb"])
    e.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("shape", [(3001, 128, 16, False), (1200, 192, 32, True)])
def test_two_gpu_sharded(tmp_path, shape):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world = 2
    N, D, q, diag = shape
    mp.spawn(_worker, args=(world, _free_port(), shape, str(tmp_path)), nprocs=world, join=True)
    X = synth_weighted(N, D, q, 0.2, tau=10.0, seed=3)[0]
    o = (WRowsDiagNoiseOracle if diag else WRowsPlateOracle)(X, q)
    o.load_state(rand_init(N, D, q, seed=1, diag=diag))
    ref = np.array([o.iterate() for _ in range(4)])
    a, b = (np.load(os.path.join(str(tmp_path), "r%d.npz" % r)) for r in range(world))
    assert np.asarray(a["qb"]).tobytes() == np.asarray(b["qb"]).tobytes() and np.array_equal(a["elbo"], b["elbo"])
    assert a["Wbar"].tobytes() == b["Wbar"].tobytes() and a["Wcov"].tobytes() == b["Wcov"].tobytes()
    assert np.max(np.abs(a["elbo"] - ref) / np.abs(ref)) < TOL
    assert tensor_rel(a["qb"], o.qb) < TOL and tensor_rel(a["Wbar"], o.Wbar) < TOL
