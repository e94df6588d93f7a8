"""GPU tests of per-dimension noise precisions (PlateEngine(..., noise="diagonal")): sweep-by-sweep parity with the oracle
on every Z-step path, the reduction to the scalar engine, INT8 against DMMA on badly scaled columns, determinism, the
error contract, a full-size run and a row-sharded run on two GPUs."""
import os

import numpy as np
import pytest
import torch

from helpers import tensor_rel
from oracle.noise_oracle import DiagNoiseOracle, synth_fa
from oracle.plate_oracle import synth_pca
from test_gpu_sparse import _free_port, densify, sparse_pca

pytestmark = pytest.mark.gpu
TOL = 1e-9


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pyvb_b200 import PlateEngine
    return PlateEngine


def rand_init(N, D, q, seed=0):
    rng = np.random.RandomState(seed)
    return {"Wbar": rng.randn(D, q), "Wvar": rng.rand(D, q) + 0.5, "mu": rng.randn(D) * 0.1, "muvar": np.ones(D),
            "Zbar": rng.randn(N, q), "Sig": np.tile(np.eye(q), (N, 1, 1)) * (rng.rand(N, 1, 1) + 0.5),
            "qb": rng.rand(D) + 0.3, "al_qb": rng.rand(q) + 0.5}


def hetero(N, D, q, missing, seed):
    rng = np.random.RandomState(seed)
    return synth_fa(N, D, q, missing, np.exp(rng.uniform(0, np.log(1e3), D)), seed=seed + 1)


def same_bound(got, ref):
    return (not np.isfinite(got)) if not np.isfinite(ref) else abs(got - ref) <= TOL * abs(ref)


# (N, D, q, algo, sparse density or None, ard): INT8 at q = 16 / 32 / 64, DMMA, generic, CSR at q = 8 / 16 / 32 / 64, N = 1
SHAPES = [(700, 128, 16, "auto", None, False), (600, 128, 32, "auto", None, True), (500, 64, 64, "auto", None, False),
          (700, 64, 16, "dmma", None, True), (300, 37, 3, "auto", None, False), (200, 37, 3, "generic", None, True),
          (1, 37, 3, "auto", None, False), (400, 45, 8, "auto", 0.6, True), (600, 300, 16, "auto", 0.1, False),
          (500, 200, 32, "auto", 0.2, False), (300, 150, 64, "auto", 0.5, True)]


@pytest.mark.parametrize("N,D,q,algo,dens,ard", SHAPES)
def test_sweeps_match_oracle(eng, N, D, q, algo, dens, ard):
    rng = np.random.RandomState(N + D)
    a0, b0 = rng.rand(D) + 0.01, 1e-3
    if dens is None:
        X = hetero(N, D, q, 0.2, seed=N + q)
        if N > 1 and ard:
            X[N // 2] = np.nan                                # an all-missing row: the bound is infinite on both sides
        A = X
    else:
        A = sparse_pca(N, D, q, dens, seed=N + D)
        X = densify(A)
    init = rand_init(N, D, q, seed=1)
    o = DiagNoiseOracle(X, q, a0=a0, b0=b0, ard=ard)
    o.load_state(init)
    if ard:
        o.al_qb = init["al_qb"].copy()
    e = eng(A, q, mode="B", algo=algo, ard=ard, a0=a0, b0=b0, noise="diagonal")
    if algo == "auto" and dens is None and D % 64 == 0:
        assert e.use_i8
    e.set_state(init)
    np.testing.assert_allclose(e.get_state_small()["qa"], o.qa, rtol=1e-15)
    for it in range(3):
        ref, got = o.iterate(), e.iterate()
        assert same_bound(got, ref), (it, got, ref)
    st = e.get_state()
    for k in ("Wbar", "Wvar", "mu", "muvar", "Zbar", "Sig", "qb", "tau"):
        assert tensor_rel(st[k], getattr(o, k)) < TOL, (k, tensor_rel(st[k], getattr(o, k)))
    if N > 1:
        np.testing.assert_allclose(st["qb"], o.qb, rtol=TOL)


@pytest.mark.parametrize("algo,dens", [("auto", None), ("dmma", None), ("generic", None), ("auto", 0.3)])
def test_equal_precisions_match_the_scalar_engine(eng, algo, dens):
    N, D, q = 900, 128, 16
    A = synth_pca(N, D, q, 0.2, seed=3) if dens is None else sparse_pca(N, D, q, dens, seed=3)
    init = rand_init(N, D, q, seed=2)
    es = eng(A, q, algo=algo)
    ed = eng(A, q, algo=algo, noise="diagonal")
    es.set_state(dict(init, qb=0.8))
    tau = es.get_state_small()["tau"]
    ed.set_state(dict(init, qb=ed.get_state_small()["qa"] / tau))
    np.testing.assert_allclose(ed.get_state_small()["tau"], tau, rtol=1e-15)
    for step in ("update_W", "update_Z", "update_Mu"):
        getattr(es, step)()
        getattr(ed, step)()
    a, b = es.get_state(), ed.get_state()
    for k in ("Wbar", "Wvar", "mu", "muvar", "Zbar", "Sig"):
        assert tensor_rel(b[k], a[k]) < 1e-12, (k, tensor_rel(b[k], a[k]))


def test_int8_matches_dmma_on_badly_scaled_columns(eng):
    """Column scales from 1e-2 to 1e3: the Z step contracts tau_d G_d, whose columns come back to one scale."""
    N, D, q = 2000, 128, 16
    X = synth_pca(N, D, q, 0.3, seed=9)
    s = np.exp(np.linspace(np.log(1e-2), np.log(1e3), D))
    X *= s[None, :]
    init = rand_init(N, D, q, seed=3)
    init["Wbar"] *= s[:, None]
    init["mu"] *= s
    init["qb"] = 1e-3 * N * s ** 2
    ei, ed = eng(X, q, noise="diagonal"), eng(X, q, algo="dmma", noise="diagonal")
    assert ei.use_i8 and not ed.use_i8
    for g in (ei, ed):
        g.set_state(init)
    for it in range(5):
        a, b = ei.iterate(), ed.iterate()
        assert abs(a - b) <= 1e-11 * abs(b), (it, a, b)
    sa, sb = ei.get_state(), ed.get_state()
    for k in ("Wbar", "mu", "Zbar", "Sig", "qb"):
        assert tensor_rel(sa[k], sb[k]) < 1e-11, (k, tensor_rel(sa[k], sb[k]))
    print("int8 guard fall-backs, column scales 1e-2..1e3:", ei.i8_fallbacks())


def test_unnormalised_feature_under_diagonal_noise(eng):
    """The data of test_gpu_i8's unnormalised-feature test at s = 1e4 (shared tau: the guard sends those Z steps to DMMA).
    With per-dimension precisions the contracted operand is tau_d G_d; the count is reported, and the result must stay on
    the all-DMMA engine."""
    N, D, q, s = 3000, 128, 16, 1e4
    X = synth_pca(N, D, q, 0.3, seed=21)
    X[:, 9] *= s
    init = rand_init(N, D, q, seed=4)
    init["Wbar"][9] *= s
    e, ed = eng(X, q, noise="diagonal"), eng(X, q, algo="dmma", noise="diagonal")
    for g in (e, ed):
        g.set_state(init)
    first = []
    for it in range(10):
        a, b = e.iterate(), ed.iterate()
        assert abs(a - b) <= 1e-9 * abs(b), (it, a, b)
        if it == 4:
            first = e.i8_fallbacks()
    last = e.i8_fallbacks()
    print("int8 guard fall-backs (Z steps, statistics) after 5 sweeps:", first, "after 10:", last,
          "-> over the last 5 sweeps:", (last[0] - first[0], last[1] - first[1]))
    e.check()


def test_runs_are_bit_identical_and_row_ranges_compose(eng):
    N, D, q = 1500, 128, 16
    X = hetero(N, D, q, 0.2, seed=5)
    init = rand_init(N, D, q, seed=5)
    res = []
    for _ in range(2):
        e = eng(X, q, ard=True, noise="diagonal")
        e.set_state(init)
        el = [e.iterate() for _ in range(3)]
        res.append((el, e.get_state()))
    assert res[0][0] == res[1][0]
    for k in ("Wbar", "Wvar", "mu", "muvar", "Zbar", "Sig", "qb", "al_qb"):
        assert np.asarray(res[0][1][k]).tobytes() == np.asarray(res[1][1][k]).tobytes(), k
    A = sparse_pca(N, 300, q, 0.05, seed=6)
    init = rand_init(N, 300, q, seed=6)
    out = []
    for split in (None, 613):
        e = eng(A, q, noise="diagonal")
        e.set_state(init)
        e.iterate()
        if split is None:
            e.update_Z()
        else:
            e.update_Z(0, split)
            e.update_Z(split, N)
        out.append((e.MZ.cpu().numpy().tobytes(), e.Sig.cpu().numpy().tobytes(), e.logdet.cpu().numpy().tobytes()))
    assert out[0] == out[1]


def test_errors(eng):
    X = synth_pca(50, 20, 4, 0.2, seed=1)
    with pytest.raises(ValueError, match="mode"):
        eng(X, 4, mode="A", noise="diagonal")
    with pytest.raises(ValueError, match="f64"):
        eng(synth_pca(64, 64, 16, 0.2, seed=1), 16, precision="f32", noise="diagonal")
    with pytest.raises(ValueError, match="a0"):
        eng(X, 4, noise="diagonal", a0=np.ones(19))
    with pytest.raises(ValueError, match="b0"):
        eng(X, 4, noise="diagonal", b0=np.ones((20, 1)))
    with pytest.raises(ValueError, match="noise"):
        eng(X, 4, noise="full")
    e = eng(X, 4, noise="diagonal")
    with pytest.raises(NotImplementedError):
        e.set_X(torch.zeros(50, 20, dtype=torch.float64, device=e.device))
    with pytest.raises(NotImplementedError):
        e.iterate_from_host(torch.zeros(50, 20, dtype=torch.float64).pin_memory())


def test_full_size_heteroscedastic(eng):
    """Config-2 shape (1M x 256, q = 16, 20 % missing), tau_d log-uniform in [1, 1e3], 50 sweeps from init_random.  Measured
    on one B200: median error 0.11 %, largest 0.51 %."""
    N, D, q = 1_000_000, 256, 16
    dev = torch.device("cuda", torch.cuda.current_device())
    g = torch.Generator(device=dev)
    g.manual_seed(17)
    tau = torch.exp(torch.rand(D, generator=g, device=dev, dtype=torch.float64) * np.log(1e3))
    W = torch.randn(D, q, generator=g, device=dev, dtype=torch.float64)
    mu = torch.randn(D, generator=g, device=dev, dtype=torch.float64)
    X = torch.empty(N, D, dtype=torch.float64, device=dev)
    for lo in range(0, N, 1 << 17):
        n = min(1 << 17, N - lo)
        Z = torch.randn(n, q, generator=g, device=dev, dtype=torch.float64)
        x = Z @ W.T + mu + torch.randn(n, D, generator=g, device=dev, dtype=torch.float64) / tau.sqrt()
        x[torch.rand(n, D, generator=g, device=dev) < 0.2] = float("nan")
        X[lo:lo + n] = x
    e = eng(X, q, noise="diagonal")
    del X
    assert e.use_i8
    e.init_random(seed=3)
    bounds = e.run(50).cpu().numpy()
    e.check()
    assert np.all(np.isfinite(bounds))
    err = np.abs(e.get_state_small()["tau"] / tau.cpu().numpy() - 1.0)
    print("tau_d relative error after 50 sweeps: median %.4f, 90%% %.4f, max %.4f; int8 fall-backs %s"
          % (np.median(err), np.quantile(err, 0.9), err.max(), e.i8_fallbacks()))
    assert np.max(err) < 0.05


def _worker(rank, world, port, shape, out_dir):
    import torch.distributed as dist
    from pyvb_b200 import PlateEngine
    from pyvb_b200.dist import shard_rows
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    N, D, q, dens = shape
    A = hetero(N, D, q, 0.2, seed=3) if dens is None else sparse_pca(N, D, q, dens, seed=3)
    init = rand_init(N, D, q, seed=1)
    lo, hi = shard_rows(N, world, rank)
    e = PlateEngine(A[lo:hi], q, device=dev, distributed=True, row_offset=lo, noise="diagonal")
    loc = dict(init)
    for k in ("Zbar", "Sig"):
        loc[k] = loc[k][lo:hi]
    e.set_state(loc)
    elbo = [e.iterate() for _ in range(4)]
    st = e.get_state_small()
    e.check()
    np.savez(os.path.join(out_dir, "r%d.npz" % rank), elbo=np.array(elbo), Wbar=st["Wbar"], qb=st["qb"])
    e.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("shape", [(3001, 128, 16, None), (1200, 200, 8, 0.05)])
def test_two_gpu_sharded(tmp_path, shape):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world = 2
    N, D, q, dens = shape
    mp.spawn(_worker, args=(world, _free_port(), shape, str(tmp_path)), nprocs=world, join=True)
    X = hetero(N, D, q, 0.2, seed=3) if dens is None else densify(sparse_pca(N, D, q, dens, seed=3))
    o = DiagNoiseOracle(X, q)
    o.load_state(rand_init(N, D, q, seed=1))
    ref = np.array([o.iterate() for _ in range(4)])
    a, b = (np.load(os.path.join(str(tmp_path), "r%d.npz" % r)) for r in range(world))
    assert a["qb"].tobytes() == b["qb"].tobytes() and np.array_equal(a["elbo"], b["elbo"])
    assert np.max(np.abs(a["elbo"] - ref) / np.abs(ref)) < TOL
    assert tensor_rel(a["qb"], o.qb) < TOL and tensor_rel(a["Wbar"], o.Wbar) < TOL
