"""GPU tests of per-entry observation weights (PlateEngine(..., weights=S)): sweep-by-sweep parity with the weighted oracle on
the DMMA, generic and sparse paths, bit identity with the unweighted engine (weights = 1, zero weights = NaN), determinism and
row ranges, the error contract, a row-sharded run on two GPUs and a full-size run."""
import os

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from helpers import tensor_rel
from oracle.weights_oracle import WeightedDiagNoiseOracle, WeightedPlateOracle, synth_weighted
from test_gpu_sparse import _free_port, densify, sparse_pca

pytestmark = pytest.mark.gpu
TOL = 1e-9


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pyvb_b200 import PlateEngine
    return PlateEngine


def rand_init(N, D, q, seed=0, diag=False, S=None):
    """A random state; with the weights S, qb puts the noise precision near the data's (tau about 10) -- a shared qb of order
    one would start tau at half the number of observations, where the q x q systems of the Z step are needlessly
    ill-conditioned."""
    rng = np.random.RandomState(seed)
    qb = (rng.rand(D) + 0.3) if diag else 0.7
    if S is not None:
        qb = 0.1 * (1.0 + 0.5 * (np.asarray(S) > 0).sum(0 if diag else None))
    return {"Wbar": rng.randn(D, q), "Wvar": rng.rand(D, q) + 0.5, "mu": rng.randn(D) * 0.1, "muvar": np.ones(D),
            "Zbar": rng.randn(N, q), "Sig": np.tile(np.eye(q), (N, 1, 1)) * (rng.rand(N, 1, 1) + 0.5),
            "qb": qb, "al_qb": rng.rand(q) + 0.5}


def weights_like(N, D, seed, zero=0.05):
    rng = np.random.RandomState(seed)
    S = 10.0 ** rng.uniform(-1.5, 1.5, size=(N, D))
    S[rng.rand(N, D) < zero] = 0.0
    return S


def same_bound(got, ref):
    return (not np.isfinite(got)) if not np.isfinite(ref) else abs(got - ref) <= TOL * abs(ref)


def sparse_weights(A, Wd):
    """The entries of the dense weights Wd at the stored entries of A, with A's stored pattern (stored zeros included)."""
    C = sp.coo_matrix(A)
    return sp.csr_matrix((Wd[C.row, C.col], (C.row, C.col)), shape=A.shape)


def data(N, D, q, dens, seed, zero_row=True):
    """(input for the engine, dense X with NaN, weights for the engine, dense weights).  zero_row: one row has weight 0
    everywhere (latent, as an all-NaN row: the reference's 0.5 / logdet term makes both bounds infinite)."""
    if dens is None:
        X, _, _ = synth_weighted(N, D, q, 0.2, tau=10.0, seed=seed)
        S = weights_like(N, D, seed + 1)
        if zero_row and N > 2:
            S[N // 3] = 0.0
        return X, X, S, S
    A = sparse_pca(N, D, q, dens, seed=seed)
    X = densify(A)
    Wd = np.where(np.isnan(X), 0.0, weights_like(N, D, seed + 1))
    if zero_row and N > 2:
        Wd[N // 3] = 0.0
    return A, X, sparse_weights(A, Wd), Wd


# (N, D, q, algo, sparse density or None): DMMA at q = 8 / 16 / 32 / 64, generic at odd shapes and N = 1, CSR at q = 8 .. 64
SHAPES = [(700, 64, 8, "auto", None), (700, 128, 16, "auto", None), (600, 128, 32, "dmma", None),
          (500, 64, 64, "auto", None), (300, 37, 3, "auto", None), (200, 64, 16, "generic", None), (1, 37, 3, "auto", None),
          (400, 45, 8, "auto", 0.6), (600, 300, 16, "auto", 0.1), (500, 200, 32, "auto", 0.2), (300, 150, 64, "auto", 0.5)]


@pytest.mark.parametrize("N,D,q,algo,dens", SHAPES)
@pytest.mark.parametrize("ard", [False, True])
@pytest.mark.parametrize("diag", [False, True])
def test_sweeps_match_oracle(eng, N, D, q, algo, dens, ard, diag):
    A, X, Wt, Wd = data(N, D, q, dens, seed=N + D + q)
    init = rand_init(N, D, q, seed=1, diag=diag, S=Wd)
    kw = {"a0": np.random.RandomState(D).rand(D) + 0.01} if diag else {}
    o = (WeightedDiagNoiseOracle if diag else WeightedPlateOracle)(X, q, Wd, ard=ard, **kw)
    o.load_state(init)
    if ard:
        o.al_qb = init["al_qb"].copy()
    e = eng(A, q, algo=algo, ard=ard, weights=Wt, noise="diagonal" if diag else "scalar", **kw)
    assert not e.use_i8
    e.set_state(init)
    np.testing.assert_allclose(e.get_state_small()["qa"], o.qa, rtol=1e-15)
    for it in range(3):
        ref, got = o.iterate(), e.iterate()
        assert same_bound(got, ref), (it, got, ref)
    st = e.get_state()
    for k in ("Wbar", "Wvar", "mu", "muvar", "Zbar", "Sig", "qb", "tau"):
        assert tensor_rel(st[k], getattr(o, k)) < TOL, (k, tensor_rel(st[k], getattr(o, k)))


def _bytes(e, sweeps):
    el = [e.iterate() for _ in range(sweeps)]
    st = e.get_state()
    return np.array(el).tobytes(), {k: np.asarray(st[k]).tobytes() for k in ("Wbar", "Wvar", "mu", "muvar", "Zbar", "Sig",
                                                                             "qb", "al_qb")}


@pytest.mark.parametrize("algo,dens,diag", [("dmma", None, False), ("generic", None, False), ("auto", 0.2, False),
                                            ("dmma", None, True), ("auto", 0.2, True)])
def test_unit_weights_are_the_unweighted_engine(eng, algo, dens, diag):
    N, D, q = 900, 128, 16
    A = synth_weighted(N, D, q, 0.2, tau=10.0, seed=3)[0] if dens is None else sparse_pca(N, D, q, dens, seed=3)
    ones = np.ones((N, D)) if dens is None else sparse_weights(A, np.ones((N, D)))
    init = rand_init(N, D, q, seed=2, diag=diag)
    noise = "diagonal" if diag else "scalar"
    out = []
    for w in (None, ones):
        e = eng(A, q, algo=algo, ard=True, noise=noise, weights=w)
        e.set_state(init)
        out.append(_bytes(e, 3))
    assert out[0] == out[1]


@pytest.mark.parametrize("algo", ["dmma", "generic"])
def test_zero_weights_are_nan_entries(eng, algo):
    N, D, q = 800, 64, 16
    X, _, _ = synth_weighted(N, D, q, 0.1, tau=10.0, seed=4)
    S = weights_like(N, D, 5, zero=0.2)
    Xn = np.where(S == 0.0, np.nan, X)
    init = rand_init(N, D, q, seed=3)
    out = []
    for x, w in ((X, S), (Xn, np.where(S == 0.0, 1.0, S))):
        e = eng(x, q, algo=algo, weights=w)
        e.set_state(init)
        out.append(_bytes(e, 3))
    assert out[0] == out[1]


def test_sparse_zero_weights_are_removed_entries(eng):
    N, D, q = 900, 200, 16
    C = sp.coo_matrix(sparse_pca(N, D, q, 0.1, seed=6))
    rng = np.random.RandomState(7)
    w = 10.0 ** rng.uniform(-1, 1, C.nnz)
    w[rng.rand(C.nnz) < 0.2] = 0.0
    keep = w > 0
    A = sp.csr_matrix((C.data, (C.row, C.col)), shape=C.shape)
    W = sp.csr_matrix((w, (C.row, C.col)), shape=C.shape)
    A2 = sp.csr_matrix((C.data[keep], (C.row[keep], C.col[keep])), shape=C.shape)
    W2 = sp.csr_matrix((w[keep], (C.row[keep], C.col[keep])), shape=C.shape)
    init = rand_init(N, D, q, seed=8)
    res = []
    for a, w in ((A, W), (A2, W2)):
        e = eng(a, q, weights=w)
        e.set_state(init)
        res.append(([e.iterate() for _ in range(3)], e.get_state()))
    for x, y in zip(res[0][0], res[1][0]):
        assert abs(x - y) <= 1e-12 * abs(y)
    for k in ("Wbar", "mu", "Zbar", "Sig"):
        assert tensor_rel(res[0][1][k], res[1][1][k]) < 1e-12, k


@pytest.mark.parametrize("algo,dens", [("dmma", None), ("generic", None), ("auto", 0.05)])
def test_runs_are_bit_identical_and_row_ranges_compose(eng, algo, dens):
    N, D, q = 1500, 128, 16
    A, _, Wt, _ = data(N, D, q, dens, seed=11, zero_row=False)
    init = rand_init(N, D, q, seed=5)
    runs = []
    for _ in range(2):
        e = eng(A, q, algo=algo, ard=True, weights=Wt)
        e.set_state(init)
        runs.append(_bytes(e, 3))
    assert runs[0] == runs[1]
    out = []
    for split in (None, 640):
        e = eng(A, q, algo=algo, weights=Wt)
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
    N, D, q = 50, 20, 4
    X, S, _ = synth_weighted(N, D, q, 0.2, tau=10.0, seed=1)
    for kw in ({"mode": "A"}, {"algo": "i8"}):
        with pytest.raises(ValueError, match="weights"):
            eng(X, q, weights=S, **kw)
    with pytest.raises(ValueError, match="weights"):
        eng(synth_weighted(64, 64, 16, 0.2, tau=10.0, seed=1)[0], 16, precision="f32", weights=np.ones((64, 64)))
    with pytest.raises(ValueError, match="shape"):
        eng(X, q, weights=S[:, :-1])
    obs = np.argwhere(~np.isnan(X))[0]
    for bad in (-1.0, np.nan, np.inf):
        B = S.copy()
        B[tuple(obs)] = bad
        with pytest.raises(ValueError, match="weights"):
            eng(X, q, weights=B)
    B = S.copy()
    B[np.isnan(X)] = np.nan                                   # weights of missing entries are not looked at
    eng(X, q, weights=B)
    A = sp.csr_matrix(sparse_pca(N, 40, 8, 0.3, seed=2))
    W = sparse_weights(A, np.full(A.shape, 2.0))
    eng(A, 8, weights=W)
    r, c = np.argwhere(np.isnan(densify(A)))[0]
    C = W.tocoo()
    W2 = sp.csr_matrix((np.r_[C.data, 1.0], (np.r_[C.row, r], np.r_[C.col, c])), shape=A.shape)
    with pytest.raises(ValueError, match="pattern"):
        eng(A, 8, weights=W2)
    with pytest.raises(ValueError, match="weights"):
        eng(A, 8, weights=W.toarray())
    W.data[0] = -1.0
    with pytest.raises(ValueError, match="weights"):
        eng(A, 8, weights=W)
    W.data[0] = np.inf
    with pytest.raises(ValueError, match="weights"):
        eng(A, 8, weights=W)
    e = eng(X, q, weights=S)
    with pytest.raises(NotImplementedError):
        e.set_X(torch.zeros(N, D, dtype=torch.float64, device=e.device))
    with pytest.raises(NotImplementedError):
        e.iterate_from_host(torch.zeros(N, D, dtype=torch.float64).pin_memory())


def _principal_angle(A, B):
    qa, _ = np.linalg.qr(A)
    qb, _ = np.linalg.qr(B)
    s = np.clip(np.linalg.svd(qa.T @ qb, compute_uv=False), -1.0, 1.0)
    return float(np.degrees(np.arccos(s.min())))


def test_full_size_weighted_fit(eng):
    """Config-2 shape (1M x 256, q = 16, 20 % missing), per-entry precisions tau * s_nd with s log-uniform over three decades,
    50 sweeps from init_random; the weighted fit against an unweighted fit of the same data (DESIGN 5d has the numbers)."""
    N, D, q, tau = 1_000_000, 256, 16, 4.0
    dev = torch.device("cuda", torch.cuda.current_device())
    g = torch.Generator(device=dev)
    g.manual_seed(23)
    W = torch.randn(D, q, generator=g, device=dev, dtype=torch.float64)
    mu = torch.randn(D, generator=g, device=dev, dtype=torch.float64)
    X = torch.empty(N, D, dtype=torch.float64, device=dev)
    S = torch.empty(N, D, dtype=torch.float64, device=dev)
    for lo in range(0, N, 1 << 17):
        n = min(1 << 17, N - lo)
        Z = torch.randn(n, q, generator=g, device=dev, dtype=torch.float64)
        s = 10.0 ** (3.0 * torch.rand(n, D, generator=g, device=dev, dtype=torch.float64) - 1.5)
        x = Z @ W.T + mu + torch.randn(n, D, generator=g, device=dev, dtype=torch.float64) / (tau * s).sqrt()
        x[torch.rand(n, D, generator=g, device=dev) < 0.2] = float("nan")
        X[lo:lo + n], S[lo:lo + n] = x, s
    Wt = W.cpu().numpy()
    res = {}
    for name, w in (("weighted", S), ("unweighted", None)):
        e = eng(X, q, weights=w)
        e.init_random(seed=3)
        b = e.run(50).cpu().numpy()
        e.check()
        assert np.all(np.isfinite(b))
        res[name] = (b, _principal_angle(e.get_state_small()["Wbar"], Wt), e.get_state_small()["tau"])
        del e
        torch.cuda.empty_cache()
    b, ang_w, tau_w = res["weighted"]
    ang_u = res["unweighted"][1]
    print("largest principal angle to the true W: weighted %.4f deg, unweighted %.4f deg; tau %.4f (true %.1f); "
          "bound rises over sweeps 10..50: %s" % (ang_w, ang_u, tau_w, tau, bool(np.all(np.diff(b[10:]) >= -1e-9 * np.abs(b[11:])))))
    assert np.all(np.diff(b[10:]) >= -1e-9 * np.abs(b[11:]))
    assert abs(tau_w / tau - 1.0) < 0.02
    assert ang_w < ang_u


def _worker(rank, world, port, shape, out_dir):
    import torch.distributed as dist
    from pyvb_b200 import PlateEngine
    from pyvb_b200.dist import shard_rows
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    N, D, q, dens, diag = shape
    A, _, _, Wd = data(N, D, q, dens, seed=3, zero_row=False)
    init = rand_init(N, D, q, seed=1, diag=diag, S=Wd)
    lo, hi = shard_rows(N, world, rank)
    if dens is None:
        a, w = A[lo:hi], Wd[lo:hi]
    else:
        a = sp.csr_matrix(A)[lo:hi]
        w = sparse_weights(a, Wd[lo:hi])
    e = PlateEngine(a, q, device=dev, distributed=True, row_offset=lo, weights=w, noise="diagonal" if diag else "scalar")
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


@pytest.mark.parametrize("shape", [(3001, 128, 16, None, False), (1200, 200, 8, 0.05, True)])
def test_two_gpu_sharded(tmp_path, shape):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world = 2
    N, D, q, dens, diag = shape
    mp.spawn(_worker, args=(world, _free_port(), shape, str(tmp_path)), nprocs=world, join=True)
    _, X, _, Wd = data(N, D, q, dens, seed=3, zero_row=False)
    o = (WeightedDiagNoiseOracle if diag else WeightedPlateOracle)(X, q, Wd)
    o.load_state(rand_init(N, D, q, seed=1, diag=diag, S=Wd))
    ref = np.array([o.iterate() for _ in range(4)])
    a, b = (np.load(os.path.join(str(tmp_path), "r%d.npz" % r)) for r in range(world))
    assert np.asarray(a["qb"]).tobytes() == np.asarray(b["qb"]).tobytes() and np.array_equal(a["elbo"], b["elbo"])
    assert a["Wbar"].tobytes() == b["Wbar"].tobytes()
    assert np.max(np.abs(a["elbo"] - ref) / np.abs(ref)) < TOL
    assert tensor_rel(a["qb"], o.qb) < TOL and tensor_rel(a["Wbar"], o.Wbar) < TOL
