"""GPU tests of the sparse-observation path (CSR input, kernels_sparse.cu): sweep-by-sweep parity with the oracle on the
densified matrix, step-by-step agreement with the dense engine, row ranges, determinism, one run at scale against the
dense default path, the error contract, and a row-sharded run on two GPUs."""
import os
import socket

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from helpers import numpy_stats, tensor_rel
from oracle.plate_oracle import PlateOracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pyvb_b200 import PlateEngine
    return PlateEngine


def sparse_pca(N, D, q, density, seed=0, noise_prec=20.0):
    """A PCA-shaped data set with `density` of its entries stored (scipy CSR) -- and a few stored zeros.  Every row stores
    at least one entry: a row without any has logdet 0, and the reference's bound term 0.5 / logdet is then infinite."""
    rng = np.random.RandomState(seed)
    W, Z, mu = rng.randn(D, q), rng.randn(N, q), rng.randn(D)
    keep = rng.rand(N, D) < density
    empty = np.nonzero(~keep.any(1))[0]
    keep[empty, rng.randint(0, D, empty.size)] = True
    r, c = np.nonzero(keep)
    v = np.einsum("nq,nq->n", Z[r], W[c]) + mu[c] + rng.randn(r.size) / np.sqrt(noise_prec)
    if v.size > 4:
        v[rng.choice(v.size, max(1, v.size // 50), replace=False)] = 0.0
    return sp.csr_matrix((v, (r, c)), shape=(N, D))


def densify(A):
    X = np.full(A.shape, np.nan)
    C = A.tocoo()
    X[C.row, C.col] = C.data
    return X


def rand_init(N, D, q, seed=0):
    rng = np.random.RandomState(seed)
    return {"Wbar": rng.randn(D, q), "Wvar": rng.rand(D, q) + 0.5, "mu": rng.randn(D) * 0.1, "muvar": np.ones(D),
            "Zbar": rng.randn(N, q), "Sig": np.tile(np.eye(q), (N, 1, 1)) * (rng.rand(N, 1, 1) + 0.5), "qb": 0.7,
            "al_qb": rng.rand(q) + 0.5}


# (N, D, q, density, ard): every q of the CSR path, D not a multiple of 8 / 16 / 64, 1 % .. 60 % observed, N = 1.  The
# sparse shapes keep >= 2q observations per row: a row with fewer leaves directions of qprec at the prior precision next to
# tau * n_obs ~ 1e5 ones, and the batched solve shared with the dense DMMA path (Gauss-Jordan at q = 16, 32) then agrees
# with the oracle's Cholesky only to cond * eps (~1e-9 on Zbar); test_zstep_and_stats_match_dense_engine covers such rows
SHAPES = [(300, 3, 8, 0.6, False), (257, 37, 16, 0.1, True), (3000, 3300, 16, 0.01, False), (3000, 650, 32, 0.1, False),
          (3000, 1300, 64, 0.1, True), (120, 37, 64, 0.6, False), (1, 37, 16, 0.6, False), (500, 45, 8, 0.6, True),
          (4000, 1700, 8, 0.01, False)]


def same_bound(got, ref):
    """1e-9 relative.  A row without observations has logdet = +-0, and the reference's term 0.5 / logdet makes the bound
    infinite (its sign follows the sign of that zero): then both must be infinite."""
    return (not np.isfinite(got)) if not np.isfinite(ref) else abs(got - ref) <= 1e-9 * abs(ref)


@pytest.mark.parametrize("N,D,q,density,ard", SHAPES)
def test_sparse_sweeps_match_oracle(eng, N, D, q, density, ard):
    A = sparse_pca(N, D, q, density, seed=N + D)
    X = densify(A)
    init = rand_init(N, D, q, seed=1)
    o = PlateOracle(X, q, mode="B", ard=ard)
    o.load_state(init)
    if ard:
        o.al_qb = init["al_qb"].copy()
    e = eng(A, q, mode="B", ard=ard)
    assert e.sparse and e.i8_fallbacks() == (0, 0)
    e.set_state(init)
    for it in range(5):
        ref = o.iterate()
        got = e.iterate()
        assert abs(got - ref) <= 1e-9 * abs(ref), (it, got, ref)
        st = e.get_state()
        for k in ("Wbar", "Wvar", "mu", "muvar", "Zbar", "Sig"):
            assert tensor_rel(st[k], getattr(o, k)) < 1e-9, (it, k)
        assert abs(st["qb"] - o.qb) <= 1e-9 * abs(o.qb)
    e.check()


def test_missing_rows_columns_and_stored_zeros(eng):
    N, D, q = 200, 37, 16
    A = sparse_pca(N, D, q, 0.3, seed=4).tolil()
    A[5, :] = 0
    A[:, 11] = 0
    A = A.tocsr()
    A.eliminate_zeros()                  # row 5 and column 11 hold nothing: all missing
    A[7, 3] = 0.0                        # stored zeros: observed values
    A[9, 20] = 0.0
    X = densify(A)
    assert np.isnan(X[5]).all() and np.isnan(X[:, 11]).all() and X[7, 3] == 0.0
    init = rand_init(N, D, q, seed=2)
    o = PlateOracle(X, q, mode="B")
    o.load_state(init)
    e = eng(A, q)
    e.set_state(init)
    for it in range(5):
        ref, got = o.iterate(), e.iterate()
        assert same_bound(got, ref), (it, got, ref)
    st = e.get_state()
    for k in ("Wbar", "Wvar", "mu", "Zbar", "Sig"):
        assert tensor_rel(st[k], getattr(o, k)) < 1e-9, k
    assert float(e.logdet[5]) == 0.0 and np.allclose(st["Zbar"][5], 0.0) and np.allclose(st["Sig"][5], np.eye(q))


def test_torch_csr_input_on_device_and_host(eng):
    N, D, q = 300, 64, 16
    A = sparse_pca(N, D, q, 0.2, seed=8)
    t = torch.sparse_csr_tensor(torch.as_tensor(A.indptr, dtype=torch.int64), torch.as_tensor(A.indices, dtype=torch.int64),
                                torch.as_tensor(A.data), size=A.shape)
    init = rand_init(N, D, q, seed=3)
    out = []
    for X in (A, t, t.to("cuda")):
        e = eng(X, q)
        e.set_state(init)
        out.append([e.iterate() for _ in range(2)] + [e.get_state()["Wbar"]])
    for r in out[1:]:
        assert r[0] == out[0][0] and r[1] == out[0][1] and np.array_equal(r[2], out[0][2])


@pytest.mark.parametrize("D,q,algo", [(37, 16, "generic"), (200, 8, "generic"), (64, 16, "dmma"), (96, 32, "dmma"),
                                      (128, 64, "dmma"), (48, 8, "dmma")])
def test_zstep_and_stats_match_dense_engine(eng, D, q, algo):
    N = 700
    A = sparse_pca(N, D, q, 0.15, seed=D + q)
    X = densify(A)
    init = rand_init(N, D, q, seed=4)
    es, ed = eng(A, q), eng(X, q, algo=algo)
    for e in (es, ed):
        e.set_state(init)
        e.update_Z()
    a, b = es.get_state(), ed.get_state()
    for k in ("Zbar", "Sig"):
        assert tensor_rel(a[k], b[k]) < 1e-12, k
    assert tensor_rel(es.logdet.cpu().numpy(), ed.logdet.cpu().numpy()) < 1e-12
    # statistics of the new rows, once with K2's partials (full-range Z step) and once after set_state (none)
    from pyvb_b200._layout import StatLayout, SC_LOGDETZ, SC_NE, SC_NROWS, SC_QLDZ, SC_SXX
    L = StatLayout(D, q)
    for with_zsums in (True, False):
        if not with_zsums:
            st = es.get_state()
            es.set_state({k: st[k] for k in ("Wbar", "Wvar", "mu", "muvar", "Zbar", "Sig", "qb")})
            assert not es._zsums_valid
        else:
            assert es._zsums_valid
        es._ensure_stats()
        got = es.stats.cpu().numpy()
        ref = numpy_stats(X, a["Zbar"], a["Sig"], q)
        gv, rv = L.views(got), L.views(ref)
        for k in ("T1", "Bst", "Ast", "cnt", "colx", "S", "zsum"):
            assert tensor_rel(gv[k], rv[k]) < 1e-12, (with_zsums, k)
        for s in (SC_SXX, SC_NE, SC_NROWS):
            assert abs(gv["scal"][s] - rv["scal"][s]) <= 1e-12 * abs(rv["scal"][s]), (with_zsums, s)
        ld = es.logdet.cpu().numpy()
        assert abs(gv["scal"][SC_LOGDETZ] - ld.sum()) <= 1e-12 * np.abs(ld).sum()
        assert abs(gv["scal"][SC_QLDZ] - (0.5 / ld).sum()) <= 1e-12 * np.abs(0.5 / ld).sum()


@pytest.mark.parametrize("q,k", [(16, 333), (64, 57), (8, 1)])
def test_row_ranges_are_bit_identical(eng, q, k):
    N, D = 1000, 77
    A = sparse_pca(N, D, q, 0.1, seed=q)
    init = rand_init(N, D, q, seed=5)
    e1, e2 = eng(A, q), eng(A, q)
    for e in (e1, e2):
        e.set_state(init)
    e1.update_Z()
    e2.update_Z(0, k)
    e2.update_Z(k, N)
    torch.cuda.synchronize()
    for name in ("MZ", "Sig", "logdet"):
        assert torch.equal(getattr(e1, name), getattr(e2, name)), name
    # and the statistics (with / without K2's partials) agree to rounding; then the sweeps continue normally
    e1._ensure_stats()
    e2._ensure_stats()
    assert tensor_rel(e2.stats.cpu().numpy(), e1.stats.cpu().numpy()) < 1e-12
    assert np.isfinite(e2.iterate())


def test_two_engines_are_bit_identical(eng):
    N, D, q = 3000, 200, 16
    A = sparse_pca(N, D, q, 0.05, seed=6)
    init = rand_init(N, D, q, seed=6)
    res = []
    for _ in range(2):
        e = eng(A, q, ard=True)
        e.set_state(init)
        el = [e.iterate() for _ in range(3)]
        st = e.get_state()
        res.append((el, st))
    assert res[0][0] == res[1][0]
    for k in ("Wbar", "Wvar", "mu", "muvar", "Zbar", "Sig", "al_qb"):
        assert np.asarray(res[0][1][k]).tobytes() == np.asarray(res[1][1][k]).tobytes(), k


def test_errors(eng):
    A = sparse_pca(50, 20, 16, 0.3, seed=1)
    with pytest.raises(ValueError, match="mode"):
        eng(A, 16, mode="A")
    with pytest.raises(ValueError, match="f64"):
        eng(A, 16, precision="f32")
    with pytest.raises(ValueError, match="q in"):
        eng(A, 12)
    with pytest.raises(ValueError, match="auto"):
        eng(A, 16, algo="dmma")
    bad = A.copy()
    bad.data[0] = np.nan
    with pytest.raises(ValueError, match="NaN"):
        eng(bad, 16)
    e = eng(A, 16)
    with pytest.raises(NotImplementedError):
        e.set_X(torch.zeros(50, 20, dtype=torch.float64, device=e.device))
    with pytest.raises(NotImplementedError):
        e.iterate_from_host(np.zeros((50, 20)))


def test_at_scale_against_dense_default_path(eng):
    """N = 1M, D = 4096, q = 16, 1 % observed: 3 sweeps from the same init_random state on the sparse engine and on the dense
    default path (32 GB of NaN-filled X)."""
    N, D, q, dens = 1_000_000, 4096, 16, 0.01
    dev = torch.device("cuda", torch.cuda.current_device())
    g = torch.Generator(device=dev)
    g.manual_seed(11)
    crow = torch.zeros(N + 1, dtype=torch.int64, device=dev)
    cols, step = [], 1 << 16
    for lo in range(0, N, step):
        m = torch.rand(min(step, N - lo), D, generator=g, device=dev) < dens
        r, c = m.nonzero(as_tuple=True)
        crow[lo + 1:lo + 1 + m.shape[0]] = m.sum(1)
        cols.append(c)
    crow = torch.cumsum(crow, 0)
    col = torch.cat(cols)
    val = torch.randn(col.numel(), generator=g, device=dev, dtype=torch.float64)
    Xs = torch.sparse_csr_tensor(crow, col, val, size=(N, D))
    es = eng(Xs, q)
    es.init_random(seed=5)
    ls = [es.iterate() for _ in range(3)]
    es.check()
    st_s = {k: getattr(es, k).clone() for k in ("Wbar", "Wvar", "mu", "muvar", "Zbar", "Sig")}
    qb_s = es.get_state_small()["qb"]
    del es
    torch.cuda.empty_cache()
    Xd = torch.full((N, D), float("nan"), dtype=torch.float64, device=dev)
    rows = torch.repeat_interleave(torch.arange(N, device=dev), crow[1:] - crow[:-1])
    Xd[rows, col] = val
    del rows, Xs
    ed = eng(Xd, q)
    del Xd
    ed.init_random(seed=5)
    ld = [ed.iterate() for _ in range(3)]
    ed.check()
    assert all(np.isfinite(ls))
    for a, b in zip(ls, ld):
        assert abs(a - b) <= 1e-9 * abs(b), (ls, ld)
    for k, v in st_s.items():
        ref = getattr(ed, k)
        err = float((v - ref).abs().max() / ref.abs().max())
        assert err < 1e-9, (k, err)
    assert abs(qb_s - ed.get_state_small()["qb"]) <= 1e-9 * abs(qb_s)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, comm, shape, out_dir):
    import torch.distributed as dist
    from pyvb_b200 import PlateEngine
    from pyvb_b200.dist import shard_rows
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["PYVB_COMM"] = comm
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    N, D, q, dens = shape
    A = sparse_pca(N, D, q, dens, seed=3)
    init = rand_init(N, D, q, seed=1)
    lo, hi = shard_rows(N, world, rank)
    e = PlateEngine(A[lo:hi], q, device=dev, distributed=True, row_offset=lo)
    assert (e.peers is not None) == (comm == "peer")
    loc = dict(init)
    for k in ("Zbar", "Sig"):
        loc[k] = loc[k][lo:hi]
    e.set_state(loc)
    elbo = [e.iterate() for _ in range(4)]
    st = e.get_state_small()
    e.check()
    np.savez(os.path.join(out_dir, "r%d_%s.npz" % (rank, comm)), elbo=np.array(elbo), Wbar=st["Wbar"], mu=st["mu"],
             qb=st["qb"], Zbar=e.Zbar.cpu().numpy())
    e.close()
    dist.destroy_process_group()


@pytest.mark.parametrize("shape", [(3001, 77, 16, 0.1), (1200, 200, 8, 0.03)])
def test_two_gpu_sparse_sharded(tmp_path, shape):
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world = 2
    N, D, q, dens = shape
    for comm in ("peer", "nccl"):
        mp.spawn(_worker, args=(world, _free_port(), comm, shape, str(tmp_path)), nprocs=world, join=True)
    X = densify(sparse_pca(N, D, q, dens, seed=3))
    init = rand_init(N, D, q, seed=1)
    o = PlateOracle(X, q, mode="B")
    o.load_state(init)
    ref = np.array([o.iterate() for _ in range(4)])
    got = {(r, c): np.load(os.path.join(str(tmp_path), "r%d_%s.npz" % (r, c))) for r in range(world) for c in ("peer", "nccl")}
    for c in ("peer", "nccl"):
        a, b = got[(0, c)], got[(1, c)]
        assert np.array_equal(a["elbo"], b["elbo"]) and np.array_equal(a["Wbar"], b["Wbar"])
        assert np.max(np.abs(a["elbo"] - ref) / np.abs(ref)) < 1e-9
        assert tensor_rel(a["Wbar"], o.Wbar) < 1e-9 and tensor_rel(a["mu"], o.mu) < 1e-9
        assert abs(float(a["qb"]) - o.qb) <= 1e-9 * abs(o.qb)
        assert tensor_rel(np.concatenate([a["Zbar"], b["Zbar"]], 0), o.Zbar) < 1e-9
