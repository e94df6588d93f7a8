"""CPU tests of the host side: graph crawl order, plate compilation / scheduling (with a recording
engine in place of the CUDA one) and the C-ABI library surface.  No GPU compute."""
import ctypes
import os
import re

import numpy as np
import pytest

from helpers import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class RecorderEngine(object):
    """Stands in for PlateEngine: records operator calls, holds the injected state."""
    def __init__(self, X, q, **kw):
        self.X, self.q, self.kw, self.calls, self.state = np.array(X), q, kw, [], None

    def set_state(self, st):
        self.state = st

    def update_W(self, lo, hi): self.calls.append(("W", lo, hi))
    def update_Z(self, lo, hi): self.calls.append(("Z", lo, hi))
    def update_X(self, lo, hi): self.calls.append(("X", lo, hi))
    def update_Mu(self): self.calls.append(("M",))
    def update_Beta(self): self.calls.append(("B",))
    def update_Alpha(self, lo, hi): self.calls.append(("L", lo, hi))


@pytest.fixture()
def recorder(monkeypatch):
    from pyvb_b200 import plate
    monkeypatch.setattr(plate.PCAPlate, "ENGINE", RecorderEngine)
    return plate


def _build(nodes, X, q, ard=False):
    N, d = X.shape
    if ard:
        Alphas = [nodes.Gamma(d, 1e-3, 1e-3) for i in range(q)]
        Ws = [nodes.Gaussian(d, np.zeros((d, 1)), Alphas[i]) for i in range(q)]
    else:
        Ws = [nodes.Gaussian(d, np.zeros((d, 1)), np.eye(d) * 1e-3) for i in range(q)]
    W = nodes.hstack(Ws)
    Mu = nodes.Gaussian(d, np.zeros((d, 1)), np.eye(d) * 1e-3)
    Beta = nodes.Gamma(d, 1e-3, 1e-3)
    Zs = [nodes.Gaussian(q, np.zeros((q, 1)), np.eye(q)) for i in range(N)]
    Xs = [nodes.Gaussian(d, W * z + Mu, Beta) for z in Zs]
    [xnode.observe(xval.reshape(d, 1)) for xnode, xval in zip(Xs, X)]
    return Ws, W, Mu, Beta, Zs, Xs


@pytest.mark.parametrize("name,seed", [("small_a.npz", 2), ("ard.npz", 5)])
def test_fetch_order_and_init_match_reference(recorder, name, seed):
    from pyvb_b200 import nodes, Network
    g = load_golden(name)
    ard = bool(int(g["ard"]))
    np.random.seed(seed)
    Ws, W, Mu, Beta, Zs, Xs = _build(nodes, g["X"], int(g["q"]), ard=ard)
    net = Network(); net.verbose = False
    net.addnode(W); net.fetch_network(); net.find_iterable()
    kinds = {id(Mu): "M", id(Beta): "B"}
    kinds.update({id(w): "W" for w in Ws}); kinds.update({id(z): "Z" for z in Zs}); kinds.update({id(x): "X" for x in Xs})
    order = "".join(kinds.get(id(n), "L") for n in net.iterable_nodes)
    assert order == str(g["order"])                     # the reference's Gauss-Seidel order (SURVEY 0.6)
    pl = recorder.bind(W)
    st = pl.engine.state
    for k in ("Wbar", "Wvar", "mu", "muvar", "Zbar", "Sig", "Xhat", "V"):
        assert np.array_equal(st[k], g["init_" + k]), k  # identical random initialisation, bit for bit
    assert st["qb"] == float(g["init_qb"])
    assert np.array_equal(np.isnan(pl.engine.X), np.isnan(g["X"]))
    sched = pl.schedule(net.iterable_nodes)
    N, q = g["X"].shape[0], int(g["q"])
    want = [("W", 0, q), ("Z", 0, N)] + ([("L", 0, q)] if ard else []) + [("X", 0, 1), ("M", 0, 1), ("X", 1, N), ("B", 0, 1)]
    assert sched == want
    pl.sweep(sched)
    assert pl.engine.calls[0] == ("W", 0, q) and pl.engine.calls[-1] == ("B",)
    Zs[3].update()
    assert pl.engine.calls[-1] == ("Z", 3, 4)


def test_error_conventions(recorder):
    from pyvb_b200 import nodes
    with pytest.raises(AssertionError):
        nodes.Gaussian(3, np.zeros((2, 1)), np.eye(3))
    with pytest.raises(AssertionError):
        nodes.Gaussian(3, np.zeros((3, 1)), np.eye(2))
    with pytest.raises(nodes.ConjugacyError):      # right shape, illegal type (gaussian.py:58-61)
        cols = [nodes.Gaussian(3, np.zeros((3, 1)), np.eye(3)) for _ in range(3)]
        nodes.Gaussian(3, np.zeros((3, 1)), nodes.hstack(cols))
    with pytest.raises(nodes.ConjugacyError):      # illegal mean parent (gaussian.py:49-52)
        nodes.Gaussian(3, nodes.hstack([nodes.Gaussian(3, np.zeros((3, 1)), np.eye(3))]), np.eye(3))
    assert issubclass(nodes.ConjugacyError, ValueError)
    g = nodes.Gaussian(2, np.zeros((2, 1)), np.eye(2))
    with pytest.raises(AssertionError):
        g.observe(np.zeros((3, 1)))
    with pytest.raises(AssertionError):
        nodes.Multiplication(nodes.Constant(np.eye(3)), nodes.Constant(np.zeros((2, 1))))
    # a graph outside the VB-PCA pattern is refused loudly (no CPU message passing)
    a = nodes.Gaussian(2, np.zeros((2, 1)), np.eye(2))
    with pytest.raises(NotImplementedError):
        a.update()
    with pytest.raises(NotImplementedError):
        nodes.Wishart(2, 1.0, np.eye(2))


def test_observe_classification():
    from pyvb_b200 import nodes
    x = nodes.Gaussian(3, np.zeros((3, 1)), np.eye(3))
    x.observe(np.array([[np.nan], [np.nan], [np.nan]]))
    assert not x.observed and not x.partially_observed
    x.observe(np.array([[1.0], [np.nan], [2.0]]))
    assert x.partially_observed and list(x.obs_index) == [0, 2] and list(x.missing_index) == [1]
    y = nodes.Gaussian(2, np.zeros((2, 1)), np.eye(2))
    v = np.array([[1.0], [2.0]])
    y.observe(v)
    assert y.observed and y.qmu is v and np.all(y.qcov == 0)


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "pyvb_b200.h")).read()
    names = set(re.findall(r"\b(pyvb_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 12
    from pyvb_b200 import _cabi
    L = _cabi.lib()
    for n in names:
        assert hasattr(L, n), n
    assert set(_cabi.SIGNATURES) == names
    assert L.pyvb_version() >= 100
    # layout mirror
    from pyvb_b200._layout import StatLayout
    for D, q in [(5, 2), (256, 16), (1024, 32), (512, 64)]:
        assert StatLayout(D, q).len == L.pyvb_stats_len(D, q)
        p = L.pyvb_gw_pitch(q)
        assert p >= q * (q + 1) // 2 + q + 1 and p % 8 == 4
    assert ctypes.sizeof(_cabi.Consts) == 14 * 8 + 8


def test_zsums_len_is_what_the_k2_kernel_writes():
    """The K2 partial buffer (pyvb_zsums_len) holds exactly the partials the K2 kernel of q writes, one per CTA, at most one CTA
    per SM (no compute: size queries only)."""
    from pyvb_b200 import _cabi
    L = _cabi.lib()
    for q in (8, 16, 32, 64):
        for N in (1, 7, 100, 1000, 40000, 1000000):
            blocks = L.pyvb_zsums_blocks(N, q)
            assert 1 <= blocks <= 148, (q, N, blocks)
            assert L.pyvb_zsums_len(N, q) == blocks * L.pyvb_zsums_kw(q), (q, N)


class _DumpEngine(object):
    """Stands in for PlateEngine in bench.dump_outputs (host tensors, keep_sigma=False layout)."""
    def __init__(self, N, D, q, seed):
        import torch
        rng = np.random.RandomState(seed)
        ii, jj = np.tril_indices(q)
        self.N, self.q, self.Sig = N, q, None
        self.Zbar = torch.as_tensor(rng.randn(N, q))
        self.sig_packed = rng.rand(N, len(ii))
        self.M2 = torch.as_tensor(self.sig_packed + self.Zbar.numpy()[:, ii] * self.Zbar.numpy()[:, jj])
        self.trace = torch.as_tensor(rng.randn(16))
        self.small = {"Wbar": rng.randn(D, q), "mu": rng.randn(D), "qb": 0.5, "alpha": np.ones(q)}

    def get_state_small(self):
        return self.small


@pytest.mark.parametrize("N,q", [(50, 3), (20000, 64)])
def test_bench_dump_outputs_writes_a_fixed_row_sample_in_float64(tmp_path, N, q):
    import bench
    e = _DumpEngine(N, 8, q, seed=1)
    names = bench.dump_outputs(e, [5, 6, 7], str(tmp_path / "a"))
    bench.dump_outputs(_DumpEngine(N, 8, q, seed=1), [5, 6, 7], str(tmp_path / "b"))
    total = 0
    for name in names:
        a = np.load(str(tmp_path / "a" / (name + ".npy")))
        assert a.dtype == np.float64 and np.array_equal(a, np.load(str(tmp_path / "b" / (name + ".npy")))), name
        total += a.nbytes
    assert total <= 64 << 20
    rows = np.load(str(tmp_path / "a" / "rows.npy")).astype(np.int64)
    assert len(rows) == min(N, bench.DUMP_ROW_BYTES // (8 * (q + q * q))) and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(str(tmp_path / "a" / "elbo.npy")), e.trace.numpy()[5:8])
    assert np.array_equal(np.load(str(tmp_path / "a" / "Zbar.npy")), e.Zbar.numpy()[rows])
    Sig = np.load(str(tmp_path / "a" / "Sig.npy"))
    ii, jj = np.tril_indices(q)
    assert np.allclose(Sig[:, ii, jj], e.sig_packed[rows], rtol=0, atol=1e-12) and np.array_equal(Sig, Sig.transpose(0, 2, 1))


def test_engine_refuses_to_run_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from pyvb_b200 import PlateEngine
    with pytest.raises(RuntimeError):
        PlateEngine(np.zeros((4, 3)), 2)
