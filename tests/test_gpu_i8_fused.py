"""GPU: the INT8 statistics with the digit planes made in shared memory (stats_i8_fused_kernel, D <= 256) against the
two-kernel path it replaces there (digitize_kernel + stats_i8_kernel, PYVB_I8_FUSED=0).  Same chunks, same integer sums,
same recombination: the chunk partials, the statistics and whole sweeps are BIT-identical."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

from oracle.plate_oracle import synth_pca
from test_gpu_parity import rand_init

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pyvb_b200 import PlateEngine
    return PlateEngine


def _bits(t):
    return t.detach().contiguous().view(torch.int64).cpu().numpy()


def _stats_pass(eng, X, q, init, fused, monkeypatch, poison_row=None):
    """One Z step, then the INT8 statistics of its rows on a zeroed workspace."""
    monkeypatch.setenv("PYVB_I8_FUSED", "1" if fused else "0")
    e = eng(X, q, mode="B", algo="i8")
    assert e.use_i8_stats
    if init is None:
        e.init_random(seed=11)
    else:
        e.set_state(init)
    e._ensure_stats()               # the X-only sums (the INT8 statistics need them)
    e.update_Z()
    if poison_row is not None:      # a non-PD row as the Z step leaves it: NaN / inf in its MZ entries
        e.MZ[poison_row, ::2] = float("nan")
        e.MZ[poison_row, 1::2] = float("inf")
    e.ws.zero_()
    e._ensure_stats()
    torch.cuda.synchronize()
    assert getattr(e, "i8_stats_calls", 0) == 1
    return e


def _assert_same_pass(a, b, what):
    assert np.array_equal(_bits(a.stats), _bits(b.stats)), what
    assert torch.equal(a.ws, b.ws), what                  # the chunk partials, byte for byte
    assert a.i8_fallbacks() == b.i8_fallbacks(), what


@pytest.mark.parametrize("q", [16, 32, 64])
@pytest.mark.parametrize("D", [64, 192, 256])
@pytest.mark.parametrize("N", [1, 64, 777, 5000, 100000])
def test_fused_stats_bit_identical(eng, monkeypatch, N, D, q):
    X = synth_pca(N, D, q, 0.3, seed=N + D + q)
    ef = _stats_pass(eng, X, q, None, True, monkeypatch)
    eo = _stats_pass(eng, X, q, None, False, monkeypatch)
    assert ef.ZI is None and eo.ZI is not None
    _assert_same_pass(ef, eo, (N, D, q))


@pytest.mark.parametrize("shape", [(5000, 256, 16), (777, 192, 32), (2100, 64, 64)])
def test_fused_stats_edge_rows(eng, monkeypatch, shape):
    """all-missing rows, fully observed rows and a non-PD row (NaN / inf in its MZ entries: zero digits on both paths)"""
    N, D, q = shape
    X = synth_pca(N, D, q, 0.25, seed=5)
    X[2, :] = np.nan
    X[N - 1, :] = np.nan
    X[5, :] = 1.0
    X[N - 2, :] = -2.0
    init = rand_init(N, D, q, seed=3)
    init["Wbar"][:, 0] *= 1e3       # columns on very different scales
    init["Wbar"][:, 1] *= 1e-4
    ef = _stats_pass(eng, X, q, init, True, monkeypatch, poison_row=7)
    eo = _stats_pass(eng, X, q, init, False, monkeypatch, poison_row=7)
    assert np.array_equal(_bits(ef.stats), _bits(eo.stats)), shape
    ef2 = _stats_pass(eng, X, q, init, True, monkeypatch)
    eo2 = _stats_pass(eng, X, q, init, False, monkeypatch)
    _assert_same_pass(ef2, eo2, shape)


@pytest.mark.parametrize("shape", [(100000, 256, 16), (5000, 192, 32), (777, 256, 64)])
def test_fused_sweeps_bit_identical(eng, monkeypatch, shape):
    """whole sweeps (auto path): the bound of every sweep and the state"""
    N, D, q = shape
    X = synth_pca(N, D, q, 0.2, seed=9)
    out = []
    for fused in (True, False):
        monkeypatch.setenv("PYVB_I8_FUSED", "1" if fused else "0")
        e = eng(X, q, mode="B", algo="auto")
        e.init_random(seed=4)
        tr = [e.iterate() for _ in range(4)]
        assert getattr(e, "i8_stats_calls", 0) >= 3 and e.i8_fallbacks() == (0, 0)
        out.append((tr, e.get_state()))
    (tf, sf), (to, so) = out
    assert tf == to, (tf, to)
    for k in sf:
        a, b = np.ascontiguousarray(sf[k]), np.ascontiguousarray(so[k])
        assert a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8)), k


def test_switch_is_read_per_call(eng, monkeypatch):
    """one engine, both paths: ZI is allocated when the switch turns the fused path off after construction"""
    N, D, q = 3000, 256, 16
    X = synth_pca(N, D, q, 0.2, seed=2)
    monkeypatch.setenv("PYVB_I8_FUSED", "1")
    e = eng(X, q, mode="B", algo="i8")
    assert e.ZI is None and e.lib.pyvb_stats_i8_fused(D, q) == 1
    e.init_random(seed=1)
    e.iterate()
    res = []
    for fused in ("1", "0", "1"):
        monkeypatch.setenv("PYVB_I8_FUSED", fused)
        e._stats_fresh = False
        e.ws.zero_()
        e._ensure_stats()
        res.append(_bits(e.stats))
    assert e.ZI is not None
    assert np.array_equal(res[0], res[1]) and np.array_equal(res[1], res[2])


def test_null_zi_rejected_off_the_fused_path(eng, monkeypatch):
    from pyvb_b200 import _cabi
    N, D, q = 700, 128, 16
    X = synth_pca(N, D, q, 0.2, seed=2)
    e = _stats_pass(eng, X, q, rand_init(N, D, q), True, monkeypatch)
    monkeypatch.setenv("PYVB_I8_FUSED", "0")
    assert e.lib.pyvb_stats_i8_fused(D, q) == 0
    rc = e.lib.pyvb_stats_i8_f64(N, D, q, e.X.data_ptr(), D, e.maskT.data_ptr(), e.MZ.data_ptr(), e.ldmz,
                                 e.logdet.data_ptr(), 0, e.i8_scratch.data_ptr(), e.stats.data_ptr(), e.ws.data_ptr(),
                                 e.ws_bytes, e.xcache.data_ptr(), 0, None, e._stream())
    with pytest.raises(_cabi.PyvbError):
        _cabi.check(rc, "pyvb_stats_i8_f64")


def test_d512_keeps_the_two_kernel_path(eng, monkeypatch):
    N, D, q = 1500, 512, 16
    X = synth_pca(N, D, q, 0.3, seed=8)
    init = rand_init(N, D, q, seed=2)
    e1 = _stats_pass(eng, X, q, init, True, monkeypatch)
    assert e1.lib.pyvb_stats_i8_fused(D, q) == 0 and e1.ZI is not None
    e0 = _stats_pass(eng, X, q, init, False, monkeypatch)
    _assert_same_pass(e1, e0, "D=512")


def test_forced_fallback_on_the_fused_path(eng):
    """PYVB_I8_GUARD=force (read once per process, hence the subprocess): every statistics pass of the fused path is redone
    on the FP64 tensor cores and the result is the DMMA one."""
    code = textwrap.dedent("""
        import numpy as np, torch, sys
        sys.path.insert(0, %r)
        from pyvb_b200 import PlateEngine
        from oracle.plate_oracle import synth_pca
        X = synth_pca(3000, 256, 16, 0.3, seed=1)
        ed, ei = PlateEngine(X, 16, mode="B", algo="dmma"), PlateEngine(X, 16, mode="B", algo="auto")
        assert ei.use_i8_stats and ei.ZI is None
        for e in (ed, ei):
            e.init_random(seed=3)
            for _ in range(3):
                e.iterate()
        assert ei.i8_fallbacks() == (3, 3), ei.i8_fallbacks()
        rel = lambda a, b: float((a - b).abs().max() / b.abs().max())
        assert rel(ei.MZ, ed.MZ) < 1e-11 and rel(ei.Wbar, ed.Wbar) < 1e-11 and rel(ei.trace[:3], ed.trace[:3]) < 1e-11
        print("forced ok")
    """ % ROOT)
    env = dict(os.environ, PYVB_I8_GUARD="force")
    env.pop("PYVB_I8_FUSED", None)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "forced ok" in r.stdout, r.stdout + r.stderr
