"""GPU: how stats_i8_fused_kernel receives the MZ rows.  A tensor map over the columns [0, P + q) of MZ delivers them into
a ring of slots per converter warp, several K steps ahead; rows past N and the rest of the row pitch arrive as zeros.
The fused partials must stay bit-identical to digitize_kernel + stats_i8_kernel (PYVB_I8_FUSED=0) across ring
wrap-around from one work item to the next, partial last K steps, empty row chunks and item counts that are not a
multiple of the grid."""
from math import gcd

import numpy as np
import pytest
import torch

from oracle.plate_oracle import synth_pca

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from pyvb_b200 import PlateEngine
    return PlateEngine


def _bits(t):
    return t.detach().contiguous().view(torch.int64).cpu().numpy()


def _stats(eng, X, q, fused, monkeypatch, pad_fill=None):
    """One Z step, then the INT8 statistics of its rows on a zeroed workspace (pad_fill: written into every MZ column
    from P + q to the end of the pitch first)."""
    monkeypatch.setenv("PYVB_I8_FUSED", "1" if fused else "0")
    e = eng(X, q, mode="B", algo="i8")
    assert e.use_i8_stats
    e.init_random(seed=17)
    e._ensure_stats()
    e.update_Z()
    if pad_fill is not None:
        P = q * (q + 1) // 2
        assert e.ldmz > P + q
        e.MZ[:, P + q:] = pad_fill
    e.ws.zero_()
    e._ensure_stats()
    torch.cuda.synchronize()
    assert getattr(e, "i8_stats_calls", 0) == 1
    assert (e.ZI is None) == fused
    return e


def _assert_same(a, b, what):
    assert np.array_equal(_bits(a.stats), _bits(b.stats)), what
    assert torch.equal(a.ws, b.ws), what
    assert a.i8_fallbacks() == b.i8_fallbacks(), what


def _ncols(q):
    return (q * (q + 1) // 2 + q + 31) & ~31


def _chunks(N, D, q):
    """(chunk count, rows per chunk) as stats_i8_nchunks / stats_i8_rows_per_chunk choose them (clusters of two)"""
    ncl = 74
    per = ((D + 127) // 128 + 1) // 2 * (_ncols(q) // 32)
    step = ncl // gcd(ncl, per)
    by_rows = max(N // 2048, 1)
    c = max((6 * ncl + per * step - 1) // (per * step), 1) * step
    if c > by_rows:
        c = by_rows // step * step if by_rows >= step else by_rows
    c = min(max(c, (N + (1 << 23) - 1) >> 23), 1024)
    r = max(((N + c - 1) // c + 63) // 64 * 64, 64)
    return c, r


@pytest.mark.parametrize("q", [16, 32, 64])
def test_pitch_past_zbar_is_never_read(eng, monkeypatch, q):
    """NaN or 1e300 in the MZ columns past P + q: the statistics do not change"""
    N, D = 4097, 256
    X = synth_pca(N, D, q, 0.25, seed=q)
    ref = _stats(eng, X, q, True, monkeypatch)
    two = _stats(eng, X, q, False, monkeypatch, pad_fill=float("nan"))
    _assert_same(ref, two, ("two-kernel", q))
    for fill in (float("nan"), 1e300):
        got = _stats(eng, X, q, True, monkeypatch, pad_fill=fill)
        _assert_same(got, ref, (fill, q))


@pytest.mark.parametrize("q", [16, 32, 64])
@pytest.mark.parametrize("N", [63, 65, 4097, 2 ** 16 + 1, 69633, 300001])
def test_fused_feed_bit_identical(eng, monkeypatch, N, q):
    D = 256
    X = synth_pca(N, D, q, 0.2, seed=N % 1000 + q)
    ef = _stats(eng, X, q, True, monkeypatch)
    eo = _stats(eng, X, q, False, monkeypatch)
    _assert_same(ef, eo, (N, q))


def test_shapes_cover_the_feed_cases():
    """the shapes above reach what the ring has to get right"""
    c, r = _chunks(69633, 256, 16)
    assert (c - 1) * r >= 69633                                  # an empty row chunk (its items have no K step)
    c, r = _chunks(2 ** 16 + 1, 256, 32)
    items = c * _ncols(32) // 32
    assert items > 148 and items % 148 != 0                     # items not a multiple of the grid
    assert (2 ** 16 + 1) % 64 != 0                               # a partial last K step
