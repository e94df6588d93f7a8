"""The converter warps of stats_i8_fused_kernel (oracle/i8_fused_oracle.py) leave byte for byte the SWIZZLE_64B image of the
ZI tile that digitize_kernel wrote and TMA delivered: every plane, column and row, tail rows past N and pad columns past
P + q included, with NaN / inf rows as zero digits; and every one of their shared-memory stores is free of bank conflicts."""
import numpy as np
import pytest

from oracle.i8_fused_oracle import converter_image, mz_pitch, ncols, tma_sw64_image, tri, zi_tile, CT, BKB


def _rows(N, q, seed):
    rng = np.random.RandomState(seed)
    MZ = np.zeros((N, mz_pitch(q)))
    nv = tri(q) + q
    MZ[:, :nv] = rng.randn(N, nv) * np.exp(rng.uniform(-20, 20, size=nv))[None, :]
    MZ[3, :] = np.nan                       # a non-PD row
    MZ[5, :nv:2] = np.inf
    MZ[7, :nv] = -MZ[7, :nv]
    with np.errstate(invalid="ignore"):
        m = np.nanmax(np.where(np.isfinite(MZ), np.abs(MZ), 0.0), axis=0)
    _, e = np.frexp(m)
    zscale = np.where(m > 0, np.ldexp(1.0, e), 1.0)[:ncols(q)]
    zscale = np.concatenate([zscale, np.ones(ncols(q) - len(zscale))])
    MZ[9, 0] = zscale[0]                    # |t| = 2^54 exactly: the largest value kept
    MZ[11, 1] = zscale[1] * (2.5 / 2 ** 54)   # a tie: rounds to even
    return MZ, zscale


@pytest.mark.parametrize("q", [16, 32, 64])
@pytest.mark.parametrize("N", [100, 128, 64 * 3 + 17])
def test_converter_image_is_the_tma_image_of_the_zi_tile(q, N):
    MZ, zscale = _rows(N, q, seed=q + N)
    nct = ncols(q) // CT
    for kb in range((N + BKB - 1) // BKB):
        for ct in sorted({0, nct // 2, nct - 1}):       # the last tile holds the pad columns
            img, banks = converter_image(MZ, N, q, zscale, kb, ct)
            want = tma_sw64_image(zi_tile(MZ, N, q, zscale, kb, ct))
            assert np.array_equal(img, want), (q, N, kb, ct, np.nonzero(img != want)[0][:8])
            for b in banks:
                assert len(set(b.tolist())) == 32, (q, kb, ct, b)


def test_zero_digits_past_n_and_past_the_valid_columns():
    q, N = 16, 70
    MZ, zscale = _rows(N, q, seed=1)
    t = zi_tile(MZ, N, q, zscale, 1, ncols(q) // CT - 1)
    assert not np.any(t[:, N - BKB:])                    # rows N ... 127 of step 1
    nv_last = tri(q) + q - (ncols(q) - CT)               # valid columns of the last tile
    cols = np.arange(7 * CT) % CT
    assert not np.any(t[cols >= nv_last])
    assert np.any(t[cols < nv_last])
