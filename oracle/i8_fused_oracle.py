"""TEST INFRASTRUCTURE (never the product): lane-level numpy restatement of the converter warps of stats_i8_fused_kernel
(pyvb_b200/csrc/kernels_i8.cu), which make the digit planes of the MZ rows in shared memory instead of reading them from
ZI.  The MMA reads the tile through a K-major SWIZZLE_64B descriptor, so the converters must leave exactly the bytes that
a TMA load of the ZI tile used to deliver.  Three restatements, compared by tests/test_oracle_i8_fused.py:

  zi_tile          the [224][64] tile ZI[kb][ct] that digitize_kernel writes, from the definition of the balanced base-256
                   digits (the recursion of pack_g_i8_kernel, not the BIAS trick the kernels use)
  tma_sw64_image   the 14 KB a SWIZZLE_64B TMA box of that tile lands as in shared memory
  converter_image  which lane of which converter warp stores which 32-bit word at which offset (the kernel's arithmetic,
                   __byte_perm included), plus the shared-memory bank of every lane of every store instruction
"""
import numpy as np

from oracle.i8_oracle import NPL, TWO54

CT, BKB = 32, 64                        # columns per tile, rows (K bytes) per step
TILE_B = NPL * CT * BKB                 # 14336
LANE = np.arange(32)
BIAS = np.uint64(0x0080808080808080)


def tri(i):
    return i * (i + 1) // 2


def mz_pitch(q):
    """pyvb_mz_pitch: [packed P | pad to 8 | zbar q] + 1 column, rounded to 4 (mod 8)"""
    p = ((tri(q) + 7) & ~7) + q + 1
    while p % 8 != 4:
        p += 1
    return p


def ncols(q):
    """stats_i8_ncols: the digit columns [packed | zbar], rounded to whole tiles of 32"""
    return (tri(q) + q + 31) & ~31


def _scaled(x, inv):
    """x * 2^54 / zscale_c, with NaN / inf (a non-PD row) -> 0, rounded to nearest even: the kernels' __double2ll_rn"""
    with np.errstate(invalid="ignore", over="ignore"):
        t = x * inv
        t = np.where(np.abs(t) <= TWO54, t, 0.0)
    return np.rint(t).astype(np.int64)


def zi_tile(MZ, N, q, zscale, kb, ct):
    """ZI[kb][ct] as [7 * 32][64] int8: plane p, tile column c, row n of the step at [p * 32 + c][n]; zero for rows >= N and
    columns >= P + q."""
    nvalid = tri(q) + q
    tile = np.zeros((NPL * CT, BKB), np.int8)
    for c in range(CT):
        col = ct * CT + c
        if col >= nvalid:
            continue
        rows = np.arange(kb * BKB, min((kb + 1) * BKB, N))
        vs = _scaled(MZ[rows, col], TWO54 / zscale[col]).tolist()
        for i, v in enumerate(vs):
            for p in range(NPL):
                d = ((v + 128) & 255) - 128          # balanced digit in [-128, 127]
                tile[p * CT + c, rows[i] - kb * BKB] = d
                v = (v - d) >> 8
            assert v == 0
    return tile


def tma_sw64_image(tile):
    """The bytes of a SWIZZLE_64B TMA box of `tile` (64-byte rows) in shared memory: the 16-byte chunk ch of row R goes to
    chunk ch ^ ((R >> 1) & 3)."""
    img = np.zeros(TILE_B, np.uint8)
    src = tile.view(np.uint8)
    for R in range(NPL * CT):
        for ch in range(4):
            dst = R * BKB + ((ch ^ ((R >> 1) & 3)) << 4)
            img[dst:dst + 16] = src[R, ch * 16:ch * 16 + 16]
    return img


def byte_perm(x, y, s):
    """__byte_perm(x, y, s) for uint32 arrays (selector nibbles 0-7, no sign replication)"""
    b = [(x >> (8 * i)) & 0xFF for i in range(4)] + [(y >> (8 * i)) & 0xFF for i in range(4)]
    out = np.zeros_like(x)
    for i in range(4):
        out |= b[(s >> (4 * i)) & 7] << (8 * i)
    return out


def converter_image(MZ, N, q, zscale, kb, ct):
    """The digit tile of step kb, column tile ct as the four converter warps of one group leave it in the ring stage.
    Returns (image, banks): banks[i] = the 32 lanes' banks of store instruction i.  Asserts that every byte is written
    exactly once."""
    nvalid = tri(q) + q
    ldmz = MZ.shape[1]
    img = np.zeros(TILE_B, np.uint8)
    hits = np.zeros(TILE_B, np.int32)
    banks = []
    c = ct * CT + LANE
    cv = c < nvalid
    inv = np.where(cv, TWO54 / zscale[np.minimum(c, len(zscale) - 1)], 0.0)
    rot = LANE >> 3                                        # lane group l / 8 starts at row quad l / 8
    for rq in range(4):                                    # warp cw of the group: rows 16 (cw % 4) ... + 15 of the step
        wbase = LANE * 64 + ((rq ^ ((LANE >> 1) & 3)) << 4)
        nb = kb * BKB + rq * 16
        xv = {}
        for g in range(4):
            for kk in range(4):
                n = nb + 4 * ((g + rot) & 3) + kk
                ok = cv & (n < N)
                xv[g, kk] = np.where(ok, MZ[np.minimum(n, N - 1), np.minimum(c, ldmz - 1)], 0.0)
        for g in range(4):
            qd = (g + rot) & 3
            lo, hi = [], []
            for kk in range(4):
                u = (_scaled(xv[g, kk], inv).astype(np.uint64) + BIAS) ^ BIAS
                lo.append(u & np.uint64(0xFFFFFFFF))
                hi.append(u >> np.uint64(32))
            for p in range(NPL):
                w = lo if p < 4 else hi
                sel = (p & 3) | ((4 + (p & 3)) << 4)
                word = byte_perm(byte_perm(w[0], w[1], sel), byte_perm(w[2], w[3], sel), 0x5410)
                off = p * (CT * BKB) + wbase + qd * 4
                banks.append((off >> 2) & 31)
                for lane in range(32):
                    o = int(off[lane])
                    img[o:o + 4] = np.frombuffer(np.uint32(word[lane]).tobytes(), np.uint8)
                    hits[o:o + 4] += 1
    assert np.all(hits == 1), "bytes written %s times" % sorted(set(hits.tolist()))
    return img, banks
