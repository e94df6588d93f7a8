// Exact FP64 mask contractions on the INT8 tensor cores (tcgen05.mma kind::i8, INT32 accumulators in TMEM).
//
// The dominant part of the Z step, qprec_n = P0 + tau * sum_d O_nd G_d (Multiplication.pass_up_m1_m2's
// m1 = tr(<w_i w_j^T> Lambda_n), nodes/node.py:213-227, with a masked precision), multiplies a 0/1 matrix with a small
// real one.  The mask is exact in int8; every column of G is written in fixed point with its own scale,
//     G[d][c] = scale_c 2^-54 sum_{t<7} digit_t[d][c] 256^t,     digit_t in [-128, 127]   (balanced base 256),
// scale_c = the power of two above max_d |G[d][c]|, so that |round(G / scale_c 2^54)| < 2^54 < 2^55 = the range of seven
// balanced digits, the scaling itself is exact, every entry is rounded once to scale_c 2^-55, and entries within a factor
// 4 of the column maximum are represented EXACTLY (finer than FP64 for the column's large entries).  Then
//     mask @ G = scale_c 2^-54 sum_t 256^t (mask @ digit_t)
// where every mask @ digit_t is an EXACT integer GEMM (|sum| <= 128 D << 2^31).  The seven INT32 results per output
// are recombined in the epilogue (two exact 64-bit integer halves, one FP64 FMA): no accumulation error at all, one
// rounding at the end -- at least as accurate as an FP64 accumulation, at the INT8 tensor rate instead of the FP64 one.
// The eta columns (both operands real) stay on the DMMA kernel (ZT<Q, true> in kernels_dmma.cu).
//
// Tiling: CTA tile = 128 rows x 32 output columns x 7 digit planes = one tcgen05.mma with N = 224 per 32-byte K step.
// The 128 x D mask block of a row tile stays RESIDENT in shared memory (D / 64 chunks of 128 x 64 bytes, each with its
// own full / empty mbarrier) while the CTA walks over the column tiles; only the 14 KB digit tiles stream through a
// ring of up to 8 stages (as many as fit next to the mask block; they come from L2: the digit array is a few MB).  TMEM holds two accumulators (2 x 256 columns)
// so that the epilogue of one tile overlaps the MMAs of the next.  Warp 0: TMA producer, warp 1: MMA issuer, warps
// 2-9: epilogue (two warps per TMEM lane quarter, 16 columns each; one TMA tensor store per warp and tile).  Operands
// are K-major TMA tiles with 64-byte rows (SWIZZLE_64B), tile-major in global memory so that every box is one
// contiguous block.  K3-i8 (the mask-type statistics) further down uses the same machinery with the roles turned.
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>

#include "common.cuh"
#include "kernels.h"
#include "ptx.cuh"
#include "umma.cuh"

namespace pyvb {

namespace {

__host__ __device__ constexpr int i_tri(int i) { return i * (i + 1) / 2; }
__host__ __device__ constexpr int i_nc8(int q) { return (i_tri(q) + 31) & ~31; }          // packed columns rounded to 32
constexpr int NPL = 7;                                                                    // digit planes
constexpr int BM = 128, BKB = 64, ST = 16, CT = 32;      // rows per tile, K bytes per chunk, max digit stages, columns per tile
constexpr int A_B = BM * BKB, B_B = NPL * CT * BKB;      // 8192, 14336
constexpr int NTHR = 10 * 32;

// smallest power of two > m (1 for m = 0, NaN, inf): a fixed-point scale whose reciprocal multiplies exactly
__device__ __forceinline__ double pow2_above(double m) {
    if (!(m > 0.0 && m < 1e300)) return 1.0;
    int e;
    frexp(m, &e);                                        // m = f 2^e, f in [0.5, 1)
    return ldexp(1.0, e);
}

// ------------------------------------------------------------------ operand preparation
// mask[rb][kb][128 rows][64 bytes] (rb = n / 128, kb = d / 64): every TMA box of the kernel is one contiguous 8 KB block
// (64-byte rows at a stride of D bytes were half cache lines: twice the L2 requests per byte); rows >= N are zero
__global__ void __launch_bounds__(256)
prepare_mask_i8_kernel(long long N, int D, const double *__restrict__ X, long long ldx, signed char *__restrict__ mask) {
    const long long npad = (N + BM - 1) / BM * BM;
    const int nk = D / BKB;
    const long long total = npad * (long long)(D / 4);
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long n = e / (D / 4);
        const int d = (int)(e - n * (D / 4)) * 4;
        char4 m = make_char4(0, 0, 0, 0);
        if (n < N) {
            const double2 a = *reinterpret_cast<const double2 *>(X + n * ldx + d);
            const double2 b = *reinterpret_cast<const double2 *>(X + n * ldx + d + 2);
            m.x = (a.x == a.x) ? 1 : 0;
            m.y = (a.y == a.y) ? 1 : 0;
            m.z = (b.x == b.x) ? 1 : 0;
            m.w = (b.y == b.y) ? 1 : 0;
        }
        const size_t dst = (((size_t)(n / BM) * nk + d / BKB) * BM + (size_t)(n % BM)) * BKB + (d % BKB);
        *reinterpret_cast<char4 *>(mask + dst) = m;
    }
}

// one CTA per output column c: scale_c = max_d |G[d][c]|, then the seven balanced base-256 digits of
// round(G / scale_c * 2^54).  G[d][c] is column c of the packed Gw row d (pack_gw_kernel: the same w_i w_j (+ v_i) bits, or
// tau_d times them with per-dimension noise).  GI[kb][ct][plane][c % 32][64] (int8), kb = d / 64, ct = c / 32: the B tile of (kb, ct) is
// one contiguous [224 rows][64 bytes] block.
__global__ void __launch_bounds__(256)
pack_g_i8_kernel(int D, int q, const double *__restrict__ Gw, int ldg, signed char *__restrict__ GI,
                 double *__restrict__ gscale, double *__restrict__ gl) {
    __shared__ double sh[33];
    const int P = i_tri(q);
    const int c = blockIdx.x;
    if (c == 0 && threadIdx.x == 0) gl[PYVB_GL_I8BAD] = 0.0;           // guard counter of the Z step that follows (K2 adds to it)
    double mx = 0.0;
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        const double g = (c < P) ? Gw[(size_t)d * ldg + c] : 0.0;
        mx = fmax(mx, fabs(g));
    }
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x < 32) {
        double t = (threadIdx.x < (blockDim.x >> 5)) ? sh[threadIdx.x] : 0.0;
        for (int o = 16; o > 0; o >>= 1) t = fmax(t, __shfl_xor_sync(0xffffffffu, t, o));
        if (threadIdx.x == 0) sh[32] = t;
    }
    __syncthreads();
    // the scale is the power of two above the column maximum: g * (2^54 / scale) is then an EXACT scaling, so every entry is
    // rounded once, to scale 2^-55, and entries within a factor 4 of the column maximum are represented exactly
    const double scale = pow2_above(sh[32]);
    if (threadIdx.x == 0) gscale[c] = scale;
    const double inv = 18014398509481984.0 / scale;                     // 2^54 / scale
    const int nct = gridDim.x / CT;
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        const double g = (c < P) ? Gw[(size_t)d * ldg + c] : 0.0;
        long long v = __double2ll_rn(g * inv);
#pragma unroll
        for (int t = 0; t < NPL; ++t) {
            const long long dg = ((v + 128) & 255) - 128;               // balanced digit in [-128, 127]
            GI[((((size_t)(d / BKB) * nct + (c >> 5)) * NPL + t) * CT + (c & 31)) * BKB + (d % BKB)] = (signed char)dg;
            v = (v - dg) >> 8;
        }
    }
}

// ------------------------------------------------------------------ tensor maps (uint8)
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode_i8() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)ptr;
    }
    return fn;
}
// [planes][rows][cols] bytes, row pitch = cols
cudaError_t make_map_u8_3d(CUtensorMap *m, const void *base, uint64_t cols, uint64_t rows, uint64_t planes,
                           uint32_t box_cols, uint32_t box_rows) {
    EncodeTiledFn enc = get_encode_i8();
    if (!enc) return cudaErrorNotSupported;
    cuuint64_t dims[3] = {cols, rows, planes};
    cuuint64_t strides[2] = {cols, cols * rows};
    cuuint32_t box[3] = {box_cols, box_rows, 1};
    cuuint32_t es[3] = {1, 1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void *>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}
__device__ __forceinline__ void tma_load_3d_i8(void *dst_smem, const void *tmap, int c0, int c1, int c2, uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
            smem_u32(dst_smem)),
        "l"(tmap), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
        : "memory");
}
// the same box delivered to the same shared-memory offset of every CTA in `mask` (and complete_tx on each CTA's barrier)
__device__ __forceinline__ void tma_load_3d_i8_mc(void *dst_smem, const void *tmap, int c0, int c1, int c2, uint64_t *bar,
                                                  uint16_t mask) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%2, %3, "
        "%4}], [%5], %6;" ::"r"(smem_u32(dst_smem)),
        "l"(tmap), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar)), "h"(mask)
        : "memory");
}
// CTA pair: the box lands in THIS CTA's shared memory, the transaction bytes are signalled on a barrier of the LEADER CTA
// (`bar_cluster` = shared::cluster address, umma::map_to_cta)
__device__ __forceinline__ void tma_load_3d_i8_pair(void *dst_smem, const void *tmap, int c0, int c1, int c2, uint32_t bar_cluster) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
            smem_u32(dst_smem)),
        "l"(tmap), "r"(c0), "r"(c1), "r"(c2), "r"(bar_cluster)
        : "memory");
}
// tcgen05.commit that arrives on the barrier at this offset in every CTA of `mask`
__device__ __forceinline__ void mma_commit_mc(uint64_t *bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"(mask)
                 : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "r"(taddr)
                 : "memory");
}
// exact int32 -> double without the conversion unit: 2^52 + 2^31 + a has the integer in its low mantissa word
__device__ __forceinline__ double i2d(int a) {
    return __hiloint2double(0x43300000, (int)((unsigned)a ^ 0x80000000u)) - 4503601774854144.0;
}
// sum_t 256^t a_t for seven INT32 accumulators (|a_t| <= 2^18): two exact 64-bit integer halves (multiply-add-wide),
// each converted through the 2^52 + 2^51 bit pattern (exact for |x| < 2^51), then ONE rounding in the final FMA
__device__ __forceinline__ double combine7(const int (&a)[NPL]) {
    const long long lo = (long long)a[3] * 16777216LL + ((long long)a[2] * 65536LL + ((long long)a[1] * 256LL + (long long)a[0]));
    const long long hi = (long long)a[6] * 65536LL + ((long long)a[5] * 256LL + (long long)a[4]);
    const double dlo = __longlong_as_double(0x4338000000000000LL + lo) - 6755399441055744.0;
    const double dhi = __longlong_as_double(0x4338000000000000LL + hi) - 6755399441055744.0;
    return fma(dhi, 4294967296.0, dlo);
}
// 2-D tiled TMA store shared -> global (rows / columns outside the tensor are clipped)
__device__ __forceinline__ void tma_store_2d(const void *tmap, int c0, int c1, const void *src_smem) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%1, %2}], [%3];" ::"l"(tmap), "r"(c0), "r"(c1),
                 "r"(smem_u32(src_smem))
                 : "memory");
}

struct I8Geom {
    int P, PP, NC8, NCT;
    __host__ __device__ explicit I8Geom(int q) {
        P = i_tri(q);
        PP = (P + 7) & ~7;
        NC8 = i_nc8(q);
        NCT = NC8 / CT;
    }
};
constexpr int OUT_B = 8 * 32 * 16 * 8;                  // epilogue staging: 8 warps x (32 rows x 16 columns) doubles
// hstage: the epilogue stages (and stores) 8 columns at a time: half the staging memory, one more digit stage at D = 1024
// pair: cta_group::2 -- a CTA holds HALF of every digit tile (7 KB per stage)
// adbl: TWO mask blocks (the next row block's is fetched while the current one is multiplied)
size_t i8_smem_bytes(int D, int q, int nst, int hstage, int pair = 0, int adbl = 0) {
    const I8Geom g(q);
    const int nk = D / BKB * (adbl ? 2 : 1);
    return 1024 + (size_t)nk * A_B + (size_t)nst * (pair ? B_B / 2 : B_B) + (hstage ? OUT_B / 2 : OUT_B) + (size_t)(2 * g.NC8) * 8 +
           (size_t)(2 * nk + 2 * nst + 4) * 8 + 16;
}
int i8_stages(int D, int q, int hstage, int pair = 0, int adbl = 0) {  // digit-tile stages that fit next to the resident mask block(s)
    for (int nst = pair ? ST : ST / 2; nst >= 2; --nst)
        if (i8_smem_bytes(D, q, nst, hstage, pair, adbl) <= 227 * 1024) return nst;
    return 0;
}
int i8_hstage(int D, int q) {                            // half staging only where it buys a stage and stages are scarce
    const int full = i8_stages(D, q, 0);
    return (full < 6 && i8_stages(D, q, 1) > full) ? 1 : 0;
}

// ------------------------------------------------------------------ K1-i8: qprec columns of the MZ rows
// CL > 1: clusters of CL CTAs (consecutive row blocks) share every digit tile: each CTA fetches 1 / CL of it and the
// copy is multicast to all of them (the digit tiles come from L2 and their traffic, not the MMAs, bounds the kernel);
// a stage is released by the MMA commits of ALL the CTAs (multicast tcgen05.commit on every CTA's `empty` barrier).
// PAIR (with CL = 2): tcgen05.mma.cta_group::2 -- the CTA pair is ONE 256-row MMA; a CTA holds its own 128 x D mask block and
// HALF of every digit tile (7 KB instead of 14: twice the ring depth next to the resident mask block), the leader CTA issues
// the MMAs for both, every CTA drains its own 128 TMEM lanes.  No multicast: each CTA fetches only its half.
template <int CL, bool PAIR = false>
__global__ void __launch_bounds__(NTHR, 1)
zstep_i8_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmO8, long long N, int D, int q,
                const double *__restrict__ P0, const double *__restrict__ gscale, const double *__restrict__ gl, int nrb,
                int nst, int hstage, int adbl, long long *prof, int ks) {
    const I8Geom G(q);
    long long w0 = 0, w1 = 0, w2 = 0;                          // PYVB_I8_PROF: clocks spent waiting, per role
    const long long tstart = clock64();
#define PROF_WAIT(acc, stmt)                    \
    do {                                        \
        if (prof) {                             \
            const long long t_ = clock64();     \
            stmt;                               \
            acc += clock64() - t_;              \
        } else {                                \
            stmt;                               \
        }                                       \
    } while (0)
    extern __shared__ unsigned char smem_dyn[];
    unsigned char *smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    static_assert(!PAIR || CL == 2, "a CTA pair is a cluster of two");
    constexpr int BSZ = PAIR ? B_B / 2 : B_B;                                  // bytes of a digit stage in THIS CTA
    const int nk = D / BKB;
    // adbl: two mask blocks -- the block of row block rl + 1 is fetched while row block rl is multiplied (without it every
    // row block starts with the latency of its 128 x D mask load: a quarter of the kernel at D = 256)
    const int nab = adbl ? 2 : 1;
    unsigned char *a_base = smem;                                              // [nab][nk][128 x 64 B] resident mask block(s)
    // ks: K chunks (digit tiles) per ring stage.  One tile per stage makes the producer's and the issuer's per-stage latency
    // (barrier round trip, TMA / MMA issue, commit: ~300 clocks each) as long as the two MMAs of a tile (257 clocks)
    const int SB = ks * BSZ;                                                   // bytes of a ring stage in THIS CTA
    unsigned char *b_base = smem + (size_t)nab * nk * A_B;                     // [nst][ks][224 (PAIR: 112) x 64 B] digit tiles
    unsigned char *o_base = b_base + (size_t)nst * SB;                         // [8 warps][32 rows x 128 B] output staging (swizzled)
    double *p0v = reinterpret_cast<double *>(o_base + (hstage ? OUT_B / 2 : OUT_B));   // [NC8]: packed P0, zero pad
    double *fcol = p0v + G.NC8;                                                // [NC8]: tau * scale_c * 2^-54
    uint64_t *afull = reinterpret_cast<uint64_t *>(fcol + G.NC8);              // [nab][nk]
    uint64_t *aempty = afull + nab * nk;                                       // [nab][nk]
    uint64_t *full = aempty + nab * nk;                                        // [nst]
    uint64_t *empty = full + nst;                                              // [nst]
    uint64_t *tfull = empty + nst;                                             // [2]
    uint64_t *tempty = tfull + 2;                                              // [2]
    uint32_t *tbase = reinterpret_cast<uint32_t *>(tempty + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const double tau = gl[PYVB_GL_TAU];
    const int crank = (CL > 1) ? (int)cluster_ctarank() : 0;
    // every CTA of a cluster runs the same number of row blocks (a CTA past the last block works on zero-filled rows)
    const int first = (int)blockIdx.x - crank;
    const int niter = (first < nrb) ? (nrb - first + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    int niter_mma = niter;                                     // (PAIR: zero in the non-leader CTA)
    constexpr uint16_t CMASK = (uint16_t)((1u << CL) - 1u);
    // every cluster walks the (column tile, K chunk) grid from its own starting point: 148 CTAs stepping through the
    // same few MB of digit tiles in lockstep would all hit the same L2 lines at the same time
    const int rot = (int)(blockIdx.x / CL) % (G.NCT * nk);
    const int ct0 = rot / nk, kb0 = rot % nk;

    for (int p = tid; p < G.NC8; p += NTHR) {
        double v = 0.0;
        if (p < G.P) {
            int i, j;
            unpack_p(p, i, j);
            v = P0[i * q + j];
        }
        p0v[p] = v;
    }
    for (int c = tid; c < G.NC8; c += NTHR) fcol[c] = tau * gscale[c] * 5.5511151231257827e-17;   // 2^-54
    if (tid == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        tma_prefetch_desc(&tmO);
        tma_prefetch_desc(&tmO8);
        for (int k = 0; k < nab * nk; ++k) {
            mbar_init(&afull[k], 1);
            mbar_init(&aempty[k], 1);
        }
        for (int s = 0; s < nst; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], PAIR ? 1 : CL);                   // PAIR: one multicast commit of the leader per use
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&tfull[b], 1);
            mbar_init(&tempty[b], PAIR ? 16 : 8);                  // PAIR: the epilogue warps of BOTH CTAs release the leader's buffer
        }
        mbar_fence_init();
    }
    if (warp == 1) {
        if (PAIR) umma::tmem_alloc2(tbase, 512);
        else umma::tmem_alloc(tbase, 512);
    }
    umma::fence_before_sync();
    __syncthreads();
    if (CL > 1) cluster_sync_all();                            // the peers' barriers are initialised before anyone signals them
    umma::fence_after_sync();
    const uint32_t tmem = *tbase;

    if (warp == 0) {
        // ===================== TMA producer (whole warp, one elected lane issues) =====================
        const bool leader = elect_one();
        const uint32_t afull_l = PAIR ? umma::map_to_cta(afull, 0) : 0u, full_l = PAIR ? umma::map_to_cta(full, 0) : 0u;
        int s = 0;
        uint32_t ph = 0;
        for (int rl = 0; rl < niter; ++rl) {
            for (int ci = 0; ci < G.NCT; ++ci) {
                const int ct = (ci + ct0 < G.NCT) ? ci + ct0 : ci + ct0 - G.NCT;
                for (int ki = 0; ki < nk; ki += ks) {
                    if (ci == 0) {
                        for (int h = 0; h < ks; ++h) {
                            const int kb = (ki + h + kb0 < nk) ? ki + h + kb0 : ki + h + kb0 - nk;
                            // mask chunk kb of row block r into buffer r % nab, once that buffer's previous user (row block r - nab)
                            // has been consumed by its last column tile.  Two buffers: row block rl + 1 is fetched NOW, a whole
                            // row block ahead of its use (and row block 0 with it).
                            for (int r = (nab == 2 && rl > 0) ? rl + 1 : rl; r <= rl + nab - 1 && r < niter; ++r) {
                                const int ab = (r & (nab - 1)) * nk + kb;
                                const int rbr = (int)blockIdx.x + r * (int)gridDim.x;
                                PROF_WAIT(w1, umma::mbar_wait_bounded(&aempty[ab], (uint32_t)(((r / nab) & 1) ^ 1)));
                                if (leader) {
                                    if (PAIR) {    // both CTAs' chunks complete on the LEADER's barrier (armed by the leader for both)
                                        if (crank == 0) mbar_arrive_expect_tx(&afull[ab], (uint32_t)(2 * A_B));
                                        tma_load_3d_i8_pair(a_base + (size_t)ab * A_B, &tmA, 0, (rbr * nk + kb) * BM, 0, afull_l + (uint32_t)ab * 8u);
                                    } else {
                                        mbar_arrive_expect_tx(&afull[ab], (uint32_t)A_B);
                                        tma_load_3d_i8(a_base + (size_t)ab * A_B, &tmA, 0, (rbr * nk + kb) * BM, 0, &afull[ab]);   // past the end: zero fill
                                    }
                                }
                            }
                        }
                    }
                    PROF_WAIT(w0, umma::mbar_wait_bounded(&empty[s], ph ^ 1));
                    if (leader) {
                        if (PAIR) {
                            if (crank == 0) mbar_arrive_expect_tx(&full[s], (uint32_t)(ks * B_B));
                        } else {
                            mbar_arrive_expect_tx(&full[s], (uint32_t)(ks * B_B));
                        }
                        for (int h = 0; h < ks; ++h) {
                            const int kb = (ki + h + kb0 < nk) ? ki + h + kb0 : ki + h + kb0 - nk;
                            unsigned char *dst = b_base + s * SB + h * BSZ;
                            if (PAIR) {            // this CTA's half of the tile (rows crank * 112 ...) into its own stage
                                tma_load_3d_i8_pair(dst, &tmB, 0, (kb * G.NCT + ct) * (NPL * CT) + crank * (NPL * CT / 2), 0,
                                                    full_l + (uint32_t)s * 8u);
                            } else if (CL == 1) {
                                tma_load_3d_i8(dst, &tmB, 0, (kb * G.NCT + ct) * (NPL * CT), 0, &full[s]);   // 7 planes x 32 columns
                            } else {                                                                           // this CTA's slice, to everybody
                                tma_load_3d_i8_mc(dst + crank * (B_B / CL), &tmB, 0,
                                                  (kb * G.NCT + ct) * (NPL * CT) + crank * (NPL * CT / CL), 0, &full[s], CMASK);
                            }
                        }
                    }
                    __syncwarp();
                    if (++s == nst) {
                        s = 0;
                        ph ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (whole warp, one elected lane issues; PAIR: the leader CTA alone) ============
        const bool leader = elect_one() && (!PAIR || crank == 0);
        if (PAIR && crank != 0) niter_mma = 0;
        const uint32_t idesc = umma::idesc_s8_s32(PAIR ? 2 * BM : BM, NPL * CT);
        // descriptors: the start-address field counts 16-byte units, so stage / chunk / K-step offsets are plain adds
        const uint64_t adesc0 = umma::desc_kmajor_sw64(smem_u32(a_base), 0), bdesc0 = umma::desc_kmajor_sw64(smem_u32(b_base), 0);
        int s = 0, tl = 0;
        uint32_t ph = 0;
        for (int rl = 0; rl < niter_mma; ++rl) {
            for (int ci = 0; ci < G.NCT; ++ci, ++tl) {
                const int buf = tl & 1;
                PROF_WAIT(w1, umma::mbar_wait_bounded(&tempty[buf], (uint32_t)(((tl >> 1) & 1) ^ 1)));
                umma::fence_after_sync();
                const uint32_t dacc = tmem + (uint32_t)(buf * 256);
                for (int ki = 0; ki < nk; ki += ks) {
                    if (ci == 0)
                        for (int h = 0; h < ks; ++h) {
                            const int kb = (ki + h + kb0 < nk) ? ki + h + kb0 : ki + h + kb0 - nk;
                            const int ab = (rl & (nab - 1)) * nk + kb;       // mask chunk kb of this row block's buffer
                            PROF_WAIT(w2, umma::mbar_wait_bounded(&afull[ab], (uint32_t)((rl / nab) & 1)));
                        }
                    PROF_WAIT(w0, umma::mbar_wait_bounded(&full[s], ph));
                    umma::fence_after_sync();
                    if (leader) {
                        for (int h = 0; h < ks; ++h) {
                            const int kb = (ki + h + kb0 < nk) ? ki + h + kb0 : ki + h + kb0 - nk;
                            const int ab = (rl & (nab - 1)) * nk + kb;
                            const uint64_t ad = adesc0 + (uint64_t)(ab * (A_B >> 4)), bd = bdesc0 + (uint64_t)((s * SB + h * BSZ) >> 4);
                            if (PAIR) {
                                umma::mma_i8_pair(dacc, ad, bd, idesc, (ki + h) ? 1u : 0u);
                                umma::mma_i8_pair(dacc, ad + 2, bd + 2, idesc, 1u);
                                if (ci == G.NCT - 1) umma::mma_commit_pair(&aempty[ab]);
                            } else {
                                umma::mma_i8(dacc, ad, bd, idesc, (ki + h) ? 1u : 0u);
                                umma::mma_i8(dacc, ad + 2, bd + 2, idesc, 1u);
                                if (ci == G.NCT - 1) umma::mma_commit(&aempty[ab]);
                            }
                        }
                        if (PAIR) umma::mma_commit_pair(&empty[s]);                      // frees the stage in both CTAs
                        else if (CL == 1) umma::mma_commit(&empty[s]);
                        else mma_commit_mc(&empty[s], CMASK);
                    }
                    __syncwarp();
                    if (++s == nst) {
                        s = 0;
                        ph ^= 1;
                    }
                }
                if (leader) {
                    if (PAIR) umma::mma_commit_pair(&tfull[buf]);            // the accumulators of both CTAs are complete
                    else umma::mma_commit(&tfull[buf]);
                }
                __syncwarp();
            }
        }
    } else {
        // ===================== epilogue: 7 INT32 planes -> FP64 -> P0 + f_c * v -> MZ row ========
        const int wq = warp & 3;                               // TMEM lane quarter this warp may access
        const int half = (warp - 2) >> 2;                      // which 16 of the tile's 32 columns
        const uint32_t tempty_l = PAIR ? umma::map_to_cta(tempty, 0) : 0u;
        int tl = 0;
        for (int rl = 0; rl < niter; ++rl) {
            const long long rowbase = ((long long)blockIdx.x + (long long)rl * gridDim.x) * BM + wq * 32;
            for (int ci = 0; ci < G.NCT; ++ci, ++tl) {
                const int ct = (ci + ct0 < G.NCT) ? ci + ct0 : ci + ct0 - G.NCT;
                const int c0 = ct * CT + half * 16;
                const int buf = tl & 1;
                PROF_WAIT(w0, umma::mbar_wait_bounded(&tfull[buf], (uint32_t)((tl >> 1) & 1)));
                umma::fence_after_sync();
                const uint32_t taddr = tmem + (uint32_t)(buf * 256 + half * 16) + ((uint32_t)(wq * 32) << 16);
                uint32_t a[2][NPL][8];
#pragma unroll
                for (int ch = 0; ch < 2; ++ch)
#pragma unroll
                    for (int p = 0; p < NPL; ++p) tmem_ld8(taddr + (uint32_t)(p * CT + ch * 8), a[ch][p]);
                umma::tmem_ld_wait();
                umma::fence_before_sync();
                __syncwarp();
                if (lane == 0) {                                // the accumulator buffer is free again
                    if (PAIR) umma::mbar_arrive_cluster(tempty_l + (uint32_t)buf * 8u);   // (the leader's barrier counts both CTAs)
                    else mbar_arrive(&tempty[buf]);
                }
                // lane = row: 16 outputs per lane, staged in this warp's [32 rows][128 B] tile (16-byte chunks XOR-swizzled
                // with the row, the SWIZZLE_128B pattern of the store map: conflict-free 16-byte shared-memory stores)
                // and written by ONE TMA tensor store (rows >= N and columns >= PP are clipped by the map).  Per-lane
                // 16-byte global stores touched 32 rows per instruction and a shuffle transposition cost ~25 instructions
                // per output: both made the epilogue, not the MMAs, the limit.
                if (!hstage) {
                    unsigned char *stage = o_base + (warp - 2) * 4096;
                    if (lane == 0) PROF_WAIT(w1, bulk_wait_read_all());   // the previous store of this warp has read the tile
                    __syncwarp();
#pragma unroll
                    for (int ch = 0; ch < 2; ++ch) {
                        if (c0 + ch * 8 >= G.PP) continue;      // a chunk of 8 columns is entirely in or out
#pragma unroll
                        for (int k = 0; k < 8; k += 2) {
                            int d0[NPL], d1[NPL];
#pragma unroll
                            for (int p = 0; p < NPL; ++p) {
                                d0[p] = (int)a[ch][p][k];
                                d1[p] = (int)a[ch][p][k + 1];
                            }
                            const int c = c0 + ch * 8 + k;
                            const double2 f2 = *reinterpret_cast<const double2 *>(&fcol[c]);
                            const double2 p2 = *reinterpret_cast<const double2 *>(&p0v[c]);
                            double2 o;
                            o.x = fma(f2.x, combine7(d0), p2.x);
                            o.y = fma(f2.y, combine7(d1), p2.y);
                            const int chunk = ch * 4 + (k >> 1);
                            *reinterpret_cast<double2 *>(stage + lane * 128 + ((chunk ^ (lane & 7)) << 4)) = o;
                        }
                    }
                    fence_async_smem();
                    __syncwarp();
                    if (lane == 0 && c0 < G.PP) {
                        tma_store_2d(&tmO, c0, (int)rowbase, stage);
                        bulk_commit();
                    }
                } else {
                    // half staging: 8 columns (64-byte rows, SWIZZLE_64B pattern: chunk ^ ((row >> 1) & 3)) per store
                    unsigned char *stage = o_base + (warp - 2) * 2048;
#pragma unroll
                    for (int ch = 0; ch < 2; ++ch) {
                        if (c0 + ch * 8 >= G.PP) continue;      // warp-uniform
                        if (lane == 0) PROF_WAIT(w1, bulk_wait_read_all());
                        __syncwarp();
#pragma unroll
                        for (int k = 0; k < 8; k += 2) {
                            int d0[NPL], d1[NPL];
#pragma unroll
                            for (int p = 0; p < NPL; ++p) {
                                d0[p] = (int)a[ch][p][k];
                                d1[p] = (int)a[ch][p][k + 1];
                            }
                            const int c = c0 + ch * 8 + k;
                            const double2 f2 = *reinterpret_cast<const double2 *>(&fcol[c]);
                            const double2 p2 = *reinterpret_cast<const double2 *>(&p0v[c]);
                            double2 o;
                            o.x = fma(f2.x, combine7(d0), p2.x);
                            o.y = fma(f2.y, combine7(d1), p2.y);
                            *reinterpret_cast<double2 *>(stage + lane * 64 + ((((k >> 1) ^ ((lane >> 1) & 3))) << 4)) = o;
                        }
                        fence_async_smem();
                        __syncwarp();
                        if (lane == 0) {
                            tma_store_2d(&tmO8, c0 + ch * 8, (int)rowbase, stage);
                            bulk_commit();
                        }
                    }
                }
            }
        }
        if (lane == 0) bulk_wait_read_all();
    }
#undef PROF_WAIT
    if (prof && lane == 0 && warp < 3) {    // (all lanes of a role wait together: lane 0's clocks are the role's)   // [producer: empty, aempty, -][MMA: full, tempty, afull][epilogue warp 2: tfull, store-read, -][total]
        long long *o = prof + (size_t)blockIdx.x * 10 + warp * 3;
        o[0] = w0;
        o[1] = w1;
        o[2] = w2;
        if (warp == 0) prof[(size_t)blockIdx.x * 10 + 9] = clock64() - tstart;
    }
    umma::fence_before_sync();
    __syncthreads();
    if (CL > 1) cluster_sync_all();        // no CTA leaves while a peer may still multicast into it or signal its barriers
    if (warp == 1) {
        if (PAIR) umma::tmem_dealloc2(tmem, 512);
        else umma::tmem_dealloc(tmem, 512);
    }
}

// launch with a cluster dimension (cl = 1: plain launch)
template <typename... KArgs, typename... Args>
cudaError_t launch_cluster(void (*kern)(KArgs...), int grid, int block, size_t smem, int cl, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid, 1, 1);
    cfg.blockDim = dim3((unsigned)block, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)cl;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = cl > 1 ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}
constexpr int I8_CL = 2;                    // CTAs per cluster of K1-i8 (1 for tiny problems) and K3-i8

// =====================================================================================================================
// K3-i8: the mask-type sufficient statistics  T1 = O^T vec<zz^T>,  Bst = O^T Zbar  (hstack, nodes/nodes_todo.py:50-61)
// on the INT8 tensor cores.  Same idea as K1-i8 with the roles turned: the contraction index is the ROW n, so both
// operands are needed "n contiguous":
//   maskT [n / 64][D][64]                int8, the transposed mask (static, prepared once per data set)
//   ZI    [n / 64][ct][plane][c % 32][64] int8, the seven balanced base-256 digit planes of the MZ columns
//                                        (tile-major: every TMA box is one contiguous 8 KB / 14 KB block -- with a
//                                        plain [column][n] layout a box touched 224 different 2 MB pages at N = 1.25M)
//                                        c in [0, P + q) = [<zz^T> packed | zbar], rewritten after every Z step with one
//                                        fixed-point scale per column, zscale_c = max_n |MZ[n][c]| (colmax pass)
// Work item = (block of 128 data dimensions, column tile of 32, row chunk): one TMEM accumulator (224 columns) summed
// over the whole chunk, then recombined to FP64 and written to the chunk's partial-sum buffer (the deterministic
// second stage, stats_reduce_kernel, adds the chunks).  Items are dealt round-robin to 148 persistent CTAs, chunk-major,
// so that the CTAs running at the same time share their operand tiles through L2.
constexpr int SST = 9;                                   // stages of the K3-i8 ring (22 KB each)
constexpr int SST_PAIR = 13;                             // ... with cta_group::2 (15 KB each: half of the digit tile per CTA)
constexpr int CM_BLOCKS = 148 * 4;                       // partial column maxima

// The partials K2 would have left for a block of rows -- [column sums (ldmz - 4) | sum 0.5/logdet, sum logdet, rows, 0 |
// column maxima of |.| (ldmz - 4)] -- in ONE pass over the MZ rows, for the cases where K2 leaves none (q = 64, or rows
// written from outside the kernels): replaces three passes (column sums, per-row scalars, column maxima).  A warp takes
// a slice of 32 x 17 columns and every (8 / slices)-th row; the warps of a slice are combined in a fixed order.
constexpr int MZP_KPL = 17;
__global__ void __launch_bounds__(256)
mzpart_kernel(long long N, int ldmz, int orow, const double *__restrict__ MZ, const double *__restrict__ logdet,
              double *__restrict__ part, long long rows_per_blk) {
    extern __shared__ double mz_sh[];                       // [sums ldmz | maxima ldmz | 4 scalars]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int kw = 2 * orow + 4;                            // orow = gw_woff(q) + q: the used columns of a row
    const int ns = (ldmz + 32 * MZP_KPL - 1) / (32 * MZP_KPL);         // column slices: 1, 2 or 4
    const int slice = warp % ns, rg = warp / ns, nrg = 8 / ns;
    const long long r0 = (long long)blockIdx.x * rows_per_blk;
    long long r1 = r0 + rows_per_blk;
    if (r1 > N) r1 = N;
    double sm[MZP_KPL], mx[MZP_KPL], s_qld = 0.0, s_ld = 0.0, s_n = 0.0;
#pragma unroll
    for (int k = 0; k < MZP_KPL; ++k) sm[k] = mx[k] = 0.0;
    const int cbase = slice * 32 * MZP_KPL + lane;
    for (long long n = r0 + rg; n < r1; n += nrg) {
        const double *row = MZ + n * ldmz;
#pragma unroll
        for (int k = 0; k < MZP_KPL; ++k) {
            const int c = cbase + 32 * k;
            if (c < ldmz) {
                const double v = row[c];
                sm[k] += v;
                mx[k] = fmax(mx[k], fabs(v));
            }
        }
        if (slice == 0 && lane == 0) {
            const double ld = logdet[n];
            s_qld += 0.5 / ld;
            s_ld += ld;
            s_n += 1.0;
        }
    }
    double *ssum = mz_sh, *smax = mz_sh + ldmz, *ssc = mz_sh + 2 * ldmz;
    for (int w = 0; w < 8; ++w) {                           // fixed order: deterministic sums
        if (warp == w) {
#pragma unroll
            for (int k = 0; k < MZP_KPL; ++k) {
                const int c = cbase + 32 * k;
                if (c < ldmz) {
                    ssum[c] = (rg == 0) ? sm[k] : ssum[c] + sm[k];
                    smax[c] = (rg == 0) ? mx[k] : fmax(smax[c], mx[k]);
                }
            }
            if (slice == 0 && lane == 0) {
                ssc[0] = (rg == 0) ? s_qld : ssc[0] + s_qld;
                ssc[1] = (rg == 0) ? s_ld : ssc[1] + s_ld;
                ssc[2] = (rg == 0) ? s_n : ssc[2] + s_n;
            }
        }
        __syncthreads();
    }
    double *out = part + (size_t)blockIdx.x * kw;
    for (int c = threadIdx.x; c < orow; c += 256) {
        out[c] = ssum[c];
        out[orow + 4 + c] = smax[c];
    }
    if (threadIdx.x < 4) out[orow + threadIdx.x] = (threadIdx.x < 3) ? ssc[threadIdx.x] : 0.0;
}

// one warp per column: max over the row-block partials
__global__ void __launch_bounds__(256)
colmax_reduce_kernel(int ncols, int nvalid, int ldmz, const double *__restrict__ pm, int nblk, double *__restrict__ zscale) {
    const int c = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (c >= ncols) return;
    double m = 0.0;
    if (c < nvalid)
        for (int b = lane; b < nblk; b += 32) m = fmax(m, pm[(size_t)b * ldmz + c]);
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) zscale[c] = pow2_above(m);              // NaN / inf rows (non-PD) are reported by K2, not here
}

// MZ rows -> digit planes, transposed: CTA = 128 rows x 32 columns
__global__ void __launch_bounds__(256)
digitize_kernel(long long N, long long npad, int ldmz, int nvalid, const double *__restrict__ MZ,
                const double *__restrict__ zscale, signed char *__restrict__ ZI) {
    constexpr int PITCH = 132;                              // bytes per (plane, column) row in shared memory: 33 words
    __shared__ __align__(16) signed char sh[NPL * CT * PITCH];
    const int ct = blockIdx.y;
    const long long n0 = (long long)blockIdx.x * 128;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = ct * CT + lane;
    const bool cv = c < nvalid;
    const double inv = cv ? 18014398509481984.0 / zscale[c] : 0.0;    // 2^54 / scale
    // v + sum_t 128 256^t has the unsigned bytes (digit_t + 128); flipping bit 7 of every byte gives the signed digits.
    // A warp takes 16 consecutive rows, four at a time: one 32-bit shared-memory store per plane and four rows.
    constexpr unsigned long long BIAS = 0x0080808080808080ULL;
    double xv[16];                                           // all 16 loads of this thread in flight before the first use
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const long long n = n0 + warp * 16 + k;
        xv[k] = (cv && n < N) ? MZ[n * ldmz + c] : 0.0;
    }
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        const int r = warp * 16 + g * 4;
        unsigned int lo[4], hi[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            double t = xv[g * 4 + k] * inv;
            t = (fabs(t) <= 18014398509481984.0) ? t : 0.0;  // NaN / inf (a non-PD row, reported separately) -> 0
            const unsigned long long u = ((unsigned long long)__double2ll_rn(t) + BIAS) ^ BIAS;
            lo[k] = (unsigned int)u;
            hi[k] = (unsigned int)(u >> 32);
        }
#pragma unroll
        for (int p = 0; p < NPL; ++p) {
            const unsigned int *w = (p < 4) ? lo : hi;
            const unsigned int sel = (unsigned)(p & 3) | ((unsigned)(4 + (p & 3)) << 4);
            const unsigned int w01 = __byte_perm(w[0], w[1], sel), w23 = __byte_perm(w[2], w[3], sel);
            *reinterpret_cast<unsigned int *>(&sh[(p * CT + lane) * PITCH + r]) = __byte_perm(w01, w23, 0x5410);
        }
    }
    __syncthreads();
    // two contiguous 14 KB tiles (64 rows each): ZI[(kb * nct + ct)][plane * 32 + column][64]
    const int nct = gridDim.y;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const long long kb = n0 / 64 + h;
        unsigned int *dst = reinterpret_cast<unsigned int *>(ZI + ((size_t)(kb * nct + ct) * (NPL * CT)) * 64);
        for (int w = threadIdx.x; w < NPL * CT * 16; w += 256)
            dst[w] = *reinterpret_cast<const unsigned int *>(&sh[(w >> 4) * PITCH + h * 64 + (w & 15) * 4]);
    }
}

// X [N][ldx] -> maskT [D][npad] (1 = observed); CTA = 128 rows x 32 data dimensions
__global__ void __launch_bounds__(256)
prepare_maskT_kernel(long long N, int D, long long npad, const double *__restrict__ X, long long ldx,
                     signed char *__restrict__ maskT) {
    constexpr int PITCH = 132;
    __shared__ __align__(16) signed char sh[32 * PITCH];
    const int d0 = blockIdx.y * 32;
    const long long n0 = (long long)blockIdx.x * 128;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int d = d0 + lane;
    for (int r = warp; r < 128; r += 8) {
        const long long n = n0 + r;
        signed char m = 0;
        if (d < D && n < N) {
            const double x = X[n * ldx + d];
            m = (x == x) ? 1 : 0;
        }
        sh[lane * PITCH + r] = m;
    }
    __syncthreads();
    // maskT[kb][d][64]: 32 data dimensions x 64 bytes per k tile
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const long long kb = n0 / 64 + h;
        for (int w = threadIdx.x; w < 32 * 16; w += 256) {
            const int row = w >> 4;
            if (d0 + row < D)
                *reinterpret_cast<unsigned int *>(maskT + ((size_t)kb * D + d0 + row) * 64 + (w & 15) * 4) =
                    *reinterpret_cast<const unsigned int *>(&sh[row * PITCH + h * 64 + (w & 15) * 4]);
        }
    }
}

constexpr int CHK_BLOCKS = 0;                             // (the guard block needs no per-CTA storage)
// one CTA per data dimension d: warp w sums T1[d][ii] over the chunks for i = w, w + 4, ... (lanes over chunks)
__global__ void __launch_bounds__(128)
stats_i8_check_kernel(int D, int q, const double *__restrict__ ws, int nchunks, const double *__restrict__ cnt,
                      const double *__restrict__ zscale, double *__restrict__ guard, double tol) {
    __shared__ double sh[8];
    const StatLayout L(D, q);
    const int P = i_tri(q), warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int d = blockIdx.x;
    double sz = 0.0;
    for (int c = threadIdx.x; c < P; c += 128) sz = fmax(sz, zscale[c]);
    double dm = 0.0;
    for (int i = warp; i < q; i += 4) {
        const size_t off = L.t1 + (size_t)d * P + i_tri(i) + i;
        double t = 0.0;
        for (int ch = lane; ch < nchunks; ch += 32) t += ws[(size_t)ch * L.len + off];
        dm = fmax(dm, warp_sum(t));
    }
    for (int o = 16; o > 0; o >>= 1) sz = fmax(sz, __shfl_xor_sync(0xffffffffu, sz, o));
    if (lane == 0) {
        sh[warp] = sz;
        sh[4 + warp] = dm;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        sz = fmax(fmax(sh[0], sh[1]), fmax(sh[2], sh[3])) * 2.7755575615628914e-17;      // max_c zscale_c * 2^-55
        dm = fmax(fmax(sh[4], sh[5]), fmax(sh[6], sh[7]));
        if (cnt[d] * sz > tol * dm) atomicAdd(guard + 3, 1.0);
        __threadfence();
        const unsigned int done = atomicAdd(reinterpret_cast<unsigned int *>(guard + 2), 1u);
        if (done == gridDim.x - 1) {           // the last CTA publishes the verdict and re-arms the counters
            __threadfence();
            const double t = *reinterpret_cast<volatile double *>(guard + 3);
            guard[0] = t;
            if (t > 0.0) guard[1] += 1.0;
            guard[3] = 0.0;
            *reinterpret_cast<unsigned int *>(guard + 2) = 0u;
        }
    }
}

size_t si8_smem_bytes(int q, int pair = 0) {
    const int ns = pair ? SST_PAIR : SST;
    return 1024 + (size_t)ns * (A_B + (pair ? B_B / 2 : B_B)) + (size_t)((i_tri(q) + q + 31) & ~31) * 8 + (size_t)(2 * ns + 4) * 8 + 16;
}

// CL > 1: the CTAs of a cluster take CL consecutive blocks of data dimensions of the same (column tile, chunk) item and
// share its digit tiles by multicast, as in K1-i8.
// PAIR (CL = 2): tcgen05.mma.cta_group::2 -- the two blocks of data dimensions are ONE 256-row MMA, each CTA stages its own
// maskT tile and HALF of the digit tile (15 KB per stage instead of 22: more stages, half the L2 traffic of the digits).
template <int CL, bool PAIR = false>
__global__ void __launch_bounds__(NTHR, 1)
stats_i8_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, long long N, int D, int q,
                const double *__restrict__ zscale, double *__restrict__ ws, long long rows_per_chunk, int nchunks, int ndb,
                int nct, int ks) {
    extern __shared__ unsigned char smem_dyn[];
    unsigned char *smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    static_assert(!PAIR || CL == 2, "a CTA pair is a cluster of two");
    constexpr int BSZ = PAIR ? B_B / 2 : B_B, STG = A_B + BSZ, NSMAX = PAIR ? SST_PAIR : SST;
    // ks K steps (64 rows each) per ring stage: half the barrier round trips, TMA arms and commits per MMA (see K1-i8)
    const int NS = NSMAX / ks, SB = ks * STG;
    const int P = i_tri(q), NCZ = (P + q + 31) & ~31;
    unsigned char *st_base = smem;                                             // [NS][A 8 KB | B 14 KB (PAIR: 7 KB)]
    double *fcol = reinterpret_cast<double *>(smem + (size_t)NSMAX * STG);      // [NCZ]: zscale_c * 2^-54
    uint64_t *full = reinterpret_cast<uint64_t *>(fcol + NCZ);
    uint64_t *empty = full + NSMAX;
    uint64_t *tfull = empty + NSMAX;
    uint64_t *tempty = tfull + 2;
    uint32_t *tbase = reinterpret_cast<uint32_t *>(tempty + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int crank = (CL > 1) ? (int)cluster_ctarank() : 0;
    const int ndg = (ndb + CL - 1) / CL;                       // groups of CL blocks of data dimensions
    const int nitems = ndg * nct * nchunks;                    // items of a CLUSTER
    const int cid = (int)blockIdx.x / CL, ncl = (int)gridDim.x / CL;
    constexpr uint16_t CMASK = (uint16_t)((1u << CL) - 1u);
    for (int c = tid; c < NCZ; c += NTHR) fcol[c] = zscale[c] * 5.5511151231257827e-17;   // 2^-54
    if (tid == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        for (int s = 0; s < NSMAX; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], PAIR ? 1 : CL);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&tfull[b], 1);
            mbar_init(&tempty[b], PAIR ? 16 : 8);
        }
        mbar_fence_init();
    }
    if (warp == 1) {
        if (PAIR) umma::tmem_alloc2(tbase, 512);
        else umma::tmem_alloc(tbase, 512);
    }
    umma::fence_before_sync();
    __syncthreads();
    if (CL > 1) cluster_sync_all();
    umma::fence_after_sync();
    const uint32_t tmem = *tbase;

    // item -> (chunk, group of blocks of data dimensions, ct), chunk-major; K steps of the chunk
    auto item_geom = [&](int item, int &chunk, int &db, int &ct, long long &r0, int &nsteps) {
        chunk = item / (ndg * nct);
        const int rem = item - chunk * (ndg * nct);
        const int dg = rem / nct;
        ct = rem - dg * nct;
        db = dg * CL + crank;                                   // may be >= ndb (an odd block count): its rows are discarded
        r0 = (long long)chunk * rows_per_chunk;
        long long r1 = r0 + rows_per_chunk;
        if (r1 > N) r1 = N;
        nsteps = (r1 > r0) ? (int)((r1 - r0 + BKB - 1) / BKB) : 0;
    };

    if (warp == 0) {
        // TMA producer: whole warp, one elected lane issues (see elect_one)
        const bool leader = elect_one();
        const uint32_t full_l = PAIR ? umma::map_to_cta(full, 0) : 0u;
        int s = 0;
        uint32_t ph = 0;
        for (int item = cid; item < nitems; item += ncl) {
            int chunk, db, ct, nsteps;
            long long r0;
            item_geom(item, chunk, db, ct, r0, nsteps);
            for (int k = 0; k < nsteps; k += ks) {
                const int kc = (nsteps - k < ks) ? nsteps - k : ks;          // K steps in this stage (the chunk's tail: fewer)
                umma::mbar_wait_bounded(&empty[s], ph ^ 1);
                if (leader) {
                    if (PAIR) {                // both CTAs' tiles complete on the LEADER's barrier (armed by the leader for both)
                        if (crank == 0) mbar_arrive_expect_tx(&full[s], (uint32_t)(2 * kc * STG));
                    } else {
                        mbar_arrive_expect_tx(&full[s], (uint32_t)(kc * (A_B + B_B)));
                    }
                    for (int h = 0; h < kc; ++h) {
                        unsigned char *st = st_base + (size_t)s * SB + (size_t)h * STG;
                        const long long kb = r0 / BKB + k + h;
                        if (PAIR) {
                            tma_load_3d_i8_pair(st, &tmA, 0, (int)(kb * D + db * BM), 0, full_l + (uint32_t)s * 8u);
                            tma_load_3d_i8_pair(st + A_B, &tmB, 0, (int)((kb * nct + ct) * (NPL * CT) + crank * (NPL * CT / 2)), 0,
                                                full_l + (uint32_t)s * 8u);
                        } else {
                            tma_load_3d_i8(st, &tmA, 0, (int)(kb * D + db * BM), 0, &full[s]);               // 128 data dimensions x 64 rows
                            if (CL == 1)
                                tma_load_3d_i8(st + A_B, &tmB, 0, (int)((kb * nct + ct) * (NPL * CT)), 0, &full[s]);   // 7 planes x 32 columns x 64 rows
                            else
                                tma_load_3d_i8_mc(st + A_B + crank * (B_B / CL), &tmB, 0,
                                                  (int)((kb * nct + ct) * (NPL * CT) + crank * (NPL * CT / CL)), 0, &full[s], CMASK);
                        }
                    }
                }
                __syncwarp();
                if (++s == NS) {
                    s = 0;
                    ph ^= 1;
                }
            }
        }
    } else if (warp == 1) {
        // MMA issuer: whole warp, one elected lane issues (PAIR: the leader CTA alone, for both)
        const bool leader = elect_one() && (!PAIR || crank == 0);
        const uint32_t idesc = umma::idesc_s8_s32(PAIR ? 2 * BM : BM, NPL * CT);
        const uint64_t adesc0 = umma::desc_kmajor_sw64(smem_u32(st_base), 0), bdesc0 = umma::desc_kmajor_sw64(smem_u32(st_base + A_B), 0);
        int s = 0, tl = 0;
        uint32_t ph = 0;
        for (int item = (PAIR && crank != 0) ? nitems : cid; item < nitems; item += ncl, ++tl) {
            int chunk, db, ct, nsteps;
            long long r0;
            item_geom(item, chunk, db, ct, r0, nsteps);
            const int buf = tl & 1;
            umma::mbar_wait_bounded(&tempty[buf], (uint32_t)(((tl >> 1) & 1) ^ 1));
            umma::fence_after_sync();
            const uint32_t dacc = tmem + (uint32_t)(buf * 256);
            for (int k = 0; k < nsteps; k += ks) {
                const int kc = (nsteps - k < ks) ? nsteps - k : ks;
                umma::mbar_wait_bounded(&full[s], ph);
                umma::fence_after_sync();
                if (leader) {
                    for (int h = 0; h < kc; ++h) {
                        const uint64_t off = (uint64_t)((s * SB + h * STG) >> 4);
                        if (PAIR) {
                            umma::mma_i8_pair(dacc, adesc0 + off, bdesc0 + off, idesc, (k + h) ? 1u : 0u);
                            umma::mma_i8_pair(dacc, adesc0 + off + 2, bdesc0 + off + 2, idesc, 1u);
                        } else {
                            umma::mma_i8(dacc, adesc0 + off, bdesc0 + off, idesc, (k + h) ? 1u : 0u);
                            umma::mma_i8(dacc, adesc0 + off + 2, bdesc0 + off + 2, idesc, 1u);
                        }
                    }
                    if (PAIR) umma::mma_commit_pair(&empty[s]);
                    else if (CL == 1) umma::mma_commit(&empty[s]);
                    else mma_commit_mc(&empty[s], CMASK);
                }
                __syncwarp();
                if (++s == NS) {
                    s = 0;
                    ph ^= 1;
                }
            }
            if (leader) {
                if (PAIR) umma::mma_commit_pair(&tfull[buf]);
                else umma::mma_commit(&tfull[buf]);
            }
            __syncwarp();
        }
    } else {
        const StatLayout L(D, q);
        const int wq = warp & 3, half = (warp - 2) >> 2;
        const uint32_t tempty_l = PAIR ? umma::map_to_cta(tempty, 0) : 0u;
        int tl = 0;
        for (int item = cid; item < nitems; item += ncl, ++tl) {
            int chunk, db, ct, nsteps;
            long long r0;
            item_geom(item, chunk, db, ct, r0, nsteps);
            const int buf = tl & 1;
            const int d = db * BM + wq * 32 + lane;
            const int c0 = ct * CT + half * 16;
            double *out = ws + (size_t)chunk * L.len;
            umma::mbar_wait_bounded(&tfull[buf], (uint32_t)((tl >> 1) & 1));
            umma::fence_after_sync();
            const uint32_t taddr = tmem + (uint32_t)(buf * 256 + half * 16) + ((uint32_t)(wq * 32) << 16);
#pragma unroll
            for (int ch = 0; ch < 2; ++ch) {
                uint32_t a[NPL][8];
                if (nsteps > 0) {                                  // an empty chunk contributes zeros (nothing was accumulated)
#pragma unroll
                    for (int p = 0; p < NPL; ++p) tmem_ld8(taddr + (uint32_t)(p * CT + ch * 8), a[p]);
                    umma::tmem_ld_wait();
                }
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    double v = 0.0;
                    if (nsteps > 0) {
#pragma unroll
                        for (int p = NPL - 1; p >= 0; --p) v = fma(v, 256.0, i2d((int)a[p][k]));   // |a| <= 128 rows: exact steps
                    }
                    const int c = c0 + ch * 8 + k;
                    if (d < D) {
                        if (c < P) out[L.t1 + (size_t)d * P + c] = fcol[c] * v;
                        else if (c < P + q) out[L.bst + (size_t)d * q + (c - P)] = fcol[c] * v;
                    }
                }
            }
            umma::fence_before_sync();
            __syncwarp();
            if (lane == 0) {
                if (PAIR) umma::mbar_arrive_cluster(tempty_l + (uint32_t)buf * 8u);
                else mbar_arrive(&tempty[buf]);
            }
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (CL > 1) cluster_sync_all();
    if (warp == 1) {
        if (PAIR) umma::tmem_dealloc2(tmem, 512);
        else umma::tmem_dealloc(tmem, 512);
    }
}

// K3-i8 with the digit planes made in shared memory (D <= 256: at most two blocks of 128 data dimensions).  digitize_kernel
// writes 7 bytes per MZ entry to ZI and stats_i8_kernel reads them back (1.1 GB each way per sweep at N = 1M, q = 16), for
// data that only ever feeds the MMA.  Here converter warps take the MZ rows from TMA tiles and write the digit tile straight
// into the ring stage, byte for byte the SWIZZLE_64B image TMA delivered from ZI (oracle/i8_fused_oracle.py).
// Work item = (column tile of 32, row chunk) over ALL blocks of data dimensions: each digit tile is made once and feeds
// the MMAs of both blocks (two TMEM accumulators of 224 columns).  Same chunks and the same integer sums as
// stats_i8_kernel, recombined by the same epilogue: bit-identical partials.
// Warps: 0 TMA producer (the maskT tiles), 1 MMA issuer, 2-9 epilogue, 10-17 converters (two groups of four that take
// alternate K steps, a warp = 16 rows of a 64-row step).  Ring stage = [maskT block 0 | maskT block 1 | digit tile]; each
// converter warp also has its own ring of MZ tiles.
constexpr int SF_CONV = 8;
constexpr int SF_NTHR = (2 + 8 + SF_CONV) * 32;
constexpr int SF_STG = 2 * A_B + B_B;                    // 30 KB
constexpr int SF_ZB = 16 * CT * 8;                       // 4 KB: a converter warp's MZ values of one step (16 rows x 32 columns)
constexpr int SF_NSMAX = 8;
constexpr int SF_PROF = 24;                              // PYVB_I8_PROF clock slots per CTA

size_t sf_smem_bytes(int q, int ns, int nz) {
    return 1024 + (size_t)ns * SF_STG + (size_t)SF_CONV * nz * SF_ZB + (size_t)stats_i8_ncols(q) * 8 +
           (size_t)(2 * ns + 2 + SF_CONV * nz) * 8 + 16;
}
// Two MZ slots per converter warp (64 KB, 32 KB of it in flight while a step is converted), the rest of the 227 KB in ring
// stages: at C2 (q = 16) 5 stages + 2 slots ran the kernel in 0.382 ms, 4 + 3 in 0.392, 3 + 4 in 0.409, 2 + 5 in 0.424 (one
// B200, 1000 W).  The converters barely wait for their TMA loads at any depth; ring stages decouple them from the MMAs.
constexpr int SF_NZ = 2;
int sf_stages(int q) {
    int ns = SF_NSMAX;
    while (ns > 2 && sf_smem_bytes(q, ns, SF_NZ) > 227 * 1024) --ns;
    return ns;
}

// 2-D tiled TMA load with an L2 cache policy (createpolicy)
__device__ __forceinline__ void tma_load_2d_hint(const void *dst_smem, const void *tmap, int c0, int c1, uint64_t *bar,
                                                 uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], "
        "%5;" ::"r"(smem_u32(dst_smem)),
        "l"(tmap), "r"(c0), "r"(c1), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}

__global__ void __launch_bounds__(SF_NTHR, 1)
stats_i8_fused_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmZ, long long N, int D, int q,
                      const double *__restrict__ zscale, double *__restrict__ ws, long long rows_per_chunk, int nchunks,
                      int ndb, int nct, int ns, int nz, long long *prof) {
    long long w0 = 0, w1 = 0;                                  // PYVB_I8_PROF: clocks spent waiting, per role
    const long long tstart = clock64();
#define PROF_WAIT(acc, stmt)                    \
    do {                                        \
        if (prof) {                             \
            const long long t_ = clock64();     \
            stmt;                               \
            acc += clock64() - t_;              \
        } else {                                \
            stmt;                               \
        }                                       \
    } while (0)
    extern __shared__ unsigned char smem_dyn[];
    unsigned char *smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    const int P = i_tri(q), NCZ = nct * CT;
    unsigned char *st_base = smem;                                             // [ns][A0 8 KB | A1 8 KB | B 14 KB]
    unsigned char *zbuf = smem + (size_t)ns * SF_STG;                          // [SF_CONV][nz][16 rows x 32 doubles]
    double *fcol = reinterpret_cast<double *>(zbuf + (size_t)SF_CONV * nz * SF_ZB);   // [NCZ]: zscale_c * 2^-54
    uint64_t *full = reinterpret_cast<uint64_t *>(fcol + NCZ);                // [ns]: producer (tx bytes) + 4 converter warps
    uint64_t *empty = full + ns;                                               // [ns]: MMA commit
    uint64_t *tfull = empty + ns;
    uint64_t *tempty = tfull + 1;
    uint64_t *zfull = tempty + 1;                                              // [SF_CONV][nz]: tmZ tx bytes
    uint32_t *tbase = reinterpret_cast<uint32_t *>(zfull + SF_CONV * nz);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nitems = nct * nchunks;
    for (int c = tid; c < NCZ; c += SF_NTHR) fcol[c] = zscale[c] * 5.5511151231257827e-17;   // 2^-54
    if (tid == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmZ);
        for (int s = 0; s < ns; ++s) {
            mbar_init(&full[s], 1 + SF_CONV / 2);
            mbar_init(&empty[s], 1);
        }
        mbar_init(tfull, 1);
        mbar_init(tempty, 8);
        for (int i = 0; i < SF_CONV * nz; ++i) mbar_init(&zfull[i], 1);
        mbar_fence_init();
    }
    if (warp == 1) umma::tmem_alloc(tbase, 512);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = *tbase;

    // item -> (chunk, column tile), chunk-major as in stats_i8_kernel; K steps of the chunk
    auto item_geom = [&](int item, int &chunk, int &ct, long long &r0, int &nsteps) {
        chunk = item / nct;
        ct = item - chunk * nct;
        r0 = (long long)chunk * rows_per_chunk;
        long long r1 = r0 + rows_per_chunk;
        if (r1 > N) r1 = N;
        nsteps = (r1 > r0) ? (int)((r1 - r0 + BKB - 1) / BKB) : 0;
    };

    if (warp == 0) {
        // TMA producer: the maskT tiles (128 data dimensions x 64 rows) of every block
        const bool leader = elect_one();
        int s = 0;
        uint32_t ph = 0;
        for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
            int chunk, ct, nsteps;
            long long r0;
            item_geom(item, chunk, ct, r0, nsteps);
            for (int k = 0; k < nsteps; ++k) {
                PROF_WAIT(w0, umma::mbar_wait_bounded(&empty[s], ph ^ 1));
                if (leader) {
                    mbar_arrive_expect_tx(&full[s], (uint32_t)(ndb * A_B));
                    const long long kb = r0 / BKB + k;
                    for (int b = 0; b < ndb; ++b)
                        tma_load_3d_i8(st_base + (size_t)s * SF_STG + b * A_B, &tmA, 0, (int)(kb * D + b * BM), 0, &full[s]);
                }
                __syncwarp();
                if (++s == ns) {
                    s = 0;
                    ph ^= 1;
                }
            }
        }
    } else if (warp == 1) {
        // MMA issuer: per K step two MMAs (K = 2 x 32 bytes) per block of data dimensions, on the same digit tile
        const bool leader = elect_one();
        const uint32_t idesc = umma::idesc_s8_s32(BM, NPL * CT);
        const uint64_t adesc0 = umma::desc_kmajor_sw64(smem_u32(st_base), 0);
        const uint64_t bdesc0 = umma::desc_kmajor_sw64(smem_u32(st_base + 2 * A_B), 0);
        int s = 0, tl = 0;
        uint32_t ph = 0;
        for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++tl) {
            int chunk, ct, nsteps;
            long long r0;
            item_geom(item, chunk, ct, r0, nsteps);
            PROF_WAIT(w1, umma::mbar_wait_bounded(tempty, (uint32_t)((tl & 1) ^ 1)));   // the epilogue has drained the accumulators
            umma::fence_after_sync();
            for (int k = 0; k < nsteps; ++k) {
                PROF_WAIT(w0, umma::mbar_wait_bounded(&full[s], ph));
                umma::fence_after_sync();
                if (leader) {
                    const uint64_t off = (uint64_t)((s * SF_STG) >> 4);
                    for (int b = 0; b < ndb; ++b) {
                        const uint32_t dacc = tmem + (uint32_t)(b * 256);
                        const uint64_t ad = adesc0 + off + (uint64_t)(b * (A_B >> 4));
                        umma::mma_i8(dacc, ad, bdesc0 + off, idesc, k ? 1u : 0u);
                        umma::mma_i8(dacc, ad + 2, bdesc0 + off + 2, idesc, 1u);
                    }
                    umma::mma_commit(&empty[s]);
                }
                __syncwarp();
                if (++s == ns) {
                    s = 0;
                    ph ^= 1;
                }
            }
            if (leader) umma::mma_commit(tfull);
            __syncwarp();
        }
    } else if (warp < 10) {
        // epilogue: the recombination of stats_i8_kernel, for each block of data dimensions
        const StatLayout L(D, q);
        const int wq = warp & 3, half = (warp - 2) >> 2;
        int tl = 0;
        for (int item = blockIdx.x; item < nitems; item += gridDim.x, ++tl) {
            int chunk, ct, nsteps;
            long long r0;
            item_geom(item, chunk, ct, r0, nsteps);
            const int c0 = ct * CT + half * 16;
            double *out = ws + (size_t)chunk * L.len;
            PROF_WAIT(w0, umma::mbar_wait_bounded(tfull, (uint32_t)(tl & 1)));
            umma::fence_after_sync();
            for (int b = 0; b < ndb; ++b) {
                const int d = b * BM + wq * 32 + lane;
                const uint32_t taddr = tmem + (uint32_t)(b * 256 + half * 16) + ((uint32_t)(wq * 32) << 16);
#pragma unroll
                for (int ch = 0; ch < 2; ++ch) {
                    uint32_t a[NPL][8];
                    if (nsteps > 0) {                              // an empty chunk contributes zeros (nothing was accumulated)
#pragma unroll
                        for (int p = 0; p < NPL; ++p) tmem_ld8(taddr + (uint32_t)(p * CT + ch * 8), a[p]);
                        umma::tmem_ld_wait();
                    }
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        double v = 0.0;
                        if (nsteps > 0) {
#pragma unroll
                            for (int p = NPL - 1; p >= 0; --p) v = fma(v, 256.0, i2d((int)a[p][k]));
                        }
                        const int c = c0 + ch * 8 + k;
                        if (d < D) {
                            if (c < P) out[L.t1 + (size_t)d * P + c] = fcol[c] * v;
                            else if (c < P + q) out[L.bst + (size_t)d * q + (c - P)] = fcol[c] * v;
                        }
                    }
                }
            }
            umma::fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty);
        }
    } else {
        // converters: the arithmetic of digitize_kernel (2^54 / zscale_c, NaN / inf -> 0, the BIAS / xor byte split), written
        // as the SWIZZLE_64B image of the K-major tile: plane p, column l of the tile, row n of the step at byte
        // (p * 32 + l) * 64 + (((n >> 4) ^ ((l >> 1) & 3)) << 4) + (n & 15).  Warp cw owns rows 16 (cw % 4) ... + 15 of every
        // other step; a lane owns one column and puts four rows into one 32-bit word per plane.  Lane group l / 8 starts at
        // row quad l / 8 of the warp's 16 rows (and cycles): with the swizzle the 32 words of every store instruction fall
        // into 32 different banks.
        // The MZ values arrive by TMA (tmZ: 16 rows x 32 columns, 4 KB) in a ring of nz slots private to the warp, nz steps
        // ahead: rows >= N and columns >= P + q (the pitch past zbar among them) arrive as zeros, so no column past zbar is
        // ever read.
        const int cw = warp - 10, grp = cw >> 2, rq = cw & 3, rot = lane >> 3;
        const int nvalid = P + q;
        constexpr unsigned long long BIAS = 0x0080808080808080ULL;
        const uint32_t wbase = (uint32_t)(lane * 64 + ((rq ^ ((lane >> 1) & 3)) << 4));
        const double *zring = reinterpret_cast<const double *>(zbuf + (size_t)cw * nz * SF_ZB);
        uint64_t *zb = zfull + cw * nz;
        const bool zlead = elect_one();
        uint64_t policy = 0;
        if (zlead) asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));   // MZ is read once
        // position (item, K step of the item) of this warp's steps: the CTA's steps j = grp, grp + 2, ... in order
        struct Pos {
            int item, k, nsteps, ct;
            long long r0;
        };
        auto settle = [&](Pos &p) {                            // past the end of an item: into the next non-empty one
            while (p.item < nitems && p.k >= p.nsteps) {
                p.k -= p.nsteps;
                p.item += gridDim.x;
                int chunk;
                if (p.item < nitems) item_geom(p.item, chunk, p.ct, p.r0, p.nsteps);
            }
        };
        auto issue = [&](const Pos &p, int slot) {            // (elected lane) this warp's 16 rows of the step at p
            mbar_arrive_expect_tx(&zb[slot], (uint32_t)SF_ZB);
            tma_load_2d_hint(zring + slot * (SF_ZB / 8), &tmZ, p.ct * CT, (int)(p.r0 + (long long)p.k * BKB + rq * 16), &zb[slot],
                             policy);
        };
        Pos cur;
        cur.item = blockIdx.x;
        cur.k = grp;
        cur.nsteps = 0;
        {
            int chunk;
            if (cur.item < nitems) item_geom(cur.item, chunk, cur.ct, cur.r0, cur.nsteps);
        }
        settle(cur);
        Pos ahead = cur;                                       // the step whose values are loaded next
        for (int i = 0; i < nz && ahead.item < nitems; ++i) {
            if (zlead) issue(ahead, i);
            ahead.k += 2;
            settle(ahead);
        }
        int ict = -1;
        double inv = 0.0;
        for (int j = grp, zt = 0; cur.item < nitems; j += 2, ++zt) {
            const int zs = zt % nz;
            PROF_WAIT(w0, umma::mbar_wait_bounded(&zb[zs], (uint32_t)((zt / nz) & 1)));
            double xv[16];
            const double *zr = zring + zs * (SF_ZB / 8) + lane;   // row r of the slot: 32 contiguous doubles
#pragma unroll
            for (int g = 0; g < 4; ++g)
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) xv[g * 4 + kk] = zr[(4 * ((g + rot) & 3) + kk) * CT];
            // the slot is refilled: the generic-proxy reads of all lanes before the async-proxy write
            __syncwarp();
            fence_async_smem();
            if (ahead.item < nitems) {
                if (zlead) issue(ahead, zs);
                ahead.k += 2;
                settle(ahead);
            }
            if (cur.ct != ict) {
                ict = cur.ct;
                const int c = ict * CT + lane;
                inv = c < nvalid ? 18014398509481984.0 / zscale[c] : 0.0;    // 2^54 / scale
            }
            const int s = j % ns;
            PROF_WAIT(w1, umma::mbar_wait_bounded(&empty[s], (uint32_t)(((j / ns) & 1) ^ 1)));
            unsigned char *bt = st_base + (size_t)s * SF_STG + 2 * A_B;
#pragma unroll
            for (int g = 0; g < 4; ++g) {
                const int qd = (g + rot) & 3;
                unsigned int lo[4], hi[4];
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    double t = xv[g * 4 + kk] * inv;
                    t = (fabs(t) <= 18014398509481984.0) ? t : 0.0;
                    const unsigned long long u = ((unsigned long long)__double2ll_rn(t) + BIAS) ^ BIAS;
                    lo[kk] = (unsigned int)u;
                    hi[kk] = (unsigned int)(u >> 32);
                }
#pragma unroll
                for (int p = 0; p < NPL; ++p) {
                    const unsigned int *w = (p < 4) ? lo : hi;
                    const unsigned int sel = (unsigned)(p & 3) | ((unsigned)(4 + (p & 3)) << 4);
                    const unsigned int w01 = __byte_perm(w[0], w[1], sel), w23 = __byte_perm(w[2], w[3], sel);
                    *reinterpret_cast<unsigned int *>(bt + p * (CT * BKB) + wbase + qd * 4) = __byte_perm(w01, w23, 0x5410);
                }
            }
            fence_async_smem();                                 // generic-proxy stores before the MMA's async-proxy reads
            __syncwarp();
            if (lane == 0) mbar_arrive(&full[s]);
            cur.k += 2;
            settle(cur);
        }
    }
#undef PROF_WAIT
    // [producer: empty][MMA: full, tempty][epilogue warp 2: tfull][converters: loads 8][converters: empty 8][total]
    if (prof && lane == 0 && (warp < 3 || warp >= 10)) {       // (all lanes of a role wait together: lane 0's clocks are the role's)
        long long *o = prof + (size_t)blockIdx.x * SF_PROF;
        if (warp < 2) {
            o[warp] = w0;
            if (warp == 1) o[2] = w1;
        } else if (warp == 2) {
            o[3] = w0;
        } else {
            o[4 + (warp - 10)] = w0;
            o[12 + (warp - 10)] = w1;
        }
        if (warp == 0) o[20] = clock64() - tstart;
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 1) umma::tmem_dealloc(tmem, 512);
}


// ---- microbenchmark: back-to-back tcgen05.mma on fixed shared-memory operands (no loads): the tensor-core rate of the
// box for kind::i8 (kind = 0) or kind::f16 / bf16 (kind = 1) at M = 128, N = n, one K step of 32 bytes per instruction.
// mode bits: 1 = rotate through 4 operand stage buffers, 2 = tcgen05.commit to an mbarrier after every pair of MMAs,
//            4 = warp 1 streams 14 KB bulk copies from global memory into other shared-memory buffers meanwhile
__global__ void __launch_bounds__(128, 1) bench_umma_kernel(int iters, int n, int kind, int mode, const unsigned char *src,
                                                           long long *clk_out) {
    extern __shared__ unsigned char smem_dyn[];
    unsigned char *smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    constexpr int STG = A_B + 256 * BKB;                    // 24 KB per stage
    __shared__ uint64_t bar, cbar[4], lbar[2];
    __shared__ uint32_t tb;
    __shared__ int stop;
    for (int i = threadIdx.x; i < 4 * STG / 4; i += 128) reinterpret_cast<uint32_t *>(smem)[i] = 0x01010101u;
    if (threadIdx.x == 0) {
        mbar_init(&bar, 1);
        for (int i = 0; i < 4; ++i) mbar_init(&cbar[i], 1);
        mbar_init(&lbar[0], 1);
        mbar_init(&lbar[1], 1);
        stop = 0;
        mbar_fence_init();
    }
    if (threadIdx.x < 32) umma::tmem_alloc(&tb, 512);
    fence_async_smem();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = tb;
    if (threadIdx.x == 0) {
        const uint32_t idesc = kind == 0 ? umma::idesc_s8_s32(BM, n) : umma::idesc_bf16_f32(BM, n, 0, 0);
        const long long t0 = clock64();
        for (int it = 0; it < iters; ++it) {
            const uint32_t d = tmem + (uint32_t)((it & 1) * 256);
            const uint32_t a0 = smem_u32(smem) + ((mode & 1) ? (uint32_t)((it & 3) * STG) : 0u), b0 = a0 + A_B;
            if (kind == 0) {
                umma::mma_i8(d, umma::desc_kmajor_sw64(a0, 0), umma::desc_kmajor_sw64(b0, 0), idesc, 1u);
                umma::mma_i8(d, umma::desc_kmajor_sw64(a0, 1), umma::desc_kmajor_sw64(b0, 1), idesc, 1u);
            } else {
                umma::mma_bf16(d, umma::desc_kmajor_sw64(a0, 0), umma::desc_kmajor_sw64(b0, 0), idesc, 1u);
                umma::mma_bf16(d, umma::desc_kmajor_sw64(a0, 1), umma::desc_kmajor_sw64(b0, 1), idesc, 1u);
            }
            if (mode & 2) umma::mma_commit(&cbar[it & 3]);
        }
        umma::mma_commit(&bar);
        umma::mbar_wait_bounded(&bar, 0);
        clk_out[blockIdx.x] = clock64() - t0;
        *reinterpret_cast<volatile int *>(&stop) = 1;
    } else if (threadIdx.x == 32 && (mode & 4)) {
        // background fill traffic: 14 KB copies, two in flight, into a scratch area behind the operand stages
        unsigned char *dst = smem + 4 * STG;
        uint32_t ph[2] = {0, 0};
        int k = 0;
        const unsigned char *g = src + (size_t)blockIdx.x * (1 << 20);
        mbar_arrive_expect_tx(&lbar[0], B_B);
        bulk_g2s(dst, g, B_B, &lbar[0]);
        mbar_arrive_expect_tx(&lbar[1], B_B);
        bulk_g2s(dst + B_B, g + B_B, B_B, &lbar[1]);
        while (!*reinterpret_cast<volatile int *>(&stop)) {
            const int b = k & 1;
            umma::mbar_wait_bounded(&lbar[b], ph[b]);
            ph[b] ^= 1;
            ++k;
            mbar_arrive_expect_tx(&lbar[b], B_B);
            bulk_g2s(dst + b * B_B, g + (size_t)((k * B_B) & ((1 << 20) - 32768)), B_B, &lbar[b]);
        }
        umma::mbar_wait_bounded(&lbar[0], ph[0]);
        umma::mbar_wait_bounded(&lbar[1], ph[1]);
        clk_out[148 + blockIdx.x] = k;
    }
    umma::fence_before_sync();
    __syncthreads();
    if (threadIdx.x < 32) umma::tmem_dealloc(tmem, 512);
}

}  // namespace

cudaError_t launch_bench_umma(int blocks, int iters, int n, int kind, int mode, const void *src, long long *clk_out,
                              cudaStream_t st) {
    const size_t smem = 1024 + 4 * (A_B + 256 * BKB) + 2 * B_B;
    cudaError_t e = cudaFuncSetAttribute(bench_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    bench_umma_kernel<<<blocks, 128, smem, st>>>(iters, n, kind, mode, static_cast<const unsigned char *>(src), clk_out);
    return cudaGetLastError();
}

bool i8_supported(int D, int q) {
    return (q == 16 || q == 32 || q == 64) && D >= 64 && (D % 64) == 0 && i8_stages(D, q, 1) >= 2;
}
size_t i8_digits_bytes(int D, int q) { return (size_t)(i_nc8(q) / CT) * NPL * CT * D; }
size_t i8_mask_bytes(long long N, int D) { return (size_t)((N + BM - 1) / BM * BM) * (size_t)D; }
int i8_ncols(int q) { return i_nc8(q); }

cudaError_t launch_prepare_mask_i8(long long N, int D, const double *X, long long ldx, void *mask, cudaStream_t st) {
    if (N <= 0) return cudaSuccess;
    long long b = (((N + BM - 1) / BM * BM) * (long long)(D / 4) + 255) / 256;
    if (b > 148 * 16) b = 148 * 16;
    prepare_mask_i8_kernel<<<(unsigned)b, 256, 0, st>>>(N, D, X, ldx, static_cast<signed char *>(mask));
    return cudaGetLastError();
}

cudaError_t launch_pack_g_i8(int D, int q, const double *Gw, int ldg, void *GI, double *gscale, double *gl, cudaStream_t st) {
    pack_g_i8_kernel<<<i_nc8(q), 256, 0, st>>>(D, q, Gw, ldg, static_cast<signed char *>(GI), gscale, gl);
    return cudaGetLastError();
}

cudaError_t launch_zstep_i8(long long N, int D, int q, const void *mask, const void *GI, const double *P0,
                            const double *gscale, const double *gl, double *MZ, int ldmz, cudaStream_t st) {
    if (N <= 0) return cudaSuccess;
    if (!i8_supported(D, q)) return cudaErrorNotSupported;
    const I8Geom g(q);
    const long long nrb = (N + BM - 1) / BM;
    const int cl = (nrb < 2LL * I8_CL) ? 1 : I8_CL;          // tiny problems: no point in pairing
    CUtensorMap tmA, tmB;
    const uint64_t nk = (uint64_t)(D / BKB);
    if ((uint64_t)nrb * nk * BM >= (1ULL << 31)) return cudaErrorNotSupported;
    cudaError_t e = make_map_u8_3d(&tmA, mask, BKB, (uint64_t)nrb * nk * BM, 1, BKB, BM);
    if (e != cudaSuccess) return e;
    e = make_map_u8_3d(&tmB, GI, BKB, nk * g.NCT * (NPL * CT), 1, BKB, NPL * CT / cl);
    if (e != cudaSuccess) return e;
    CUtensorMap tmO;
    {   // the qprec columns [0, PP) of the MZ rows, as [N][PP] doubles with the row pitch ldmz: 16-column x 32-row boxes
        EncodeTiledFn enc = get_encode_i8();
        if (!enc) return cudaErrorNotSupported;
        cuuint64_t dims[2] = {(cuuint64_t)g.PP, (cuuint64_t)N};
        cuuint64_t strides[1] = {(cuuint64_t)ldmz * sizeof(double)};
        cuuint32_t box[2] = {16, 32}, es[2] = {1, 1};
        CUresult r = enc(&tmO, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, MZ, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
    }
    // tcgen05.mma.cta_group::2 where digit stages are scarce (D = 1024: 5 stages of 14 KB next to the 128 KB mask block -> 10 of
    // 7 KB; K1 4.49 -> 4.19 ms on the config-3 shard).  Where eight full stages fit anyway (D <= 512) the pair only couples the
    // two CTAs' epilogues (D = 256: 0.43 -> 0.54 ms): plain clusters with multicast there.
    const int pair = (cl == 2 && i8_stages(D, q, i8_hstage(D, q), 0) < 8) ? 1 : 0;
    const int hstage = pair ? ((i8_stages(D, q, 0, 1) < 12 && i8_stages(D, q, 1, 1) > i8_stages(D, q, 0, 1)) ? 1 : 0) : i8_hstage(D, q);
    // a second mask block where it costs no digit stage (D <= 256)
    const int adbl = (!pair && i8_stages(D, q, hstage, 0, 1) >= ST / 2) ? 1 : 0;
    int nst = i8_stages(D, q, hstage, pair, adbl);
    if (nst < 2) return cudaErrorNotSupported;
    const size_t smem = i8_smem_bytes(D, q, nst, hstage, pair, adbl);
    // two K chunks per ring stage: half as many barrier round trips, TMA arms and commits per MMA -- with one tile per stage the
    // producer's and the issuer's per-stage latency (~300 clocks each) was as long as the tile's two MMAs (257 clocks).  Measured
    // under ncu on one box: config-3 shard 5.07 -> 4.02 ms, config 2 0.450 -> 0.388 ms, D = 512 / q = 64 unchanged.
    const int ks = ((nk % 2) != 0 || nst < 4) ? 1 : 2;
    if (ks == 2) nst /= 2;                                   // same bytes: the ring keeps its depth in K chunks
    CUtensorMap tmO8;
    {   // the same rows as 8-column x 32-row boxes (64-byte rows, SWIZZLE_64B) for the half-staging epilogue
        EncodeTiledFn enc = get_encode_i8();
        cuuint64_t dims[2] = {(cuuint64_t)g.PP, (cuuint64_t)N};
        cuuint64_t strides[1] = {(cuuint64_t)ldmz * sizeof(double)};
        cuuint32_t box[2] = {8, 32}, es[2] = {1, 1};
        CUresult r = enc(&tmO8, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, MZ, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
    }
    long long gl_ = (nrb + cl - 1) / cl * cl;
    const int grid = (int)(gl_ < 148 ? gl_ : 148 / cl * cl);
    auto kern = pair ? zstep_i8_kernel<I8_CL, true> : cl == I8_CL ? zstep_i8_kernel<I8_CL> : zstep_i8_kernel<1>;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    static long long *prof = nullptr;
    static int prof_on = -1;
    if (prof_on < 0) {
        prof_on = getenv("PYVB_I8_PROF") ? 1 : 0;
        if (prof_on && cudaMalloc(&prof, 148 * 10 * sizeof(long long)) != cudaSuccess) prof_on = 0;
    }
    e = launch_cluster(kern, grid, NTHR, smem, cl, st, tmA, tmB, tmO, tmO8, N, D, q, P0, gscale, gl, (int)nrb, nst, hstage, adbl,
                       prof_on ? prof : (long long *)nullptr, ks);
    if (prof_on && e == cudaSuccess) {      // diagnosis only: synchronises
        long long h[148 * 10];
        cudaStreamSynchronize(st);
        cudaMemcpy(h, prof, sizeof(h), cudaMemcpyDeviceToHost);
        double a[10] = {0};
        for (int b = 0; b < grid; ++b)
            for (int k = 0; k < 10; ++k) a[k] += (double)h[b * 10 + k] / grid;
        fprintf(stderr, "[i8 prof] N=%lld D=%d q=%d cl=%d nst=%d total %.0f clk | producer: empty %.0f aempty %.0f | mma: full %.0f tempty %.0f afull %.0f | epilogue(w2): tfull %.0f store-read %.0f\n",
                N, D, q, cl, nst, a[9], a[0], a[1], a[3], a[4], a[5], a[6], a[7]);
    }
    return e;
}

// ---- K3-i8 host side
bool stats_i8_supported(int D, int q) { return (q == 16 || q == 32 || q == 64) && D >= 16 && (D % 16) == 0; }
int stats_i8_ncols(int q) { return (i_tri(q) + q + 31) & ~31; }
long long stats_i8_npad(long long N) { return (N + 127) / 128 * 128; }
size_t stats_i8_digits_bytes(long long N, int q) { return (size_t)stats_i8_ncols(q) * NPL * (size_t)stats_i8_npad(N); }
size_t stats_i8_maskt_bytes(long long N, int D) { return (size_t)D * (size_t)stats_i8_npad(N) + (size_t)BM * BKB; }
size_t stats_i8_scratch_len(int q, int ldmz) { return (size_t)CM_BLOCKS * 2 * ldmz + stats_i8_ncols(q) + 8 + CHK_BLOCKS; }
double *stats_i8_guard(double *scratch, int q, int ldmz) { return scratch + (size_t)CM_BLOCKS * 2 * ldmz + stats_i8_ncols(q); }

// Accuracy guard of the INT8 statistics: T1[d][c] carries at most cnt_d * zscale_c * 2^-55 of fixed-point rounding.  A data
// dimension whose largest diagonal entry max_i T1[d][ii] (a sum of cnt_d non-negative terms) does not dominate that bound by
// 1 / tol fails; guard[0] = number of failing dimensions (the conditional DMMA statistics redo the pass when it is > 0).
// guard: [0] failing dimensions of the last call, [1] fall-backs so far, [2] CTA counter, [3] running count (all zero at first).
cudaError_t launch_stats_i8_check(int D, int q, const double *ws, int nchunks, const double *xcache, double *scratch,
                                  int ldmz, double tol, cudaStream_t st) {
    stats_i8_check_kernel<<<D, 128, 0, st>>>(D, q, ws, nchunks, xcache, scratch + (size_t)CM_BLOCKS * 2 * ldmz,
                                                  stats_i8_guard(scratch, q, ldmz), tol);
    return cudaGetLastError();
}

static long long gcd_ll(long long a, long long b) { return b ? gcd_ll(b, a % b) : a; }
// chunks: items = ndb * nct * nchunks a whole number of rounds over 148 CTAs, chunks of >= 32 K steps, <= 2^23 rows
int stats_i8_nchunks(long long N, int D, int q) {
    const int cl = I8_CL;
    const long long ncl = 148 / cl;
    const long long per = (long long)(((D + BM - 1) / BM + cl - 1) / cl) * (stats_i8_ncols(q) / CT);   // items of a cluster per chunk
    const long long step = ncl / gcd_ll(ncl, per);
    long long by_rows = N / (32LL * BKB);
    if (by_rows < 1) by_rows = 1;
    long long k = (6 * ncl + per * step - 1) / (per * step);        // ~6 items per cluster
    if (k < 1) k = 1;
    long long c = k * step;
    if (c > by_rows) c = (by_rows >= step) ? (by_rows / step) * step : by_rows;
    const long long cmin = (N + (1LL << 23) - 1) >> 23;
    if (c < cmin) c = cmin;
    if (c > 1024) c = 1024;
    return (int)c;
}
long long stats_i8_rows_per_chunk(long long N, int nchunks) {
    long long rpc = (N + nchunks - 1) / nchunks;
    rpc = (rpc + BKB - 1) / BKB * BKB;
    return rpc < BKB ? BKB : rpc;
}

cudaError_t launch_prepare_maskT_i8(long long N, int D, const double *X, long long ldx, void *maskT, cudaStream_t st) {
    if (N <= 0) return cudaSuccess;
    dim3 grid((unsigned)((N + 127) / 128), (unsigned)((D + 31) / 32));
    prepare_maskT_kernel<<<grid, 256, 0, st>>>(N, D, stats_i8_npad(N), X, ldx, static_cast<signed char *>(maskT));
    return cudaGetLastError();
}

// PYVB_I8_FUSED=0 keeps digitize_kernel + stats_i8_kernel where the fused kernel applies.  Read on every call, so that one
// process can compare the two paths.
bool stats_i8_fused(int D) {
    const char *e = getenv("PYVB_I8_FUSED");
    return (D + BM - 1) / BM <= 2 && !(e && e[0] == '0');
}

// colmax -> zscale -> digit planes of the MZ rows -> T1, Bst partial sums of every row chunk in ws[chunk][stat layout]
// (D <= 256: stats_i8_fused_kernel makes the digit planes in shared memory and ZI is not touched; it may be NULL)
// zsums (nullable): K2's per-CTA partials [column sums | 4 scalars | bounds on the column maxima] (nzblk partials of zkw
// doubles).  Without them (or when `trusted` is 0: a K2 kernel that leaves no maxima) one pass over the MZ rows builds the same
// partials in `scratch` (logdet needed); *zs_out / *nzblk_out / *zkw_out say which partials the second stage must add up.
cudaError_t launch_stats_i8(long long N, int D, int q, const void *maskT, const double *MZ, int ldmz, void *ZI,
                            double *scratch, double *ws, int nchunks, const double *zsums, int nzblk, int zkw, int trusted,
                            const double *logdet, const double **zs_out, int *nzblk_out, int *zkw_out, cudaStream_t st) {
    if (N <= 0) return cudaSuccess;
    const int P = i_tri(q), NCZ = stats_i8_ncols(q), nct = NCZ / CT, ndb = (D + BM - 1) / BM;
    const long long npad = stats_i8_npad(N);
    const int orow = gw_woff(q) + q;                        // [packed | pad | zbar] columns of an MZ row (K2's partial layout)
    double *pm = scratch, *zscale = scratch + (size_t)CM_BLOCKS * 2 * ldmz;
    if (!(zsums != nullptr && nzblk > 0 && trusted)) {
        if (logdet == nullptr) return cudaErrorInvalidValue;
        int nblk = CM_BLOCKS;
        long long rpb = (N + nblk - 1) / nblk;
        if (rpb < 64) rpb = 64;
        nblk = (int)((N + rpb - 1) / rpb);
        mzpart_kernel<<<nblk, 256, (size_t)(2 * ldmz + 4) * sizeof(double), st>>>(N, ldmz, orow, MZ, logdet, pm, rpb);
        zsums = pm;
        nzblk = nblk;
        zkw = 2 * orow + 4;
    }
    *zs_out = zsums;
    *nzblk_out = nzblk;
    *zkw_out = zkw;
    colmax_reduce_kernel<<<(NCZ + 7) / 8, 256, 0, st>>>(NCZ, P + q, zkw, zsums + orow + 4, nzblk, zscale);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    const cuuint64_t nkb = (cuuint64_t)(npad / BKB);
    EncodeTiledFn enc = get_encode_i8();
    if (!enc) return cudaErrorNotSupported;
    if (nkb * (cuuint64_t)D + BM >= (1ULL << 31) || nkb * nct * (NPL * CT) >= (1ULL << 31)) return cudaErrorNotSupported;
    const cuuint32_t es[3] = {1, 1, 1};
    CUtensorMap tmA;
    {   // maskT [npad / 64][D][64] (+ one box of slack: the last block of data dimensions may reach past D)
        cuuint64_t da[3] = {BKB, nkb * D + BM, 1}, sa[2] = {BKB, (nkb * D + BM) * BKB};
        cuuint32_t ba[3] = {BKB, BM, 1};
        CUresult r = enc(&tmA, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void *>(maskT), da, sa, ba, es,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
    }
    const long long rpc = stats_i8_rows_per_chunk(N, nchunks);
    if (stats_i8_fused(D)) {
        CUtensorMap tmZ;
        {   // the MZ columns [0, P + q) as [N][P + q] doubles with the row pitch ldmz (16-byte aligned, C-ABI): 32-column x
            // 16-row boxes, rows >= N and columns >= P + q zero-filled
            cuuint64_t dz[2] = {(cuuint64_t)(P + q), (cuuint64_t)N}, sz[1] = {(cuuint64_t)ldmz * sizeof(double)};
            cuuint32_t bz[2] = {CT, 16};
            CUresult r = enc(&tmZ, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double *>(MZ), dz, sz, bz, es,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
            if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
        }
        const int ns = sf_stages(q), nz = SF_NZ;
        const size_t smem = sf_smem_bytes(q, ns, nz);
        e = cudaFuncSetAttribute(stats_i8_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        const long long nitems = (long long)nct * nchunks;
        const int grid = (int)(nitems < 148 ? nitems : 148);
        static long long *prof = nullptr;
        static int prof_on = -1;
        if (prof_on < 0) {
            prof_on = getenv("PYVB_I8_PROF") ? 1 : 0;
            if (prof_on && cudaMalloc(&prof, 148 * SF_PROF * sizeof(long long)) != cudaSuccess) prof_on = 0;
        }
        stats_i8_fused_kernel<<<grid, SF_NTHR, smem, st>>>(tmA, tmZ, N, D, q, (const double *)zscale, ws, rpc, nchunks, ndb, nct,
                                                           ns, nz, prof_on ? prof : (long long *)nullptr);
        e = cudaGetLastError();
        if (prof_on && e == cudaSuccess) {      // diagnosis only: synchronises
            long long h[148 * SF_PROF];
            cudaStreamSynchronize(st);
            cudaMemcpy(h, prof, sizeof(h), cudaMemcpyDeviceToHost);
            double a[SF_PROF] = {0};
            for (int b = 0; b < grid; ++b)
                for (int k = 0; k < SF_PROF; ++k) a[k] += (double)h[b * SF_PROF + k] / grid;
            double cl = 0, ce = 0;
            for (int w = 0; w < SF_CONV; ++w) {
                cl += a[4 + w] / SF_CONV;
                ce += a[12 + w] / SF_CONV;
            }
            fprintf(stderr, "[i8 stats prof] N=%lld D=%d q=%d ns=%d nz=%d total %.0f clk | producer: empty %.0f | mma: full %.0f tempty %.0f | epilogue(w2): tfull %.0f | converters: loads %.0f empty %.0f\n",
                    N, D, q, ns, nz, a[20], a[0], a[1], a[2], a[3], cl, ce);
        }
        return e;
    }
    if (ZI == nullptr) return cudaErrorInvalidValue;
    dim3 gd((unsigned)((N + 127) / 128), (unsigned)nct);
    digitize_kernel<<<gd, 256, 0, st>>>(N, npad, ldmz, P + q, MZ, zscale, static_cast<signed char *>(ZI));
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    CUtensorMap tmB;
    {   // ZI [npad / 64][nct][224][64]
        cuuint64_t db[3] = {BKB, nkb * nct * (NPL * CT), 1}, sb[2] = {BKB, nkb * nct * (NPL * CT) * BKB};
        cuuint32_t bb[3] = {BKB, (cuuint32_t)(NPL * CT / I8_CL), 1};
        CUresult r = enc(&tmB, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, ZI, db, sb, bb, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
    }
    const int cl = I8_CL;
    const int pair = (cl == 2 && ndb >= 2 && D >= 512) ? 1 : 0;   // tcgen05.mma.cta_group::2
    const size_t smem = si8_smem_bytes(q, pair);
    auto kern = pair ? stats_i8_kernel<I8_CL, true> : stats_i8_kernel<I8_CL>;
    e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const long long nitems = (long long)((ndb + cl - 1) / cl) * nct * nchunks;
    const int grid = (int)(nitems < 148 / cl ? nitems : 148 / cl) * cl;
    // K steps per ring stage (as in K1-i8; ncu on one box: config-3 shard 4.17 -> 3.34 ms, config 2 284 -> 265 us; 3 and 4 are slower)
    const int ks = 2;
    return launch_cluster(kern, grid, NTHR, smem, cl, st, tmA, tmB, N, D, q, (const double *)zscale, ws, rpc, nchunks, ndb,
                          nct, ks);
}

}  // namespace pyvb
