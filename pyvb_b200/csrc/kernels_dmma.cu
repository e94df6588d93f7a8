// FP64 tensor-core (DMMA.8x8x4) kernels fed by TMA -- the throughput path.
//
//   zstep_dmma_kernel<Q>  K1: [O | O.(X-mu)] (rows x D)  @  Gw (D x (P+q))  -> per-row [qprec packed | eta],
//                             written into the MZ row (one bulk store per row)
//                             (WT: per-entry observation weights S, a second TMA tile next to X: [S.O | S.O.(X-mu)])
//   K2 (launch_zsolve below, kernels in kernels_k2*.cu): per-row q x q SPD inverse / solve IN PLACE on the MZ rows,
//                             [qprec | eta] -> [<zz^T> packed | zbar].  Separate kernels on purpose: K2 is a
//                             latency-bound DFMA chain; fused behind K1 it kept the CTA's registers and the
//                             DMMA pipe idle half of the time (profiles/r01_ncu_*.md)
//   stats_dmma_kernel<Q>  K3: [O | O.X]^T (D x rows) @ [<zz^T> | zbar] (rows x (P+q)) -> T1, Bst, Ast
//                             (WT: [S.O | S.O.X]^T, the S sub-tiles next to the X sub-tiles)
//
// Reference arithmetic: nodes/node.py:203-227 (K1), nodes/gaussian.py:117-123 (K2), nodes/nodes_todo.py:50-61 (K3).
//
// Data movement: 2-D TMA tensor tiles (cp.async.bulk.tensor.2d, SASS UTMALDG) with 128-byte (64-byte)
// swizzle for X, 1-D bulk copies (UBLKCP) for contiguous blocks, mbarrier full/empty pipeline; warp 0 of the
// CTA issues the copies ST-1 stages ahead and is otherwise a normal MMA warp.  Math: mma.sync.m8n8k4.f64
// (the only FP64 tensor shape the hardware has; measured 37.0 TF on B200 = the roofline of this path).
// Every fragment load is bank-conflict free: the MMA row <-> tile row assignment is permuted so that the
// four rows a half-warp touches differ in the swizzle bits, and row pitches of the non-swizzled tiles are
// 32 or 96 bytes mod 128.
#include <cuda.h>

#include "common.cuh"
#include "kernels.h"
#include "ptx.cuh"

namespace pyvb {

// ------------------------------------------------------------------ compile-time geometry
__host__ __device__ constexpr int c_tri(int i) { return i * (i + 1) / 2; }
__host__ __device__ constexpr int c_gw_pitch(int q) {
    int p = ((c_tri(q) + 7) & ~7) + q + 1;
    while ((p % 8) != 4) ++p;
    return p;
}
// start of row k in the "even padded" packed lower-triangular layout (every row starts 16-byte aligned)
__host__ __device__ constexpr int c_off(int k) {
    return (k & 1) ? 2 * ((k - 1) / 2 + 1) * ((k - 1) / 2 + 1) : 2 * (k / 2) * (k / 2 + 1);
}
__host__ __device__ constexpr int c_srow(int need) {
    int s = need + (need & 1);
    while ((s % 16) != 2) s += 2;
    return s;
}
__host__ __device__ constexpr int c_max(int a, int b) { return a > b ? a : b; }

// Swizzled X tile with KC doubles per row (KC = 16: 128-byte rows, SWIZZLE_128B; KC = 8: 64-byte rows,
// SWIZZLE_64B).  Byte offset of element (row, col) inside a tile whose base is 1024-byte aligned:
template <int KC>
__device__ __forceinline__ int xt_off(int row, int col) {
    if (KC == 16) return row * 128 + ((((col >> 1) ^ (row & 7)) << 4) | ((col & 1) << 3));
    return row * 64 + ((((col >> 1) ^ ((row >> 1) & 3)) << 4) | ((col & 1) << 3));
}
// MMA row g (0..7) -> tile row inside a group of 8 such that the rows g = 0..3 (one half-warp) differ in the
// swizzle bits: KC = 16 -> {0,2,4,6 | 1,3,5,7}; KC = 8 -> {0,1,4,5 | 2,3,6,7}
template <int KC>
__device__ __forceinline__ int row_perm(int g) {
    if (KC == 16) return ((g & 3) << 1) | (g >> 2);
    return (g & 1) | (((g >> 1) & 1) << 2) | ((g >> 2) << 1);
}

// ------------------------------------------------------------------ host: tensor maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode() {
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
// row-major FP64 matrix [outer][inner] with row pitch `pitch` (doubles); box = box_outer x box_inner
static cudaError_t make_map(CUtensorMap *m, const void *base, uint64_t inner, uint64_t outer, uint64_t pitch,
                            uint32_t box_inner, uint32_t box_outer, CUtensorMapSwizzle sw) {
    EncodeTiledFn enc = get_encode();
    if (!enc) return cudaErrorNotSupported;
    cuuint64_t dims[2] = {inner, outer};
    cuuint64_t strides[1] = {pitch * sizeof(double)};
    cuuint32_t box[2] = {box_inner, box_outer};
    cuuint32_t es[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<void *>(base), dims, strides, box, es,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}

// NCT > 1: the output columns are split into NCT column tiles, one CTA each (q = 64: 268 column groups do not
// fit one CTA's accumulators); consecutive CTAs share the X tile through L2
template <int Q> struct ZC;
// (measured and rejected for q = 16: KC = 8 with 6 stages, 4 stages, one 8-warp CTA per SM, a dedicated producer
//  warp -- all within 1 % of this configuration; what did help was making the kernel persistent)
template <> struct ZC<8>  { static constexpr int WM = 4, WN = 1, RGW = 4, KC = 16, ST = 3, OCC = 2, NCT = 1; };
template <> struct ZC<16> { static constexpr int WM = 4, WN = 1, RGW = 2, KC = 16, ST = 3, OCC = 2, NCT = 1; };
template <> struct ZC<32> { static constexpr int WM = 2, WN = 4, RGW = 2, KC = 8,  ST = 3, OCC = 1, NCT = 1; };
template <> struct ZC<64> { static constexpr int WM = 2, WN = 4, RGW = 2, KC = 8,  ST = 3, OCC = 1, NCT = 4; };

__host__ __device__ constexpr int c_pitch4(int need) {      // smallest pitch >= need with pitch = 4 (mod 8)
    int p = need;
    while ((p % 8) != 4) ++p;
    return p;
}

// ETA = true: only the eta column groups [NGO, NG) (the O.(X - mu) @ <W> part); all warps line up along the rows.
// Used together with the int8 mask contraction (kernels_i8.cu), which produces the qprec columns.
// WT = true: per-entry weights S (same layout as X) -- every stage carries an S tile of the X tile's box and swizzle, and the
// A operand becomes [S.O | S.O.(X - mu)]; at q = 8 (two 4-warp CTAs per SM) the doubled stages leave room for two of them.
template <int Q, bool ETA = false, bool WT = false> struct ZT {
    using C = ZC<Q>;
    static constexpr int P = c_tri(Q), PP = (P + 7) & ~7, NGO = PP / 8, NGE = Q / 8, NG = NGO + NGE;
    // ETA: 2 x Q / 8 tensor-core instructions per 4 x 8 data entries -- the kernel streams X at HBM speed only with many
    // small stages in flight (8 stages, 2 CTAs per SM: > 100 KB outstanding per SM)
    // (ETA always takes 16 data dimensions per stage: its Gw tile is tiny, and half as many barrier round trips per byte)
    static constexpr int WM = ETA ? C::WM * C::WN : C::WM, WN = ETA ? 1 : C::WN, RGW = C::RGW, KC = ETA ? 16 : C::KC;
    static constexpr int ST = ETA ? (Q <= 16 ? 8 : 5) : ((WT && Q == 8) ? 2 : C::ST), OCC = ETA ? 2 : C::OCC;
    static constexpr int NCT = ETA ? 1 : C::NCT;
    static constexpr bool TILED = ETA || NCT > 1;
    static constexpr int CG0 = ETA ? NGO : 0;          // first column group this kernel computes
    static constexpr int NGT = ETA ? NGE : (NG + NCT - 1) / NCT;   // column groups per column tile
    static constexpr int NGW = (NGT + WN - 1) / WN;
    static constexpr int R = WM * RGW * 8;
    static constexpr int NCW = WM * WN;
    static constexpr int NTHR = NCW * 32;       // no dedicated producer warp: warp 0 also issues the copies
    static constexpr int LDG = c_gw_pitch(Q);   // pitch of Gw rows and of the interleaved MZ rows
    static constexpr int MUCOL = PP + Q;
    static constexpr int GP = TILED ? c_pitch4(NGT * 8 + 2) : LDG;   // pitch of the Gw tile in shared memory
    static constexpr int MUL = TILED ? NGT * 8 : MUCOL;              // where mu sits in a shared-memory Gw row
    static constexpr int XT_B = R * KC * 8;     // swizzled X tile (bytes), multiple of 1024
    static constexpr int XS_B = WT ? 2 * XT_B : XT_B;   // data bytes of a stage: the X tile (+ the S tile behind it)
    static constexpr int GS_B = KC * GP * 8;
    static constexpr int OROW = NGT * 8;        // doubles per output row (segment) [packed | pad | eta]
    static constexpr int SROW = c_srow(OROW);   // staging pitch
    static constexpr int MAIN_B = (ST * (XS_B + GS_B) + 15) & ~15;
    static constexpr size_t SMEM = 1024 + (size_t)MAIN_B + (size_t)(P + Q) * 8 + 2 * ST * 8;
    static_assert(XT_B % 1024 == 0, "swizzled tiles must stay 1024-byte aligned");
    static_assert(!WT || OCC * (SMEM + 1024) <= 228 * 1024, "the weighted CTAs of an SM must fit its shared memory");
};

// ------------------------------------------------------------------ Z step, part 1 (K1): tensor-core contraction
// Persistent: every CTA walks over (row tile, column tile) pairs; the TMA pipeline runs CONTINUOUSLY across the
// tiles (the copies of the next tile are in flight while the current one finishes), and the accumulators leave
// straight from registers with 16-byte stores (8 rows x 64 contiguous bytes per warp instruction), so there is no
// staging buffer, no per-tile prologue and no pipeline drain between tiles.
template <int Q, bool ETA, bool WT>
__global__ void __launch_bounds__(ZT<Q, ETA, WT>::NTHR, ZT<Q, ETA, WT>::OCC)
zstep_dmma_kernel(const __grid_constant__ CUtensorMap tmX, long long N, int D, const double *__restrict__ Gw,
                  const double *__restrict__ P0, const double *__restrict__ h0, const double *__restrict__ gl,
                  double *__restrict__ MZ, long long ntiles, const double *__restrict__ cond,
                  const __grid_constant__ CUtensorMap tmS) {
    using T = ZT<Q, ETA, WT>;
    if (cond != nullptr && !(*cond > 0.0)) return;              // conditional (fall-back) launch of the INT8 path
    extern __shared__ unsigned char smem_dyn[];
    // 1024-byte aligned base (swizzled TMA tiles); pointer arithmetic on the __shared__ array keeps the
    // shared address space so that fragment loads compile to LDS, not generic LD
    unsigned char *smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    unsigned char *xs_base = smem;                              // ST swizzled X tiles
    unsigned char *ss_base = smem + T::ST * T::XT_B;            // WT: ST swizzled S tiles
    unsigned char *gs_base = smem + T::ST * T::XS_B;            // ST Gw chunks
    double *p0v = reinterpret_cast<double *>(smem + T::MAIN_B);
    double *h0s = p0v + T::P;
    uint64_t *full = reinterpret_cast<uint64_t *>(h0s + Q);
    uint64_t *empty = full + T::ST;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nk = D / T::KC;
    // tiles of this CTA: blockIdx.x, blockIdx.x + gridDim.x, ...; column tile fastest (neighbours share the X tile in L2)
    const long long my_tiles = (ntiles > (long long)blockIdx.x) ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const long long total_it = my_tiles * nk;                   // pipeline steps of this CTA

    for (int p = tid; p < T::P; p += T::NTHR) {
        int i, j;
        unpack_p(p, i, j);
        p0v[p] = P0[i * Q + j];
    }
    if (tid < Q) h0s[tid] = h0[tid];
    if (tid == 0) {
        tma_prefetch_desc(&tmX);
        if (WT) tma_prefetch_desc(&tmS);
        for (int s = 0; s < T::ST; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], T::NCW);
        }
        mbar_fence_init();
    }
    __syncthreads();

    // ===================== producer role (warp 0, one lane): pipeline step `it` = chunk it % nk of tile it / nk =====
    // (the producer keeps its own (tile, chunk, stage, parity) counters: no divisions on the critical path)
    long long p_tile = blockIdx.x, p_it = 0;
    int p_kc = 0, p_s = 0;
    uint32_t p_ph = 0;
    auto produce = [&]() {
        const int s = p_s;
        const uint32_t ph = p_ph;
        const long long tile = p_tile;
        const int kc = p_kc;
        const int ct = T::NCT > 1 ? (int)((unsigned long long)tile % (unsigned)T::NCT) : 0;
        const long long row0 = (T::NCT > 1 ? (long long)((unsigned long long)tile / (unsigned)T::NCT) : tile) * T::R;
        const int cgb = T::CG0 + ct * T::NGT;
        const int ngt = (T::NG - cgb < T::NGT) ? (T::NG - cgb) : T::NGT;
        const bool need_mu = cgb + ngt > T::NGO;
        mbar_wait(&empty[s], ph ^ 1);
        if (!T::TILED || ETA) {
            // ETA: Gw is the compact [wbar (Q) | mu | pad] array with row pitch GP (pack_weta_kernel): the chunk is one copy
            if (elect_one()) {
                mbar_arrive_expect_tx(&full[s], (uint32_t)(T::XS_B + T::GS_B));
                tma_load_2d(xs_base + s * T::XT_B, &tmX, kc * T::KC, (int)row0, &full[s]);   // rows past N: zero fill
                if (WT) tma_load_2d(ss_base + s * T::XT_B, &tmS, kc * T::KC, (int)row0, &full[s]);
                bulk_g2s(gs_base + s * T::GS_B, Gw + (size_t)kc * T::KC * (ETA ? T::GP : T::LDG), T::GS_B, &full[s]);
            }
        } else {
            // one Gw row segment per lane (+ the mu pair for the tile that holds the eta columns)
            if (elect_one()) {
                mbar_arrive_expect_tx(&full[s], (uint32_t)(T::XS_B + T::KC * (ngt * 64 + (need_mu ? 16 : 0))));
                tma_load_2d(xs_base + s * T::XT_B, &tmX, kc * T::KC, (int)row0, &full[s]);
                if (WT) tma_load_2d(ss_base + s * T::XT_B, &tmS, kc * T::KC, (int)row0, &full[s]);
            }
            __syncwarp();
            if (lane < T::KC) {
                double *dst = reinterpret_cast<double *>(gs_base + s * T::GS_B) + lane * T::GP;
                const double *src = Gw + (size_t)(kc * T::KC + lane) * T::LDG;
                bulk_g2s(dst, src + cgb * 8, (uint32_t)(ngt * 64), &full[s]);
                if (need_mu) bulk_g2s(dst + T::MUL, src + T::MUCOL, 16, &full[s]);
            }
        }
        __syncwarp();
        ++p_it;
        if (++p_kc == nk) {
            p_kc = 0;
            p_tile += gridDim.x;
        }
        if (++p_s == T::ST) {
            p_s = 0;
            p_ph ^= 1;
        }
    };
    if (warp == 0)
        while (p_it < T::ST - 1 && p_it < total_it) produce();

    // ===================== DMMA main loop =====================
    const int wm = warp / T::WN, wn = warp % T::WN;
    const int gid = lane >> 2, qd = lane & 3;
    const int prow = row_perm<T::KC>(gid);                 // tile row (within a group of 8) of MMA row gid
    const int lg0 = wn * T::NGW;                            // first group of this warp inside the tile
    const double tau = gl[PYVB_GL_TAU];
    int xo[T::KC / 4];                                      // swizzled byte offsets of this lane's X element
#pragma unroll
    for (int kk = 0; kk < T::KC / 4; ++kk) xo[kk] = xt_off<T::KC>(wm * T::RGW * 8 + prow, kk * 4 + qd);
    int s = 0;
    uint32_t ph = 0;
    for (long long tl = 0; tl < my_tiles; ++tl) {
        const long long tile = (long long)blockIdx.x + tl * gridDim.x;
        const int ct = T::NCT > 1 ? (int)((unsigned long long)tile % (unsigned)T::NCT) : 0;
        const long long row0 = (T::NCT > 1 ? (long long)((unsigned long long)tile / (unsigned)T::NCT) : tile) * T::R;
        const int cgb = T::CG0 + ct * T::NGT;
        const int ngt = (T::NG - cgb < T::NGT) ? (T::NG - cgb) : T::NGT;
        const int cg0 = cgb + lg0;
        const int ncg = (ngt - lg0 < T::NGW) ? (ngt - lg0) : T::NGW;
        double acc[T::RGW][T::NGW][2];
#pragma unroll
        for (int rg = 0; rg < T::RGW; ++rg)
#pragma unroll
            for (int j = 0; j < T::NGW; ++j) acc[rg][j][0] = acc[rg][j][1] = 0.0;
        for (int kc = 0; kc < nk; ++kc) {
            if (warp == 0 && p_it < total_it) produce();       // keeps the pipeline ST - 1 steps ahead
            mbar_wait(&full[s], ph);
            const unsigned char *xs = xs_base + s * T::XT_B;
            const unsigned char *ss = ss_base + s * T::XT_B;
            const double *gs = reinterpret_cast<const double *>(gs_base + s * T::GS_B) + qd * T::GP;
#pragma unroll
            for (int kk = 0; kk < T::KC / 4; ++kk) {
                const double *grow = gs + kk * 4 * T::GP;
                const double muv = grow[T::MUL];
                double ao[T::RGW], ax[T::RGW];
#pragma unroll
                for (int rg = 0; rg < T::RGW; ++rg) {
                    // rows of group rg sit 8 tile rows further: +8 rows keeps (row & 7) and ((row >> 1) & 3)
                    const double x = *reinterpret_cast<const double *>(xs + xo[kk] + rg * 8 * T::KC * 8);
                    const bool ob = (x == x);          // NaN = not observed
                    if (WT) {                          // (the weight of an unobserved entry is not read: it may be NaN)
                        const double w = *reinterpret_cast<const double *>(ss + xo[kk] + rg * 8 * T::KC * 8);
                        ao[rg] = ob ? w : 0.0;
                        ax[rg] = ob ? w * (x - muv) : 0.0;
                    } else {
                        ao[rg] = ob ? 1.0 : 0.0;
                        ax[rg] = ob ? (x - muv) : 0.0;
                    }
                }
#pragma unroll
                for (int j = 0; j < T::NGW; ++j) {
                    if (T::WN > 1 && j >= ncg) continue;
                    const int cg = cg0 + j;
                    const double b = grow[(lg0 + j) * 8 + gid];
                    const bool otype = cg < T::NGO;
#pragma unroll
                    for (int rg = 0; rg < T::RGW; ++rg)
                        dmma884(acc[rg][j][0], acc[rg][j][1], otype ? ao[rg] : ax[rg], b);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);
            if (++s == T::ST) {
                s = 0;
                ph ^= 1;
            }
        }
        // ---- epilogue of the tile: qprec = P0 + tau*acc, eta = h0 + tau*acc, registers -> MZ rows
#pragma unroll
        for (int rg = 0; rg < T::RGW; ++rg) {
            const long long row = row0 + wm * T::RGW * 8 + rg * 8 + prow;
            if (row >= N) continue;
            double *orow = MZ + row * T::LDG;
#pragma unroll
            for (int j = 0; j < T::NGW; ++j) {
                if (T::WN > 1 && j >= ncg) continue;
                const int cg = cg0 + j;
                const int c = cg * 8 + 2 * qd;
                double2 v;
                if (cg < T::NGO) {   // packed qprec columns; the pad columns [P, PP) come out as exact zeros
                    v.x = (c < T::P) ? fma(tau, acc[rg][j][0], p0v[c]) : 0.0;
                    v.y = (c + 1 < T::P) ? fma(tau, acc[rg][j][1], p0v[c + 1]) : 0.0;
                } else {
                    v.x = fma(tau, acc[rg][j][0], h0s[c - T::PP]);
                    v.y = fma(tau, acc[rg][j][1], h0s[c + 1 - T::PP]);
                }
                *reinterpret_cast<double2 *>(orow + c) = v;
            }
        }
    }
}

// pure-DMMA loop: the FP64 tensor roofline of the box (see pyvb_bench_dmma_f64)
__global__ void __launch_bounds__(256) bench_dmma_kernel(double *out, int iters, double a, double b) {
    double c[8][2];
#pragma unroll
    for (int i = 0; i < 8; ++i) c[i][0] = c[i][1] = threadIdx.x * 1e-9;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i) dmma884(c[i][0], c[i][1], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += c[i][0] + c[i][1];
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

cudaError_t launch_bench_dmma(int blocks, int iters, double *scratch, cudaStream_t st) {
    bench_dmma_kernel<<<blocks, 256, 0, st>>>(scratch, iters, 1.0000001, 0.9999999);
    return cudaGetLastError();
}

bool dmma_supported(int D, int q) { return (q == 8 || q == 16 || q == 32 || q == 64) && D >= 16 && (D % 16) == 0; }

template <int Q, bool ETA>
static cudaError_t launch_k1_q(long long N, int D, const double *X, long long ldx, const double *Gw, const double *P0,
                               const double *h0, double *gl, double *MZ, cudaStream_t st) {
    using T = ZT<Q, ETA>;
    CUtensorMap tmX;
    cudaError_t e = make_map(&tmX, X, (uint64_t)D, (uint64_t)N, (uint64_t)ldx, T::KC, T::R,
                             T::KC == 16 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(zstep_dmma_kernel<Q, ETA, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T::SMEM);
    if (e != cudaSuccess) return e;
    const long long ntiles = ((N + T::R - 1) / T::R) * T::NCT;
    const long long blocks = ntiles < 148LL * T::OCC ? ntiles : 148LL * T::OCC;
    zstep_dmma_kernel<Q, ETA, false><<<(unsigned)blocks, T::NTHR, T::SMEM, st>>>(tmX, N, D, Gw, P0, h0, gl, MZ, ntiles, nullptr,
                                                                               tmX);
    return cudaGetLastError();
}

// compact copy of the [wbar | mu] columns of Gw: weta[d][0..q) = wbar_d, weta[d][q] = mu_d, zero pad to the pitch
__global__ void __launch_bounds__(256)
pack_weta_kernel(int D, int q, int ldg, int pp, int gp, const double *__restrict__ Gw, double *__restrict__ weta) {
    const int e = blockIdx.x * 256 + threadIdx.x;
    if (e >= D * gp) return;
    const int d = e / gp, c = e - d * gp;
    weta[e] = (c <= q) ? Gw[(size_t)d * ldg + pp + c] : 0.0;
}
int zstep_eta_pitch(int q) { return c_pitch4(q + 2); }

// the eta columns alone (see ZT<Q, true>): MZ rows get [.. | eta] with the qprec columns left untouched.
// weta: scratch of D * zstep_eta_pitch(q) doubles
cudaError_t launch_zstep_eta_dmma(long long N, int D, int q, const double *X, long long ldx, const double *Gw,
                                  double *weta, const double *P0, const double *h0, double *gl, double *MZ,
                                  cudaStream_t st) {
    if (N <= 0) return cudaSuccess;
    const int gp = zstep_eta_pitch(q);
    pack_weta_kernel<<<(D * gp + 255) / 256, 256, 0, st>>>(D, q, c_gw_pitch(q), (c_tri(q) + 7) & ~7, gp, Gw, weta);
    switch (q) {
        case 16: return launch_k1_q<16, true>(N, D, X, ldx, weta, P0, h0, gl, MZ, st);
        case 32: return launch_k1_q<32, true>(N, D, X, ldx, weta, P0, h0, gl, MZ, st);
        case 64: return launch_k1_q<64, true>(N, D, X, ldx, weta, P0, h0, gl, MZ, st);
    }
    return cudaErrorNotSupported;
}

template <int Q, bool WT>
static cudaError_t launch_k1w_q(long long N, int D, const double *X, long long ldx, const double *S, long long lds,
                                const double *Gw, const double *P0, const double *h0, double *gl, double *MZ,
                                cudaStream_t st, const double *cond) {
    using T = ZT<Q, false, WT>;
    const CUtensorMapSwizzle sw = T::KC == 16 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    CUtensorMap tmX, tmS;
    cudaError_t e = make_map(&tmX, X, (uint64_t)D, (uint64_t)N, (uint64_t)ldx, T::KC, T::R, sw);
    if (e != cudaSuccess) return e;
    tmS = tmX;                                                  // (not read without weights)
    if (WT) e = make_map(&tmS, S, (uint64_t)D, (uint64_t)N, (uint64_t)lds, T::KC, T::R, sw);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(zstep_dmma_kernel<Q, false, WT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T::SMEM);
    if (e != cudaSuccess) return e;
    const long long ntiles = ((N + T::R - 1) / T::R) * T::NCT;
    const long long blocks = ntiles < 148LL * ZC<Q>::OCC ? ntiles : 148LL * ZC<Q>::OCC;
    zstep_dmma_kernel<Q, false, WT><<<(unsigned)blocks, T::NTHR, T::SMEM, st>>>(tmX, N, D, Gw, P0, h0, gl, MZ, ntiles, cond,
                                                                              tmS);
    return cudaGetLastError();
}

template <int Q>
static cudaError_t launch_zstep_q(long long N, int D, const double *X, long long ldx, const double *S, long long lds,
                                  const double *Gw, const double *P0, const double *h0, double *gl, double *MZ, double *Sig,
                                  double *logdet, double *zsums, int k1_only, cudaStream_t st, const double *cond) {
    cudaError_t e = S ? launch_k1w_q<Q, true>(N, D, X, ldx, S, lds, Gw, P0, h0, gl, MZ, st, cond)
                      : launch_k1w_q<Q, false>(N, D, X, ldx, S, lds, Gw, P0, h0, gl, MZ, st, cond);
    if (e != cudaSuccess || k1_only) return e;
    return launch_zsolve(N, Q, MZ, Sig, logdet, gl, zsums, st, cond);
}

cudaError_t launch_zstep_dmma(long long N, int D, int q, const double *X, long long ldx, const double *Gw, int ldg,
                              const double *P0, const double *h0, double *gl, double *MZ, double *Sig,
                              double *logdet, double *zsums, int k1_only, cudaStream_t st, const double *cond,
                              const double *S, long long lds) {
    if (N <= 0) return cudaSuccess;
    if (ldg != c_gw_pitch(q)) return cudaErrorInvalidValue;
    switch (q) {
        case 8: return launch_zstep_q<8>(N, D, X, ldx, S, lds, Gw, P0, h0, gl, MZ, Sig, logdet, zsums, k1_only, st, cond);
        case 16: return launch_zstep_q<16>(N, D, X, ldx, S, lds, Gw, P0, h0, gl, MZ, Sig, logdet, zsums, k1_only, st, cond);
        case 32: return launch_zstep_q<32>(N, D, X, ldx, S, lds, Gw, P0, h0, gl, MZ, Sig, logdet, zsums, k1_only, st, cond);
        case 64: return launch_zstep_q<64>(N, D, X, ldx, S, lds, Gw, P0, h0, gl, MZ, Sig, logdet, zsums, k1_only, st, cond);
    }
    return cudaErrorNotSupported;
}

// K2, one kernel per q (DESIGN.md 5 has the measurements behind the choice): thread per matrix at q = 8 (kernels_k2t.cu),
// Gauss-Jordan in registers at q = 16, 32 (kernels_k2g.cu), blocked symmetric sweep on swizzled tiles at q = 64 (kernels_k2s.cu)
void zsolve_partials(long long N, int q, int &nblk, int &kw) {
    nblk = kw = 0;
    if (N <= 0) return;
    switch (q) {
        case 8: kw = zsolve_tpm_kw(q), nblk = zsolve_tpm_blocks(N, q); break;
        case 16:
        case 32: kw = zsolve_gj_kw(q), nblk = zsolve_gj_blocks(N, q); break;
        case 64: kw = zsolve_sweep_kw(q), nblk = zsolve_sweep_blocks(N, q); break;
    }
}

cudaError_t launch_zsolve(long long N, int q, double *MZ, double *Sig, double *logdet, double *gl, double *zsums,
                          cudaStream_t st, const double *cond, I8Check chk) {
    if (N <= 0) return cudaSuccess;
    // the Gauss-Jordan and sweep kernels move the rows with bulk copies: 16-byte aligned rows (the pitch is a multiple of 32 bytes)
    const bool aligned = (reinterpret_cast<uintptr_t>(MZ) & 15) == 0;
    switch (q) {
        case 8: return launch_zsolve_tpm(N, q, MZ, Sig, logdet, gl, zsums, st, cond, chk);
        case 16:
        case 32:
            if (!aligned) return cudaErrorMisalignedAddress;
            return launch_zsolve_gj(N, q, MZ, Sig, logdet, gl, zsums, st, cond, chk);
        case 64:
            if (!aligned) return cudaErrorMisalignedAddress;
            return launch_zsolve_sweep(N, q, MZ, Sig, logdet, gl, zsums, st, cond, chk);
    }
    return cudaErrorNotSupported;
}

// ------------------------------------------------------------------ statistics kernel (K3)
template <int Q> struct SC;
template <> struct SC<8>  { static constexpr int WM = 4, WN = 1, RGW = 4, KC = 16, ST = 3, OCC = 1, NCT = 1; };
template <> struct SC<16> { static constexpr int WM = 8, WN = 1, RGW = 2, KC = 16, ST = 3, OCC = 1, NCT = 1; };
template <> struct SC<32> { static constexpr int WM = 2, WN = 4, RGW = 2, KC = 8,  ST = 3, OCC = 1, NCT = 1; };
template <> struct SC<64> { static constexpr int WM = 2, WN = 4, RGW = 2, KC = 8,  ST = 3, OCC = 1, NCT = 4; };

// XO = true: only the X-type statistics Ast = (O.X)^T Zbar (the mask-type ones come from the INT8 kernel, kernels_i8.cu):
// all warps line up along the data dimensions, the MZ tile is just the zbar columns (+ the 4 pad columns that follow
// them, which keeps the shared-memory pitch = 4 (mod 8): conflict-free B fragments)
// WT = true: per-entry weights S (same layout as X): every stage carries the S sub-tiles behind the X sub-tiles, and the A
// operand becomes [S.O | S.O.X]
template <int Q, bool XO = false, bool WT = false> struct STT {
    using C = SC<Q>;
    static constexpr int P = c_tri(Q), PP = (P + 7) & ~7;
    static constexpr int NGO = XO ? 0 : (PP + Q) / 8, NGX = Q / 8, NG = NGO + NGX;   // O-type: [<zz^T> | pad | zbar]; X-type: zbar
    static constexpr int WM = XO ? C::WM * C::WN : C::WM, WN = XO ? 1 : C::WN, RGW = C::RGW, KC = XO ? 16 : C::KC, ST = XO ? 4 : C::ST;
    static constexpr int NCT = XO ? 1 : C::NCT;
    static constexpr bool TILED = NCT > 1;      // output columns split over NCT CTAs (q = 64)
    static constexpr int NGT = (NG + NCT - 1) / NCT;
    static constexpr int NGW = (NGT + WN - 1) / WN;
    static constexpr int DT = WM * RGW * 8;     // data dimensions per CTA (multiple of 16)
    static constexpr int NSUB = DT / 16;        // swizzled X sub-tiles [KC rows][16 d] per stage
    static constexpr int NCW = WM * WN;
    static constexpr int NTHR = NCW * 32;       // warp 0 doubles as the producer
    static constexpr int VP = c_gw_pitch(Q);    // pitch of the MZ rows in global memory
    static constexpr int VPS = XO ? Q + 4 : (TILED ? c_pitch4(NGT * 8) : VP);   // ... and of the (column tile of the) rows in shared memory
    static constexpr bool BTILE = XO || VP <= 256;    // MZ tile through one tensor copy (box dims are limited to 256)
    static constexpr int SUB_B = KC * 128;
    static constexpr int AS_B = NSUB * SUB_B, VS_B = KC * VPS * 8;
    static constexpr int AW_B = WT ? 2 * AS_B : AS_B;   // data bytes of a stage: the X sub-tiles (+ the S sub-tiles)
    static constexpr size_t SMEM = 1024 + (size_t)ST * (AW_B + VS_B) + 2 * ST * 8;
    static_assert(SMEM <= 227 * 1024, "one CTA must fit the shared memory of an SM");
    static_assert(DT % 16 == 0 && SUB_B % 1024 == 0, "sub-tiles must stay 1024-byte aligned");
};

// grid.x = number of d tiles, grid.y = row chunks.  Partial sums go to ws[chunk][stat layout]; a second
// kernel adds the chunks in a fixed order (deterministic).
template <int Q, bool XO, bool WT>
__global__ void __launch_bounds__(STT<Q, XO, WT>::NTHR, SC<Q>::OCC)
stats_dmma_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmV, long long N, int D,
                  const double *__restrict__ MZ, double *__restrict__ ws, long long rows_per_chunk,
                  const double *__restrict__ cond, const __grid_constant__ CUtensorMap tmS) {
    using T = STT<Q, XO, WT>;
    if (cond != nullptr && !(*cond > 0.0)) return;              // conditional (fall-back) launch of the INT8 statistics
    extern __shared__ unsigned char smem_dyn[];
    // 1024-byte aligned base (swizzled TMA tiles); pointer arithmetic on the __shared__ array keeps the
    // shared address space so that fragment loads compile to LDS, not generic LD
    unsigned char *smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    unsigned char *as_base = smem;                          // ST x NSUB swizzled X sub-tiles
    unsigned char *ws_base = smem + T::ST * T::AS_B;        // WT: ST x NSUB swizzled S sub-tiles
    unsigned char *vs_base = smem + T::ST * T::AW_B;        // ST MZ tiles [KC][VP]
    uint64_t *full = reinterpret_cast<uint64_t *>(smem + T::ST * (T::AW_B + T::VS_B));
    uint64_t *empty = full + T::ST;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr bool virt = false;
    const int ct = T::TILED ? (int)(blockIdx.x % T::NCT) : 0;            // column tile
    const int cgb = ct * T::NGT;
    const int ngt = (T::NG - cgb < T::NGT) ? (T::NG - cgb) : T::NGT;
    // MZ columns the tile needs: its O-type groups (the X-type groups re-use the zbar columns, which are the
    // last O-type groups of the same -- the last -- tile)
    const int vcols = (((cgb + ngt < T::NGO) ? (cgb + ngt) : T::NGO) - cgb) * 8;
    const int d0 = (int)(blockIdx.x / T::NCT) * T::DT;
    const int dvalid = (D - d0 < T::DT) ? (D - d0) : T::DT;
    const int nsub = dvalid / 16;
    const long long r0 = (long long)blockIdx.y * rows_per_chunk;
    long long r1 = r0 + rows_per_chunk;
    if (r1 > N) r1 = N;
    const int nsteps = (r1 > r0) ? (int)((r1 - r0 + T::KC - 1) / T::KC) : 0;

    if (tid == 0) {
        tma_prefetch_desc(&tmX);
        tma_prefetch_desc(&tmV);
        if (WT) tma_prefetch_desc(&tmS);
        for (int s = 0; s < T::ST; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], T::NCW);
        }
        mbar_fence_init();
    }
    __syncthreads();

    // ===================== producer role (warp 0) =====================
    auto produce = [&](int it) {
        const int s = it % T::ST;
        const uint32_t ph = (uint32_t)((it / T::ST) & 1);
        mbar_wait(&empty[s], ph ^ 1);
        const long long nb = r0 + (long long)it * T::KC;     // chunk boundaries are multiples of KC; rows >= N are
        double *vs = reinterpret_cast<double *>(vs_base + s * T::VS_B);   // zero filled by the tensor copies
        if (T::BTILE) {
            if (elect_one()) {        // (not `lane == 0`: that wraps every TMA instruction in an election loop)
                mbar_arrive_expect_tx(&full[s], (uint32_t)((WT ? 2 : 1) * nsub * T::SUB_B + T::VS_B));
                for (int t = 0; t < nsub; ++t)
                    tma_load_2d(as_base + s * T::AS_B + t * T::SUB_B, &tmX, d0 + t * 16, (int)nb, &full[s]);
                if (WT)
                    for (int t = 0; t < nsub; ++t)
                        tma_load_2d(ws_base + s * T::AS_B + t * T::SUB_B, &tmS, d0 + t * 16, (int)nb, &full[s]);
                tma_load_2d(vs, &tmV, 0, (int)nb, &full[s]);
            }
        } else {
            const int nval = (N - nb < T::KC) ? (int)(N - nb) : T::KC;
            const int wcols = T::TILED ? vcols : (T::PP + Q);
            for (int r = nval; r < T::KC; ++r)
                for (int c = lane; c < T::VPS; c += 32) vs[r * T::VPS + c] = 0.0;
            __syncwarp();
            if (elect_one()) {
                mbar_arrive_expect_tx(&full[s], (uint32_t)((WT ? 2 : 1) * nsub * T::SUB_B + nval * wcols * 8));
                for (int t = 0; t < nsub; ++t)
                    tma_load_2d(as_base + s * T::AS_B + t * T::SUB_B, &tmX, d0 + t * 16, (int)nb, &full[s]);
                if (WT)
                    for (int t = 0; t < nsub; ++t)
                        tma_load_2d(ws_base + s * T::AS_B + t * T::SUB_B, &tmS, d0 + t * 16, (int)nb, &full[s]);
            }
            __syncwarp();
            if (lane < nval)
                bulk_g2s(vs + lane * T::VPS, MZ + (nb + lane) * T::VP + cgb * 8, (uint32_t)(wcols * 8), &full[s]);
        }
        __syncwarp();
    };
    if (warp == 0)
        for (int it = 0; it < T::ST - 1 && it < nsteps; ++it) produce(it);

    // ===================== DMMA main loop =====================
    const int wm = warp / T::WN, wn = warp % T::WN;
    const int gid = lane >> 2, qd = lane & 3;
    const int lg0 = wn * T::NGW;                            // first group of this warp inside the column tile
    const int cg0 = cgb + lg0;
    const int ncg = (ngt - lg0 < T::NGW) ? (ngt - lg0) : T::NGW;
    const int blk0 = wm * T::RGW;                           // first group of 8 d's of this warp inside the tile
    // MMA row gid -> d inside a 16-wide sub-tile (first or second half chosen by the group parity): the four
    // rows of a half-warp must sit in chunks that differ in bit 2 -> {0,1,8,9 | 2,3,10,11} (+4 for odd groups)
    const int dperm = (gid & 1) + 8 * ((gid >> 1) & 1) + 2 * (gid >> 2);
    const bool active = virt ? (wm == 0) : (blk0 * 8 < dvalid);   // warp-uniform
    double acc[T::RGW][T::NGW][2];
#pragma unroll
    for (int rg = 0; rg < T::RGW; ++rg)
#pragma unroll
        for (int j = 0; j < T::NGW; ++j) acc[rg][j][0] = acc[rg][j][1] = 0.0;
    int aoff[T::RGW];                                       // sub-tile offset + swizzle-independent part
    int dl[T::RGW];
#pragma unroll
    for (int rg = 0; rg < T::RGW; ++rg) {
        const int blk = blk0 + rg;
        dl[rg] = 4 * (blk & 1) + dperm;
        aoff[rg] = (blk >> 1) * T::SUB_B + ((dl[rg] & 1) << 3);
    }
    {
        int s = 0;
        uint32_t ph = 0;
        for (int it = 0; it < nsteps; ++it) {
            if (warp == 0 && it + T::ST - 1 < nsteps) produce(it + T::ST - 1);
            mbar_wait(&full[s], ph);
            if (active) {
                const unsigned char *as = as_base + s * T::AS_B;
                const unsigned char *wsb = ws_base + s * T::AS_B;
                const double *vs = reinterpret_cast<const double *>(vs_base + s * T::VS_B) + qd * T::VPS + gid;
#pragma unroll
                for (int kk = 0; kk < T::KC / 4; ++kk) {
                    const int row = kk * 4 + qd;
                    double ao[T::RGW], ax[T::RGW];
#pragma unroll
                    for (int rg = 0; rg < T::RGW; ++rg) {
                        if (virt) {
                            ao[rg] = (rg == 0 && gid == 0) ? 1.0 : 0.0;
                            ax[rg] = 0.0;
                        } else {
                            const bool in = (blk0 + rg) * 8 < dvalid;
                            const int off = aoff[rg] + row * 128 + ((((dl[rg] >> 1) ^ (row & 7))) << 4);
                            const double x = *reinterpret_cast<const double *>(as + off);   // stale data if !in
                            const bool ob = in && (x == x);
                            if (WT) {
                                const double w = *reinterpret_cast<const double *>(wsb + off);
                                ao[rg] = ob ? w : 0.0;
                                ax[rg] = ob ? w * x : 0.0;
                            } else {
                                ao[rg] = ob ? 1.0 : 0.0;
                                ax[rg] = ob ? x : 0.0;
                            }
                        }
                    }
#pragma unroll
                    for (int j = 0; j < T::NGW; ++j) {
                        if (T::WN > 1 && j >= ncg) continue;
                        const int cg = cg0 + j;
                        const bool otype = cg < T::NGO;
                        // X-type groups re-use the zbar columns of the tile
                        const int col = XO ? cg * 8 : ((otype ? cg * 8 : (T::PP + (cg - T::NGO) * 8)) - cgb * 8);
                        const double b = vs[kk * 4 * T::VPS + col];
#pragma unroll
                        for (int rg = 0; rg < T::RGW; ++rg)
                            dmma884(acc[rg][j][0], acc[rg][j][1], otype ? ao[rg] : ax[rg], b);
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);
            if (++s == T::ST) {
                s = 0;
                ph ^= 1;
            }
        }
    }
    if (!active) return;
    // ===================== store partial sums =====================
    const StatLayout L(D, Q);
    double *out = ws + (size_t)blockIdx.y * L.len;
#pragma unroll
    for (int rg = 0; rg < T::RGW; ++rg) {
        const int d = d0 + ((blk0 + rg) >> 1) * 16 + dl[rg];
#pragma unroll
        for (int j = 0; j < T::NGW; ++j) {
            if (T::WN > 1 && j >= ncg) continue;
            const int cg = cg0 + j;
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int c = cg * 8 + 2 * qd + e;
                const double v = acc[rg][j][e];
                if (virt) {
                    if (rg == 0 && gid == 0 && cg < T::NGO) {
                        if (c < T::P) out[L.S + c] = v;
                        else if (c >= T::PP) out[L.zsum + (c - T::PP)] = v;
                    }
                } else if (d < D && (blk0 + rg) * 8 < dvalid) {
                    if (cg < T::NGO) {
                        if (c < T::P) out[L.t1 + (size_t)d * T::P + c] = v;
                        else if (c >= T::PP) out[L.bst + (size_t)d * Q + (c - T::PP)] = v;
                    } else {
                        out[L.ast + (size_t)d * Q + (c - T::NGO * 8)] = v;
                    }
                }
            }
        }
    }
}

static long long gcdll(long long a, long long b) { return b ? gcdll(b, a % b) : a; }

int stats_dmma_nchunks(long long N, int D, int q) {
    int kc = 16, dt = 128, nct = 1;
    if (q >= 32) { kc = 8; dt = 32; }
    if (q == 64) nct = SC<64>::NCT;
    const int ndt = ((D + dt - 1) / dt) * nct;               // CTAs per row chunk
    // CTAs = ndt * nchunks should be a whole number of waves of 148 SMs (1 CTA/SM): nchunks = k * step
    const long long step = 148 / gcdll(148, ndt);
    long long by_rows = (N + 64LL * kc - 1) / (64LL * kc);     // at least 64 pipeline steps per chunk
    long long k = (4 * 148LL) / (step * ndt);                  // ~4 waves
    if (k < 1) k = 1;
    long long c = k * step;
    if (c > by_rows) c = (by_rows / step) * step;              // few rows: fewer whole waves ...
    if (c < 1) c = by_rows < 1 ? 1 : by_rows;                  // ... or simply one chunk per 64 steps
    if (c > 1024) c = 1024;
    return (int)c;
}

template <int Q, bool XO = false, bool WT = false>
static cudaError_t launch_stats_q(long long N, int D, const double *X, long long ldx, const double *MZ, double *ws,
                                  int nchunks, cudaStream_t st, const double *cond = nullptr, const double *S = nullptr,
                                  long long lds = 0) {
    using T = STT<Q, XO, WT>;
    CUtensorMap tmX, tmV, tmS;
    cudaError_t e = make_map(&tmX, X, (uint64_t)D, (uint64_t)N, (uint64_t)ldx, 16, T::KC, CU_TENSOR_MAP_SWIZZLE_128B);
    if (e != cudaSuccess) return e;
    tmS = tmX;                                                  // (not read without weights)
    if (WT) e = make_map(&tmS, S, (uint64_t)D, (uint64_t)N, (uint64_t)lds, 16, T::KC, CU_TENSOR_MAP_SWIZZLE_128B);
    if (e != cudaSuccess) return e;
    if (XO) {   // the zbar columns [PP, PP + Q) and the 4 pad columns behind them
        e = make_map(&tmV, MZ + T::PP, (uint64_t)(Q + 4), (uint64_t)N, (uint64_t)T::VP, Q + 4, T::KC, CU_TENSOR_MAP_SWIZZLE_NONE);
        if (e != cudaSuccess) return e;
    } else if (T::BTILE) {
        e = make_map(&tmV, MZ, (uint64_t)T::VP, (uint64_t)N, (uint64_t)T::VP, T::VP, T::KC, CU_TENSOR_MAP_SWIZZLE_NONE);
        if (e != cudaSuccess) return e;
    } else {
        tmV = tmX;   // unused
    }
    e = cudaFuncSetAttribute(stats_dmma_kernel<Q, XO, WT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T::SMEM);
    if (e != cudaSuccess) return e;
    long long rpc = (N + nchunks - 1) / nchunks;
    rpc = ((rpc + T::KC - 1) / T::KC) * T::KC;                 // chunk boundaries on pipeline-step boundaries
    if (rpc < T::KC) rpc = T::KC;
    const int ndt = ((D + T::DT - 1) / T::DT) * T::NCT;
    dim3 grid((unsigned)ndt, (unsigned)nchunks);
    stats_dmma_kernel<Q, XO, WT><<<grid, T::NTHR, T::SMEM, st>>>(tmX, tmV, N, D, MZ, ws, rpc, cond, tmS);
    return cudaGetLastError();
}

// Ast alone, `nchunks` row chunks of `rpc` rows (a multiple of 64: the INT8 kernel's chunks) into ws[chunk][stat layout]
cudaError_t launch_stats_x_dmma(long long N, int D, int q, const double *X, long long ldx, const double *MZ,
                                double *ws_main, int nchunks, cudaStream_t st) {
    if (N <= 0) return cudaSuccess;
    switch (q) {
        case 16: return launch_stats_q<16, true>(N, D, X, ldx, MZ, ws_main, nchunks, st);
        case 32: return launch_stats_q<32, true>(N, D, X, ldx, MZ, ws_main, nchunks, st);
        case 64: return launch_stats_q<64, true>(N, D, X, ldx, MZ, ws_main, nchunks, st);
    }
    return cudaErrorNotSupported;
}

cudaError_t launch_stats_dmma(long long N, int D, int q, const double *X, long long ldx, const double *MZ,
                              double *ws_main, int nchunks, cudaStream_t st, const double *cond, const double *S,
                              long long lds) {
    if (N <= 0) return cudaSuccess;
    if (S) {
        switch (q) {
            case 8: return launch_stats_q<8, false, true>(N, D, X, ldx, MZ, ws_main, nchunks, st, cond, S, lds);
            case 16: return launch_stats_q<16, false, true>(N, D, X, ldx, MZ, ws_main, nchunks, st, cond, S, lds);
            case 32: return launch_stats_q<32, false, true>(N, D, X, ldx, MZ, ws_main, nchunks, st, cond, S, lds);
            case 64: return launch_stats_q<64, false, true>(N, D, X, ldx, MZ, ws_main, nchunks, st, cond, S, lds);
        }
        return cudaErrorNotSupported;
    }
    switch (q) {
        case 8: return launch_stats_q<8>(N, D, X, ldx, MZ, ws_main, nchunks, st, cond);
        case 16: return launch_stats_q<16>(N, D, X, ldx, MZ, ws_main, nchunks, st, cond);
        case 32: return launch_stats_q<32>(N, D, X, ldx, MZ, ws_main, nchunks, st, cond);
        case 64: return launch_stats_q<64>(N, D, X, ldx, MZ, ws_main, nchunks, st, cond);
    }
    return cudaErrorNotSupported;
}

}  // namespace pyvb
