// K2, thread per matrix (FP64 rows at q = 8, FP32 rows at q = 16): batched q x q SPD inverse / solve where every LANE owns
// one matrix.
//
// Replaces cho_factor / cho_solve(., I) / dot(qcov, .) / q_ln_det of Gaussian.update (nodes/gaussian.py:117-123).
// A warp takes 32 consecutive rows of MZ.  The rows are loaded cooperatively (coalesced) into shared memory as
// [element][33] (element-major, one matrix per column, pitch 33: conflict-free both for the cooperative copies and for
// the per-lane accesses), then each lane runs the whole factorisation on ITS matrix with 8 x 8 triangles held in
// registers -- straight-line, fully unrolled DFMA code, no shuffles, no divergence, one rsqrt chain shared by the 32
// matrices of the warp.  Per 16 x 16 matrix: potrf / trtri / lauum on 8 x 8 blocks,
//     L00, X00 = L00^-1 | L10 = A10 X00^T | A11 -= L10 L10^T | L11, X11 | X10 = -X11 (L10 X00) | Sigma = X^T X,
// off-diagonal blocks streamed row- or column-wise through shared memory.  ~155 instructions per matrix (the
// one-warp-per-matrix kernels need 1400-2000): the kernel runs at the HBM rate instead of the issue rate.
#include <cuda_bf16.h>

#include "common.cuh"
#include "kernels.h"
#include "ptx.cuh"

namespace pyvb {

namespace {

__host__ __device__ constexpr int t_tri(int i) { return i * (i + 1) / 2; }
__host__ __device__ constexpr int t_idx(int i, int j) { return i * (i + 1) / 2 + j; }   // i >= j
__host__ __device__ constexpr int t_pitch(int q) {
    int p = ((t_tri(q) + 7) & ~7) + q + 1;
    while ((p % 8) != 4) ++p;
    return p;
}

// Outer row / column loops of the 16 x 16 phases: rolled, two iterations in flight.  Fully unrolled the body was ~70 KB of
// code -- instruction-cache misses were the second largest stall of the kernel (ncu: no_instruction) -- and the scheduler
// hoisted loads until it spilled; rolled: 0.89 -> 0.81 ms per 1M rows (1 / 2 / 4 iterations in flight: 0.808 / 0.807 / 0.826).
constexpr int TPM_ROLL = 2;

template <int Q, bool F32> struct TIO;
template <int Q> struct TIO<Q, false> {
    using type = double;
    static constexpr int PITCH = t_pitch(Q), POFF = 0, ZOFF = (t_tri(Q) + 7) & ~7;
};
template <int Q> struct TIO<Q, true> {
    using type = float;
    static constexpr int PITCH = (Q + t_tri(Q) + 63) & ~63, POFF = Q, ZOFF = 0;
};

template <int Q> struct TK {
    static constexpr int P = t_tri(Q), PP = (P + 7) & ~7, OROW = PP + Q;
    static constexpr int NE = P + Q;                      // elements per matrix in shared memory: packed | eta, then z
    static constexpr int LP = 33;                         // lane pitch
    static constexpr int WARPS = 5;
    static constexpr int WARP_D = NE * LP;
    static constexpr int NU = (P + 31) / 32;              // packed elements per lane in the cooperative copies
    static constexpr int KW = 2 * OROW + PYVB_ZS_EXTRA;   // [column sums OROW | 4 scalars | column maxima of |.| OROW]
    static constexpr size_t SMEM = (size_t)WARPS * WARP_D * 8 + (size_t)WARPS * KW * 8;
};

// 8 x 8 lower triangle in registers (packed, A[t_idx(i, j)]).  In: SPD block.  Out: X = chol(A)^-1 (lower triangular);
// lp *= prod_k 1/l_kk.
__device__ __forceinline__ void chol_inv8(double (&A)[36], double &lp) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const double rinv = rsqrt(A[t_idx(k, k)]);
        lp *= rinv;
        A[t_idx(k, k)] = rinv;
#pragma unroll
        for (int i = k + 1; i < 8; ++i) A[t_idx(i, k)] *= rinv;
#pragma unroll
        for (int j = k + 1; j < 8; ++j)
#pragma unroll
            for (int i = j; i < 8; ++i) A[t_idx(i, j)] = fma(-A[t_idx(i, k)], A[t_idx(j, k)], A[t_idx(i, j)]);
    }
    // in-place inverse of L (its diagonal already holds 1 / l_kk), column by column
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
        for (int i = j + 1; i < 8; ++i) {
            double s = A[t_idx(i, j)] * A[t_idx(j, j)];
#pragma unroll
            for (int k = j + 1; k < i; ++k) s = fma(A[t_idx(i, k)], A[t_idx(k, j)], s);
            A[t_idx(i, j)] = -s * A[t_idx(i, i)];
        }
}

// S = X^T X for a lower-triangular 8 x 8 X (packed); S packed lower
__device__ __forceinline__ void xtx8(const double (&X)[36], double (&S)[36]) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j <= i; ++j) {
            double s = 0.0;
#pragma unroll
            for (int k = i; k < 8; ++k) s = fma(X[t_idx(k, i)], X[t_idx(k, j)], s);
            S[t_idx(i, j)] = s;
        }
}

// 8-byte asynchronous global -> shared copy (LDGSTS): no register staging, so a whole batch can be in flight
__device__ __forceinline__ void cp_async8(void *dst_smem, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async4(void *dst_smem, const void *src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

__device__ __forceinline__ void split3_store(__nv_bfloat16 *dst, size_t plane, float v) {
    const __nv_bfloat16 h = __float2bfloat16(v);
    const float r1 = v - __bfloat162float(h);
    const __nv_bfloat16 m = __float2bfloat16(r1);
    dst[0] = h;
    dst[plane] = m;
    dst[2 * plane] = __float2bfloat16(r1 - __bfloat162float(m));
}

// MP (FP32 rows only): bf16 [3][nalloc][PITCH], already offset to the first row; a row range keeps the plane stride of
// the whole allocation
template <int Q, bool F32>
__global__ void __launch_bounds__(32 * TK<Q>::WARPS, 1)
zsolve_tpm_kernel(long long N, typename TIO<Q, F32>::type *__restrict__ MZ, double *__restrict__ Sig,
                  double *__restrict__ logdet, double *gl, double *__restrict__ zsums, __nv_bfloat16 *__restrict__ MP,
                  long long nalloc, const double *__restrict__ cond, const I8Check chk) {
    using T = TK<Q>;
    if (cond != nullptr && !(*cond > 0.0)) return;                 // conditional (fall-back) launch: nothing to redo
    __shared__ double s_chk[T::WARPS + 1];
    using IO = TIO<Q, F32>;
    using io_t = typename IO::type;
    constexpr int P = T::P, LP = T::LP;
    extern __shared__ __align__(16) double smem_t[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double *sm = smem_t + (size_t)warp * T::WARP_D;
    double *wsum = smem_t + (size_t)T::WARPS * T::WARP_D + (size_t)warp * T::KW;
#define EL(e) sm[(e) * LP + lane]
    // INT8 guard (kernels.h: I8Check): a row whose largest diagonal entry is below `thr` carries too much fixed-point rounding
    double thr = -1.0;
    if (chk.gscale != nullptr) {                                   // kernel-uniform
        double m = 0.0;
        for (int c = threadIdx.x; c < chk.ncols; c += 32 * T::WARPS) m = fmax(m, chk.gscale[c]);
        for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0) s_chk[warp] = m;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < T::WARPS; ++w) m = fmax(m, s_chk[w]);
            s_chk[T::WARPS] = gl[PYVB_GL_TAU] * chk.fac * m;
        }
        __syncthreads();
        thr = s_chk[T::WARPS];
    }
    if (cond != nullptr && blockIdx.x == 0 && threadIdx.x == 0) gl[PYVB_GL_I8FALL] += 1.0;
    // column sums of the finished rows, kept in registers: packed element lane + 32 u, zbar element lane (if < Q)
    double cs[T::NU], cz = 0.0, s_qld = 0.0, s_ld = 0.0, s_n = 0.0;
    // ... and upper bounds on their maxima of |.| (the scales of the INT8 statistics): the maximum of the high words of
    // |v| as integers (two integer instructions per element), rounded up by one unit of the high word at the end
    int cm[T::NU], czm = 0;
#pragma unroll
    for (int u = 0; u < T::NU; ++u) {
        cs[u] = 0.0;
        cm[u] = 0;
    }

    const long long nwarps = (long long)gridDim.x * T::WARPS;
    const long long nbatch = (N + 31) / 32;
    for (long long b = (long long)blockIdx.x * T::WARPS + warp; b < nbatch; b += nwarps) {
        const long long n0 = b * 32;
        const int nval = (N - n0 < 32) ? (int)(N - n0) : 32;
        if (lane == 0 && (b + nwarps) * 32 + 32 <= N)
            prefetch_l2(MZ + (b + nwarps) * 32 * IO::PITCH, (uint32_t)(32 * IO::PITCH * sizeof(io_t)));
        // ---- cooperative, coalesced load of the batch: matrix m -> column m of the [element][33] array
#pragma unroll 4
        for (int m = 0; m < 32; ++m) {
            if (m < nval) {
                const io_t *row = MZ + (n0 + m) * IO::PITCH;
#pragma unroll
                for (int u = 0; u < T::NU; ++u) {
                    const int e = lane + 32 * u;
                    if (e < P) {                                   // all copies of the batch in flight at once
                        if (F32) cp_async4(&sm[e * LP + m], row + IO::POFF + e);   // float into the slot, widened below
                        else cp_async8(&sm[e * LP + m], row + IO::POFF + e);
                    }
                }
                if (lane < Q) {
                    if (F32) cp_async4(&sm[(P + lane) * LP + m], row + IO::ZOFF + lane);
                    else cp_async8(&sm[(P + lane) * LP + m], row + IO::ZOFF + lane);
                }
            } else {                                               // tail of the last batch: the identity, never stored
#pragma unroll
                for (int u = 0; u < T::NU; ++u) {
                    const int e = lane + 32 * u;
                    if (e < P) sm[e * LP + m] = 0.0;
                }
                if (lane < Q) {
                    sm[(P + lane) * LP + m] = 0.0;
                    sm[t_idx(lane, lane) * LP + m] = 1.0;
                }
            }
        }
        cp_async_wait_all();
        __syncwarp();
        if (F32) {                                                 // widen the FP32 rows in place (own column only)
            if (lane < nval) {
#pragma unroll 8
                for (int e = 0; e < T::NE; ++e) {
                    const float f = *reinterpret_cast<const float *>(&sm[e * LP + lane]);
                    sm[e * LP + lane] = (double)f;
                }
            }
            __syncwarp();
        }

        // ---- every lane factors / inverts ITS matrix.  Register budget: at most two 8 x 8 triangles (72 doubles) live
        //      at a time; PHASE() keeps the compiler from hoisting the next phase's loads over the current one
#define PHASE() asm volatile("" ::: "memory")
        if (thr >= 0.0) {
            double dmax = 0.0;
#pragma unroll
            for (int i = 0; i < Q; ++i) dmax = fmax(dmax, EL(t_idx(i, i)));
            if (lane < nval && thr > dmax) atomicAdd(&gl[PYVB_GL_I8BAD], 1.0);
        }
        double lp = 1.0;
        if (Q == 16) {
            {   // X00 = chol(A00)^-1 ; L10 = A10 X00^T, row by row, in place (block (1,0): rows 8..15, columns 0..7)
                double A0[36];
#pragma unroll
                for (int e = 0; e < 36; ++e) A0[e] = EL(e);
                chol_inv8(A0, lp);
#pragma unroll TPM_ROLL
                for (int r = 8; r < 16; ++r) {
                    double a[8], l[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) a[k] = EL(t_idx(r, k));
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        double s = a[0] * A0[t_idx(j, 0)];
#pragma unroll
                        for (int k = 1; k <= j; ++k) s = fma(a[k], A0[t_idx(j, k)], s);
                        l[j] = s;
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j) EL(t_idx(r, j)) = l[j];
                }
#pragma unroll
                for (int e = 0; e < 36; ++e) EL(e) = A0[e];        // X00 -> shared memory
            }
            PHASE();
            {   // A11 -= L10 L10^T (stream the columns of L10) ; X11 = chol(A11)^-1 -> shared memory
                double A1[36];
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j <= i; ++j) A1[t_idx(i, j)] = EL(t_idx(8 + i, 8 + j));
#pragma unroll TPM_ROLL
                for (int k = 0; k < 8; ++k) {
                    double c[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) c[i] = EL(t_idx(8 + i, k));
#pragma unroll
                    for (int i = 0; i < 8; ++i)
#pragma unroll
                        for (int j = 0; j <= i; ++j) A1[t_idx(i, j)] = fma(-c[i], c[j], A1[t_idx(i, j)]);
                }
                chol_inv8(A1, lp);
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j <= i; ++j) EL(t_idx(8 + i, 8 + j)) = A1[t_idx(i, j)];
            }
            PHASE();
            double S0[36];
            {   // T = L10 X00 (row-wise, in place) ; S0 = X00^T X00
                double X0[36];
#pragma unroll
                for (int e = 0; e < 36; ++e) X0[e] = EL(e);
#pragma unroll TPM_ROLL
                for (int r = 8; r < 16; ++r) {
                    double l[8], t[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) l[k] = EL(t_idx(r, k));
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        double s = l[j] * X0[t_idx(j, j)];
#pragma unroll
                        for (int k = j + 1; k < 8; ++k) s = fma(l[k], X0[t_idx(k, j)], s);
                        t[j] = s;
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j) EL(t_idx(r, j)) = t[j];
                }
                xtx8(X0, S0);
            }
            PHASE();
            {
                double X1[36];
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j <= i; ++j) X1[t_idx(i, j)] = EL(t_idx(8 + i, 8 + j));
                // X10 = -X11 T (column-wise, in place)
#pragma unroll TPM_ROLL
                for (int j = 0; j < 8; ++j) {
                    double t[8], x[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) t[k] = EL(t_idx(8 + k, j));
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        double s = X1[t_idx(i, 0)] * t[0];
#pragma unroll
                        for (int k = 1; k <= i; ++k) s = fma(X1[t_idx(i, k)], t[k], s);
                        x[i] = -s;
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i) EL(t_idx(8 + i, j)) = x[i];
                }
                PHASE();
                // Sigma00 = S0 + X10^T X10 (stream the rows of X10) -> shared memory
#pragma unroll TPM_ROLL
                for (int k = 8; k < 16; ++k) {
                    double x[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) x[i] = EL(t_idx(k, i));
#pragma unroll
                    for (int i = 0; i < 8; ++i)
#pragma unroll
                        for (int j = 0; j <= i; ++j) S0[t_idx(i, j)] = fma(x[i], x[j], S0[t_idx(i, j)]);
                }
#pragma unroll
                for (int e = 0; e < 36; ++e) EL(e) = S0[e];
                PHASE();
                // Sigma10 = X11^T X10 (column-wise, in place)
#pragma unroll TPM_ROLL
                for (int j = 0; j < 8; ++j) {
                    double x[8], sv[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) x[k] = EL(t_idx(8 + k, j));
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        double a = X1[t_idx(i, i)] * x[i];
#pragma unroll
                        for (int k = i + 1; k < 8; ++k) a = fma(X1[t_idx(k, i)], x[k], a);
                        sv[i] = a;
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i) EL(t_idx(8 + i, j)) = sv[i];
                }
                PHASE();
                // Sigma11 = X11^T X11
                double S1[36];
                xtx8(X1, S1);
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j <= i; ++j) EL(t_idx(8 + i, 8 + j)) = S1[t_idx(i, j)];
            }
        } else {
            double A0[36], S0[36];
#pragma unroll
            for (int e = 0; e < 36; ++e) A0[e] = EL(e);
            chol_inv8(A0, lp);
            xtx8(A0, S0);
#pragma unroll
            for (int e = 0; e < 36; ++e) EL(e) = S0[e];
        }
        PHASE();
        // ---- zbar = Sigma eta (Sigma symmetric, packed in shared memory), then <zz^T> = Sigma + zbar zbar^T in place
        double eta[Q], z[Q];
#pragma unroll
        for (int i = 0; i < Q; ++i) {
            eta[i] = EL(P + i);
            z[i] = 0.0;
        }
        double *sg = (Sig != nullptr && lane < nval) ? (Sig + (n0 + lane) * P) : nullptr;
#pragma unroll
        for (int i = 0; i < Q; ++i)
#pragma unroll
            for (int j = 0; j <= i; ++j) {
                const double v = EL(t_idx(i, j));
                z[i] = fma(v, eta[j], z[i]);
                if (j < i) z[j] = fma(v, eta[i], z[j]);
            }
#pragma unroll
        for (int i = 0; i < Q; ++i) {
            EL(P + i) = z[i];                                      // z takes eta's place
#pragma unroll
            for (int j = 0; j <= i; ++j) {
                const double v = EL(t_idx(i, j));
                if (sg) sg[t_idx(i, j)] = v;                       // (uncoalesced; Sigma output is optional)
                EL(t_idx(i, j)) = fma(z[i], z[j], v);
            }
        }
#undef PHASE
        // ln prod diag chol = -ln prod 1/l_kk
        const double ld = -log(lp);
        if (lane < nval) {
            logdet[n0 + lane] = ld;
            s_qld += 0.5 / ld;
            s_ld += ld;
            s_n += 1.0;
            if (!(ld - ld == 0.0)) atomicAdd(&gl[PYVB_GL_NONPD], 1.0);   // NaN / inf <=> a pivot was <= 0
        }
        __syncwarp();

        // ---- cooperative, coalesced store of the finished rows (+ column sums, + bf16 x 3 planes for the FP32 rows)
#pragma unroll 4
        for (int m = 0; m < 32; ++m) {
            if (m >= nval) break;
            io_t *row = MZ + (n0 + m) * IO::PITCH;
#pragma unroll
            for (int u = 0; u < T::NU; ++u) {
                const int e = lane + 32 * u;
                if (e < P) {
                    const double v = sm[e * LP + m];
                    row[IO::POFF + e] = (io_t)v;
                    if (F32) split3_store(MP + (n0 + m) * IO::PITCH + IO::POFF + e, (size_t)nalloc * IO::PITCH, (float)v);
                    cs[u] += v;
                    if (!F32) cm[u] = max(cm[u], __double2hiint(v) & 0x7fffffff);
                }
            }
            if (lane < Q) {
                const double v = sm[(P + lane) * LP + m];
                row[IO::ZOFF + lane] = (io_t)v;
                if (F32) split3_store(MP + (n0 + m) * IO::PITCH + IO::ZOFF + lane, (size_t)nalloc * IO::PITCH, (float)v);
                cz += v;
                if (!F32) czm = max(czm, __double2hiint(v) & 0x7fffffff);
            }
        }
        __syncwarp();
    }
#undef EL
    if (zsums == nullptr) return;                                  // kernel-uniform
    // ---- CTA partial of the column sums: [packed P | pad | zbar q | sum 0.5/logdet | sum logdet | rows | 0]
    for (int c = lane; c < T::KW; c += 32) wsum[c] = 0.0;
    __syncwarp();
#pragma unroll
    for (int u = 0; u < T::NU; ++u)
        if (lane + 32 * u < P) {
            wsum[lane + 32 * u] = cs[u];
            wsum[T::OROW + 4 + lane + 32 * u] = cm[u] ? __hiloint2double(cm[u] + 1, 0) : 0.0;
        }
    if (lane < Q) {
        wsum[T::PP + lane] = cz;
        wsum[T::OROW + 4 + T::PP + lane] = czm ? __hiloint2double(czm + 1, 0) : 0.0;
    }
    s_qld = warp_sum(s_qld);
    s_ld = warp_sum(s_ld);
    s_n = warp_sum(s_n);
    if (lane == 0) {
        wsum[T::OROW] = s_qld;
        wsum[T::OROW + 1] = s_ld;
        wsum[T::OROW + 2] = s_n;
    }
    __syncthreads();
    double *out = zsums + (size_t)blockIdx.x * T::KW;
    const double *w0 = smem_t + (size_t)T::WARPS * T::WARP_D;
    for (int c = threadIdx.x; c < T::KW; c += 32 * T::WARPS) {
        double a = 0.0;
        if (c < T::OROW + 4)
            for (int w = 0; w < T::WARPS; ++w) a += w0[(size_t)w * T::KW + c];
        else
            for (int w = 0; w < T::WARPS; ++w) a = fmax(a, w0[(size_t)w * T::KW + c]);
        out[c] = a;
    }
}

template <int Q, bool F32>
cudaError_t launch_tpm_q(long long N, void *MZ, double *Sig, double *logdet, double *gl, double *zsums, void *MP,
                         long long nalloc, cudaStream_t st, const double *cond = nullptr, I8Check chk = I8Check()) {
    using T = TK<Q>;
    cudaError_t e =
        cudaFuncSetAttribute(zsolve_tpm_kernel<Q, F32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)T::SMEM);
    if (e != cudaSuccess) return e;
    const int blocks = zsolve_tpm_blocks(N, Q);
    zsolve_tpm_kernel<Q, F32><<<blocks, 32 * T::WARPS, T::SMEM, st>>>(N, static_cast<typename TIO<Q, F32>::type *>(MZ), Sig,
                                                                    logdet, gl, zsums, static_cast<__nv_bfloat16 *>(MP),
                                                                    nalloc, cond, chk);
    return cudaGetLastError();
}

}  // namespace

int zsolve_tpm_blocks(long long N, int q) {
    if (q != 8 && q != 16) return 0;
    const int warps = 5;
    long long b = ((N + 31) / 32 + warps - 1) / warps;
    if (b > 148) b = 148;
    if (b < 1) b = 1;
    return (int)b;
}
int zsolve_tpm_kw(int q) { return q == 8 ? TK<8>::KW : q == 16 ? TK<16>::KW : 0; }

cudaError_t launch_zsolve_tpm(long long N, int q, double *MZ, double *Sig, double *logdet, double *gl, double *zsums,
                              cudaStream_t st, const double *cond, I8Check chk) {
    if (N <= 0) return cudaSuccess;
    if (q == 8) return launch_tpm_q<8, false>(N, MZ, Sig, logdet, gl, zsums, nullptr, 0, st, cond, chk);
    return cudaErrorNotSupported;
}
cudaError_t launch_zsolve_tpm_f32(long long N, long long nalloc, int q, float *MZ32, void *MP, double *Sig, double *logdet,
                                  double *gl, double *zsums, cudaStream_t st) {
    if (N <= 0) return cudaSuccess;
    if (q == 16) return launch_tpm_q<16, true>(N, MZ32, Sig, logdet, gl, zsums, MP, nalloc, st);
    return cudaErrorNotSupported;
}

}  // namespace pyvb
