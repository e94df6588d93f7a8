// K2, blocked: batched q x q SPD inverse / solve with the FP64 tensor cores (DMMA.8x8x4), one warp per matrix.
//
// Replaces, per row n, the reference's  cho_factor(qprec) / cho_solve(., I) / dot(qcov, .)  and
// q_ln_det = .5/log(prod(diag(chol)))  (nodes/gaussian.py:117-123) for the FP32 rows at q = 32, 64 (the FP64 rows have a
// faster kernel at every q: launch_zsolve, DESIGN.md 5).
//
// The matrix lives in shared memory as NB x NB lower-triangular storage of 8 x 8 blocks (NB = q/8, 64 doubles per
// block, 32-byte chunks XOR-swizzled so that every DMMA fragment pattern -- row-wise, transposed, accumulator --
// is bank-conflict free without padding).  Three in-place block sweeps, LAPACK potrf / trtri / lauum style:
//   1. left-looking Cholesky:   C_ij = A_ij - sum_k L_ik L_jk^T (DMMA);  diagonal block factored AND inverted in
//      registers with warp shuffles (it already sits in the accumulator layout);  L_ij = C_ij X_jj^T (DMMA)
//   2. X = L^-1:                X_ik = -X_ii sum_j L_ij X_jk   (DMMA, a block row at a time)
//   3. Sigma = X^T X:           S_ij = sum_k X_ki^T X_kj       (DMMA)
// then zbar = Sigma eta, <zz^T> = Sigma + zbar zbar^T, ln prod diag chol from the pivots.  Only the 8 x 8 diagonal
// blocks run on the FP64 FMA pipe (8 sequential pivots each); everything else is tensor-core work.
#include <cuda_bf16.h>

#include "chol8.cuh"
#include "common.cuh"
#include "kernels.h"
#include "ptx.cuh"

namespace pyvb {

namespace {

__host__ __device__ constexpr int kb_tri(int i) { return i * (i + 1) / 2; }
__host__ __device__ constexpr int kb_pitch(int q) {          // == pyvb_gw_pitch(q)
    int p = ((kb_tri(q) + 7) & ~7) + q + 1;
    while ((p % 8) != 4) ++p;
    return p;
}
// element (r, c) of a swizzled 8 x 8 block
__host__ __device__ constexpr int kb_sw(int r, int c) { return r * 8 + ((((c >> 2) ^ ((r >> 1) & 1))) << 2) + (c & 3); }
// block (i, j), i >= j
__host__ __device__ constexpr int kb_boff(int i, int j) { return (kb_tri(i) + j) * 64; }

template <int Q> struct KBC;
// MPW: matrices per warp, processed as interleaved instruction streams (the 8 x 8 diagonal blocks are a chain of
// 8 dependent pivots each; a second matrix fills the latency)
// (measured: MPW = 2 does not help -- the kernel is issue-bound, not latency-bound -- so MPW = 1 everywhere)
template <> struct KBC<32> { static constexpr int WARPS = 10, OCC = 2, MPW = 1; static constexpr bool ZS = true; };
template <> struct KBC<64> { static constexpr int WARPS = 11, OCC = 1, MPW = 1; static constexpr bool ZS = false; };

template <int Q> struct KB {
    static constexpr int NB = Q / 8, NBLK = kb_tri(NB);
    static constexpr int P = kb_tri(Q), PP = (P + 7) & ~7, OROW = PP + Q, LDG = kb_pitch(Q);
    static constexpr int WARPS = KBC<Q>::WARPS, OCC = KBC<Q>::OCC, MPW = KBC<Q>::MPW;
    static constexpr bool ZS = KBC<Q>::ZS;
    static constexpr int KW = 2 * OROW + PYVB_ZS_EXTRA;   // [column sums OROW | 4 scalars | bounds on the column maxima OROW]
    static constexpr int MAT_D = NBLK * 64 + 2 * Q;                             // per matrix: blocks | eta | z
    static constexpr int WARP_D = MPW * MAT_D + (ZS ? OROW : 0) + 4 + (ZS ? 2 * Q : 0);   // ... | column sums | scalars | max <z_i^2>, max |z_i|
    static constexpr int TAB_B = ((P * 4) + 15) & ~15;                         // one uint32 table
    static constexpr int UNR = (P / 32 >= 16) ? 16 : (P + 31) / 32;            // global loads in flight per lane
    static constexpr size_t SMEM = (size_t)TAB_B + (size_t)WARPS * WARP_D * 8;
};

// Row format of the batched solve.  FP64: the interleaved MZ rows [packed (P) | pad | eta/zbar (q)], pitch
// pyvb_mz_pitch(q).  FP32 variant: float rows [eta/zbar (q) | packed (P) | pad] of pitch pyvb_f32_pitch(q); the
// arithmetic stays FP64 (the rows are converted on load / store), and the finished row is also written as a
// three-way bf16 split (planes [3][nalloc][pitch], nalloc >= N: a row range keeps the plane stride of the whole
// allocation) -- the B operand of the FP32 statistics kernel.
template <int Q, bool F32> struct KIO;
template <int Q> struct KIO<Q, false> {
    using type = double;
    static constexpr int PITCH = kb_pitch(Q), POFF = 0, ZOFF = (kb_tri(Q) + 7) & ~7, USED = ZOFF + Q;
};
template <int Q> struct KIO<Q, true> {
    using type = float;
    static constexpr int PITCH = (Q + kb_tri(Q) + 63) & ~63, POFF = Q, ZOFF = 0, USED = Q + kb_tri(Q);
};

__device__ __forceinline__ void store_split3(__nv_bfloat16 *dst, size_t plane, float v) {
    const __nv_bfloat16 h = __float2bfloat16(v);
    const float r1 = v - __bfloat162float(h);
    const __nv_bfloat16 m = __float2bfloat16(r1);
    const float r2 = r1 - __bfloat162float(m);
    dst[0] = h;
    dst[plane] = m;
    dst[2 * plane] = __float2bfloat16(r2);
}

template <int Q, bool F32>
__global__ void __launch_bounds__(32 * KB<Q>::WARPS, KB<Q>::OCC)
zsolve_blocked_kernel(long long N, typename KIO<Q, F32>::type *__restrict__ MZ, double *__restrict__ Sig,
                      double *__restrict__ logdet, double *gl, double *__restrict__ zsums,
                      __nv_bfloat16 *__restrict__ MP, long long nalloc, const double *__restrict__ cond, const I8Check chk) {
    using T = KB<Q>;
    if (cond != nullptr && !(*cond > 0.0)) return;               // conditional (fall-back) launch: nothing to redo
    __shared__ double s_chk[T::WARPS + 1];
    using IO = KIO<Q, F32>;
    using io_t = typename IO::type;
    constexpr int NB = T::NB, MPW = T::MPW;
    extern __shared__ __align__(16) unsigned char smem_kb[];
    // packed index p -> offset in the block storage (bits 0-11) | i (bits 12-17) | j (bits 18-23)
    uint32_t *tab = reinterpret_cast<uint32_t *>(smem_kb);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    double *wbase = reinterpret_cast<double *>(smem_kb + T::TAB_B) + (size_t)warp * T::WARP_D;
    double *csum = wbase + MPW * T::MAT_D;                       // [OROW] when ZS
    double *wsc = csum + (T::ZS ? T::OROW : 0);                  // [4]
    double *wmx = wsc + 4;                                       // [2 Q] when ZS: max_n <z_i z_i>, max_n |<z_i>| of this warp's rows
    double dmx[(Q + 31) / 32], zmx[(Q + 31) / 32];
#pragma unroll
    for (int k = 0; k < (Q + 31) / 32; ++k) dmx[k] = zmx[k] = 0.0;

    for (int p = tid; p < T::P; p += 32 * T::WARPS) {
        int i, j;
        unpack_p(p, i, j);
        tab[p] = (uint32_t)(kb_boff(i >> 3, j >> 3) + kb_sw(i & 7, j & 7)) | ((uint32_t)i << 12) | ((uint32_t)j << 18);
    }
    if (T::ZS)
        for (int c = lane; c < T::OROW; c += 32) csum[c] = 0.0;
    // INT8 guard (kernels.h: I8Check): a row whose largest diagonal entry is below `thr` carries too much fixed-point rounding
    if (chk.gscale != nullptr) {                                 // kernel-uniform
        double m = 0.0;
        for (int c = tid; c < chk.ncols; c += 32 * T::WARPS) m = fmax(m, chk.gscale[c]);
        for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (lane == 0) s_chk[warp] = m;
    }
    __syncthreads();
    double thr = -1.0;
    if (chk.gscale != nullptr) {
        double m = s_chk[0];
        for (int w = 1; w < T::WARPS; ++w) m = fmax(m, s_chk[w]);
        thr = gl[PYVB_GL_TAU] * chk.fac * m;
    }
    if (cond != nullptr && blockIdx.x == 0 && tid == 0) gl[PYVB_GL_I8FALL] += 1.0;

    const int gid = lane >> 2, qd = lane & 3;
    const int oA0 = kb_sw(gid, qd), oA1 = kb_sw(gid, qd + 4);    // row-wise fragment   M[gid][qd + 4h]
    const int oT0 = kb_sw(qd, gid), oT1 = kb_sw(qd + 4, gid);    // transposed fragment M[qd + 4h][gid]
    const int oC = kb_sw(gid, 2 * qd);                           // accumulator pair    M[gid][2qd, 2qd+1]
    double s_qld = 0.0, s_ld = 0.0, s_n = 0.0;

    // every warp walks over groups of MPW consecutive rows; the MPW matrices are independent instruction streams
    const long long nwarps = (long long)gridDim.x * T::WARPS;
    const long long ngroups = (N + MPW - 1) / MPW;
    for (long long g = (long long)blockIdx.x * T::WARPS + warp; g < ngroups; g += nwarps) {
        io_t *row[MPW];
        long long nrow[MPW];
        bool valid[MPW];
        double *blk[MPW], *eta[MPW], *zv[MPW];
#pragma unroll
        for (int m = 0; m < MPW; ++m) {
            nrow[m] = g * MPW + m;
            valid[m] = nrow[m] < N;
            if (!valid[m]) nrow[m] = N - 1;                      // tail: redo the last row, store nothing
            row[m] = MZ + nrow[m] * IO::PITCH;
            blk[m] = wbase + m * T::MAT_D;
            eta[m] = blk[m] + T::NBLK * 64;
            zv[m] = eta[m] + Q;
        }
        // the group after this one: pull it into L2 now, it is read tens of thousands of cycles from now
        if (lane == 0 && (g + nwarps) * MPW + MPW <= N)
            prefetch_l2(MZ + (g + nwarps) * MPW * IO::PITCH, (uint32_t)(MPW * IO::PITCH * sizeof(io_t)));
        // ---- unpack [qprec packed | eta] into the block storage (coalesced global reads, UNR in flight)
#pragma unroll
        for (int m = 0; m < MPW; ++m) {
            const double e0 = (lane < Q) ? (double)row[m][IO::ZOFF + lane] : 0.0;
            const double e1 = (Q > 32) ? (double)row[m][IO::ZOFF + 32 + (lane & 31)] : 0.0;
#pragma unroll 1
            for (int base = 0; base < T::P; base += 32 * T::UNR) {
                double v[T::UNR];
#pragma unroll
                for (int u = 0; u < T::UNR; ++u) {
                    const int p = base + 32 * u + lane;
                    v[u] = (p < T::P) ? (double)row[m][IO::POFF + p] : 0.0;
                }
#pragma unroll
                for (int u = 0; u < T::UNR; ++u) {
                    const int p = base + 32 * u + lane;
                    if (p < T::P) blk[m][tab[p] & 0xfff] = v[u];
                }
            }
            if (lane < Q) eta[m][lane] = e0;
            if (Q > 32) eta[m][32 + lane] = e1;
        }
        __syncwarp();
        if (thr >= 0.0) {                                        // diagonal of qprec, before the factorisation overwrites it
#pragma unroll
            for (int m = 0; m < MPW; ++m) {
                double dm = 0.0;
#pragma unroll
                for (int i = lane; i < Q; i += 32) dm = fmax(dm, blk[m][kb_boff(i >> 3, i >> 3) + kb_sw(i & 7, i & 7)]);
                for (int o = 16; o > 0; o >>= 1) dm = fmax(dm, __shfl_xor_sync(0xffffffffu, dm, o));
                if (lane == 0 && valid[m] && thr > dm) atomicAdd(&gl[PYVB_GL_I8BAD], 1.0);
            }
        }

        // ---- 1. left-looking block Cholesky; diagonal blocks are replaced by their inverses X_jj
        double mant[MPW];             // prod_k 1/l_kk = mant * 2^esum, renormalised after every diagonal block
        int esum[MPW];
        bool ok[MPW];
#pragma unroll
        for (int m = 0; m < MPW; ++m) {
            mant[m] = 1.0;
            esum[m] = 0;
            ok[m] = true;
        }
#pragma unroll
        for (int jb = 0; jb < NB; ++jb) {
            double acc[MPW][NB][2];
#pragma unroll
            for (int m = 0; m < MPW; ++m) {
#pragma unroll
                for (int ib = 0; ib < NB; ++ib) acc[m][ib][0] = acc[m][ib][1] = 0.0;
#pragma unroll
                for (int kb = 0; kb < jb; ++kb) {
                    const double *Bj = blk[m] + kb_boff(jb, kb);
                    const double b0 = Bj[oA0], b1 = Bj[oA1];
#pragma unroll
                    for (int ib = jb; ib < NB; ++ib) {
                        const double *Ai = blk[m] + kb_boff(ib, kb);
                        dmma884(acc[m][ib][0], acc[m][ib][1], Ai[oA0], b0);
                        dmma884(acc[m][ib][0], acc[m][ib][1], Ai[oA1], b1);
                    }
                }
#pragma unroll
                for (int ib = jb; ib < NB; ++ib) {
                    const double2 a = *reinterpret_cast<const double2 *>(blk[m] + kb_boff(ib, jb) + oC);
                    acc[m][ib][0] = a.x - acc[m][ib][0];
                    acc[m][ib][1] = a.y - acc[m][ib][1];
                }
            }
            double d0[MPW], d1[MPW], x0[MPW], x1[MPW];
#pragma unroll
            for (int m = 0; m < MPW; ++m) {
                d0[m] = acc[m][jb][0];
                d1[m] = acc[m][jb][1];
            }
            diag_chol_inv<MPW>(d0, d1, x0, x1, mant);
#pragma unroll
            for (int m = 0; m < MPW; ++m) {
                ok[m] = ok[m] && (mant[m] - mant[m] == 0.0);     // NaN / inf <=> a pivot was <= 0
                const long long bits = __double_as_longlong(mant[m]);
                esum[m] += (int)((bits >> 52) & 0x7ff) - 1023;
                mant[m] = __longlong_as_double((bits & 0x800fffffffffffffLL) | 0x3ff0000000000000LL);
                *reinterpret_cast<double2 *>(blk[m] + kb_boff(jb, jb) + oC) = make_double2(x0[m], x1[m]);
#pragma unroll
                for (int ib = jb + 1; ib < NB; ++ib)
                    *reinterpret_cast<double2 *>(blk[m] + kb_boff(ib, jb) + oC) = make_double2(acc[m][ib][0], acc[m][ib][1]);
            }
            __syncwarp();
            if (jb + 1 < NB) {
                // L_ij = C_ij X_jj^T
#pragma unroll
                for (int m = 0; m < MPW; ++m) {
                    const double *Xj = blk[m] + kb_boff(jb, jb);
                    const double xb0 = Xj[oA0], xb1 = Xj[oA1];
#pragma unroll
                    for (int ib = jb + 1; ib < NB; ++ib) {
                        const double *Ci = blk[m] + kb_boff(ib, jb);
                        acc[m][ib][0] = acc[m][ib][1] = 0.0;
                        dmma884(acc[m][ib][0], acc[m][ib][1], Ci[oA0], xb0);
                        dmma884(acc[m][ib][0], acc[m][ib][1], Ci[oA1], xb1);
                    }
                }
                __syncwarp();
#pragma unroll
                for (int m = 0; m < MPW; ++m)
#pragma unroll
                    for (int ib = jb + 1; ib < NB; ++ib)
                        *reinterpret_cast<double2 *>(blk[m] + kb_boff(ib, jb) + oC) =
                            make_double2(acc[m][ib][0], acc[m][ib][1]);
                __syncwarp();
            }
        }

        // ---- 2. X = L^-1, one block row at a time:  X_ik = -X_ii * sum_{k <= j < i} L_ij X_jk
#pragma unroll
        for (int ib = 1; ib < NB; ++ib) {
            double acc[MPW][NB][2];
#pragma unroll
            for (int m = 0; m < MPW; ++m) {
#pragma unroll
                for (int kb = 0; kb < NB; ++kb) acc[m][kb][0] = acc[m][kb][1] = 0.0;
#pragma unroll
                for (int jb = 0; jb < ib; ++jb) {
                    const double *Lij = blk[m] + kb_boff(ib, jb);
                    const double a0 = Lij[oA0], a1 = Lij[oA1];
#pragma unroll
                    for (int kb = 0; kb <= jb; ++kb) {
                        const double *Xjk = blk[m] + kb_boff(jb, kb);
                        dmma884(acc[m][kb][0], acc[m][kb][1], a0, Xjk[oT0]);
                        dmma884(acc[m][kb][0], acc[m][kb][1], a1, Xjk[oT1]);
                    }
                }
            }
            __syncwarp();
#pragma unroll
            for (int m = 0; m < MPW; ++m)
#pragma unroll
                for (int kb = 0; kb < ib; ++kb)
                    *reinterpret_cast<double2 *>(blk[m] + kb_boff(ib, kb) + oC) = make_double2(acc[m][kb][0], acc[m][kb][1]);
            __syncwarp();
#pragma unroll
            for (int m = 0; m < MPW; ++m) {
                const double *Xii = blk[m] + kb_boff(ib, ib);
                const double xa0 = Xii[oA0], xa1 = Xii[oA1];
#pragma unroll
                for (int kb = 0; kb < ib; ++kb) {
                    const double *S = blk[m] + kb_boff(ib, kb);
                    acc[m][kb][0] = acc[m][kb][1] = 0.0;
                    dmma884(acc[m][kb][0], acc[m][kb][1], xa0, S[oT0]);
                    dmma884(acc[m][kb][0], acc[m][kb][1], xa1, S[oT1]);
                }
            }
            __syncwarp();
#pragma unroll
            for (int m = 0; m < MPW; ++m)
#pragma unroll
                for (int kb = 0; kb < ib; ++kb)
                    *reinterpret_cast<double2 *>(blk[m] + kb_boff(ib, kb) + oC) =
                        make_double2(-acc[m][kb][0], -acc[m][kb][1]);
            __syncwarp();
        }

        // ---- 3. Sigma = X^T X (lower blocks, diagonal blocks come out full):  S_ij = sum_{k >= i} X_ki^T X_kj
#pragma unroll
        for (int i = 0; i < NB; ++i) {
            double acc[MPW][NB][2];
#pragma unroll
            for (int m = 0; m < MPW; ++m) {
#pragma unroll
                for (int j = 0; j < NB; ++j) acc[m][j][0] = acc[m][j][1] = 0.0;
#pragma unroll
                for (int k = i; k < NB; ++k) {
                    const double *Xki = blk[m] + kb_boff(k, i);
                    const double a0 = Xki[oT0], a1 = Xki[oT1];
#pragma unroll
                    for (int j = 0; j <= i; ++j) {
                        const double *Xkj = blk[m] + kb_boff(k, j);
                        dmma884(acc[m][j][0], acc[m][j][1], a0, Xkj[oT0]);
                        dmma884(acc[m][j][0], acc[m][j][1], a1, Xkj[oT1]);
                    }
                }
            }
            __syncwarp();
#pragma unroll
            for (int m = 0; m < MPW; ++m)
#pragma unroll
                for (int j = 0; j <= i; ++j)
                    *reinterpret_cast<double2 *>(blk[m] + kb_boff(i, j) + oC) = make_double2(acc[m][j][0], acc[m][j][1]);
        }
        __syncwarp();

        // ---- zbar = Sigma eta on the tensor cores: B = eta_j broadcast over the 8 columns, so every accumulator
        //      column holds the block row's part of z
#pragma unroll
        for (int m = 0; m < MPW; ++m) {
#pragma unroll
            for (int i = 0; i < NB; ++i) {
                double z0 = 0.0, z1 = 0.0;
#pragma unroll
                for (int j = 0; j < NB; ++j) {
                    const double *B = blk[m] + (j <= i ? kb_boff(i, j) : kb_boff(j, i));
                    const double a0 = B[j <= i ? oA0 : oT0], a1 = B[j <= i ? oA1 : oT1];
                    dmma884(z0, z1, a0, eta[m][j * 8 + qd]);
                    dmma884(z0, z1, a1, eta[m][j * 8 + qd + 4]);
                }
                if (qd == 0) zv[m][i * 8 + gid] = z0;
            }
        }
        __syncwarp();

        // ---- outputs: [<zz^T> packed | pad (left as it is: zeros) | zbar], optional Sigma, log-det
#pragma unroll
        for (int m = 0; m < MPW; ++m) {
            const double ldsum = ok[m] ? -fma((double)esum[m], 0.69314718055994530942, log(mant[m]))
                                       : __longlong_as_double(0x7ff8000000000000LL);
            if (!valid[m]) continue;                             // warp-uniform
            const long long n = nrow[m];
            double *sg = (Sig != nullptr) ? (Sig + n * T::P) : nullptr;
#pragma unroll 4
            for (int p = lane; p < T::P; p += 32) {
                const uint32_t t = tab[p];
                const double s = blk[m][t & 0xfff];
                const double mm = fma(zv[m][(t >> 12) & 63], zv[m][t >> 18], s);
                row[m][IO::POFF + p] = (io_t)mm;
                if (F32) store_split3(MP + n * IO::PITCH + IO::POFF + p, (size_t)nalloc * IO::PITCH, (float)mm);
                if (sg) sg[p] = s;
                if (T::ZS) csum[p] += mm;
            }
#pragma unroll
            for (int k = 0; k < (Q + 31) / 32; ++k) {
                const int c = lane + 32 * k;
                if (c >= Q) continue;
                const double z = zv[m][c];
                row[m][IO::ZOFF + c] = (io_t)z;
                if (F32) store_split3(MP + n * IO::PITCH + IO::ZOFF + c, (size_t)nalloc * IO::PITCH, (float)z);
                if (T::ZS) {
                    csum[T::PP + c] += z;
                    // <z_c z_c> = Sigma_cc + z_c^2: with the diagonal maxima, |<z_i z_j>| <= sqrt(<z_i z_i> <z_j z_j>) bounds
                    // every column of the packed rows (the fixed-point scales of the INT8 statistics)
                    dmx[k] = fmax(dmx[k], fma(z, z, blk[m][kb_boff(c >> 3, c >> 3) + kb_sw(c & 7, c & 7)]));
                    zmx[k] = fmax(zmx[k], fabs(z));
                }
            }
            if (lane == 0) {
                logdet[n] = ldsum;
                s_qld += 0.5 / ldsum;
                s_ld += ldsum;
                s_n += 1.0;
                if (!(ldsum - ldsum == 0.0)) atomicAdd(&gl[PYVB_GL_NONPD], 1.0);   // NaN / inf <=> a pivot was <= 0
            }
        }
        __syncwarp();
    }

    if (!T::ZS || zsums == nullptr) return;
    if (lane == 0) {
        wsc[0] = s_qld;
        wsc[1] = s_ld;
        wsc[2] = s_n;
        wsc[3] = 0.0;
    }
#pragma unroll
    for (int k = 0; k < (Q + 31) / 32; ++k)
        if (lane + 32 * k < Q) {
            wmx[lane + 32 * k] = dmx[k];
            wmx[Q + lane + 32 * k] = zmx[k];
        }
    __syncthreads();
    double *out = zsums + (size_t)blockIdx.x * T::KW;
    const double *w0 = reinterpret_cast<const double *>(smem_kb + T::TAB_B) + MPW * T::MAT_D;   // csum of warp 0
    for (int c = tid; c < T::OROW + 4; c += 32 * T::WARPS) {
        double a = 0.0;
        for (int w = 0; w < T::WARPS; ++w) a += w0[(size_t)w * T::WARP_D + c];   // [csum OROW | scalars 4] is contiguous
        out[c] = a;
    }
    // CTA maxima of the diagonal second moments and of |z| (fold the warps into warp 0's slots), then the column bounds
    double *m0 = const_cast<double *>(w0) + T::OROW + 4;
    __syncthreads();
    for (int c = tid; c < 2 * Q; c += 32 * T::WARPS) {
        double a = 0.0;
        for (int w = 0; w < T::WARPS; ++w) a = fmax(a, m0[(size_t)w * T::WARP_D + c]);
        m0[c] = a;
    }
    __syncthreads();
    for (int c = tid; c < T::OROW; c += 32 * T::WARPS) {
        double a = 0.0;
        if (c < T::P) {
            const uint32_t t = tab[c];
            a = sqrt(m0[(t >> 12) & 63] * m0[t >> 18]);
        } else if (c >= T::PP) {
            a = m0[Q + c - T::PP];
        }
        out[T::OROW + 4 + c] = a;
    }
}

template <int Q>
int blocked_blocks(long long N) {
    using T = KB<Q>;
    long long b = (N + (long long)T::MPW * T::WARPS - 1) / ((long long)T::MPW * T::WARPS);
    if (b > 148LL * T::OCC) b = 148LL * T::OCC;
    if (b < 1) b = 1;
    return (int)b;
}

template <int Q>
cudaError_t launch_blocked_q(long long N, long long nalloc, float *MZ32, void *MP, double *Sig, double *logdet, double *gl,
                             double *zsums, cudaStream_t st) {
    using T = KB<Q>;
    cudaError_t e = cudaFuncSetAttribute(zsolve_blocked_kernel<Q, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)T::SMEM);
    if (e != cudaSuccess) return e;
    zsolve_blocked_kernel<Q, true><<<blocked_blocks<Q>(N), 32 * T::WARPS, T::SMEM, st>>>(
        N, MZ32, Sig, logdet, gl, T::ZS ? zsums : nullptr, static_cast<__nv_bfloat16 *>(MP), nalloc, nullptr, I8Check());
    return cudaGetLastError();
}

}  // namespace

// q = 16: the thread-per-matrix kernel (kernels_k2t.cu); q = 64: no column-sum partials, so pyvb_stats_f32 (which has no
// other source for the sums over the rows) rejects q = 64
void zsolve_partials_f32(long long N, int q, int &nblk, int &kw) {
    kw = (q == 16) ? zsolve_tpm_kw(q) : (q == 32) ? KB<32>::KW : 0;
    nblk = (kw == 0 || N <= 0) ? 0 : (q == 16) ? zsolve_tpm_blocks(N, q) : blocked_blocks<32>(N);
}

// FP32 rows (see KIO): in place on MZ32, plus the bf16 x 3 split of the finished rows into MP [3][nalloc][pitch]
cudaError_t launch_zsolve_f32(long long N, long long nalloc, int q, float *MZ32, void *MP, double *Sig, double *logdet,
                              double *gl, double *zsums, cudaStream_t st) {
    if (N <= 0) return cudaSuccess;
    switch (q) {
        case 16: return launch_zsolve_tpm_f32(N, nalloc, q, MZ32, MP, Sig, logdet, gl, zsums, st);
        case 32: return launch_blocked_q<32>(N, nalloc, MZ32, MP, Sig, logdet, gl, zsums, st);
        case 64: return launch_blocked_q<64>(N, nalloc, MZ32, MP, Sig, logdet, gl, zsums, st);
    }
    return cudaErrorNotSupported;
}

}  // namespace pyvb
