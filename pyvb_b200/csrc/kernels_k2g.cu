// K2, Gauss-Jordan in registers: batched q x q SPD inverse / solve, LPM = q / RPL lanes per matrix, every lane owns RPL rows.
//
// Replaces cho_factor / cho_solve(., I) / dot(qcov, .) / q_ln_det of Gaussian.update (nodes/gaussian.py:117-123).
//
// The other K2 kernels are Cholesky based (potrf / trtri / lauum): three triangular phases whose operands have to be
// re-laid-out between the phases, which is what binds them (thread per matrix: 40 KB of shared memory per warp -> 5 warps per
// SM, latency; blocked DMMA: 1,300 shared-memory wavefronts + 3,000 instructions per 32 x 32 matrix).  Here the inverse comes
// from ONE phase, the in-place Gauss-Jordan elimination without pivoting (backward stable on SPD input; measured against a
// long-double inverse it is as accurate as LAPACK's Cholesky route at cond 1e2 .. 1e6, oracle-side check in
// tests/test_host_logic.py), organised so that nothing but a broadcast column ever leaves the registers:
//
//   lane (m, l) holds rows  l, l + LPM, ..  of matrix m as FULL rows a[r][0..q)  (q = 32, RPL = 2: 128 registers)
//   step k:   every lane publishes its column-k entry b_i (one STS.64 per row), the warp reads the q published values back as
//             broadcast LDS.128 (one shared-memory wavefront per two columns and per TWO rows of arithmetic), and
//             a[r][j] += t_r * b_j  for all j != k,  t_r = -a[r][k] / d,  d = b_k          (q - 1 DFMA per row)
//   the pivot row is NOT scaled inside the loop (its lane keeps t = 0 and gets a 1 in column k): scaling row k by 1 / d is
//   deferred to the end (one multiplication per entry), which keeps the inner loop free of per-lane selects.  A row that is
//   already pivoted therefore holds d_i times its true value, and (U, K) / (K, U) blocks of the Gauss-Jordan iterate differ by
//   their sign: the published entry is  b_i = a[r][k] * sinv_i  with  sinv_i = 1 before row i's pivot and -1 / d_i after it.
//
// ln prod diag chol = -1/2 sum_i ln(1 / d_i): one logarithm per lane at the end.  zbar = Sigma eta and <zz^T> = Sigma + zbar zbar^T
// use the same broadcast scheme.  The rows of a group (MPW matrices) travel as ONE bulk copy each way (global -> shared ->
// registers ... registers -> shared -> global, in place), column sums / maxima bounds / log-det scalars per CTA as in the
// other K2 kernels (zsums partial layout of the blocked kernel).
#include "common.cuh"
#include "kernels.h"
#include "ptx.cuh"

namespace pyvb {

namespace {

__host__ __device__ constexpr int g_tri(int i) { return i * (i + 1) / 2; }
__host__ __device__ constexpr int g_pitch(int q) {          // == pyvb_mz_pitch(q)
    int p = ((g_tri(q) + 7) & ~7) + q + 1;
    while ((p % 8) != 4) ++p;
    return p;
}

// RPL rows per lane, WARPS per CTA (one CTA per SM: the register file allows 65536 / (32 WARPS) registers per thread)
template <int Q, int RPL_, int WARPS_> struct GJ {
    static constexpr int RPL = RPL_, WARPS = WARPS_;
    static constexpr int LPM = Q / RPL;                       // lanes per matrix
    static constexpr int MPW = 32 / LPM;                      // matrices per warp (= rows of MZ per group)
    static constexpr int P = g_tri(Q), PP = (P + 7) & ~7, OROW = PP + Q, PITCH = g_pitch(Q);
    static constexpr int KW = 2 * OROW + PYVB_ZS_EXTRA;       // [column sums OROW | 4 scalars | bounds on the column maxima OROW]
    static constexpr int STAGE_D = MPW * PITCH;               // the rows of a group as they lie in HBM
    static constexpr int BC_P = MPW * (Q + 2);                // published columns of the warp's matrices + the next pivot row's diagonal
    static constexpr int BC_D = 2 * BC_P;                     // two parities
    static constexpr int WARP_D = 2 * STAGE_D + BC_D + OROW + 4 + 2 * Q + 2;   // two stages | .. | csum | scalars | maxima | 2 mbarriers
    static constexpr size_t SMEM = (size_t)WARPS * WARP_D * 8;
    static_assert(LPM <= 32 && (32 % LPM) == 0, "a matrix lives in one warp");
    static_assert((STAGE_D % 2) == 0 && (BC_D % 2) == 0 && (OROW % 2) == 0, "16-byte alignment of the per-warp arrays");
    // published entry j of matrix m: the pairs (j, j + 1) of the warp's matrices are interleaved, so that one broadcast LDS.128
    // of all lanes touches ONE contiguous 16 MPW bytes
    __host__ __device__ static constexpr int bidx(int m, int j) { return ((j >> 1) * MPW + m) * 2 + (j & 1); }
};

// 1 / d to the last bit or so: MUFU.RCP64H seed (20 bits) + two Newton steps; no special-case branch (d <= 0 is flagged by the
// caller through the logarithm of the pivots)
__device__ __forceinline__ double rcp_nr(double d) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    double e = fma(-d, r, 1.0);
    r = fma(r, e, r);
    e = fma(-d, r, 1.0);
    return fma(r, e, r);
}

template <int Q, int RPL_, int WARPS_>
__global__ void __launch_bounds__(32 * WARPS_, 1)
zsolve_gj_kernel(long long N, double *__restrict__ MZ, double *__restrict__ Sig, double *__restrict__ logdet, double *gl,
                 double *__restrict__ zsums, const double *__restrict__ cond, const I8Check chk) {
    using T = GJ<Q, RPL_, WARPS_>;
    constexpr int RPL = T::RPL, LPM = T::LPM, MPW = T::MPW, P = T::P, PP = T::PP, PITCH = T::PITCH;
    if (cond != nullptr && !(*cond > 0.0)) return;               // conditional (fall-back) launch: nothing to redo
    __shared__ double s_chk[T::WARPS + 1];
    extern __shared__ __align__(16) double smem_gj[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int m = lane / LPM, l = lane % LPM;
    double *stage = smem_gj + (size_t)warp * T::WARP_D;
    double *bc = stage + 2 * T::STAGE_D;
    double *csum = bc + T::BC_D;                                  // [OROW]
    double *wsc = csum + T::OROW;                                 // [4]
    double *wmx = wsc + 4;                                        // [2 Q]: max_n <z_i z_i>, max_n |<z_i>| of this warp's rows
    uint64_t *bar = reinterpret_cast<uint64_t *>(wmx + 2 * Q);

    for (int c = lane; c < T::OROW; c += 32) csum[c] = 0.0;
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_init(bar + 1, 1);
    }
    // INT8 guard (kernels.h: I8Check): a row whose largest diagonal entry is below `thr` carries too much fixed-point rounding
    if (chk.gscale != nullptr) {                                 // kernel-uniform
        double mx = 0.0;
        for (int c = tid; c < chk.ncols; c += 32 * T::WARPS) mx = fmax(mx, chk.gscale[c]);
        for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        if (lane == 0) s_chk[warp] = mx;
    }
    mbar_fence_init();
    __syncthreads();
    double thr = -1.0;
    if (chk.gscale != nullptr) {
        double mx = s_chk[0];
        for (int w = 1; w < T::WARPS; ++w) mx = fmax(mx, s_chk[w]);
        thr = gl[PYVB_GL_TAU] * chk.fac * mx;
    }
    if (cond != nullptr && blockIdx.x == 0 && tid == 0) gl[PYVB_GL_I8FALL] += 1.0;

    int row[RPL], trow[RPL];
#pragma unroll
    for (int r = 0; r < RPL; ++r) {
        row[r] = l + r * LPM;
        trow[r] = g_tri(row[r]);
    }
    double dmx[RPL], zmx[RPL], s_qld = 0.0, s_ld = 0.0, s_n = 0.0;
#pragma unroll
    for (int r = 0; r < RPL; ++r) dmx[r] = zmx[r] = 0.0;

    const long long nwarps = (long long)gridDim.x * T::WARPS;
    const long long ngroups = (N + MPW - 1) / MPW;
    long long g = (long long)blockIdx.x * T::WARPS + warp;
    // Two stages: while group g is inverted in stage s, the bulk copy of the warp's next group lands in stage s ^ 1 (whose
    // store -- the group before g -- has been read by then).  With one stage every group paid the store's read + the next
    // load's latency with the warp idle, and an issue-bound kernel at two warps per scheduler cannot hide an idle warp.
    if (g < ngroups && lane == 0) {                               // the first group of this warp
        const long long left = N - g * MPW;
        const uint32_t bytes = (uint32_t)((left < MPW ? left : MPW) * PITCH * 8);
        mbar_arrive_expect_tx(bar, bytes);
        bulk_g2s(stage, MZ + g * MPW * PITCH, bytes, bar);
    }
    for (int it = 0; g < ngroups; g += nwarps, ++it) {
        const int sidx = it & 1;
        double *stg = stage + sidx * T::STAGE_D;                  // this group's rows
        double *st = stg + m * PITCH;                             // this lane's matrix
        const long long n0 = g * MPW;
        const int nval = (N - n0 < MPW) ? (int)(N - n0) : MPW;
        const bool valid = m < nval;
        const long long gn = g + nwarps;                         // the warp's next group: into the other stage now
        if (lane == 0 && gn < ngroups) {
            bulk_wait_read_all();                                // (the store of the group before this one has read that stage)
            const long long left = N - gn * MPW;
            const uint32_t bytes = (uint32_t)((left < MPW ? left : MPW) * PITCH * 8);
            mbar_arrive_expect_tx(bar + (sidx ^ 1), bytes);
            bulk_g2s(stage + (sidx ^ 1) * T::STAGE_D, MZ + gn * MPW * PITCH, bytes, bar + (sidx ^ 1));
        }
        mbar_wait(bar + sidx, (uint32_t)((it >> 1) & 1));

        // ---- rows of the packed lower triangle -> full rows in registers
        double a[RPL][Q];
#pragma unroll
        for (int r = 0; r < RPL; ++r)
#pragma unroll
            for (int j = 0; j < Q; ++j) {
                int idx;
                if (j / LPM < r) idx = trow[r] + j;                      // always below the diagonal
                else if (j / LPM > r) idx = g_tri(j) + row[r];           // always above: the transposed entry
                else idx = (j <= row[r]) ? trow[r] + j : g_tri(j) + row[r];
                a[r][j] = st[idx];
            }
        if (thr >= 0.0) {                                        // diagonal of qprec (kernel-uniform branch)
            double dm = 0.0;
#pragma unroll
            for (int r = 0; r < RPL; ++r) dm = fmax(dm, st[trow[r] + row[r]]);
#pragma unroll
            for (int o = LPM / 2; o > 0; o >>= 1) dm = fmax(dm, __shfl_xor_sync(0xffffffffu, dm, o));
            if (l == 0 && valid && thr > dm) atomicAdd(&gl[PYVB_GL_I8BAD], 1.0);
        }

        // ---- Gauss-Jordan sweep over the q pivots
        double sinv[RPL];
#pragma unroll
        for (int r = 0; r < RPL; ++r) sinv[r] = 1.0;
        // Software pipeline over the pivots, so that a single warp keeps the FP64 pipe busy (two warps per scheduler are all the
        // register file allows at q = 32):
        //  * 1 / d_{k+1} is computed ONE STEP AHEAD by every lane: the row that is pivoted next publishes its diagonal entry
        //    beside its column entry, and d_{k+1} = a_{k+1,k+1} - b_{k+1}^2 / d_k -- the MUFU + Newton chain runs under the DFMAs;
        //  * step k first updates columns k + 1, k + 2, publishes column k + 1 (the next broadcast) and only then runs the other
        //    q - 3 columns, refilling B[] IN PLACE with the next step's published values as it goes: the shared-memory round
        //    trip of step k + 1 hides behind the arithmetic of step k.
        double2 B[Q / 2];
        double dgp = 0.0;                                        // published diagonal entry of the row that is pivoted next
        {
#pragma unroll
            for (int r = 0; r < RPL; ++r) bc[T::bidx(m, row[r])] = a[r][0];
            if (1 < Q && l == (1 % LPM)) bc[MPW * Q + m] = a[1 / LPM][1];
            __syncwarp();
#pragma unroll
            for (int i = 0; i < Q / 2; ++i) B[i] = *reinterpret_cast<const double2 *>(bc + T::bidx(m, 2 * i));
            dgp = bc[MPW * Q + m];
        }
        double rc = rcp_nr(B[0].x);
#pragma unroll
        for (int k = 0; k < Q; ++k) {
            const int rk = k / LPM;                              // which of a lane's rows can be the pivot row
            const bool piv = (l == (k % LPM));
            const double *bn = bc + ((k + 1) & 1) * T::BC_P;     // where step k + 1 is published
            double t[RPL];
#pragma unroll
            for (int r = 0; r < RPL; ++r) t[r] = -a[r][k] * rc;
            t[rk] = piv ? 0.0 : t[rk];
            sinv[rk] = piv ? -rc : sinv[rk];
            // pairs of columns that go first: those of columns k + 1 and k + 2
            const int p1 = (k + 1 < Q) ? (k + 1) / 2 : -1, p2 = (k + 2 < Q) ? (k + 2) / 2 : -1;
            double rcn = 0.0;
            if (k + 1 < Q) {
                const double b1 = ((k + 1) & 1) ? B[(k + 1) / 2].y : B[(k + 1) / 2].x;
                rcn = rcp_nr(fma(-(b1 * rc), b1, dgp));
#pragma unroll
                for (int i = 0; i < Q / 2; ++i) {
                    if (i != p1 && i != p2) continue;
#pragma unroll
                    for (int r = 0; r < RPL; ++r) {
                        if (2 * i != k) a[r][2 * i] = fma(t[r], B[i].x, a[r][2 * i]);
                        if (2 * i + 1 != k) a[r][2 * i + 1] = fma(t[r], B[i].y, a[r][2 * i + 1]);
                    }
                }
                double *bw = bc + ((k + 1) & 1) * T::BC_P;
#pragma unroll
                for (int r = 0; r < RPL; ++r) bw[T::bidx(m, row[r])] = a[r][k + 1] * sinv[r];
                if (k + 2 < Q && l == ((k + 2) % LPM)) bw[MPW * Q + m] = a[(k + 2) / LPM][k + 2];
                __syncwarp();
#pragma unroll
                for (int i = 0; i < Q / 2; ++i)
                    if (i == p1 || i == p2) B[i] = *reinterpret_cast<const double2 *>(bn + T::bidx(m, 2 * i));
                if (k + 2 < Q) dgp = bn[MPW * Q + m];
            }
#pragma unroll
            for (int i = 0; i < Q / 2; ++i) {
                if (i == p1 || i == p2) continue;
#pragma unroll
                for (int r = 0; r < RPL; ++r) {
                    if (2 * i != k) a[r][2 * i] = fma(t[r], B[i].x, a[r][2 * i]);
                    if (2 * i + 1 != k) a[r][2 * i + 1] = fma(t[r], B[i].y, a[r][2 * i + 1]);
                }
                if (k + 1 < Q) B[i] = *reinterpret_cast<const double2 *>(bn + T::bidx(m, 2 * i));
            }
#pragma unroll
            for (int r = 0; r < RPL; ++r) a[r][k] = t[r];
            a[rk][k] = piv ? 1.0 : t[rk];
            rc = rcn;
        }

        // ---- ln prod diag chol = -1/2 sum ln(1 / d_i); a pivot <= 0 (or NaN) poisons the logarithm
        double pr = 1.0;
        bool pos = true;
#pragma unroll
        for (int r = 0; r < RPL; ++r) {
            pr *= -sinv[r];
            pos = pos && (-sinv[r] > 0.0);
        }
        double lg = pos ? log(pr) : __longlong_as_double(0x7ff8000000000000LL);
#pragma unroll
        for (int o = LPM / 2; o > 0; o >>= 1) lg += __shfl_xor_sync(0xffffffffu, lg, o);
        const double ldsum = -0.5 * lg;

        // ---- Sigma = deferred row scaling; zbar = Sigma eta
        double z[RPL];
#pragma unroll
        for (int r = 0; r < RPL; ++r) {
            const double s = -sinv[r];
#pragma unroll
            for (int j = 0; j < Q; ++j) a[r][j] *= s;
            z[r] = 0.0;
        }
#pragma unroll
        for (int j2 = 0; j2 < Q / 2; ++j2) {
            const double2 E = *reinterpret_cast<const double2 *>(st + PP + 2 * j2);
#pragma unroll
            for (int r = 0; r < RPL; ++r) z[r] = fma(a[r][2 * j2 + 1], E.y, fma(a[r][2 * j2], E.x, z[r]));
        }
        __syncwarp();                                            // every lane has read eta
#pragma unroll
        for (int r = 0; r < RPL; ++r) st[PP + row[r]] = z[r];    // zbar takes eta's place
        if (Sig != nullptr && valid) {                           // (uncoalesced; the Sigma output is optional)
            double *sg = Sig + (n0 + m) * P;
#pragma unroll
            for (int r = 0; r < RPL; ++r)
#pragma unroll
                for (int j = 0; j < Q; ++j) {
                    if (j / LPM > r) continue;
                    if (j / LPM < r || j <= row[r]) sg[trow[r] + j] = a[r][j];
                }
        }
        __syncwarp();
        // ---- <zz^T> = Sigma + zbar zbar^T, packed in place
#pragma unroll
        for (int j2 = 0; j2 < Q / 2; ++j2) {
            const double2 Z = *reinterpret_cast<const double2 *>(st + PP + 2 * j2);
#pragma unroll
            for (int r = 0; r < RPL; ++r) {
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int j = 2 * j2 + h;
                    if (j / LPM > r) continue;
                    const double v = fma(z[r], h ? Z.y : Z.x, a[r][j]);
                    if (j / LPM < r || j <= row[r]) st[trow[r] + j] = v;
                }
            }
        }
        if (valid) {
#pragma unroll
            for (int r = 0; r < RPL; ++r) {
                dmx[r] = fmax(dmx[r], st[trow[r] + row[r]]);     // <z_i z_i> (own write)
                zmx[r] = fmax(zmx[r], fabs(z[r]));
            }
            if (l == 0) {
                logdet[n0 + m] = ldsum;
                s_qld += 0.5 / ldsum;
                s_ld += ldsum;
                s_n += 1.0;
                if (!(ldsum - ldsum == 0.0)) atomicAdd(&gl[PYVB_GL_NONPD], 1.0);   // NaN / inf <=> a pivot was <= 0
            }
        }
        fence_async_smem();
        __syncwarp();
        // ---- rows back to HBM (one bulk store), column sums of the finished rows, next group in
        if (lane == 0) {
            bulk_s2g(MZ + n0 * PITCH, stg, (uint32_t)(nval * PITCH * 8));
            bulk_commit();
        }
        if (zsums != nullptr) {                                  // kernel-uniform
            for (int c = lane; c < T::OROW; c += 32) {
                double v = 0.0;
#pragma unroll
                for (int mm = 0; mm < MPW; ++mm)
                    if (mm < nval) v += stg[mm * PITCH + c];
                csum[c] += v;
            }
        }
        __syncwarp();
    }
    if (lane == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");

    if (zsums == nullptr) return;                                // kernel-uniform
    // ---- CTA partial: [column sums | sum 0.5/logdet | sum logdet | rows | 0 | bounds on the column maxima]
    s_qld = warp_sum(s_qld);
    s_ld = warp_sum(s_ld);
    s_n = warp_sum(s_n);
    if (lane == 0) {
        wsc[0] = s_qld;
        wsc[1] = s_ld;
        wsc[2] = s_n;
        wsc[3] = 0.0;
    }
#pragma unroll
    for (int r = 0; r < RPL; ++r) {
#pragma unroll
        for (int o = LPM; o < 32; o <<= 1) {                      // fold the matrices of the warp
            dmx[r] = fmax(dmx[r], __shfl_xor_sync(0xffffffffu, dmx[r], o));
            zmx[r] = fmax(zmx[r], __shfl_xor_sync(0xffffffffu, zmx[r], o));
        }
        if (m == 0) {
            wmx[row[r]] = dmx[r];
            wmx[Q + row[r]] = zmx[r];
        }
    }
    __syncthreads();
    double *out = zsums + (size_t)blockIdx.x * T::KW;
    const double *w0 = smem_gj + 2 * T::STAGE_D + T::BC_D;            // csum of warp 0
    for (int c = tid; c < T::OROW + 4; c += 32 * T::WARPS) {
        double v = 0.0;
        for (int w = 0; w < T::WARPS; ++w) v += w0[(size_t)w * T::WARP_D + c];   // [csum OROW | scalars 4] is contiguous
        out[c] = v;
    }
    // CTA maxima of the diagonal second moments and of |z| (folded into warp 0's slots), then the column bounds:
    // |<z_i z_j>| <= sqrt(<z_i z_i> <z_j z_j>) because <zz^T> is PSD
    const double *m0 = w0 + T::OROW + 4;
    double *fm = smem_gj;                                        // warp 0's stage is free now: [2 Q] folded maxima
    for (int c = tid; c < 2 * Q; c += 32 * T::WARPS) {
        double v = 0.0;
        for (int w = 0; w < T::WARPS; ++w) v = fmax(v, m0[(size_t)w * T::WARP_D + c]);
        fm[c] = v;
    }
    __syncthreads();
    for (int c = tid; c < T::OROW; c += 32 * T::WARPS) {
        double v = 0.0;
        if (c < P) {
            int i, j;
            unpack_p(c, i, j);
            v = sqrt(fm[i] * fm[j]);
        } else if (c >= PP) {
            v = fm[Q + c - PP];
        }
        out[T::OROW + 4 + c] = v;
    }
}

// The configuration of each q (rows per lane, warps per CTA).  Measured per launch (B200): q = 16, N = 1M: (4, 8) 0.642 ms,
// (2, 16) 0.79, (2, 12) 0.81, (2, 8) 0.89, (1, 16) 1.06; q = 32, N = 1.25M: (2, 8) 5.9 ms, (1, 12) 6.8, and 12 warps at two rows
// per lane spill (168 registers) and serialise the broadcast loads.  More rows per lane = fewer broadcast loads per DFMA.
using GJ16 = GJ<16, 4, 8>;
using GJ32 = GJ<32, 2, 8>;

template <typename T>
int gj_blocks(long long N) {
    long long b = (N + (long long)T::MPW * T::WARPS - 1) / ((long long)T::MPW * T::WARPS);
    if (b > 148) b = 148;
    if (b < 1) b = 1;
    return (int)b;
}

template <int Q, int RPL, int WARPS>
cudaError_t launch_gj_cfg(long long N, double *MZ, double *Sig, double *logdet, double *gl, double *zsums, cudaStream_t st,
                          const double *cond, I8Check chk) {
    using T = GJ<Q, RPL, WARPS>;
    cudaError_t e = cudaFuncSetAttribute(zsolve_gj_kernel<Q, RPL, WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)T::SMEM);
    if (e != cudaSuccess) return e;
    zsolve_gj_kernel<Q, RPL, WARPS><<<gj_blocks<T>(N), 32 * WARPS, T::SMEM, st>>>(N, MZ, Sig, logdet, gl, zsums, cond, chk);
    return cudaGetLastError();
}

}  // namespace

int zsolve_gj_blocks(long long N, int q) { return q == 16 ? gj_blocks<GJ16>(N) : q == 32 ? gj_blocks<GJ32>(N) : 0; }

int zsolve_gj_kw(int q) { return q == 16 ? GJ16::KW : q == 32 ? GJ32::KW : 0; }

cudaError_t launch_zsolve_gj(long long N, int q, double *MZ, double *Sig, double *logdet, double *gl, double *zsums,
                             cudaStream_t st, const double *cond, I8Check chk) {
    if (N <= 0) return cudaSuccess;
    if (q == 16) return launch_gj_cfg<16, GJ16::RPL, GJ16::WARPS>(N, MZ, Sig, logdet, gl, zsums, st, cond, chk);
    if (q == 32) return launch_gj_cfg<32, GJ32::RPL, GJ32::WARPS>(N, MZ, Sig, logdet, gl, zsums, st, cond, chk);
    return cudaErrorNotSupported;
}

}  // namespace pyvb
