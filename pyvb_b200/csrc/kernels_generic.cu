// Generic FP64 kernels of the VB-PCA hot path: any D, any q <= 64.
//
// They are the correctness path for odd shapes (the shipped workload is D=5, q=2)
// and host the small replicated updates (W columns, Mu, Gamma, ELBO).  The
// throughput path for q in {8,16,32}, D % 16 == 0 is kernels_dmma.cu.
//
// Reference arithmetic restated here (paths under /root/reference/src/pyvb):
//   zstep   : nodes/node.py:203-227 (m1, m2 for requester z) + nodes/gaussian.py:117-123
//   stats   : nodes/nodes_todo.py:50-61 (hstack sums), nodes/nodes_todo.py:136-138 (Gamma traces)
//   wupdate : nodes/nodes_todo.py:53-62 + nodes/gaussian.py:117-123 (diagonal precision)
//   wrows   : the row-wise W posterior (DESIGN 5e), one q x q block per data dimension solved by K2
//   global  : nodes/node.py:105-109 (Mu), nodes/nodes_todo.py:130-157, nodes/gaussian.py:136-151
//   impute  : nodes/gaussian.py:125-134
#include "common.cuh"
#include "kernels.h"

namespace pyvb {

// =============================================================== pack Gw
// ND: per-dimension noise precisions (include/pyvb_b200.h, "nd" block) folded into the row: [tau_d G_d | pad | tau_d wbar_d |
// mu_d], so that every Z-step contraction computes sum_d O_nd tau_d G_d and sum_d O_nd (x_nd - mu_d) tau_d wbar_d unchanged
// WR: row-wise W posterior -- G_d = wbar_d wbar_d^T + Sigma_d with the packed row covariances Wcov [D][P] (Wvar is not read)
template <bool ND, bool WR = false>
__global__ void pack_gw_kernel(int D, int q, const double *__restrict__ Wbar, const double *__restrict__ Wvar,
                               const double *__restrict__ mu, const double *__restrict__ tau_d, double *__restrict__ Gw,
                               int ldg, const double *__restrict__ Wcov = nullptr) {
    const int d = blockIdx.x;
    if (d >= D) return;
    const int P = tri(q), Pp = gw_woff(q);
    const double *w = Wbar + (size_t)d * q;
    const double *v = Wvar + (size_t)d * q;
    double *g = Gw + (size_t)d * ldg;
    const double t = ND ? tau_d[d] : 1.0;
    for (int idx = threadIdx.x; idx < q * q; idx += blockDim.x) {
        const int i = idx / q, j = idx % q;
        if (j <= i) {
            double val = w[i] * w[j];
            if (WR) val += Wcov[(size_t)d * P + tri(i) + j];
            else if (i == j) val += v[i];
            if (ND) val *= t;
            g[tri(i) + j] = val;
        }
    }
    for (int c = P + threadIdx.x; c < ldg; c += blockDim.x) {
        double val = 0.0;
        if (c >= Pp && c < Pp + q) val = ND ? t * w[c - Pp] : w[c - Pp];
        else if (c == Pp + q) val = mu[d];
        g[c] = val;
    }
}

cudaError_t launch_pack_gw(int D, int q, const double *Wbar, const double *Wvar, const double *mu, const double *tau_d,
                           double *Gw, int ldg, cudaStream_t st, const double *Wcov) {
    if (Wcov) {
        if (tau_d) pack_gw_kernel<true, true><<<D, 128, 0, st>>>(D, q, Wbar, nullptr, mu, tau_d, Gw, ldg, Wcov);
        else pack_gw_kernel<false, true><<<D, 128, 0, st>>>(D, q, Wbar, nullptr, mu, nullptr, Gw, ldg, Wcov);
    } else if (tau_d) pack_gw_kernel<true><<<D, 128, 0, st>>>(D, q, Wbar, Wvar, mu, tau_d, Gw, ldg);
    else pack_gw_kernel<false><<<D, 128, 0, st>>>(D, q, Wbar, Wvar, mu, nullptr, Gw, ldg);
    return cudaGetLastError();
}

// =============================================================== Z step (K1+K2), one warp per row
// K2 follows the reference literally (nodes/gaussian.py:118-123): Cholesky factor of qprec, then
// cho_solve against the identity (two triangular solves per column; lane j owns column j), then
// qmu = qcov . (pprec.pmu + sum m2).  ln prod diag chol comes from the factor's diagonal.
// WT: per-entry observation weights S [N][lds]: qprec_n = P0 + tau sum_d s_nd G_d, eta_n = h0 + tau sum_d s_nd (x_nd - mu_d) wbar_d
// (an entry of weight 0 is skipped, as a NaN)
// KN: the last kn of the q dimensions are known per row, c_n = Cv[n][0, kn) (row covariates, DESIGN.md 5f): between the
// contraction and the factorisation the row is conditioned on them in shared memory (eta_z -= qprec_zc c, qprec_zc = 0,
// qprec_cc = I, eta_c = c: kernels_known.cu's condition), and the finished row gets zbar_c = c, <z z^T>_cc = c_i c_j
template <int NT, int WPB, bool WT, bool KN = false>
__global__ void __launch_bounds__(32 * WPB)
zstep_generic_kernel(long long N, int D, int q, const double *__restrict__ X, long long ldx,
                     const double *__restrict__ Gw, int ldg, const double *__restrict__ P0,
                     const double *__restrict__ h0, double *gl, double *__restrict__ Zbar, long long ldz,
                     double *__restrict__ M2, long long ldm, double *__restrict__ Sig,
                     double *__restrict__ logdet, const double *__restrict__ S, long long lds,
                     const double *__restrict__ Cv, long long ldc, int kn) {
    extern __shared__ double smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int P = tri(q), Pp = gw_woff(q), C = P + q;
    const int pitch = q + 1;
    const int per_warp = 2 * q * pitch + 2 * q;
    double *a = smem + (size_t)warp * per_warp;   // qprec, overwritten by its Cholesky factor (lower)
    double *sv = a + q * pitch;                   // solution columns: sv[i*pitch + j], column j <- lane j
    double *eta = sv + q * pitch;
    double *zb = eta + q;
    const double tau = gl[PYVB_GL_TAU];
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);

    for (long long n = (long long)blockIdx.x * WPB + warp; n < N; n += (long long)gridDim.x * WPB) {
        double acc[NT];
#pragma unroll
        for (int t = 0; t < NT; ++t) acc[t] = 0.0;
        const double *xr = X + n * ldx;
        for (int d0 = 0; d0 < D; d0 += 32) {
            const int d = d0 + lane;
            const double xv = (d < D) ? xr[d] : qnan;
            const double sv = (WT && d < D) ? S[n * lds + d] : 1.0;
            const int dmax = min(32, D - d0);
            for (int dd = 0; dd < dmax; ++dd) {
                const double x = __shfl_sync(0xffffffffu, xv, dd);
                if (x != x) continue;  // not observed: warp-uniform
                const double *g = Gw + (size_t)(d0 + dd) * ldg;
                if (WT) {
                    const double w = __shfl_sync(0xffffffffu, sv, dd);
                    if (w == 0.0) continue;
                    const double xm = w * (x - g[Pp + q]);
#pragma unroll
                    for (int t = 0; t < NT; ++t) {
                        const int c = lane + 32 * t;
                        if (c < P) acc[t] = fma(w, g[c], acc[t]);
                        else if (c < C) acc[t] = fma(xm, g[c - P + Pp], acc[t]);
                    }
                    continue;
                }
                const double xm = x - g[Pp + q];
#pragma unroll
                for (int t = 0; t < NT; ++t) {
                    const int c = lane + 32 * t;
                    if (c < P) acc[t] += g[c];
                    else if (c < C) acc[t] = fma(xm, g[c - P + Pp], acc[t]);
                }
            }
        }
        __syncwarp();
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            const int c = lane + 32 * t;
            if (c < P) {
                int i, j;
                unpack_p(c, i, j);
                a[i * pitch + j] = P0[i * q + j] + tau * acc[t];   // lower triangle
            } else if (c < C) {
                eta[c - P] = h0[c - P] + tau * acc[t];
            }
        }
        __syncwarp();
        if (KN) {
            const double *cn = Cv + n * ldc;
            const int qf = q - kn;
            for (int i = lane; i < qf; i += 32) {
                double e = eta[i];
                for (int j = 0; j < kn; ++j) e = fma(-a[(qf + j) * pitch + i], cn[j], e);
                eta[i] = e;
            }
            __syncwarp();                           // every zc entry is read before the tail rows are overwritten
            for (int r = qf + lane; r < q; r += 32) {
                for (int m = 0; m <= r; ++m) a[r * pitch + m] = (m == r) ? 1.0 : 0.0;
                eta[r] = cn[r - qf];
            }
            __syncwarp();
        }
        // ---- left-looking Cholesky, lanes over rows
        double ld = 0.0;
        bool ok = true;
        for (int k = 0; k < q; ++k) {
            for (int r = k + lane; r < q; r += 32) {
                double v = a[r * pitch + k];
                for (int m = 0; m < k; ++m) v = fma(-a[r * pitch + m], a[k * pitch + m], v);
                a[r * pitch + k] = v;
            }
            __syncwarp();
            const double dkk = a[k * pitch + k];
            if (!(dkk > 0.0)) ok = false;
            const double lkk = sqrt(dkk);
            ld += log(lkk);
            __syncwarp();
            for (int r = k + lane; r < q; r += 32) a[r * pitch + k] = (r == k) ? lkk : a[r * pitch + k] / lkk;
            __syncwarp();
        }
        // ---- cho_solve(L, I): column j by lane j
        for (int j = lane; j < q; j += 32) {
            for (int i = 0; i < q; ++i) {           // forward: L y = e_j
                double t = (i == j) ? 1.0 : 0.0;
                for (int m = 0; m < i; ++m) t = fma(-a[i * pitch + m], sv[m * pitch + j], t);
                sv[i * pitch + j] = t / a[i * pitch + i];
            }
            for (int i = q - 1; i >= 0; --i) {      // backward: L^T s = y
                double t = sv[i * pitch + j];
                for (int m = i + 1; m < q; ++m) t = fma(-a[m * pitch + i], sv[m * pitch + j], t);
                sv[i * pitch + j] = t / a[i * pitch + i];
            }
        }
        __syncwarp();
        for (int r = lane; r < q; r += 32) {
            double z = 0.0;
            for (int j = 0; j < q; ++j) z = fma(sv[r * pitch + j], eta[j], z);
            if (KN && r >= q - kn) z = Cv[n * ldc + r - (q - kn)];
            zb[r] = z;
            Zbar[n * ldz + r] = z;
        }
        __syncwarp();
        for (int p = lane; p < P; p += 32) {
            int i, j;
            unpack_p(p, i, j);
            const double sg = 0.5 * (sv[i * pitch + j] + sv[j * pitch + i]);
            if (KN && j >= q - kn) M2[n * ldm + p] = zb[i] * zb[j];      // <c c^T>: no variance
            else M2[n * ldm + p] = fma(zb[i], zb[j], sg);
            if (Sig) Sig[n * P + p] = sg;
        }
        if (lane == 0) {
            logdet[n] = ld;
            if (!ok) atomicAdd(&gl[PYVB_GL_NONPD], 1.0);
        }
        __syncwarp();
    }
}

cudaError_t launch_zstep_generic(long long N, int D, int q, const double *X, long long ldx, const double *Gw,
                                 int ldg, const double *P0, const double *h0, double *gl, double *Zbar,
                                 long long ldz, double *M2, long long ldm, double *Sig, double *logdet,
                                 cudaStream_t st, const double *S, long long lds, const double *Cv, long long ldc, int kn) {
    if (N <= 0) return cudaSuccess;
    const int C = tri(q) + q;
    const int nt = (C + 31) / 32;
    const int wpb = (q > 32) ? 2 : 4;
    const size_t smem = (size_t)wpb * (2 * q * (q + 1) + 2 * q) * sizeof(double);
    long long blocks = (N + wpb - 1) / wpb;
    if (blocks > 148 * 16) blocks = 148 * 16;
#define PYVB_LAUNCH_ZK(NT, WPB, WT, KN)                                                                        \
    do {                                                                                                       \
        cudaError_t e = cudaFuncSetAttribute(zstep_generic_kernel<NT, WPB, WT, KN>,                            \
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);          \
        if (e != cudaSuccess) return e;                                                                        \
        zstep_generic_kernel<NT, WPB, WT, KN><<<(unsigned)blocks, 32 * WPB, smem, st>>>(                       \
            N, D, q, X, ldx, Gw, ldg, P0, h0, gl, Zbar, ldz, M2, ldm, Sig, logdet, S, lds, Cv, ldc, kn);       \
    } while (0)
#define PYVB_LAUNCH_ZW(NT, WPB, WT)                                                                            \
    do {                                                                                                       \
        if (Cv) PYVB_LAUNCH_ZK(NT, WPB, WT, true);                                                             \
        else PYVB_LAUNCH_ZK(NT, WPB, WT, false);                                                               \
    } while (0)
#define PYVB_LAUNCH_Z(NT, WPB)                                                                                 \
    do {                                                                                                       \
        if (S) PYVB_LAUNCH_ZW(NT, WPB, true);                                                                  \
        else PYVB_LAUNCH_ZW(NT, WPB, false);                                                                   \
    } while (0)
    if (nt <= 1) PYVB_LAUNCH_Z(1, 4);
    else if (nt <= 2) PYVB_LAUNCH_Z(2, 4);
    else if (nt <= 5) PYVB_LAUNCH_Z(5, 4);
    else if (nt <= 18) PYVB_LAUNCH_Z(18, 4);
    else PYVB_LAUNCH_Z(67, 2);
#undef PYVB_LAUNCH_Z
#undef PYVB_LAUNCH_ZW
#undef PYVB_LAUNCH_ZK
    return cudaGetLastError();
}

// =============================================================== statistics (K3), generic
// One thread per output element, rows of a chunk in the inner loop.  Outputs are per-chunk partial
// sums (deterministic two-stage reduction).  WT: every observed entry counts with its weight s_nd (S [N][lds]): T1, Bst, Ast,
// cnt = sum s, colx = sum s x.
template <bool WT>
__global__ void __launch_bounds__(256)
stats_generic_kernel(long long N, int D, int q, const double *__restrict__ X, long long ldx,
                     const double *__restrict__ Zbar, long long ldz, const double *__restrict__ M2,
                     long long ldm, double *__restrict__ ws, long long rows_per_chunk, const double *__restrict__ S,
                     long long lds) {
    const StatLayout L(D, q);
    const int P = L.P;
    const int CT = P + 2 * q + 2;
    const long long nout = (long long)D * CT + P + q;
    const long long r0 = (long long)blockIdx.y * rows_per_chunk;
    const long long r1 = min(N, r0 + rows_per_chunk);
    double *out = ws + (size_t)blockIdx.y * L.len;
    for (long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x; o < nout;
         o += (long long)gridDim.x * blockDim.x) {
        double acc = 0.0;
        size_t dest;
        if (o < (long long)D * CT) {
            const int d = (int)(o / CT), c = (int)(o % CT);
            if (c < P) {
                for (long long n = r0; n < r1; ++n) {
                    const double x = X[n * ldx + d];
                    if (x == x) acc = WT ? fma(S[n * lds + d], M2[n * ldm + c], acc) : acc + M2[n * ldm + c];
                }
                dest = L.t1 + (size_t)d * P + c;
            } else if (c < P + q) {
                const int i = c - P;
                for (long long n = r0; n < r1; ++n) {
                    const double x = X[n * ldx + d];
                    if (x == x) acc = WT ? fma(S[n * lds + d], Zbar[n * ldz + i], acc) : acc + Zbar[n * ldz + i];
                }
                dest = L.bst + (size_t)d * q + i;
            } else if (c < P + 2 * q) {
                const int i = c - P - q;
                for (long long n = r0; n < r1; ++n) {
                    const double x = X[n * ldx + d];
                    if (x == x) acc = fma(WT ? S[n * lds + d] * x : x, Zbar[n * ldz + i], acc);
                }
                dest = L.ast + (size_t)d * q + i;
            } else if (c == P + 2 * q) {
                for (long long n = r0; n < r1; ++n) {
                    const double x = X[n * ldx + d];
                    if (x == x) acc += WT ? S[n * lds + d] : 1.0;
                }
                dest = L.cnt + d;
            } else {
                for (long long n = r0; n < r1; ++n) {
                    const double x = X[n * ldx + d];
                    if (x == x) acc = WT ? fma(S[n * lds + d], x, acc) : acc + x;
                }
                dest = L.colx + d;
            }
        } else {
            const int c = (int)(o - (long long)D * CT);
            if (c < P) {
                for (long long n = r0; n < r1; ++n) acc += M2[n * ldm + c];
                dest = L.S + c;
            } else {
                for (long long n = r0; n < r1; ++n) acc += Zbar[n * ldz + (c - P)];
                dest = L.zsum + (c - P);
            }
        }
        out[dest] = acc;
    }
}

int stats_generic_nchunks(long long N) {
    long long c = (N + 255) / 256;
    if (c < 1) c = 1;
    if (c > 64) c = 64;
    return (int)c;
}

cudaError_t launch_stats_generic(long long N, int D, int q, const double *X, long long ldx, const double *Zbar,
                                 long long ldz, const double *M2, long long ldm, double *ws_main, int nchunks,
                                 cudaStream_t st, const double *S, long long lds) {
    const int P = tri(q);
    const long long nout = (long long)D * (P + 2 * q + 2) + P + q;
    long long bx = (nout + 255) / 256;
    if (bx > 4096) bx = 4096;
    const long long rpc = (N + nchunks - 1) / nchunks;
    dim3 grid((unsigned)bx, (unsigned)nchunks);
    if (S)
        stats_generic_kernel<true><<<grid, 256, 0, st>>>(N, D, q, X, ldx, Zbar, ldz, M2, ldm, ws_main, rpc > 0 ? rpc : 1, S, lds);
    else
        stats_generic_kernel<false><<<grid, 256, 0, st>>>(N, D, q, X, ldx, Zbar, ldz, M2, ldm, ws_main, rpc > 0 ? rpc : 1,
                                                          nullptr, 0);
    return cudaGetLastError();
}

// =============================================================== column sums of the mask and of O.X
// (the DMMA statistics kernel leaves cnt / colsumX to this HBM-bound pass)
// WT: weighted sums, cnt = sum s, colsumX = sum s x (S [N][lds])
template <int ROWS, bool WT>
__global__ void __launch_bounds__(128)
colsums2_kernel(long long N, int D, int q, const double *__restrict__ X, long long ldx, double *__restrict__ ws,
                long long rows_per_chunk, const double *__restrict__ S, long long lds) {
    const StatLayout L(D, q);
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    const long long r0 = (long long)blockIdx.y * rows_per_chunk;
    long long r1 = r0 + rows_per_chunk;
    if (r1 > N) r1 = N;
    if (d >= D) return;
    double c[ROWS], s[ROWS];
#pragma unroll
    for (int u = 0; u < ROWS; ++u) c[u] = s[u] = 0.0;
    long long n = r0;
    for (; n + ROWS <= r1; n += ROWS) {
#pragma unroll
        for (int u = 0; u < ROWS; ++u) {
            const double x = X[(n + u) * ldx + d];
            if (x == x) {
                if (WT) {
                    const double w = S[(n + u) * lds + d];
                    c[u] += w;
                    s[u] = fma(w, x, s[u]);
                } else {
                    c[u] += 1.0;
                    s[u] += x;
                }
            }
        }
    }
    for (; n < r1; ++n) {
        const double x = X[n * ldx + d];
        if (x == x) {
            if (WT) {
                const double w = S[n * lds + d];
                c[0] += w;
                s[0] = fma(w, x, s[0]);
            } else {
                c[0] += 1.0;
                s[0] += x;
            }
        }
    }
    double ct = 0.0, stot = 0.0;
#pragma unroll
    for (int u = 0; u < ROWS; ++u) {
        ct += c[u];
        stot += s[u];
    }
    double *out = ws + (size_t)blockIdx.y * L.len;
    out[L.cnt + d] = ct;
    out[L.colx + d] = stot;
}

cudaError_t launch_colsums(long long N, int D, int q, const double *X, long long ldx, double *ws_main, int nchunks,
                           cudaStream_t st, const double *S, long long lds) {
    long long rpc = (N + nchunks - 1) / nchunks;
    if (rpc < 1) rpc = 1;
    dim3 grid((unsigned)((D + 127) / 128), (unsigned)nchunks);
    if (S) colsums2_kernel<8, true><<<grid, 128, 0, st>>>(N, D, q, X, ldx, ws_main, rpc, S, lds);
    else colsums2_kernel<8, false><<<grid, 128, 0, st>>>(N, D, q, X, ldx, ws_main, rpc, nullptr, 0);
    return cudaGetLastError();
}

// =============================================================== column sums of [M2 | zbar] -> S, zsum
template <int ROWS>
__global__ void __launch_bounds__(128)
mzsums_kernel(long long N, int D, int q, const double *__restrict__ Zbar, long long ldz,
              const double *__restrict__ M2, long long ldm, double *__restrict__ ws, long long rows_per_chunk) {
    const StatLayout L(D, q);
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= L.P + q) return;
    const long long r0 = (long long)blockIdx.y * rows_per_chunk;
    long long r1 = r0 + rows_per_chunk;
    if (r1 > N) r1 = N;
    const double *src = (c < L.P) ? (M2 + c) : (Zbar + (c - L.P));
    const long long ld = (c < L.P) ? ldm : ldz;
    double s[ROWS];
#pragma unroll
    for (int u = 0; u < ROWS; ++u) s[u] = 0.0;
    long long n = r0;
    for (; n + ROWS <= r1; n += ROWS) {
#pragma unroll
        for (int u = 0; u < ROWS; ++u) s[u] += src[(n + u) * ld];
    }
    for (; n < r1; ++n) s[0] += src[n * ld];
    double t = 0.0;
#pragma unroll
    for (int u = 0; u < ROWS; ++u) t += s[u];
    double *out = ws + (size_t)blockIdx.y * L.len;
    if (c < L.P) out[L.S + c] = t;
    else out[L.zsum + (c - L.P)] = t;
}

cudaError_t launch_mzsums(long long N, int D, int q, const double *Zbar, long long ldz, const double *M2,
                          long long ldm, double *ws_main, int nchunks, cudaStream_t st) {
    long long rpc = (N + nchunks - 1) / nchunks;
    if (rpc < 1) rpc = 1;
    const int C = tri(q) + q;
    dim3 grid((unsigned)((C + 127) / 128), (unsigned)nchunks);
    mzsums_kernel<8><<<grid, 128, 0, st>>>(N, D, q, Zbar, ldz, M2, ldm, ws_main, rpc);
    return cudaGetLastError();
}

// =============================================================== per-row scalars (K4)
// WT (mode B): sxx = sum s x^2 over the observed entries, nE = the NUMBER of observed entries of positive weight
template <bool WT>
__global__ void __launch_bounds__(256)
rowscalars_kernel(long long N, int D, const double *__restrict__ X, long long ldx, const double *__restrict__ V,
                  const double *__restrict__ Xorig, const double *__restrict__ qldX,
                  const double *__restrict__ logdet, double *__restrict__ ws_sc, int skip_x, const double *__restrict__ S,
                  long long lds) {
    __shared__ double sh[33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    double sxx = 0, sumv = 0, ne = 0, qz = 0, ldz = 0, latq = 0, nlat = 0, pnm = 0, plnv = 0, nrows = 0;
    for (long long n = (long long)blockIdx.x * nwarp + warp; n < N; n += (long long)gridDim.x * nwarp) {
        const double *xr = X + n * ldx;
        int nmiss = 0;
        double lnv = 0.0;
        for (int d = lane; d < D && !skip_x; d += 32) {
            const double x = xr[d];
            if (x == x) {
                if (WT) {
                    const double w = S[n * lds + d];
                    sxx = fma(w * x, x, sxx);
                    ne += (w > 0.0) ? 1.0 : 0.0;
                } else {
                    sxx = fma(x, x, sxx);
                    ne += 1.0;
                }
                if (V) sumv += V[n * (long long)D + d];
            }
            if (Xorig) {
                const double xo = Xorig[n * ldx + d];
                if (xo != xo) {
                    ++nmiss;
                    lnv += log(V[n * (long long)D + d]);
                }
            }
        }
        if (Xorig) {
            nmiss = __reduce_add_sync(0xffffffffu, nmiss);
            if (nmiss == D) {
                if (lane == 0) {
                    nlat += 1.0;
                    latq += qldX[n];
                }
            } else if (nmiss > 0) {
                plnv += lnv;
                if (lane == 0) pnm += (double)nmiss;
            }
        }
        if (lane == 0) {
            const double l = logdet[n];
            qz += 0.5 / l;
            ldz += l;
            nrows += 1.0;
        }
    }
    double *out = ws_sc + (size_t)blockIdx.x * PYVB_NSCAL;
    double r;
    r = block_sum(sxx, sh);   if (threadIdx.x == 0) out[PYVB_SC_SXX] = r;
    r = block_sum(sumv, sh);  if (threadIdx.x == 0) out[PYVB_SC_SUMV] = r;
    r = block_sum(ne, sh);    if (threadIdx.x == 0) out[PYVB_SC_NE] = r;
    r = block_sum(qz, sh);    if (threadIdx.x == 0) out[PYVB_SC_QLDZ] = r;
    r = block_sum(ldz, sh);   if (threadIdx.x == 0) out[PYVB_SC_LOGDETZ] = r;
    r = block_sum(latq, sh);  if (threadIdx.x == 0) out[PYVB_SC_LATQLD] = r;
    r = block_sum(nlat, sh);  if (threadIdx.x == 0) out[PYVB_SC_NLAT] = r;
    r = block_sum(pnm, sh);   if (threadIdx.x == 0) out[PYVB_SC_PNMISS] = r;
    r = block_sum(plnv, sh);  if (threadIdx.x == 0) out[PYVB_SC_PLNV] = r;
    r = block_sum(nrows, sh); if (threadIdx.x == 0) out[PYVB_SC_NROWS] = r;
    if (threadIdx.x == 0)
        for (int k = PYVB_SC_NROWS + 1; k < PYVB_NSCAL; ++k) out[k] = 0.0;
}

int rowscalars_nblk(long long N) {
    long long b = (N + 7) / 8;
    if (b < 1) b = 1;
    if (b > 148 * 4) b = 148 * 4;
    return (int)b;
}

cudaError_t launch_rowscalars(long long N, int D, const double *X, long long ldx, const double *V,
                              const double *Xorig, const double *qldX, const double *logdet, double *ws_sc,
                              int nblk, int skip_x, cudaStream_t st, const double *S, long long lds) {
    if (S) rowscalars_kernel<true><<<nblk, 256, 0, st>>>(N, D, X, ldx, V, Xorig, qldX, logdet, ws_sc, skip_x, S, lds);
    else rowscalars_kernel<false><<<nblk, 256, 0, st>>>(N, D, X, ldx, V, Xorig, qldX, logdet, ws_sc, skip_x, nullptr, 0);
    return cudaGetLastError();
}

// =============================================================== deterministic second stage
// sum of n partials p[k * stride], four independent chains combined in a fixed order
__device__ inline double strided_sum(const double *p, int n, size_t stride) {
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
    int k = 0;
    for (; k + 4 <= n; k += 4) {
        a0 += p[(size_t)k * stride];
        a1 += p[(size_t)(k + 1) * stride];
        a2 += p[(size_t)(k + 2) * stride];
        a3 += p[(size_t)(k + 3) * stride];
    }
    for (; k < n; ++k) a0 += p[(size_t)k * stride];
    return (a0 + a1) + (a2 + a3);
}

// ---- peer exchange (multi-GPU, one process per GPU on one NVLink/NVSwitch box)
// Every rank owns a cudaMalloc'd exchange buffer that all other ranks have opened through CUDA IPC:
//   [ flags: uint64 [2][PYVB_PEER_MAXBLK] | slot 0: len doubles | slot 1: len doubles ]   (slots 256-byte aligned)
// The second stage below writes the rank's reduced statistics into its own slot (parity = epoch & 1), publishes a
// per-CTA flag (release, system scope), waits for the same CTA's flag on every peer (acquire over NVLink) and adds the
// peers' slices in rank order: the reduction of the partial sums and the all-reduce are ONE kernel, the result is
// bit-identical on every rank, and there is no host round trip.  Two slots suffice: a rank can only be one exchange
// ahead of the slowest one (it needs everybody's flags of exchange t+1 before it starts t+2).
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ double ld_relaxed_sys(const double *p) {
    double v;
    asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
    return v;
}

__host__ __device__ inline size_t peer_slot_bytes(size_t len) { return (len * sizeof(double) + 255) & ~(size_t)255; }
__host__ __device__ inline size_t peer_flag_bytes() { return 2 * (size_t)PYVB_PEER_MAXBLK * sizeof(unsigned long long); }

__global__ void __launch_bounds__(256)
stats_reduce_kernel(int D, int q, const double *__restrict__ ws_main, int nchunks, const double *__restrict__ ws_sc,
                    int nblk, double *__restrict__ stats, double *xcache, int use_xcache,
                    const double *__restrict__ zsums, int nzblk, int zkw, void *const *peer_bufs, int world, int rank,
                    unsigned long long epoch) {
    const StatLayout L(D, q);
    const int PP = gw_woff(q);
    const bool xchg = (peer_bufs != nullptr) && world > 1;
    const int par = (int)(epoch & 1ULL);
    double *mine = stats;                                   // where the local sums go
    if (xchg) mine = reinterpret_cast<double *>(static_cast<char *>(peer_bufs[rank]) + peer_flag_bytes() +
                                                (size_t)par * peer_slot_bytes(L.len));
    for (size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x; o < L.len; o += (size_t)gridDim.x * blockDim.x) {
        // slot of this entry in the X-only cache [cnt D | colx D | sxx | nE], or -1
        long long xc = -1;
        if (o >= L.cnt && o < L.S) xc = (long long)(o - L.cnt);
        else if (o == L.scal + PYVB_SC_SXX) xc = 2LL * D;
        else if (o == L.scal + PYVB_SC_NE) xc = 2LL * D + 1;
        // slot of this entry in the K2 partials [<zz^T> packed | pad | zbar | 0.5/logdet | logdet | rows], or -1
        int zc = -1;
        if (zsums != nullptr) {
            if (o >= L.S && o < L.zsum) zc = (int)(o - L.S);
            else if (o >= L.zsum && o < L.scal) zc = PP + (int)(o - L.zsum);
            else if (o == L.scal + PYVB_SC_QLDZ) zc = PP + q;
            else if (o == L.scal + PYVB_SC_LOGDETZ) zc = PP + q + 1;
            else if (o == L.scal + PYVB_SC_NROWS) zc = PP + q + 2;
        }
        double acc = 0.0;
        if (xc >= 0 && xcache != nullptr && use_xcache) {
            acc = xcache[xc];
        } else if (zc >= 0) {
            acc = strided_sum(zsums + zc, nzblk, (size_t)zkw);
        } else {
            if (o < L.scal) acc = strided_sum(ws_main + o, nchunks, L.len);
            else if (ws_sc != nullptr) acc = strided_sum(ws_sc + (o - L.scal), nblk, PYVB_NSCAL);
            if (xc >= 0 && xcache != nullptr) xcache[xc] = acc;
        }
        mine[o] = acc;
    }
    if (!xchg) return;
    // ---- publish this CTA's slice, wait for the same slice on every peer, add in rank order
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence_system();
        unsigned long long *flags = static_cast<unsigned long long *>(peer_bufs[rank]);
        st_release_sys(flags + (size_t)par * PYVB_PEER_MAXBLK + blockIdx.x, epoch);
    }
    if ((int)threadIdx.x < world && (int)threadIdx.x != rank) {
        const unsigned long long *pf = static_cast<const unsigned long long *>(peer_bufs[threadIdx.x]) +
                                       (size_t)par * PYVB_PEER_MAXBLK + blockIdx.x;
        // bounded: a dead or failed peer must not hang this GPU forever (~5 s, then the kernel traps: a CUDA error on the
        // next synchronisation instead of a wedged device)
        unsigned int spins = 0;
        while (ld_acquire_sys(pf) < epoch) {
            __nanosleep(256);
            if (++spins > (1u << 24)) __trap();
        }
    }
    __syncthreads();
    for (size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x; o < L.len; o += (size_t)gridDim.x * blockDim.x) {
        double acc = 0.0;
        for (int r = 0; r < world; ++r) {
            const double *src = reinterpret_cast<const double *>(static_cast<const char *>(peer_bufs[r]) +
                                                                 peer_flag_bytes() + (size_t)par * peer_slot_bytes(L.len));
            acc += (r == rank) ? src[o] : ld_relaxed_sys(src + o);
        }
        stats[o] = acc;
    }
}

size_t peer_buffer_bytes(size_t len) { return peer_flag_bytes() + 2 * peer_slot_bytes(len); }

cudaError_t launch_stats_reduce(int D, int q, const double *ws_main, int nchunks, const double *ws_sc, int nblk,
                                double *stats, double *xcache, int use_xcache, const double *zsums, int nzblk,
                                int zkw, void *const *peer_bufs, int world, int rank, unsigned long long epoch,
                                cudaStream_t st) {
    const StatLayout L(D, q);
    size_t b = (L.len + 255) / 256;
    // all CTAs must be co-resident when they wait for their peers: what the occupancy calculator says fits on THIS device
    // (SM count queried, not assumed), at most 2 per SM and <= PYVB_PEER_MAXBLK
    static int cap[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 0 && dev < 64 && cap[dev] == 0) {
        int sms = 0, per = 0;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, stats_reduce_kernel, 256, 0) != cudaSuccess || per <= 0) per = 1;
        if (per > 2) per = 2;
        cap[dev] = sms * per < PYVB_PEER_MAXBLK ? sms * per : PYVB_PEER_MAXBLK;
    }
    const size_t bmax = (dev >= 0 && dev < 64) ? (size_t)cap[dev] : 148;
    if (b > bmax) b = bmax;
    stats_reduce_kernel<<<(unsigned)b, 256, 0, st>>>(D, q, ws_main, nchunks, ws_sc, nblk, stats, xcache, use_xcache,
                                                     zsums, nzblk, zkw, peer_bufs, world, rank, epoch);
    return cudaGetLastError();
}

// =============================================================== W columns (Gauss-Seidel), thread per d
// tau_d (nullable): per-dimension noise precisions; NULL reads the shared tau of gl
// QT > 0: q known at compile time -- the loops unroll and w[] lives in registers (with a run-time q the array is indexed
// dynamically, i.e. it sits in local memory, and every FMA of the q^2-long dependent chain waits for a local load: 36 us at
// D = 256, q = 16); QT = 0: any q.
template <int QT>
__global__ void __launch_bounds__(128)
wupdate_kernel(int D, int q_rt, int col_lo, int col_hi, const double *__restrict__ stats,
               const double *__restrict__ mu, const double *__restrict__ gl, const double *__restrict__ tau_d,
               double *__restrict__ Wbar, double *__restrict__ Wvar) {
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= D) return;
    const int q = QT > 0 ? QT : q_rt;
    const StatLayout L(D, q);
    const int P = L.P;
    const double tau = tau_d ? tau_d[d] : gl[PYVB_GL_TAU];
    const double *T1 = stats + L.t1 + (size_t)d * P;
    const double *Bst = stats + L.bst + (size_t)d * q;
    const double *Ast = stats + L.ast + (size_t)d * q;
    double w[QT > 0 ? QT : PYVB_QMAX];
    const double m = mu[d];
    if (QT > 0) {
#pragma unroll
        for (int i = 0; i < QT; ++i) w[i] = Wbar[(size_t)d * QT + i];
#pragma unroll
        for (int i = 0; i < QT; ++i) {
            if (i < col_lo || i >= col_hi) continue;                 // (kernel-uniform)
            const double prec = gl[PYVB_GL_ALPHA + i] + tau * T1[tri(i) + i];
            double m2 = Ast[i] - m * Bst[i];
#pragma unroll
            for (int j = 0; j < QT; ++j) {
                if (j < i) m2 = fma(-T1[tri(i) + j], w[j], m2);
                if (j > i) m2 = fma(-T1[tri(j) + i], w[j], m2);
            }
            w[i] = tau * m2 / prec;
            Wvar[(size_t)d * QT + i] = 1.0 / prec;
            Wbar[(size_t)d * QT + i] = w[i];
        }
        return;
    }
    for (int i = 0; i < q; ++i) w[i] = Wbar[(size_t)d * q + i];
    for (int i = col_lo; i < col_hi; ++i) {
        const double prec = gl[PYVB_GL_ALPHA + i] + tau * T1[tri(i) + i];
        double m2 = Ast[i] - m * Bst[i];
        for (int j = 0; j < i; ++j) m2 = fma(-T1[tri(i) + j], w[j], m2);
        for (int j = i + 1; j < q; ++j) m2 = fma(-T1[tri(j) + i], w[j], m2);
        w[i] = tau * m2 / prec;
        Wvar[(size_t)d * q + i] = 1.0 / prec;
    }
    for (int i = col_lo; i < col_hi; ++i) Wbar[(size_t)d * q + i] = w[i];
}

cudaError_t launch_wupdate(int D, int q, int col_lo, int col_hi, const double *stats, const double *mu,
                           const double *gl, const double *tau_d, double *Wbar, double *Wvar, cudaStream_t st) {
    const int blocks = (D + 63) / 64;
    switch (q) {
        case 16: wupdate_kernel<16><<<blocks, 64, 0, st>>>(D, q, col_lo, col_hi, stats, mu, gl, tau_d, Wbar, Wvar); break;
        case 32: wupdate_kernel<32><<<blocks, 64, 0, st>>>(D, q, col_lo, col_hi, stats, mu, gl, tau_d, Wbar, Wvar); break;
        case 64: wupdate_kernel<64><<<blocks, 64, 0, st>>>(D, q, col_lo, col_hi, stats, mu, gl, tau_d, Wbar, Wvar); break;
        default: wupdate_kernel<0><<<(D + 127) / 128, 128, 0, st>>>(D, q, col_lo, col_hi, stats, mu, gl, tau_d, Wbar, Wvar);
    }
    return cudaGetLastError();
}

// =============================================================== W rows (row-wise posterior), warp per d
// q(W) = prod_d N(w_d | wbar_d, Sigma_d): Lambda_d = diag(<alpha>) + tau_d T1_d, eta_d = tau_d (Ast_d - mu_d Bst_d).  The
// assemble kernel writes the K2 input row [Lambda_d packed | 0 | eta_d | 0] (pitch pyvb_mz_pitch(q)); launch_zsolve turns it
// into [<w_d w_d^T> packed | 0 | wbar_d | 0] with Sigma_d and ln prod diag chol(Lambda_d) beside it; the finish kernel copies
// wbar_d and diag Sigma_d into Wbar / Wvar, which the ARD update, the bound's prior term and the state read.
// tau_d (nullable): per-dimension noise precisions; NULL reads the shared tau of gl
__global__ void __launch_bounds__(256)
wrows_assemble_kernel(int D, int q, const double *__restrict__ stats, const double *__restrict__ mu,
                      const double *__restrict__ gl, const double *__restrict__ tau_d, double *__restrict__ WM, int ldwm) {
    const int lane = threadIdx.x & 31;
    const int d = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (d >= D) return;
    const StatLayout L(D, q);
    const int P = L.P, Pp = gw_woff(q);
    const double tau = tau_d ? tau_d[d] : gl[PYVB_GL_TAU];
    const double *T1 = stats + L.t1 + (size_t)d * P;
    const double *Bst = stats + L.bst + (size_t)d * q, *Ast = stats + L.ast + (size_t)d * q;
    const double m = mu[d];
    double *r = WM + (size_t)d * ldwm;
    for (int p = lane; p < P; p += 32) {
        int i, j;
        unpack_p(p, i, j);
        r[p] = (i == j) ? fma(tau, T1[p], gl[PYVB_GL_ALPHA + i]) : tau * T1[p];
    }
    for (int c = P + lane; c < ldwm; c += 32) r[c] = (c >= Pp && c < Pp + q) ? tau * fma(-m, Bst[c - Pp], Ast[c - Pp]) : 0.0;
}

__global__ void __launch_bounds__(256)
wrows_finish_kernel(int D, int q, const double *__restrict__ WM, int ldwm, const double *__restrict__ Wcov,
                    double *__restrict__ Wbar, double *__restrict__ Wvar) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= D * q) return;
    const int d = idx / q, i = idx - d * q;
    Wbar[idx] = WM[(size_t)d * ldwm + gw_woff(q) + i];
    Wvar[idx] = Wcov[(size_t)d * tri(q) + tri(i) + i];
}

cudaError_t launch_wupdate_rows(int D, int q, const double *stats, const double *mu, double *gl, const double *tau_d,
                                double *WM, int ldwm, double *Wbar, double *Wvar, double *Wcov, double *Wld, cudaStream_t st) {
    wrows_assemble_kernel<<<(D + 7) / 8, 256, 0, st>>>(D, q, stats, mu, gl, tau_d, WM, ldwm);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = launch_zsolve(D, q, WM, Wcov, Wld, gl, nullptr, st);
    if (e != cudaSuccess) return e;
    wrows_finish_kernel<<<(D * q + 255) / 256, 256, 0, st>>>(D, q, WM, ldwm, Wcov, Wbar, Wvar);
    return cudaGetLastError();
}

// =============================================================== Mu, Gamma(s), ELBO: one CTA (+ helpers of its cluster)
// The kernel is launched as ONE thread-block cluster: rank 0 does everything below; the other CTAs only take their share of the
// D x P contraction  sum_d sum_p g_dp T1[d][p]  of the residual (0.3 of the kernel's 0.35 ms at D = 1024, q = 32 on a single SM),
// hand their partial sums to rank 0 through distributed shared memory (fixed order: deterministic, replicas stay bit-identical)
// and leave.
__device__ __forceinline__ uint32_t gk_cluster_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t gk_cluster_size() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void gk_cluster_sync() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void gk_store_remote(const double *local_smem, uint32_t rank, double v) {
    uint32_t a = (uint32_t)__cvta_generic_to_shared(local_smem), r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
    asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(r), "d"(v) : "memory");
}
// nd (nullable): the per-dimension noise block (include/pyvb_b200.h).  With it, noise_diag_kernel (kernels_noise.cu) has already
// done Mu, the per-dimension Gammas and their bound terms: this kernel skips its scalar Mu / Beta and the contraction, and adds
// the per-dimension X and Beta terms in a fixed order (one CTA).
// WT: weighted data (pyvb_global_w_f64): the X bound term also carries the data constant gl[PYVB_GL_LNS] = 1/2 sum ln s_nd.
// WR: row-wise W posterior (pyvb_global_rows_f64): the contraction reads g = wbar_i wbar_j + Sigma_d,ij from the packed row
// covariances Wcov [D][P], and the entropy part of the W term is that of D row nodes, sum_d [1/2 (0.5 / Wld_d) + q / 2]
// (Wld_d = ln prod diag chol(Lambda_d), the reference's q_ln_det quirk per node) in place of the q column nodes'.
constexpr int GK_CLUSTER = 8;

template <bool WT, bool WR = false>
__global__ void __launch_bounds__(1024)
global_kernel(int D, int q, int ops, int col_lo, int col_hi, const double *__restrict__ stats, const double *__restrict__ Wbar,
              const double *__restrict__ Wvar, double *mu, double *muvar, double *gl,
              const double *__restrict__ P0, const double *__restrict__ h0, const pyvb_consts c,
              double *elbo_out, const double *__restrict__ nd, const double *__restrict__ Wcov = nullptr,
              const double *__restrict__ Wld = nullptr) {
    __shared__ double sh[33];
    __shared__ double cl_part[GK_CLUSTER];                              // the cluster's partial sums of the D x P contraction
    __shared__ unsigned short ijtab[PYVB_QMAX * (PYVB_QMAX + 1) / 2];   // packed index -> (i << 8) | j
    const StatLayout L(D, q);
    const int P = L.P;
    const int tid = threadIdx.x, nt = blockDim.x;
    const int crank = (int)gk_cluster_rank(), csize = (int)gk_cluster_size();
    if (crank != 0 && !(ops & (PYVB_OP_BETA | PYVB_OP_ELBO))) return;   // (kernel-uniform: nobody waits for the helpers)
    for (int p = tid; p < P; p += nt) {
        int i, j;
        unpack_p(p, i, j);
        ijtab[p] = (unsigned short)((i << 8) | j);
    }
    const double *T1 = stats + L.t1, *Bst = stats + L.bst, *Ast = stats + L.ast;
    const double *cnt = stats + L.cnt, *colx = stats + L.colx, *S = stats + L.S, *zsum = stats + L.zsum;
    const double *sc = stats + L.scal;
    const double LN2PI = 1.8378770664093454835606594728112;
    const double qa = gl[PYVB_GL_QA];
    double qb = gl[PYVB_GL_QB];
    double tau = gl[PYVB_GL_TAU];
    __syncthreads();

    if ((ops & PYVB_OP_MU) && crank == 0 && !nd) {
        for (int d = tid; d < D; d += nt) {
            const double prec = c.alpha_mu + tau * cnt[d];
            double s = colx[d];
            for (int i = 0; i < q; ++i) s = fma(-Bst[(size_t)d * q + i], Wbar[(size_t)d * q + i], s);
            mu[d] = tau * s / prec;
            muvar[d] = 1.0 / prec;
        }
        __syncthreads();
    }
    // per-column sums over d: one WARP per column (lanes stride over d, fixed order), no block-wide reduction per column
    // (2 q block sums with three barriers each were most of this kernel's 65 us at D = 256, q = 16)
    __shared__ double s_ww[PYVB_QMAX], s_lv[PYVB_QMAX];
    const int lane = tid & 31, warp = tid >> 5, nwarp = nt >> 5;
    if ((ops & PYVB_OP_ALPHA) && c.ard && crank == 0) {
        for (int i = col_lo + warp; i < col_hi; i += nwarp) {
            double part = 0.0;
            for (int d = lane; d < D; d += 32) {
                const double w = Wbar[(size_t)d * q + i];
                part += fma(w, w, Wvar[(size_t)d * q + i]);
            }
            const double tot = warp_sum(part);
            if (lane == 0) {
                const double b = c.ard_b0 + 0.5 * tot;
                gl[PYVB_GL_ALQB + i] = b;
                gl[PYVB_GL_ALPHA + i] = c.al_qa / b;
            }
        }
        __threadfence_block();
        __syncthreads();
    }
    double resid2 = 0.0;
    if ((ops & (PYVB_OP_BETA | PYVB_OP_ELBO)) && !nd) {
        // (d, p) advance incrementally and (i, j) come from a table: a 64-bit division and a square root per element made
        //  this loop 0.5 ms at D = 1024, q = 32); the cluster's CTAs take contiguous slices of the D x P index range
        double dot = 0.0;
        {
            const long long tot = (long long)D * P;
            const long long per = (tot + csize - 1) / csize;
            const long long lo = per * crank, hi = (lo + per < tot) ? lo + per : tot;
            const long long i0 = lo + tid;
            int d = (int)(i0 / P), pp = (int)(i0 - (long long)d * P);
            const int dstep = nt / P, pstep = nt - (nt / P) * P;
            for (long long idx = i0; idx < hi; idx += nt) {
                const int ij = ijtab[pp], i = ij >> 8, j = ij & 255;
                double g = Wbar[(size_t)d * q + i] * Wbar[(size_t)d * q + j];
                if (WR) {
                    g += Wcov[idx];
                    if (i != j) g *= 2.0;
                } else if (i == j) g += Wvar[(size_t)d * q + i];
                else g *= 2.0;
                dot = fma(g, T1[idx], dot);
                d += dstep;
                pp += pstep;
                if (pp >= P) {
                    pp -= P;
                    ++d;
                }
            }
        }
        dot = block_sum(dot, sh);
        if (csize > 1) {
            if (tid == 0) gk_store_remote(cl_part + crank, 0, dot);
            gk_cluster_sync();
            if (crank != 0) return;
            dot = 0.0;
            for (int r = 0; r < csize; ++r) dot += cl_part[r];
        }
        double part = 0.0;
        for (int d = tid; d < D; d += nt) {
            double s1 = 0.0, s2 = 0.0;
            for (int i = 0; i < q; ++i) {
                const double w = Wbar[(size_t)d * q + i];
                s1 = fma(w, Ast[(size_t)d * q + i], s1);
                s2 = fma(w, Bst[(size_t)d * q + i], s2);
            }
            const double m = mu[d];
            part += -2.0 * (s1 + m * colx[d]) + 2.0 * m * s2 + cnt[d] * (m * m + muvar[d]);
        }
        part = block_sum(part, sh) + dot;
        resid2 = part + sc[PYVB_SC_SXX] + sc[PYVB_SC_SUMV];
        if (ops & PYVB_OP_BETA) {
            qb = c.b0 + 0.5 * resid2;
            tau = qa / qb;
        }
        if (tid == 0) {
            gl[PYVB_GL_RESID2] = resid2;
            if (ops & PYVB_OP_BETA) {
                gl[PYVB_GL_QB] = qb;
                gl[PYVB_GL_TAU] = tau;
            }
        }
    }
    if (ops & PYVB_OP_ELBO) {
        __syncthreads();
        // ---- W columns (gaussian.py:141-147; q_ln_det = .5/ln prod diag chol is a division)
        double eW = 0.0;
        for (int i = warp; i < q; i += nwarp) {
            double pw = 0.0, pl = 0.0;
            for (int d = lane; d < D; d += 32) {
                const double w = Wbar[(size_t)d * q + i], v = Wvar[(size_t)d * q + i];
                pw += fma(w, w, v);
                if (!WR) pl += log(v);
            }
            pw = warp_sum(pw);
            pl = warp_sum(pl);
            if (lane == 0) {
                s_ww[i] = pw;
                s_lv[i] = pl;
            }
        }
        __syncthreads();
        for (int i = 0; i < q; ++i) {
            const double ww = s_ww[i], lv = s_lv[i];
            const double qld = 0.5 / (-0.5 * lv);
            const double al = gl[PYVB_GL_ALPHA + i];
            const double lndet = c.ard ? D * (log(c.al_qa) - log(gl[PYVB_GL_ALQB + i])) : D * log(al);
            if (WR) eW += -0.5 * D * LN2PI + 0.5 * lndet - 0.5 * al * ww - (-0.5 * D * LN2PI - 0.5 * D);
            else eW += -0.5 * D * LN2PI + 0.5 * lndet - 0.5 * al * ww - (-0.5 * D * LN2PI - 0.5 * qld - 0.5 * D);
        }
        if (WR) {
            double pe = 0.0;
            for (int d = tid; d < D; d += nt) pe += 0.5 / Wld[d];
            eW += 0.5 * block_sum(pe, sh);
        }
        // ---- Mu
        double pm = 0.0, pl = 0.0;
        for (int d = tid; d < D; d += nt) {
            pm += fma(mu[d], mu[d], muvar[d]);
            pl += log(muvar[d]);
        }
        const double mm = block_sum(pm, sh);
        const double lvm = block_sum(pl, sh);
        const double qldm = 0.5 / (-0.5 * lvm);
        const double eMu = -0.5 * D * LN2PI + 0.5 * D * log(c.alpha_mu) - 0.5 * c.alpha_mu * mm -
                           (-0.5 * D * LN2PI - 0.5 * qldm - 0.5 * D);
        // ---- Z rows
        double pt = 0.0, pz = 0.0;
        for (int idx = tid; idx < q * q; idx += nt) {
            const int i = idx / q, j = idx % q;
            const int p = (i >= j) ? tri(i) + j : tri(j) + i;
            pt = fma(P0[idx], S[p], pt);
        }
        for (int i = tid; i < q; i += nt) pz = fma(zsum[i], h0[i], pz);
        const double trPS = block_sum(pt, sh);
        const double zh = block_sum(pz, sh);
        const double nrows = sc[PYVB_SC_NROWS];
        const double eZ = nrows * (-0.5 * q * LN2PI + 0.5 * c.lndet_P0 - 0.5 * c.m0P0m0 + 0.5 * q * LN2PI + 0.5 * q) -
                          0.5 * trPS + zh + 0.5 * sc[PYVB_SC_QLDZ];
        // ---- X rows (nodes_todo.py:144-147 uses ln<tau>)
        double eX, eB;
        if (nd) {
            // per-dimension terms of noise_diag_kernel, summed in a fixed order
            double px = 0.0, pb = 0.0, pr = 0.0;
            for (int d = tid; d < D; d += nt) {
                px += nd[(size_t)PYVB_ND_EX * D + d];
                pb += nd[(size_t)PYVB_ND_EB * D + d];
                pr += nd[(size_t)PYVB_ND_R * D + d];
            }
            eX = block_sum(px, sh);
            eB = block_sum(pb, sh);
            pr = block_sum(pr, sh);
            if (tid == 0) gl[PYVB_GL_RESID2] = pr;
        } else {
            const double nE = sc[PYVB_SC_NE];
            eX = -0.5 * nE * LN2PI + 0.5 * nE * (log(qa) - log(qb)) - 0.5 * tau * resid2;
            if (c.mode_a) {
                eX -= sc[PYVB_SC_NLAT] * (-0.5 * D * LN2PI - 0.5 * D) - 0.5 * sc[PYVB_SC_LATQLD];
                eX -= 0.5 * sc[PYVB_SC_PNMISS] * LN2PI - 0.5 * sc[PYVB_SC_PLNV] - 0.5 * sc[PYVB_SC_PNMISS];
            }
            // ---- Gammas (nodes_todo.py:149-157)
            const double El = c.psi_qa - log(qb);
            eB = (c.a0 - 1.0) * El - c.lgam_a0 + c.a0 * log(c.b0) - c.b0 * (qa / qb) -
                 ((qa - 1.0) * El - c.lgam_qa + qa * log(qb) - qa);
        }
        if (WT) eX += gl[PYVB_GL_LNS];
        double eA = 0.0;
        if (c.ard) {
            for (int i = 0; i < q; ++i) {
                const double b = gl[PYVB_GL_ALQB + i];
                const double E2 = c.psi_alqa - log(b);
                eA += (c.ard_a0 - 1.0) * E2 - c.lgam_ard_a0 + c.ard_a0 * log(c.ard_b0) - c.ard_b0 * (c.al_qa / b) -
                      ((c.al_qa - 1.0) * E2 - c.lgam_alqa + c.al_qa * log(b) - c.al_qa);
            }
        }
        if (tid == 0) {
            const double e = eW + eMu + eZ + eX + eB + eA;
            gl[PYVB_GL_ELBO] = e;
            gl[PYVB_GL_ELBO_W] = eW;
            gl[PYVB_GL_ELBO_MU] = eMu;
            gl[PYVB_GL_ELBO_Z] = eZ;
            gl[PYVB_GL_ELBO_X] = eX;
            gl[PYVB_GL_ELBO_BETA] = eB;
            gl[PYVB_GL_ELBO_ALPHA] = eA;
            if (elbo_out) *elbo_out = e;
        }
    }
}

cudaError_t launch_global(int D, int q, int ops, int col_lo, int col_hi, const double *stats, const double *Wbar, const double *Wvar,
                          double *mu, double *muvar, double *gl, const double *P0, const double *h0,
                          const pyvb_consts &c, double *elbo_out, const double *nd, cudaStream_t st, bool weighted,
                          const double *Wcov, const double *Wld) {
    // one cluster; its size follows the work of the D x P contraction (small problems, or no contraction: one CTA)
    const long long work = nd ? 0 : (long long)D * q * (q + 1) / 2;
    const int cl = work >= (1LL << 17) ? GK_CLUSTER : work >= (1LL << 15) ? 2 : 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)cl, 1, 1);
    cfg.blockDim = dim3(1024, 1, 1);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)cl;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    if (Wcov)
        return cudaLaunchKernelEx(&cfg, weighted ? global_kernel<true, true> : global_kernel<false, true>, D, q, ops, col_lo,
                                  col_hi, stats, Wbar, Wvar, mu, muvar, gl, P0, h0, c, elbo_out, nd, Wcov, Wld);
    return cudaLaunchKernelEx(&cfg, weighted ? global_kernel<true> : global_kernel<false>, D, q, ops, col_lo, col_hi, stats, Wbar,
                              Wvar, mu, muvar, gl, P0, h0, c, elbo_out, nd, (const double *)nullptr, (const double *)nullptr);
}

// =============================================================== mode A imputation, warp per row
__global__ void __launch_bounds__(256)
impute_kernel(long long N, int D, int q, const double *__restrict__ Xorig, long long ldx,
              const double *__restrict__ Wbar, const double *__restrict__ mu, const double *__restrict__ Zbar,
              long long ldz, const double *__restrict__ gl, double *__restrict__ Xhat, double *__restrict__ V,
              double *__restrict__ qldX) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    const double tau = gl[PYVB_GL_TAU];
    const double vmiss = 1.0 / tau;
    for (long long n = (long long)blockIdx.x * nwarp + warp; n < N; n += (long long)gridDim.x * nwarp) {
        const double *xo = Xorig + n * ldx;
        int nmiss = 0;
        for (int d = lane; d < D; d += 32) nmiss += (xo[d] != xo[d]) ? 1 : 0;
        nmiss = __reduce_add_sync(0xffffffffu, nmiss);
        if (nmiss == 0) continue;  // fully observed rows are never updated (gaussian.py:109-110)
        const double *z = Zbar + n * ldz;
        for (int d = lane; d < D; d += 32) {
            const double x = xo[d];
            const bool miss = (x != x);
            double m = mu[d];
            for (int i = 0; i < q; ++i) m = fma(Wbar[(size_t)d * q + i], z[i], m);
            Xhat[n * (long long)D + d] = miss ? m : x;
            V[n * (long long)D + d] = miss ? vmiss : 0.0;
        }
        if (lane == 0) qldX[n] = 0.5 / (0.5 * D * log(tau));
    }
}

cudaError_t launch_impute(long long N, int D, int q, const double *Xorig, long long ldx, const double *Wbar,
                          const double *mu, const double *Zbar, long long ldz, const double *gl, double *Xhat,
                          double *V, double *qldX, cudaStream_t st) {
    if (N <= 0) return cudaSuccess;
    long long b = (N + 7) / 8;
    if (b > 148 * 8) b = 148 * 8;
    impute_kernel<<<(unsigned)b, 256, 0, st>>>(N, D, q, Xorig, ldx, Wbar, mu, Zbar, ldz, gl, Xhat, V, qldX);
    return cudaGetLastError();
}

}  // namespace pyvb
