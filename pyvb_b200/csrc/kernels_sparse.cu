// Sparse observations (CSR input): the gather kernels of the Z step (K1-csr) and of the statistics (K3-csc).
//
// Both contractions are "a 0/1 pattern with stored values, times a dense matrix whose rows have the MZ / Gw pitch":
//   K1-csr (row-owned):    qprec_n = P0 + tau sum_{d in O_n} G_d,   eta_n = h0 + tau sum_{d in O_n} (x_nd - mu_d) wbar_d
//                          -- the rows d of Gw = [G_d packed | pad | wbar_d | mu_d] are gathered per stored entry of row n
//   K3-csc (column-owned): T1_d = sum_{n in O^d} <zz^T>_n,  Bst_d = sum zbar_n,  Ast_d = sum x_nd zbar_n
//                          -- the rows n of MZ = [<zz^T>_n packed | pad | zbar_n] are gathered per stored entry of column d
// so one device routine (gather_rows) serves both.  A group of G threads owns one output row; thread t of the group owns
// the column pairs t, t + G, t + 2G, ... of the gathered rows and loads them as 128-bit words, U entries' rows in flight
// at once.  Every sum runs over the stored entries in their stored order, in one thread, with no atomics: the result is
// bit-identical from run to run, and a Z step over a row range equals the same rows of a full-range step.
//
// K3 takes the entries in a row-blocked column-major layout (pyvb_b200/sparse.py): rows are cut into blocks whose MZ slice
// fits a share of the L2, and the work items (block, column) are dealt block-major, so the MZ rows of a block are gathered
// from the L2 while the block is being worked on.  Item (b, d) writes the T1 | Bst | Ast slice of column d into block b's
// partial ws_main[b][statlen]; the shared second stage (stats_reduce) adds the partials in block order.
#include "common.cuh"
#include "kernels.h"

namespace pyvb {

constexpr int SP_THREADS = 256;

template <int Q> struct SpT {
    static constexpr int P = Q * (Q + 1) / 2;
    static constexpr int PP = (P + 7) & ~7;              // first wbar / zbar column (gw_woff)
    static constexpr int NPAIR = (PP + Q) / 2;           // column pairs gathered per row: [packed | pad | wbar or zbar]
    static constexpr int G = (Q == 64) ? 128 : 32;       // threads per output row
    static constexpr int NT = (NPAIR + G - 1) / G;       // pairs per thread
    static constexpr int TX = (PP / 2) / G;              // first of a thread's pairs that can be a wbar / zbar pair
    static constexpr int NX = NT - TX;
    static constexpr int U = (Q == 8) ? 8 : (Q == 16) ? 4 : 2;   // entries whose rows are loaded before they are added
    static constexpr int MINB = (Q <= 16) ? 2 : 1;               // CTAs per SM (q >= 32: 138 registers, no spills)
    static_assert(P % 2 == 0 && PP % 2 == 0 && Q % 2 == 0, "pairs never straddle the packed / pad / vector boundaries");
};

// acc  += the packed columns of the gathered rows, and on the vector columns:
//   K3 = false (Z step):      acc  += (x - row[PP + Q]) * row      (row[PP + Q] is mu_d in a Gw row)
//   K3 = true  (statistics):  acc  += row,  accx += x * row
template <int Q, bool K3, typename IDX>
__device__ __forceinline__ void gather_rows(const double *__restrict__ src, long long ld, const IDX *__restrict__ idx,
                                            const double *__restrict__ val, long long e0, long long e1, int t0,
                                            double2 (&acc)[SpT<Q>::NT], double2 (&accx)[SpT<Q>::NX]) {
    using T = SpT<Q>;
    for (long long e = e0; e < e1; e += T::U) {
        long long r[T::U];
        double x[T::U], m[T::U];
        double2 v[T::U][T::NT];
#pragma unroll
        for (int u = 0; u < T::U; ++u) {
            const bool ok = e + u < e1;
            r[u] = ok ? (long long)__ldg(idx + e + u) : -1;
            x[u] = ok ? __ldg(val + e + u) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < T::U; ++u) {
            if (r[u] < 0) continue;
            const double *row = src + r[u] * ld;
            if (!K3) m[u] = __ldg(row + T::PP + Q);
#pragma unroll
            for (int t = 0; t < T::NT; ++t) {
                const int k = t0 + t * T::G;
                if (k < T::NPAIR && !(2 * k >= T::P && 2 * k < T::PP))
                    v[u][t] = __ldg(reinterpret_cast<const double2 *>(row) + k);
            }
        }
#pragma unroll
        for (int u = 0; u < T::U; ++u) {
            if (r[u] < 0) continue;
            const double xm = K3 ? x[u] : x[u] - m[u];
#pragma unroll
            for (int t = 0; t < T::NT; ++t) {
                const int k = t0 + t * T::G;
                if (k >= T::NPAIR) continue;
                if (2 * k < T::P) {
                    acc[t].x += v[u][t].x;
                    acc[t].y += v[u][t].y;
                } else if (2 * k >= T::PP) {
                    if (K3) {
                        acc[t].x += v[u][t].x;
                        acc[t].y += v[u][t].y;
                        if (t >= T::TX) {
                            accx[t - T::TX].x = fma(xm, v[u][t].x, accx[t - T::TX].x);
                            accx[t - T::TX].y = fma(xm, v[u][t].y, accx[t - T::TX].y);
                        }
                    } else {
                        acc[t].x = fma(xm, v[u][t].x, acc[t].x);
                        acc[t].y = fma(xm, v[u][t].y, acc[t].y);
                    }
                }
            }
        }
    }
}

// ------------------------------------------------------------------ K1-csr: one group per row
// indptr: the rows' own offsets into indices / values (indptr[0] need not be 0: a row range is a pointer offset)
template <int Q>
__global__ void __launch_bounds__(SP_THREADS, SpT<Q>::MINB)
zstep_csr_kernel(long long N, const long long *__restrict__ indptr, const int *__restrict__ indices,
                 const double *__restrict__ values, const double *__restrict__ Gw, int ldg, const double *__restrict__ P0,
                 const double *__restrict__ h0, const double *__restrict__ gl, double *__restrict__ MZ, int ldmz) {
    using T = SpT<Q>;
    __shared__ double prior[T::PP + Q];                  // [P0 packed | 0 | h0]: the row of an empty observation set
    for (int c = threadIdx.x; c < T::PP + Q; c += blockDim.x) {
        double v = 0.0;
        if (c < T::P) {
            int i, j;
            unpack_p(c, i, j);
            v = P0[i * Q + j];
        } else if (c >= T::PP) {
            v = h0[c - T::PP];
        }
        prior[c] = v;
    }
    __syncthreads();
    const long long n = (long long)blockIdx.x * (SP_THREADS / T::G) + threadIdx.x / T::G;
    if (n >= N) return;
    const int t0 = threadIdx.x % T::G;
    const double tau = gl[PYVB_GL_TAU];
    double2 acc[T::NT], accx[T::NX];
#pragma unroll
    for (int t = 0; t < T::NT; ++t) acc[t] = make_double2(0.0, 0.0);
    gather_rows<Q, false>(Gw, ldg, indices, values, indptr[n], indptr[n + 1], t0, acc, accx);
    double2 *out = reinterpret_cast<double2 *>(MZ + n * ldmz);
#pragma unroll
    for (int t = 0; t < T::NT; ++t) {
        const int k = t0 + t * T::G;
        if (k < T::NPAIR)      // the pad columns [P, PP) come out as exact zeros, as on the dense paths
            out[k] = make_double2(fma(tau, acc[t].x, prior[2 * k]), fma(tau, acc[t].y, prior[2 * k + 1]));
    }
}

// ------------------------------------------------------------------ K3-csc: one group per (row block, column)
// colptr [nblk * D + 1]: entries of item b * D + d are [colptr[b * D + d], colptr[b * D + d + 1]) of rows / vals, the rows
// in increasing order; rows are row indices of the shard (MZ row r at MZ + r * ldmz)
template <int Q>
__global__ void __launch_bounds__(SP_THREADS, SpT<Q>::MINB)
stats_csc_kernel(long long nitems, int D, const long long *__restrict__ colptr, const int *__restrict__ rows,
                 const double *__restrict__ vals, const double *__restrict__ MZ, int ldmz, double *__restrict__ ws,
                 size_t statlen) {
    using T = SpT<Q>;
    const long long item = (long long)blockIdx.x * (SP_THREADS / T::G) + threadIdx.x / T::G;
    if (item >= nitems) return;
    const int t0 = threadIdx.x % T::G;
    const long long b = item / D;
    const int d = (int)(item - b * D);
    double2 acc[T::NT], accx[T::NX];
#pragma unroll
    for (int t = 0; t < T::NT; ++t) acc[t] = make_double2(0.0, 0.0);
#pragma unroll
    for (int t = 0; t < T::NX; ++t) accx[t] = make_double2(0.0, 0.0);
    gather_rows<Q, true>(MZ, ldmz, rows, vals, colptr[item], colptr[item + 1], t0, acc, accx);
    const StatLayout L(D, Q);
    double *out = ws + (size_t)b * statlen;
#pragma unroll
    for (int t = 0; t < T::NT; ++t) {
        const int k = t0 + t * T::G, c = 2 * k;
        if (k >= T::NPAIR) continue;
        if (c < T::P) {
            out[L.t1 + (size_t)d * T::P + c] = acc[t].x;
            out[L.t1 + (size_t)d * T::P + c + 1] = acc[t].y;
        } else if (c >= T::PP) {
            const size_t i = (size_t)d * Q + (c - T::PP);
            out[L.bst + i] = acc[t].x;
            out[L.bst + i + 1] = acc[t].y;
            if (t >= T::TX) {
                out[L.ast + i] = accx[t - T::TX].x;
                out[L.ast + i + 1] = accx[t - T::TX].y;
            }
        }
    }
}

// ------------------------------------------------------------------ sizes and launches
bool csr_supported(int q) { return q == 8 || q == 16 || q == 32 || q == 64; }

// Row blocks of K3-csc: as many as it takes for one block's MZ slice to fit 32 MB (a quarter of the L2, so the gathered rows
// stay resident while the entries stream past), but at most 64 and no more than 1 GiB of partials (D * (P + 2q) * 8 bytes
// each): wide or q = 64 shapes get larger blocks and gather part of their rows from HBM.
int csr_stats_nblocks(long long N, int D, int q) {
    if (N <= 0) return 1;
    int pitch = gw_woff(q) + q + 1;                       // pyvb_mz_pitch(q)
    while (pitch % 8 != 4) ++pitch;
    const long long row_bytes = (long long)pitch * 8;
    long long nb = (N * row_bytes + (32LL << 20) - 1) / (32LL << 20);
    const long long by_ws = (1LL << 30) / ((long long)StatLayout(D, q).len * 8);
    if (nb > by_ws) nb = by_ws;
    if (nb > 64) nb = 64;
    if (nb > N) nb = N;
    if (nb < 1) nb = 1;
    const long long rows = (N + nb - 1) / nb;              // every block but the last holds `rows` rows
    return (int)((N + rows - 1) / rows);
}

long long csr_block_rows(long long N, int D, int q) {
    if (N <= 0) return 1;
    const int nb = csr_stats_nblocks(N, D, q);
    return (N + nb - 1) / nb;
}

template <int Q>
static cudaError_t launch_zstep_csr_q(long long N, const long long *indptr, const int *indices, const double *values,
                                      const double *Gw, int ldg, const double *P0, const double *h0, const double *gl,
                                      double *MZ, int ldmz, cudaStream_t st) {
    constexpr int GPB = SP_THREADS / SpT<Q>::G;
    const long long blocks = (N + GPB - 1) / GPB;
    zstep_csr_kernel<Q><<<(unsigned)blocks, SP_THREADS, 0, st>>>(N, indptr, indices, values, Gw, ldg, P0, h0, gl, MZ, ldmz);
    return cudaGetLastError();
}

cudaError_t launch_zstep_csr(long long N, int q, const long long *indptr, const int *indices, const double *values,
                             const double *Gw, int ldg, const double *P0, const double *h0, const double *gl, double *MZ,
                             int ldmz, cudaStream_t st) {
    if (N <= 0) return cudaSuccess;
    switch (q) {
        case 8: return launch_zstep_csr_q<8>(N, indptr, indices, values, Gw, ldg, P0, h0, gl, MZ, ldmz, st);
        case 16: return launch_zstep_csr_q<16>(N, indptr, indices, values, Gw, ldg, P0, h0, gl, MZ, ldmz, st);
        case 32: return launch_zstep_csr_q<32>(N, indptr, indices, values, Gw, ldg, P0, h0, gl, MZ, ldmz, st);
        case 64: return launch_zstep_csr_q<64>(N, indptr, indices, values, Gw, ldg, P0, h0, gl, MZ, ldmz, st);
    }
    return cudaErrorNotSupported;
}

template <int Q>
static cudaError_t launch_stats_csc_q(int D, int nblk, const long long *colptr, const int *rows, const double *vals,
                                      const double *MZ, int ldmz, double *ws_main, cudaStream_t st) {
    constexpr int GPB = SP_THREADS / SpT<Q>::G;
    const long long nitems = (long long)nblk * D;
    const long long blocks = (nitems + GPB - 1) / GPB;
    stats_csc_kernel<Q><<<(unsigned)blocks, SP_THREADS, 0, st>>>(nitems, D, colptr, rows, vals, MZ, ldmz, ws_main,
                                                                  StatLayout(D, Q).len);
    return cudaGetLastError();
}

cudaError_t launch_stats_csc(int D, int q, int nblk, const long long *colptr, const int *rows, const double *vals,
                             const double *MZ, int ldmz, double *ws_main, cudaStream_t st) {
    if (nblk <= 0) return cudaSuccess;
    switch (q) {
        case 8: return launch_stats_csc_q<8>(D, nblk, colptr, rows, vals, MZ, ldmz, ws_main, st);
        case 16: return launch_stats_csc_q<16>(D, nblk, colptr, rows, vals, MZ, ldmz, ws_main, st);
        case 32: return launch_stats_csc_q<32>(D, nblk, colptr, rows, vals, MZ, ldmz, ws_main, st);
        case 64: return launch_stats_csc_q<64>(D, nblk, colptr, rows, vals, MZ, ldmz, ws_main, st);
    }
    return cudaErrorNotSupported;
}

}  // namespace pyvb
