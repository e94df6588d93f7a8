// Known trailing latent dimensions (row covariates, DESIGN.md 5f): the Z step of a plate whose latent row is
// z'_n = [z_n ; c_n], the last k of its qt dimensions known per row.  K1 runs at qt as usual and leaves the MZ row
// [qprec' packed | pad | eta' | ...]; the known dimensions are the last ones, so their rows of the packed triangle are the
// contiguous tail [tri(qf), tri(qt)) (qf = qt - k).  Two passes touch only that tail, eta' / zbar' and c_n:
//
//   condition (between K1 and K2):  eta_z -= qprec_zc c,  qprec_zc = 0,  qprec_cc = I,  eta_c = c
//       K2 then solves the block-diagonal system blockdiag(A_n, I): its free block is the Gaussian conditioned on c_n, the
//       identity pivots add ln 1 = 0 to the log-det, and its zbar tail is c.
//   finish (after K2):  <z'z'^T>_cc = c c^T (computed directly, not as (1 + c_i c_j) - 1), zbar_c = c (so the tail holds c's
//       bits whatever sign of zero K2's block-diagonal sums left)
//
// One group of G lanes per row (G the smallest power of two covering the row's work, so a warp takes 32 / G rows); no
// atomics, fixed order: deterministic.  The partials K2 leaves (column sums and maxima) are wrong on the
// cc entries, so the callers pass none and the statistics rebuild them from the finished rows.
#include "common.cuh"
#include "kernels.h"

namespace pyvb {

namespace {

constexpr int KN_THREADS = 256;
constexpr int KN_WARPS = KN_THREADS / 32;

// lanes per row: the smallest power of two >= the row's work items (at most 32); a warp takes 32 / G rows
int lanes_per_row(int items) {
    int g = 1;
    while (g < items && g < 32) g <<= 1;
    return g;
}

// the packed row r >= r0 holding entry p (p >= tri(r0))
__device__ inline int tail_row(int p, int r0) {
    int r = r0;
    while (tri(r + 1) <= p) ++r;
    return r;
}

__global__ void __launch_bounds__(KN_THREADS) known_condition_kernel(long long N, int qt, int k, const double *__restrict__ C,
                                                                     long long ldc, double *__restrict__ MZ, long long ldmz,
                                                                     int G, const double *cond) {
    if (cond != nullptr && !(*cond > 0.0)) return;
    const int lane = threadIdx.x & 31, lig = lane & (G - 1), R = 32 / G;
    const int qf = qt - k, woff = gw_woff(qt), p0 = tri(qf), pt = tri(qt);
    const long long step = (long long)gridDim.x * KN_WARPS * R;
    for (long long base = ((long long)blockIdx.x * KN_WARPS + (threadIdx.x >> 5)) * R; base < N; base += step) {
        const long long n = base + lane / G;
        const bool ok = n < N;
        double *r = MZ + n * ldmz;
        const double *c = C + n * ldc;
        // e_i = eta_i - sum_j qprec[qf + j][i] c_j, j in order; eta_z is written here, the tail only after every lane of the row
        // has read its zc entries
        if (ok) {
            for (int i = lig; i < qf; i += G) {
                double e = r[woff + i];
                for (int j = 0; j < k; ++j) e = fma(-r[tri(qf + j) + i], c[j], e);
                r[woff + i] = e;
            }
        }
        __syncwarp();
        if (ok) {
            for (int p = p0 + lig; p < pt; p += G) {           // the contiguous tail: zc = 0, cc = I
                const int row = tail_row(p, qf);
                r[p] = (p - tri(row) == row) ? 1.0 : 0.0;
            }
            for (int j = lig; j < k; j += G) r[woff + qf + j] = c[j];
        }
    }
}

__global__ void __launch_bounds__(KN_THREADS) known_finish_kernel(long long N, int qt, int k, const double *__restrict__ C,
                                                                  long long ldc, double *__restrict__ MZ, long long ldmz, int G) {
    const int lane = threadIdx.x & 31, lig = lane & (G - 1), R = 32 / G;
    const int qf = qt - k, woff = gw_woff(qt), T0 = tri(k);
    const long long step = (long long)gridDim.x * KN_WARPS * R;
    for (long long base = ((long long)blockIdx.x * KN_WARPS + (threadIdx.x >> 5)) * R; base < N; base += step) {
        const long long n = base + lane / G;
        if (n >= N) continue;
        double *r = MZ + n * ldmz;
        const double *c = C + n * ldc;
        for (int t = lig; t < T0 + k; t += G) {
            if (t < T0) {                                      // <c_j c_i>, i <= j: row qf + j, column qf + i
                const int j = tail_row(t, 0), i = t - tri(j);
                r[tri(qf + j) + qf + i] = c[j] * c[i];
            } else {
                r[woff + qf + (t - T0)] = c[t - T0];
            }
        }
    }
}

__global__ void known_guard_scale_kernel(int qt, int k, const double *__restrict__ gscale, double cmax, double *out) {
    __shared__ double sh[32];
    const int qf = qt - k;
    const double cf = cmax > 1.0 ? cmax : 1.0;
    double m = 0.0;
    for (int p = threadIdx.x; p < tri(qt); p += blockDim.x) {
        const int row = tail_row(p, 0), col = p - tri(row);
        if (row < qf) m = fmax(m, gscale[p]);
        else if (col < qf) m = fmax(m, cf * gscale[p]);
    }
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = fmax(m, sh[w]);
        *out = fmax(m, sh[0]);
    }
}

unsigned known_blocks(long long N, int G) {
    const long long rows = (long long)KN_WARPS * (32 / G);
    const long long b = (N + rows - 1) / rows;
    return (unsigned)(b < 0x7fffffffLL ? b : 0x7fffffffLL);
}

}  // namespace

cudaError_t launch_known_condition(long long N, int qt, int k, const double *C, long long ldc, double *MZ, long long ldmz,
                                   cudaStream_t st, const double *cond) {
    if (N <= 0) return cudaSuccess;
    const int G = lanes_per_row(qt - k > k ? qt - k : k);
    known_condition_kernel<<<known_blocks(N, G), KN_THREADS, 0, st>>>(N, qt, k, C, ldc, MZ, ldmz, G, cond);
    return cudaGetLastError();
}

cudaError_t launch_known_finish(long long N, int qt, int k, const double *C, long long ldc, double *MZ, long long ldmz,
                                cudaStream_t st) {
    if (N <= 0) return cudaSuccess;
    const int G = lanes_per_row(k * (k + 1) / 2 + k);
    known_finish_kernel<<<known_blocks(N, G), KN_THREADS, 0, st>>>(N, qt, k, C, ldc, MZ, ldmz, G);
    return cudaGetLastError();
}

cudaError_t launch_known_guard_scale(int qt, int k, const double *gscale, double cmax, double *out, cudaStream_t st) {
    known_guard_scale_kernel<<<1, 256, 0, st>>>(qt, k, gscale, cmax, out);
    return cudaGetLastError();
}

}  // namespace pyvb
