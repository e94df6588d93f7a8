// Warp-cooperative 8 x 8 Cholesky + triangular inverse in the DMMA accumulator layout (shared by the blocked batched
// solve, kernels_k2.cu, and the LDS smoother, kernels_lds.cu).
#pragma once

namespace pyvb {

// 8 x 8 diagonal blocks of MPW independent matrices, accumulator layout (lane l: row l/4, columns 2(l%4), 2(l%4)+1).
// In: the SPD blocks A (lower triangle valid).  Out: X = chol(A)^-1 (lower triangular, exact zeros above the
// diagonal); lprod[m] is multiplied by prod_k 1/l_kk.  Right-looking factorisation and right-looking inversion fused
// in one sweep: per pivot one broadcast, one rsqrt, and independent multiply-adds; the MPW pivot chains interleave.
template <int MPW>
__device__ __forceinline__ void diag_chol_inv(double (&c0)[MPW], double (&c1)[MPW], double (&x0)[MPW], double (&x1)[MPW],
                                              double (&lprod)[MPW]) {
    const int lane = threadIdx.x & 31;
    const int gid = lane >> 2, qd = lane & 3;
#pragma unroll
    for (int m = 0; m < MPW; ++m) {
        x0[m] = (gid == 2 * qd) ? 1.0 : 0.0;
        x1[m] = (gid == 2 * qd + 1) ? 1.0 : 0.0;
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int kq = k >> 1;
        double rinv[MPW], lik[MPW];
#pragma unroll
        for (int m = 0; m < MPW; ++m) {
            const double ck = (k & 1) ? c1[m] : c0[m];
            const double d = __shfl_sync(0xffffffffu, ck, k * 4 + kq);                    // pivot a_kk
            rinv[m] = rsqrt(d);
            lprod[m] *= rinv[m];
            lik[m] = __shfl_sync(0xffffffffu, ck, (lane & ~3) | kq) * rinv[m];            // l_(gid, k)   (gid >= k)
            const double lj0 = __shfl_sync(0xffffffffu, ck, (2 * qd) * 4 + kq) * rinv[m];  // l_(2qd, k)
            const double lj1 = __shfl_sync(0xffffffffu, ck, (2 * qd + 1) * 4 + kq) * rinv[m];
            if (2 * qd > k) c0[m] = fma(-lik[m], lj0, c0[m]);
            if (2 * qd + 1 > k) c1[m] = fma(-lik[m], lj1, c1[m]);
        }
        // row k of X is final once scaled by 1/l_kk; eliminate it from the rows below
#pragma unroll
        for (int m = 0; m < MPW; ++m) {
            if (gid == k) {
                x0[m] *= rinv[m];
                x1[m] *= rinv[m];
            }
            const double xk0 = __shfl_sync(0xffffffffu, x0[m], k * 4 + qd);
            const double xk1 = __shfl_sync(0xffffffffu, x1[m], k * 4 + qd);
            if (gid > k) {
                x0[m] = fma(-lik[m], xk0, x0[m]);
                x1[m] = fma(-lik[m], xk1, x1[m]);
            }
        }
    }
#pragma unroll
    for (int m = 0; m < MPW; ++m) {
        if (gid < 2 * qd) x0[m] = 0.0;
        if (gid < 2 * qd + 1) x1[m] = 0.0;
    }
}

}  // namespace pyvb
