// Per-dimension noise precisions (factor analysis): the second stage of a mode-B sweep when every data dimension d has its own
// Gamma posterior Gamma(qa_d, qb_d) (DiagonalGamma, nodes/nodes_todo.py:159-204) instead of one shared tau.
//
// The Z step and the W update need no kernel of their own: pack_gw folds tau_d into the Gw rows and wupdate reads tau_d from
// the nd block.  What is left is per data dimension and runs here, one warp per d:
//   Mu     prec_d = alpha_mu + tau_d cnt_d,  mu_d = tau_d (colx_d - wbar_d . Bst_d) / prec_d            (old tau_d)
//   r_d    sum_n O_nd <(x_nd - w_d z_n - mu_d)^2> = sxx_d - 2 (wbar_d . Ast_d + mu_d colx_d) + 2 mu_d (wbar_d . Bst_d)
//          + cnt_d (mu_d^2 + muvar_d) + sum_p g_dp T1[d][p]        (the per-d slice of global_kernel's D x P contraction)
//   Gamma  qb_d = b0_d + r_d / 2, tau_d = qa_d / qb_d                                          (DiagonalGamma.update)
//   bound  eX_d = -cnt_d/2 ln 2pi + cnt_d/2 (ln qa_d - ln qb_d) - tau_d r_d / 2   (ln<tau> as the scalar path)
// WT (per-entry observation weights): the statistics' cnt_d is the weight sum sum_n s_nd, which Mu and r_d read; the bound reads
// the NUMBER of observed entries of column d from ncnt[d] instead.
//          eB_d = the Gamma bound of entry d                                       (DiagonalGamma.log_lower_bound)
// global_kernel then adds eX_d and eB_d over d in a fixed order.  No atomics: replicas on several GPUs stay bit-identical.
#include "common.cuh"
#include "kernels.h"

namespace pyvb {

constexpr int ND_WARPS = 8;

template <bool WT>
__global__ void __launch_bounds__(32 * ND_WARPS)
noise_diag_kernel(int D, int q, int ops, const double *__restrict__ stats, const double *__restrict__ Wbar,
                  const double *__restrict__ Wvar, double *__restrict__ mu, double *__restrict__ muvar, double *__restrict__ nd,
                  double alpha_mu, const double *__restrict__ ncnt) {
    __shared__ unsigned short ijtab[PYVB_QMAX * (PYVB_QMAX + 1) / 2];   // packed index -> (i << 8) | j
    const StatLayout L(D, q);
    const int P = L.P;
    for (int p = threadIdx.x; p < P; p += blockDim.x) {
        int i, j;
        unpack_p(p, i, j);
        ijtab[p] = (unsigned short)((i << 8) | j);
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int d = blockIdx.x * ND_WARPS + (threadIdx.x >> 5);
    if (d >= D) return;
    const double LN2PI = 1.8378770664093454835606594728112;
    const double *w = Wbar + (size_t)d * q, *v = Wvar + (size_t)d * q;
    const double *T1 = stats + L.t1 + (size_t)d * P;
    const double *Bst = stats + L.bst + (size_t)d * q, *Ast = stats + L.ast + (size_t)d * q;
    const double cnt = stats[L.cnt + d], colx = stats[L.colx + d];
    double *tau = nd + (size_t)PYVB_ND_TAU * D, *qb = nd + (size_t)PYVB_ND_QB * D;
    double s1 = 0.0, s2 = 0.0;                          // wbar_d . Ast_d, wbar_d . Bst_d
    for (int i = lane; i < q; i += 32) {
        s1 = fma(w[i], Ast[i], s1);
        s2 = fma(w[i], Bst[i], s2);
    }
    s1 = warp_sum(s1);
    s2 = warp_sum(s2);
    double m = mu[d], mv = muvar[d];
    if (ops & PYVB_OP_MU) {
        const double prec = alpha_mu + tau[d] * cnt;
        m = tau[d] * (colx - s2) / prec;
        mv = 1.0 / prec;
        if (lane == 0) {
            mu[d] = m;
            muvar[d] = mv;
        }
    }
    if (!(ops & (PYVB_OP_BETA | PYVB_OP_ELBO))) return;
    double dot = 0.0;
    for (int p = lane; p < P; p += 32) {
        const int ij = ijtab[p], i = ij >> 8, j = ij & 255;
        double g = w[i] * w[j];
        if (i == j) g += v[i];
        else g *= 2.0;
        dot = fma(g, T1[p], dot);
    }
    dot = warp_sum(dot);
    if (lane != 0) return;
    const double r = nd[(size_t)PYVB_ND_SXX * D + d] - 2.0 * (s1 + m * colx) + 2.0 * m * s2 + cnt * (m * m + mv) + dot;
    const double qa = nd[(size_t)PYVB_ND_QA * D + d];
    double b = qb[d], t = tau[d];
    if (ops & PYVB_OP_BETA) {
        b = nd[(size_t)PYVB_ND_B0 * D + d] + 0.5 * r;
        t = qa / b;
        qb[d] = b;
        tau[d] = t;
    }
    const double a0 = nd[(size_t)PYVB_ND_A0 * D + d], b0 = nd[(size_t)PYVB_ND_B0 * D + d];
    const double El = nd[(size_t)PYVB_ND_PSI_QA * D + d] - log(b);
    nd[(size_t)PYVB_ND_R * D + d] = r;
    const double nobs = WT ? ncnt[d] : cnt;
    nd[(size_t)PYVB_ND_EX * D + d] = -0.5 * nobs * LN2PI + 0.5 * nobs * (log(qa) - log(b)) - 0.5 * t * r;
    nd[(size_t)PYVB_ND_EB * D + d] = (a0 - 1.0) * El - nd[(size_t)PYVB_ND_LGAM_A0 * D + d] + a0 * log(b0) - b0 * t -
                                     ((qa - 1.0) * El - nd[(size_t)PYVB_ND_LGAM_QA * D + d] + qa * log(b) - qa);
}

cudaError_t launch_noise_diag(int D, int q, int ops, const double *stats, const double *Wbar, const double *Wvar, double *mu,
                              double *muvar, double *nd, double alpha_mu, cudaStream_t st, const double *ncnt) {
    if (!(ops & (PYVB_OP_MU | PYVB_OP_BETA | PYVB_OP_ELBO))) return cudaSuccess;
    const unsigned blocks = (D + ND_WARPS - 1) / ND_WARPS;
    if (ncnt)
        noise_diag_kernel<true><<<blocks, 32 * ND_WARPS, 0, st>>>(D, q, ops, stats, Wbar, Wvar, mu, muvar, nd, alpha_mu, ncnt);
    else
        noise_diag_kernel<false><<<blocks, 32 * ND_WARPS, 0, st>>>(D, q, ops, stats, Wbar, Wvar, mu, muvar, nd, alpha_mu, nullptr);
    return cudaGetLastError();
}

}  // namespace pyvb
