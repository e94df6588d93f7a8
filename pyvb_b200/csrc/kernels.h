// Internal launch interface between the C-ABI (cabi.cu) and the kernel files.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include "../../include/pyvb_b200.h"

namespace pyvb {

// Accuracy guard of the INT8 mask contraction (K1-i8): the qprec entries of a row carry at most tau * n_obs * scale_c * 2^-55
// of fixed-point rounding (scale_c = the power of two above the column maximum of G).  K2 reads the finished qprec row anyway:
// with gscale != NULL it flags every row whose bound  tau * fac * max_c scale_c  (fac = D * 2^-55 / tol) exceeds the largest
// diagonal entry of the row, i.e. whose qprec is not accurate to `tol` in the max norm, into gl[PYVB_GL_I8BAD].
struct I8Check {
    const double *gscale = nullptr;    // [ncols] fixed-point scales of the G columns (NULL: no check)
    int ncols = 0;
    double fac = 0.0;
};

// ---- generic (any D, q <= 64) ------------------------------------------------
// tau_d (nullable): per-dimension noise precisions folded into the row (pyvb_pack_gw_nd_f64)
// Wcov (nullable): row-wise W posterior, packed Sigma_d [D][P] in place of diag(Wvar) (Wvar is then not read)
cudaError_t launch_pack_gw(int D, int q, const double *Wbar, const double *Wvar, const double *mu, const double *tau_d,
                           double *Gw, int ldg, cudaStream_t st, const double *Wcov = nullptr);
// S (nullable, here and below): per-entry observation weights [N][lds] of a mode-B data set (the weight of an entry whose x is
// NaN is not read); every observed entry then counts with its weight, the statistics' cnt is the weight sum and nE the number
// of observed entries of positive weight
cudaError_t launch_zstep_generic(long long N, int D, int q, const double *X, long long ldx, const double *Gw,
                                 int ldg, const double *P0, const double *h0, double *gl, double *Zbar,
                                 long long ldz, double *M2, long long ldm, double *Sig, double *logdet,
                                 cudaStream_t st, const double *S = nullptr, long long lds = 0,
                                 const double *Cv = nullptr, long long ldc = 0, int kn = 0);
// (Cv, ldc, kn: the last kn dimensions known per row, c_n = Cv[n][0, kn), conditioned on inside the kernel: DESIGN.md 5f)
// main statistics: partial sums for `nchunks` row chunks into ws_main[nchunks][statlen]
int stats_generic_nchunks(long long N);
cudaError_t launch_stats_generic(long long N, int D, int q, const double *X, long long ldx, const double *Zbar,
                                 long long ldz, const double *M2, long long ldm, double *ws_main, int nchunks,
                                 cudaStream_t st, const double *S = nullptr, long long lds = 0);
cudaError_t launch_colsums(long long N, int D, int q, const double *X, long long ldx, double *ws_main, int nchunks,
                           cudaStream_t st, const double *S = nullptr, long long lds = 0);
// per-row scalars: partial sums into ws_sc[nblk][PYVB_NSCAL]
int rowscalars_nblk(long long N);
cudaError_t launch_rowscalars(long long N, int D, const double *X, long long ldx, const double *V,
                              const double *Xorig, const double *qldX, const double *logdet, double *ws_sc,
                              int nblk, int skip_x, cudaStream_t st, const double *S = nullptr, long long lds = 0);
// column sums of the [M2 | zbar] rows -> S, zsum partials (DMMA path)
cudaError_t launch_mzsums(long long N, int D, int q, const double *Zbar, long long ldz, const double *M2,
                          long long ldm, double *ws_main, int nchunks, cudaStream_t st);
cudaError_t launch_stats_reduce(int D, int q, const double *ws_main, int nchunks, const double *ws_sc, int nblk,
                                double *stats, double *xcache, int use_xcache, const double *zsums, int nzblk,
                                int zkw, void *const *peer_bufs, int world, int rank, unsigned long long epoch,
                                cudaStream_t st);
size_t peer_buffer_bytes(size_t len);
cudaError_t launch_wupdate(int D, int q, int col_lo, int col_hi, const double *stats, const double *mu,
                           const double *gl, const double *tau_d, double *Wbar, double *Wvar, cudaStream_t st);
// row-wise W posterior: Lambda_d, eta_d into the K2 rows WM [D][ldwm], launch_zsolve, then wbar_d, diag Sigma_d into Wbar, Wvar.
// Wcov [D][P] receives Sigma_d, Wld [D] ln prod diag chol(Lambda_d); non-PD rows are counted into gl[PYVB_GL_NONPD]
cudaError_t launch_wupdate_rows(int D, int q, const double *stats, const double *mu, double *gl, const double *tau_d,
                                double *WM, int ldwm, double *Wbar, double *Wvar, double *Wcov, double *Wld, cudaStream_t st);
// nd (nullable): per-dimension noise mode -- Mu and the Gammas are left to launch_noise_diag, which must run first
// weighted: the X bound term also carries gl[PYVB_GL_LNS]
// Wcov, Wld (nullable, both or neither): row-wise W posterior -- the contraction reads Sigma_d, the W entropy term Wld
cudaError_t launch_global(int D, int q, int ops, int col_lo, int col_hi, const double *stats, const double *Wbar, const double *Wvar,
                          double *mu, double *muvar, double *gl, const double *P0, const double *h0,
                          const pyvb_consts &c, double *elbo_out, const double *nd, cudaStream_t st, bool weighted = false,
                          const double *Wcov = nullptr, const double *Wld = nullptr);
// per-dimension noise precisions (kernels_noise.cu): Mu (PYVB_OP_MU), r_d, the Gamma of every d (PYVB_OP_BETA) and the per-d X
// and Beta bound terms (PYVB_OP_BETA | PYVB_OP_ELBO) into the nd block; one warp per data dimension, no atomics
// ncnt (nullable): weighted data -- the number of observed entries of every column, which the bound reads (stats' cnt is then
// the weight sum)
// Wcov (nullable): row-wise W posterior, r_d reads Sigma_d
cudaError_t launch_noise_diag(int D, int q, int ops, const double *stats, const double *Wbar, const double *Wvar, double *mu,
                              double *muvar, double *nd, double alpha_mu, cudaStream_t st, const double *ncnt = nullptr,
                              const double *Wcov = nullptr);
cudaError_t launch_impute(long long N, int D, int q, const double *Xorig, long long ldx, const double *Wbar,
                          const double *mu, const double *Zbar, long long ldz, const double *gl, double *Xhat,
                          double *V, double *qldX, cudaStream_t st);

// ---- FP64 tensor-core (DMMA) + TMA-bulk kernels -------------------------------
bool dmma_supported(int D, int q);
// S (nullable): per-entry observation weights, [N][lds] like X (lds even, 16-byte aligned): the contractions become
// [S.O | S.O.(X - mu)] (K1) and [S.O | S.O.X] (K3); the weight of an entry whose x is NaN is not read
cudaError_t launch_zstep_dmma(long long N, int D, int q, const double *X, long long ldx, const double *Gw,
                              int ldg, const double *P0, const double *h0, double *gl, double *MZ, double *Sig,
                              double *logdet, double *zsums, int k1_only, cudaStream_t st, const double *cond = nullptr,
                              const double *S = nullptr, long long lds = 0);
int zstep_eta_pitch(int q);
cudaError_t launch_zstep_eta_dmma(long long N, int D, int q, const double *X, long long ldx, const double *Gw,
                                  double *weta, const double *P0, const double *h0, double *gl, double *MZ,
                                  cudaStream_t st);
// K2, the batched q x q solve in place on the MZ rows, one kernel per q: thread per matrix at q = 8 (kernels_k2t.cu), Gauss-Jordan
// in registers at q = 16, 32 (kernels_k2g.cu), blocked symmetric sweep at q = 64 (kernels_k2s.cu).
// cond (nullable, device): the kernel exits at once unless *cond > 0 (the conditional fall-back launches of the INT8 path)
cudaError_t launch_zsolve(long long N, int q, double *MZ, double *Sig, double *logdet, double *gl, double *zsums,
                          cudaStream_t st, const double *cond = nullptr, I8Check chk = I8Check());
// K2 leaves nblk partials of kw doubles each in zsums (0, 0: no fast K2 for this q)
void zsolve_partials(long long N, int q, int &nblk, int &kw);
// the K2 kernels behind launch_zsolve; all of them leave the partial layout [column sums OROW | 4 scalars | column maxima OROW]
int zsolve_gj_blocks(long long N, int q);         // q in {16, 32}
int zsolve_gj_kw(int q);
cudaError_t launch_zsolve_gj(long long N, int q, double *MZ, double *Sig, double *logdet, double *gl, double *zsums,
                             cudaStream_t st, const double *cond = nullptr, I8Check chk = I8Check());
int zsolve_sweep_blocks(long long N, int q);      // q = 64
int zsolve_sweep_kw(int q);
cudaError_t launch_zsolve_sweep(long long N, int q, double *MZ, double *Sig, double *logdet, double *gl, double *zsums,
                                cudaStream_t st, const double *cond = nullptr, I8Check chk = I8Check());
int zsolve_tpm_blocks(long long N, int q);        // q in {8, 16} (q = 16: the FP32 rows)
int zsolve_tpm_kw(int q);
cudaError_t launch_zsolve_tpm(long long N, int q, double *MZ, double *Sig, double *logdet, double *gl, double *zsums,
                              cudaStream_t st, const double *cond = nullptr, I8Check chk = I8Check());
// K2 on the FP32 rows: thread per matrix at q = 16, blocked tensor-core kernel (kernels_k2.cu) at q = 32, 64.
// MP: bf16 [3][nalloc][pitch] (N <= nalloc, already offset to the first row: a row range keeps the plane stride)
cudaError_t launch_zsolve_tpm_f32(long long N, long long nalloc, int q, float *MZ32, void *MP, double *Sig, double *logdet,
                                  double *gl, double *zsums, cudaStream_t st);
cudaError_t launch_zsolve_f32(long long N, long long nalloc, int q, float *MZ32, void *MP, double *Sig, double *logdet,
                              double *gl, double *zsums, cudaStream_t st);
int stats_dmma_nchunks(long long N, int D, int q);
cudaError_t launch_stats_dmma(long long N, int D, int q, const double *X, long long ldx, const double *MZ,
                              double *ws_main, int nchunks, cudaStream_t st, const double *cond = nullptr,
                              const double *S = nullptr, long long lds = 0);

// ---- FP32 variant: tcgen05 / TMEM contraction on bf16 x 3 splits (kernels_f32.cu) ----
int f32_ncp(int q);                 // floats per MZ32 row
int f32_zoff(int q);                // first eta / zbar column of an MZ32 row (0)
int f32_poff(int q);                // first packed column (q)
bool f32_supported(int D, int q);
cudaError_t launch_prepare_x_f32(long long N, int D, const double *X, long long ldx, void *planes, cudaStream_t st);
cudaError_t launch_pack_gw_f32(int D, int q, const double *Wbar, const double *Wvar, const double *mu, void *GT, void *WT,
                               cudaStream_t st);
// nalloc: rows per plane in the planes / MP allocations (N <= nalloc: row sub-ranges keep the plane stride)
cudaError_t launch_zstep_f32(long long N, long long nalloc, int D, int q, const void *planes, const void *GT,
                             const void *WT, const double *P0, const double *h0, const double *gl, float *MZ,
                             cudaStream_t st);

int stats_f32_nchunks(long long N, int D, int q);
void zsolve_partials_f32(long long N, int q, int &nblk, int &kw);
cudaError_t launch_stats_f32(long long N, long long nalloc, int D, int q, const void *planes, const void *MP, double *ws,
                             int nchunks, cudaStream_t st);

// ---- exact mask contraction on the INT8 tensor cores (kernels_i8.cu) ----
bool i8_supported(int D, int q);
size_t i8_digits_bytes(int D, int q);          // bytes of the digit planes of G
size_t i8_mask_bytes(long long N, int D);      // bytes of the tile-major int8 mask
int i8_ncols(int q);                           // packed columns rounded up to 32 (length of gscale)
cudaError_t launch_prepare_mask_i8(long long N, int D, const double *X, long long ldx, void *mask, cudaStream_t st);
// also clears gl[PYVB_GL_I8BAD] (the guard counter of the Z step that follows)
// G is read from the packed Gw rows (pitch pyvb_gw_pitch(q)): with per-dimension noise they carry tau_d G_d
cudaError_t launch_pack_g_i8(int D, int q, const double *Gw, int ldg, void *GI, double *gscale, double *gl, cudaStream_t st);
cudaError_t launch_zstep_i8(long long N, int D, int q, const void *mask, const void *GI, const double *P0,
                            const double *gscale, const double *gl, double *MZ, int ldmz, cudaStream_t st);

// K3-i8: mask-type statistics (T1, Bst) on the INT8 tensor cores + Ast on the FP64 tensor cores
bool stats_i8_supported(int D, int q);
int stats_i8_ncols(int q);
long long stats_i8_npad(long long N);                       // rows of maskT / ZI rounded up to 128
size_t stats_i8_digits_bytes(long long N, int q);           // bytes of ZI
size_t stats_i8_maskt_bytes(long long N, int D);            // bytes of maskT
size_t stats_i8_scratch_len(int q, int ldmz);               // doubles: partial column maxima + zscale + guard block
double *stats_i8_guard(double *scratch, int q, int ldmz);   // [0] data dimensions that failed the guard, [1] fall-backs taken
// after launch_stats_i8: flags (guard[0] > 0) the data dimensions d whose T1 row is not accurate to tol in the max norm:
// cnt_d * max_c zscale_c * 2^-55 > tol * max_i T1[d][ii]  (cnt = the first D entries of xcache)
cudaError_t launch_stats_i8_check(int D, int q, const double *ws, int nchunks, const double *xcache, double *scratch,
                                  int ldmz, double tol, cudaStream_t st);
int stats_i8_nchunks(long long N, int D, int q);
bool stats_i8_fused(int D);                                 // launch_stats_i8 makes the digit planes in shared memory (ZI unused)
cudaError_t launch_prepare_maskT_i8(long long N, int D, const double *X, long long ldx, void *maskT, cudaStream_t st);
cudaError_t launch_stats_i8(long long N, int D, int q, const void *maskT, const double *MZ, int ldmz, void *ZI,
                            double *scratch, double *ws, int nchunks, const double *zsums, int nzblk, int zkw, int trusted,
                            const double *logdet, const double **zs_out, int *nzblk_out, int *zkw_out, cudaStream_t st);
cudaError_t launch_stats_x_dmma(long long N, int D, int q, const double *X, long long ldx, const double *MZ,
                                double *ws_main, int nchunks, cudaStream_t st);

// ---- sparse observations: CSR gather for the Z step, row-blocked CSC gather for the statistics (kernels_sparse.cu) ----
bool csr_supported(int q);                                  // q in {8, 16, 32, 64} (the q of launch_zsolve)
int csr_stats_nblocks(long long N, int D, int q);           // row blocks of the column-major layout (partials of K3-csc)
long long csr_block_rows(long long N, int D, int q);        // rows per block (the last one may hold fewer)
// MZ rows [0, N) <- [qprec packed | 0 | eta], the input of launch_zsolve.  weights (nullable): per entry, in the order of values
cudaError_t launch_zstep_csr(long long N, int q, const long long *indptr, const int *indices, const double *values,
                             const double *Gw, int ldg, const double *P0, const double *h0, const double *gl, double *MZ,
                             int ldmz, cudaStream_t st, const double *weights = nullptr);
// T1 | Bst | Ast of every row block b into ws_main[b][statlen] (the other entries of the partials are not written).
// wts (nullable): per entry, in the order of vals
cudaError_t launch_stats_csc(int D, int q, int nblk, const long long *colptr, const int *rows, const double *vals,
                             const double *MZ, int ldmz, double *ws_main, cudaStream_t st, const double *wts = nullptr);

// ---- known trailing latent dimensions, the row covariates of the plate (kernels_known.cu) ----
// MZ rows of width qt whose last k dimensions are known per row, c_n = C[n][0, k).  condition: on K1's rows, eta_z -= qprec_zc c,
// qprec_zc = 0, qprec_cc = I, eta_c = c (cond as launch_zsolve's).  finish: on K2's rows, <z'z'^T>_cc = c c^T and zbar_c = c.
cudaError_t launch_known_condition(long long N, int qt, int k, const double *C, long long ldc, double *MZ, long long ldmz,
                                   cudaStream_t st, const double *cond = nullptr);
// the INT8 guard's scale of a conditioned row, one double into *out: max(max of gscale over the free columns,
// max(1, cmax) * max of gscale over the zc columns); the cc columns, which condition discards, are left out
cudaError_t launch_known_guard_scale(int qt, int k, const double *gscale, double cmax, double *out, cudaStream_t st);
cudaError_t launch_known_finish(long long N, int qt, int k, const double *C, long long ldc, double *MZ, long long ldmz,
                                cudaStream_t st);

// ---- LDS smoother, batched over sequences (kernels_lds.cu) ----
size_t lds_smem_bytes(int T, int d);
cudaError_t launch_lds_iterate(int B, int T, int q, int d, const double *Y, double *X, double *Xcov3, double *A,
                               double *Avar, double *C, double *Cvar, double *Qa, double *Qb, double *Ra, double *Rb,
                               double alpha0, double a0, double b0, int niters, double *status, cudaStream_t st,
                               const double *Aknown = nullptr);

cudaError_t launch_bench_dmma(int blocks, int iters, double *scratch, cudaStream_t st);
cudaError_t launch_bench_umma(int blocks, int iters, int n, int kind, int mode, const void *src, long long *clk_out,
                              cudaStream_t st);

}  // namespace pyvb
