/*
 * pyvb_b200 -- C-ABI of the B200-native VB-PCA (missing data) hot path.
 *
 * Plain C symbols, raw DEVICE pointers (unless marked host), explicit CUDA stream
 * (passed as void* = cudaStream_t), no hidden allocation: every workspace is
 * passed in and sized by a *_len / *_bytes query.  Every entry point returns 0 on
 * success or a negative PYVB_E* code; pyvb_last_error() gives the text.  No
 * exceptions, no torch types.
 *
 * Each entry point replaces a piece of the reference's message-passing update
 * (paths relative to /root/reference/src/pyvb):
 *
 *   pyvb_pack_gw_f64     nodes/node.py:214-224      <w_i w_j^T> + Cov(w_i) per data dimension, packed
 *   pyvb_zstep_f64       nodes/node.py:203-227      m1 = tr(<w_i w_j^T> Lambda_n), m2 = <W>^T sum_m2   (K1)
 *                        nodes/gaussian.py:112-123  qprec, cho_factor, cho_solve, qmu, q_ln_det         (K2)
 *   pyvb_stats_f64       nodes/nodes_todo.py:50-61  hstack sufficient statistics over all rows         (K3)
 *                        nodes/nodes_todo.py:136-138, nodes/gaussian.py:141-151  residual / ELBO sums  (K4)
 *   pyvb_wupdate_f64     nodes/nodes_todo.py:53-62 + nodes/gaussian.py:117-123  one W column at a time
 *   pyvb_global_f64      nodes/node.py:105-109 (Mu), nodes/nodes_todo.py:130-157 (Gamma update, bounds),
 *                        nodes/gaussian.py:136-151 (Gaussian bounds), network.py:49 (ELBO sum)
 *   pyvb_impute_f64      nodes/gaussian.py:125-134  partially observed X_n (mode A imputation)
 *
 * Layouts (all float64, row-major):
 *   X      [N][ldx]   data; NaN = entry not observed (marginalised)
 *   Zbar   [N][ldz]   <z_n>
 *   M2     [N][ldm]   <z_n z_n^T>, packed lower triangle p(i,j) = i(i+1)/2 + j (i >= j), P = q(q+1)/2
 *                     The DMMA path wants the two interleaved in ONE array MZ [N][pyvb_mz_pitch(q)]:
 *                     M2 = MZ, Zbar = MZ + pyvb_gw_woff(q), ldm = ldz = pyvb_mz_pitch(q), unused columns 0
 *                     (one TMA tile then feeds the statistics GEMM, one bulk store per row leaves the Z step)
 *   Sig    [N][P]     Cov(z_n) packed (optional output)
 *   logdet [N]        ln prod diag chol(qprec_n)  (= 0.5 ln det)
 *   Gw     [D][ldg]   cols [0,P) = G_d packed, [Pp,Pp+q) = <w_d>, [Pp+q] = <mu_d>, rest zero padding;
 *                     Pp = pyvb_gw_woff(q) = P rounded up to a multiple of 8, ldg = pyvb_gw_pitch(q)
 *   Wbar, Wvar [D][q] column means / diagonal of the column covariances
 *   stats  [pyvb_stats_len(D,q)] one contiguous buffer, ready for a single all-reduce(SUM):
 *            T1 [D][P] = O^T vec<zz^T> | Bst [D][q] = O^T Zbar | Ast [D][q] = (O.X)^T Zbar |
 *            cnt [D] | colsumX [D] | S [P] = sum_n <zz^T>_n | zsum [q] | scal [PYVB_NSCAL]
 *   gl     [PYVB_GL_LEN]  device-resident globals (tau lives here so that no host sync is needed)
 */
#ifndef PYVB_B200_H
#define PYVB_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PYVB_OK 0
#define PYVB_EINVAL (-1)   /* bad argument (shape, pitch, null pointer) */
#define PYVB_ECUDA (-2)    /* CUDA runtime error; see pyvb_last_error() */
#define PYVB_ENOSUP (-3)   /* shape not supported by the requested algorithm */

#define PYVB_QMAX 64

/* scalar slots at the tail of the stats buffer */
#define PYVB_NSCAL 16
#define PYVB_SC_SXX 0        /* sum over observed entries of <x>^2              */
#define PYVB_SC_SUMV 1       /* sum of imputation variances (mode A)            */
#define PYVB_SC_NE 2         /* number of observed (effective) entries          */
#define PYVB_SC_QLDZ 3       /* sum_n 0.5/logdet_n  (gaussian.py:120 quirk)     */
#define PYVB_SC_LOGDETZ 4    /* sum_n logdet_n                                  */
#define PYVB_SC_LATQLD 5     /* mode A: sum over all-NaN rows of q_ln_det(X_n)  */
#define PYVB_SC_NLAT 6       /* mode A: number of all-NaN rows                  */
#define PYVB_SC_PNMISS 7     /* mode A: missing entries in partially observed rows */
#define PYVB_SC_PLNV 8       /* mode A: sum ln v over those entries             */
#define PYVB_SC_NROWS 9

/* multi-GPU exchange: per-CTA flags in a peer buffer (see pyvb_peer_bytes) */
#define PYVB_PEER_MAXBLK 512

/* K2 column-sum partials (zsums): per CTA [<zz^T> packed | pad | zbar] column sums followed by
 * sum 0.5/logdet, sum logdet, rows, 0 */
#define PYVB_ZS_EXTRA 4

/* device globals */
#define PYVB_GL_QA 0
#define PYVB_GL_QB 1
#define PYVB_GL_TAU 2
#define PYVB_GL_ELBO 3
#define PYVB_GL_ELBO_W 4
#define PYVB_GL_ELBO_MU 5
#define PYVB_GL_ELBO_Z 6
#define PYVB_GL_ELBO_X 7
#define PYVB_GL_ELBO_BETA 8
#define PYVB_GL_ELBO_ALPHA 9
#define PYVB_GL_RESID2 10
#define PYVB_GL_NONPD 11     /* rows whose posterior precision was not positive definite (as a double) */
#define PYVB_GL_I8BAD 12     /* INT8 path: rows of the LAST Z step whose qprec failed the accuracy guard (then redone on DMMA) */
#define PYVB_GL_I8FALL 14    /* INT8 path: Z steps that fell back to the FP64 tensor cores so far (diagnostic) */
#define PYVB_GL_ALPHA 16     /* [64] <alpha_i>  (constant prior precision when ARD is off) */
#define PYVB_GL_ALQB 80      /* [64] ARD Gamma qb_i */
#define PYVB_GL_LEN 144

/* pyvb_global_f64 op mask */
#define PYVB_OP_MU 1
#define PYVB_OP_BETA 2
#define PYVB_OP_ALPHA 4
#define PYVB_OP_ELBO 8

/* algorithm selector for zstep / stats */
#define PYVB_ALGO_AUTO 0
#define PYVB_ALGO_GENERIC 1  /* any D, q <= 64; FP64 FMA */
#define PYVB_ALGO_DMMA 2     /* FP64 tensor-core (DMMA) + TMA staging; q in {8,16,32,64}, D % 16 == 0 */
#define PYVB_ALGO_F32 4      /* FP32 variant (tcgen05): only for pyvb_stats_workspace_bytes */
#define PYVB_ALGO_DMMA_K1 3  /* measurement only (zstep): the tensor-core contraction alone; the MZ rows are
                                left as [qprec packed | eta] for pyvb_zsolve_f64 */

typedef struct pyvb_consts {
    double alpha_mu;      /* prior precision of Mu (Constant alpha*I)                    */
    double a0, b0;        /* noise Gamma prior                                           */
    double psi_qa;        /* digamma(qa), lgamma(qa), lgamma(a0): qa is fixed, host-computed */
    double lgam_qa;
    double lgam_a0;
    double ard_a0, ard_b0;
    double al_qa;         /* ARD: a0 + D/2 */
    double psi_alqa, lgam_alqa, lgam_ard_a0;
    double lndet_P0;      /* Z prior N(m0, P0^-1): ln det P0 and m0^T P0 m0              */
    double m0P0m0;
    int ard;              /* 1: W columns have Gamma (ARD) precisions                    */
    int mode_a;           /* 1: reference-exact imputation mode (adds the X entropy terms) */
} pyvb_consts;

/* Multi-GPU exchange of the statistics over NVLink peer memory (one process per GPU, one box).  bufs is a DEVICE
 * array of `world` pointers: entry r is rank r's exchange buffer (pyvb_peer_bytes(stats_len) bytes, from
 * pyvb_peer_alloc on rank r, opened here through pyvb_peer_import).  epoch: 1, 2, 3, ... -- the same on every rank,
 * incremented by the caller for every pyvb_stats_f64 call that carries the struct. */
typedef struct pyvb_peers {
    void *const *bufs;            /* device pointer */
    int world, rank;
    unsigned long long epoch;
} pyvb_peers;

int pyvb_version(void);
const char *pyvb_last_error(void);

/* sizes */
int pyvb_gw_pitch(int q);                              /* doubles per Gw row */
int pyvb_gw_woff(int q);                               /* first <w_d> column of a Gw row (= zbar offset in MZ) */
int pyvb_mz_pitch(int q);                              /* doubles per row of the interleaved [M2 | zbar] array */
size_t pyvb_stats_len(int D, int q);                   /* doubles */
size_t pyvb_stats_workspace_bytes(long long N, int D, int q, int algo);
size_t pyvb_zsums_len(long long N, int q);             /* doubles to allocate (the largest over the K2 kernels); 0 when K2 has no fast path for q */
int pyvb_zsums_blocks(long long N, int q);             /* partials the K2 kernel in use writes: the first pyvb_zsums_blocks * pyvb_zsums_kw doubles */

/* peer exchange buffers: cudaMalloc'd (zeroed) so that the CUDA IPC handle (64 bytes) names exactly this buffer */
size_t pyvb_peer_bytes(size_t stats_len);
int pyvb_peer_alloc(size_t bytes, void **dptr /* host out */);
int pyvb_peer_free(void *dptr);
int pyvb_peer_export(void *dptr, unsigned char *handle64 /* host out, 64 bytes */);
int pyvb_peer_import(const unsigned char *handle64 /* host */, void **dptr /* host out */);
int pyvb_peer_close(void *dptr);
int pyvb_algo_supported(int algo, int D, int q);       /* 1/0 */
int pyvb_zsums_kw(int q);   /* doubles per K2 partial: [column sums (Pp + q) | 4 scalars | column maxima (Pp + q)] */

int pyvb_pack_gw_f64(int D, int q, const double *Wbar, const double *Wvar, const double *mu,
                     double *Gw, int ldg, void *stream);

/* K1+K2 for rows [0,N): reads X, Gw, tau = gl[PYVB_GL_TAU]; P0 [q][q] and h0 = P0 m0 [q] are the
 * (constant) prior of z.  Sig may be NULL.  Non-PD rows are counted into gl[PYVB_GL_NONPD].
 * zsums (nullable, pyvb_zsums_len(N, q) doubles, DMMA path only): K2 leaves per-CTA partial column sums of
 * its output rows there (S = sum_n <zz^T>_n, zsum, sum 0.5/logdet, sum logdet); pyvb_stats_f64 called with the
 * same buffer and zsums_valid = 1 then skips its own pass over the MZ rows. */
int pyvb_zstep_f64(long long N, int D, int q, const double *X, long long ldx, const double *Gw, int ldg,
                   const double *P0, const double *h0, double *gl,
                   double *Zbar, long long ldz, double *M2, long long ldm, double *Sig, double *logdet,
                   double *zsums, int algo, void *stream);

/* K2 alone (DMMA-path layout): rows of MZ = [qprec packed | pad | eta] are replaced in place by
 * [<zz^T> packed | 0 | zbar]; batched q x q SPD inverse / solve, q in {8,16,32,64}.  Sig may be NULL.
 * MZ must be 16-byte aligned (the rows travel as bulk copies; the pitch is a multiple of 32 bytes). */
int pyvb_zsolve_f64(long long N, int q, double *MZ, long long ldmz, double *Sig, double *logdet, double *gl,
                    double *zsums, void *stream);

/* K3+K4 over rows [0,N) into `stats` (fully overwritten).  V, Xorig, qldX are mode-A only (NULL in
 * mode B).  ws: pyvb_stats_workspace_bytes().
 * xcache (nullable, 2*D+2 doubles, caller-owned): the sums that depend on X alone -- cnt[D], colsumX[D],
 * sum x^2, number of observed entries.  With xcache_valid = 0 they are computed and stored there; with
 * xcache_valid = 1 (X unchanged since, i.e. mode B) the two passes over X are skipped and the cached local
 * sums are used.
 * peers (nullable): with it, the second-stage kernel also performs the all-reduce(SUM) over the ranks -- it
 * publishes the local sums in this rank's exchange buffer and adds the peers' buffers over NVLink in rank order,
 * so `stats` holds the global statistics, bit-identical on every rank, when the call's kernels finish.
 * zsums / zsums_valid: the K2 partials of a pyvb_zstep_f64 / pyvb_zsolve_f64 call that covered exactly these
 * N rows (see there); with zsums_valid = 0 the sums over the MZ rows are recomputed here. */
int pyvb_stats_f64(long long N, int D, int q, const double *X, long long ldx, const double *V,
                   const double *Xorig, const double *qldX, const double *Zbar, long long ldz, const double *M2,
                   long long ldm, const double *logdet, double *stats, void *ws, size_t ws_bytes,
                   double *xcache, int xcache_valid, const double *zsums, int zsums_valid,
                   const pyvb_peers *peers /* host, nullable */, int algo, void *stream);

/* Gauss-Seidel update of W columns [col_lo, col_hi) from the (all-reduced) stats. */
int pyvb_wupdate_f64(int D, int q, int col_lo, int col_hi, const double *stats, const double *mu,
                     const double *gl, double *Wbar, double *Wvar, void *stream);

/* Replicated small updates + ELBO; ops = OR of PYVB_OP_*.  PYVB_OP_ALPHA updates the ARD Gammas of
 * columns [col_lo, col_hi).  P0/h0 as in zstep.  elbo_out may be NULL. */
int pyvb_global_f64(int D, int q, int ops, int col_lo, int col_hi, const double *stats, const double *Wbar, const double *Wvar,
                    double *mu, double *muvar, double *gl, const double *P0, const double *h0,
                    const pyvb_consts *consts /* host */, double *elbo_out, void *stream);

/* Mode A: x_hat = observed ? x : W zbar + mu, v = observed ? 0 : 1/tau for rows [0,N) that are not
 * fully observed (pointers already offset to the first row). */
int pyvb_impute_f64(long long N, int D, int q, const double *Xorig, long long ldx, const double *Wbar,
                    const double *mu, const double *Zbar, long long ldz, const double *gl,
                    double *Xhat, double *V, double *qldX, void *stream);

/* ---- exact mask contraction on the INT8 tensor cores (tcgen05.mma kind::i8) ----
 * Same reference arithmetic as pyvb_zstep_f64 (nodes/node.py:203-227 + nodes/gaussian.py:112-123) and the same result
 * to FP64 rounding: the 0/1 mask is exact in int8 and every column of G is split into seven balanced base-256 digit
 * planes of a 2^-54 fixed-point representation (relative to the column maximum), so mask @ G is a sum of exact
 * integer GEMMs recombined in FP64.  The eta columns (X real) stay on the FP64 tensor cores.  Mode B only.
 * q in {16, 32, 64}, D % 64 == 0, D small enough for the resident mask block (pyvb_i8_supported).
 *   mask   pyvb_i8_mask_bytes(N, D) bytes, int8 tiles [n / 128][d / 64][128][64], 1 = observed: pyvb_prepare_mask_i8
 *          (once per data set).  A sub-range of rows starting at a multiple of 128 starts at mask + first_row * D.
 *   GI     pyvb_i8_digits_bytes(D, q) bytes, gscale pyvb_i8_ncols(q) doubles: per-sweep scratch (filled by the call)
 *   MZ     the interleaved rows of the DMMA path (ldmz = pyvb_mz_pitch(q)); Gw as for pyvb_zstep_f64 (DMMA pitch)
 * k1_only (measurement): 1 leaves [qprec packed | eta] in the rows; 2 runs the INT8 part alone, 3 the eta part alone.
 * Accuracy guard: the fixed point is relative to the COLUMN maximum of G, so a row that observes none of a column's large
 * entries keeps at most tau * n_obs * scale_c * 2^-55 of rounding.  The batched solve checks every finished qprec row:
 * when tau * D * max_c scale_c * 2^-55 > 2^-38 * max_i qprec_ii for any row (gl[PYVB_GL_I8BAD] counts them), the whole
 * call is redone on the FP64 tensor cores by conditional launches that exit at once otherwise (gl[PYVB_GL_I8FALL] counts
 * the fall-backs).  The result is therefore accurate to 2^-38 of max_i qprec_ii per row for ANY input range; on the
 * normalised data of BASELINE.json's configurations the bound sits at ~2^-50 and the guard never fires. */
int pyvb_i8_supported(int D, int q);
size_t pyvb_i8_digits_bytes(int D, int q);
int pyvb_i8_ncols(int q);
size_t pyvb_i8_mask_bytes(long long N, int D);
int pyvb_prepare_mask_i8(long long N, int D, const double *X, long long ldx, void *mask, void *stream);
int pyvb_zstep_i8_f64(long long N, int D, int q, const double *X, long long ldx, const void *mask, const double *Wbar,
                      const double *Wvar, const double *Gw, int ldg, const double *P0, const double *h0, double *gl,
                      double *MZ, long long ldmz, void *GI, double *gscale, double *Sig, double *logdet, double *zsums,
                      int k1_only, void *stream);

/* Statistics with the mask-type sums T1 = O^T vec<zz^T>, Bst = O^T Zbar (nodes/nodes_todo.py:50-61) on the INT8 tensor
 * cores: the MZ columns are rewritten as seven balanced base-256 digit planes (fixed point, 2^-54 of the column maximum),
 * the products with the 0/1 mask are exact integer GEMMs, recombined in FP64 per row chunk.  Ast = (O.X)^T Zbar stays on
 * the FP64 tensor cores.  Mode B, interleaved MZ rows, q in {16, 32, 64}, D % 16 == 0.  Requires what pyvb_stats_f64
 * treats as optional: xcache (valid: the X-only sums of an earlier pyvb_stats_f64 call).  zsums: the K2 partials of the
 * Z step that produced these rows, or NULL (then logdet [N] is read and the MZ column sums take one more pass).
 *   maskT  pyvb_stats_i8_maskt_bytes(N, D) bytes, [n / 64][D][64] int8: pyvb_prepare_maskt_i8 (once per data set)
 *   ZI     pyvb_stats_i8_digits_bytes(N, q) bytes, per-call scratch; NULL is allowed where pyvb_stats_i8_fused(D, q) is 1
 *          (D <= 256: the digit planes are made in shared memory; PYVB_I8_FUSED=0, read on every call, turns that off)
 *   scratch pyvb_stats_i8_scratch_len(q) doubles: per-call scratch; the caller ZEROES it once (its last 8 doubles are the
 *          guard's counters, kept from call to call)
 *   ws     pyvb_stats_i8_workspace_bytes(N, D, q)
 * Accuracy guard, as for pyvb_zstep_i8_f64: a data dimension d with cnt_d * max_c zscale_c * 2^-55 > 2^-38 * max_i T1[d][ii]
 * (outlier rows that d does not observe) sends the whole pass to the FP64 tensor cores, before the exchange. */
int pyvb_stats_i8_supported(int D, int q);
long long pyvb_stats_i8_npad(long long N);
size_t pyvb_stats_i8_digits_bytes(long long N, int q);
int pyvb_stats_i8_fused(int D, int q);
size_t pyvb_stats_i8_maskt_bytes(long long N, int D);
size_t pyvb_stats_i8_scratch_len(int q);
size_t pyvb_stats_i8_guard_offset(int q);   /* scratch[off] = data dimensions that failed the guard in the last call, [off+1] = fall-backs so far */
size_t pyvb_stats_i8_workspace_bytes(long long N, int D, int q);
int pyvb_prepare_maskt_i8(long long N, int D, const double *X, long long ldx, void *maskT, void *stream);
int pyvb_stats_i8_f64(long long N, int D, int q, const double *X, long long ldx, const void *maskT, const double *MZ,
                      long long ldmz, const double *logdet, void *ZI, double *scratch, double *stats, void *ws,
                      size_t ws_bytes, const double *xcache, const double *zsums, const pyvb_peers *peers, void *stream);

/* ---- FP32 variant of the Z-step contraction (tcgen05 tensor cores, TMEM accumulators, TMA-staged bf16 x 3 splits) ----
 * Same reference arithmetic as pyvb_zstep_f64's K1 (nodes/node.py:203-227).  q in {16, 32, 64}, D % 32 == 0.
 *   planes  bf16 [3][N][D]    mask | x_h | x_m  (x = x_h + x_m to 16 bits; zeros where not observed); static over sweeps
 *   GT      bf16 [3][NCP][D]  three-way split of [-mu_d <w_d> (q) | G_d packed (P) | pad]^T,  NCP = pyvb_f32_pitch(q)
 *   WT      bf16 [3][q][D]    three-way split of <W>^T
 *   MZ32    float [N][NCP]    out: [eta (q) | qprec packed (P) | pad]: the FP32 rows keep zbar / eta FIRST
 *                             (pyvb_f32_zoff(q) = 0, packed part at pyvb_f32_poff(q) = q) */
int pyvb_f32_pitch(int q);
int pyvb_f32_zoff(int q);
int pyvb_f32_poff(int q);
int pyvb_f32_supported(int D, int q);
size_t pyvb_zsums_len_f32(long long N, int q);        /* K2 partials of the FP32 path (always the blocked kernel) */
int pyvb_prepare_x_f32(long long N, int D, const double *X, long long ldx, void *planes, void *stream);
int pyvb_pack_gw_f32(int D, int q, const double *Wbar, const double *Wvar, const double *mu, void *GT, void *WT,
                     void *stream);
int pyvb_zstep_k1_f32(long long N, int D, int q, const void *planes, const void *GT, const void *WT, const double *P0,
                      const double *h0, const double *gl, float *MZ32, void *stream);

/* FP32 Z step for rows [0,N) of arrays whose planes hold `nalloc` rows each (pointers already offset to the first
 * row): the tcgen05 contraction, then the batched solve IN PLACE on the FP32 rows (FP64 arithmetic inside the solve:
 * the q x q systems have condition numbers ~1e4): MZ32 rows become [zbar | <zz^T> packed | 0], MP bf16 [3][nalloc][NCP]
 * receives their three-way bf16 split (the B operand of pyvb_stats_f32).  Sig (double [N][P]) may be NULL; zsums as
 * in pyvb_zstep_f64. */
int pyvb_zstep_f32(long long N, long long nalloc, int D, int q, const void *planes, const void *GT, const void *WT,
                   const double *P0, const double *h0, double *gl, float *MZ32, void *MP, double *Sig, double *logdet,
                   double *zsums, void *stream);

/* FP32 statistics: T1, Bst, Ast partial sums on the tensor cores (MN-major bf16 tiles, FP32 accumulation per row
 * chunk, FP64 across chunks), then the shared fixed-order second stage (+ the peer exchange).  The sums that depend
 * on X alone (xcache) and K2's column sums (zsums) must be valid: the FP32 path has no other source for them. */
int pyvb_stats_f32(long long N, long long nalloc, int D, int q, const void *planes, const void *MP, double *stats,
                   void *ws, size_t ws_bytes, double *xcache, const double *zsums, const pyvb_peers *peers /* host */,
                   void *stream);

/* ---- sparse observations (mode B, FP64, q in {8, 16, 32, 64}, any D) ----
 * The stored entries of a CSR matrix are the observations (a stored zero is an observed 0); everything not stored is
 * missing.  The work of a sweep is per stored entry: the Z step gathers one Gw row per entry of its row, the statistics
 * gather one MZ row per entry of their column.  The callers own and validate the layouts (pyvb_b200/sparse.py builds them):
 * column indices in [0, D), sorted within a row, no duplicates, finite values.  Both calls are deterministic (fixed
 * summation order, no atomics).
 *   CSR       indptr int64 [N + 1] (the rows' own offsets: a row range [lo, hi) passes indptr + lo), indices int32,
 *             values double
 *   blocked   the same entries column-major per row block: nblk blocks of pyvb_csr_block_rows(N, D, q) consecutive
 *   CSC       rows (pyvb_csr_stats_blocks(N, D, q) of them; any nblk >= 1 is valid, these sizes keep a block's MZ rows in
 *             the L2).  colptr int64 [nblk * D + 1]: the entries of block b, column d are [colptr[b*D + d],
 *             colptr[b*D + d + 1]) of rows int32 (row index within these N rows, increasing) / vals double
 *   xcache    2*D + 2 doubles [cnt (D) | colsumX (D) | sum x^2 | number of stored entries] of these N rows, computed once by
 *             the caller (the layout of pyvb_stats_f64's cache)
 * pyvb_zstep_csr_f64: MZ rows [0, N) <- [qprec packed | 0 | eta] (rows without entries get the prior), then the batched
 * solve in place as pyvb_zsolve_f64 (zsums, Sig nullable as there).
 * pyvb_stats_csr_f64: T1 | Bst | Ast per row block, then the shared second stage with xcache and the optional peer exchange.
 * zsums: the K2 partials of the pyvb_zstep_csr_f64 call that covered exactly these N rows, or NULL (then the MZ column sums
 * and the log-det scalars take one pass each over MZ / logdet).  ws: pyvb_stats_csr_workspace_bytes(N, D, q, nblk).  An
 * empty shard (N = 0) contributes zeros and still takes part in the exchange. */
int pyvb_csr_supported(int D, int q);
int pyvb_csr_stats_blocks(long long N, int D, int q);
long long pyvb_csr_block_rows(long long N, int D, int q);
size_t pyvb_stats_csr_workspace_bytes(long long N, int D, int q, int nblk);
int pyvb_zstep_csr_f64(long long N, int D, int q, const long long *indptr, const int *indices, const double *values,
                       const double *Gw, int ldg, const double *P0, const double *h0, double *gl, double *MZ,
                       long long ldmz, double *Sig, double *logdet, double *zsums, void *stream);
int pyvb_stats_csr_f64(long long N, int D, int q, int nblk, const long long *colptr, const int *rows, const double *vals,
                       const double *MZ, long long ldmz, const double *logdet, double *stats, void *ws, size_t ws_bytes,
                       const double *xcache, const double *zsums, const pyvb_peers *peers /* host, nullable */,
                       void *stream);

/* ---- VB smoother of a linear dynamic system, batched over B independent sequences (BASELINE config 5) ----
 * Replaces the sweep of examples/Linear_Dynamic_System.py:69-76 for every sequence: all X_t.update() forwards, all
 * backwards (nodes/gaussian.py:102-123 + nodes/node.py:203-227), the columns of A and C (nodes/nodes_todo.py:43-62),
 * Q.update(), R.update() (DiagonalGamma, nodes/nodes_todo.py:187-190) -- `niters` whole iterations in one launch,
 * one warp per sequence, the sequence resident in shared memory.  q, d <= 8; 3 <= T <= pyvb_lds_max_len().
 *   Y [B][T][d] observations;  X [B][T][q] state means (in/out);  Xcov3 [B][3][q][q] out: the posterior covariances
 *   of X_0, X_1..X_{T-2}, X_{T-1} (they do not depend on t otherwise);  A, Avar [B][q][q] (row k, column i: mean and
 *   variance of A[k][i]);  C, Cvar [B][d][q];  Qa, Qb [B][q];  Ra, Rb [B][d]  (all in/out).
 *   status: device double, incremented for every sequence with a non-positive-definite posterior precision. */
int pyvb_lds_max_len(void);
int pyvb_lds_iterate_f64(int B, int T, int q, int d, const double *Y, double *X, double *Xcov3, double *A, double *Avar,
                         double *C, double *Cvar, double *Qa, double *Qb, double *Ra, double *Rb, double alpha0,
                         double a0, double b0, int niters, double *status, void *stream);
/* The same with KNOWN entries of A (examples/LDS_knowns_in_A.py:72-74: `As[i].observe(...)` with NaN = unknown makes the
 * column a partially observed Gaussian, nodes/gaussian.py:125-134; with the diagonal posterior covariance of an hstack
 * column that conditioning clamps the known entries to their values with zero variance after every column update).
 *   Aknown [B][q][q] (row k, column i), NaN = free; NULL = nothing known (= pyvb_lds_iterate_f64). */
int pyvb_lds_iterate_known_f64(int B, int T, int q, int d, const double *Y, double *X, double *Xcov3, double *A, double *Avar,
                               double *C, double *Cvar, double *Qa, double *Qb, double *Ra, double *Rb, const double *Aknown,
                               double alpha0, double a0, double b0, int niters, double *status, void *stream);

/* Measurement utility (not part of the hot path): `iters` dependent rounds of 8 independent
 * DMMA.8x8x4 per warp on `blocks` x 256 threads; flops = blocks * 8 warps * iters * 8 * 512.
 * bench.py times it with CUDA events to obtain the FP64 tensor roofline of the box it runs on. */
/* Measurement: `iters` x 2 back-to-back tcgen05.mma (M = 128, N = n, 32 bytes of K each; kind 0 = i8, 1 = bf16) per CTA;
 * clk_out[block] = SM clocks from the first issue to the completion of the last (clk_out: 2 x 148 entries).
 * mode bits: 1 rotate through four operand buffers, 2 commit to an mbarrier after every pair, 4 a second warp streams
 * 14 KB bulk copies from src (blocks MiB) into shared memory meanwhile. */
int pyvb_bench_umma(int blocks, int iters, int n, int kind, int mode, const void *src, long long *clk_out, void *stream);
int pyvb_bench_dmma_f64(int blocks, int iters, double *scratch /* blocks*256 doubles */, void *stream);

#ifdef __cplusplus
}
#endif
#endif
