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
#define PYVB_GL_LNS 13       /* weighted data: 1/2 sum of ln s_nd over the observed entries of positive weight, ALL rows (all
                                ranks); set by the caller, read by pyvb_global_w_f64 only */
#define PYVB_GL_I8FALL 14    /* INT8 path: Z steps that fell back to the FP64 tensor cores so far (diagnostic) */
#define PYVB_GL_ALPHA 16     /* [64] <alpha_i>  (constant prior precision when ARD is off) */
#define PYVB_GL_ALQB 80      /* [64] ARD Gamma qb_i */
#define PYVB_GL_LEN 144

/* per-dimension noise precisions (noise "diagonal", factor analysis): the nd block, PYVB_ND_LEN arrays of D doubles each;
 * array k starts at nd + k * D (pyvb_nd_len(D) doubles in all) */
#define PYVB_ND_TAU 0        /* tau_d = qa_d / qb_d                                  (state: updated by PYVB_OP_BETA) */
#define PYVB_ND_QB 1         /* qb_d                                                 (state: updated by PYVB_OP_BETA) */
#define PYVB_ND_QA 2         /* qa_d = a0_d + cnt_d / 2, cnt_d the GLOBAL observed count of column d   (constant)   */
#define PYVB_ND_PSI_QA 3     /* digamma(qa_d)                                                           (constant)   */
#define PYVB_ND_LGAM_QA 4    /* lgamma(qa_d)                                                            (constant)   */
#define PYVB_ND_A0 5         /* prior Gamma(a0_d, b0_d)                                                 (constant)   */
#define PYVB_ND_B0 6
#define PYVB_ND_LGAM_A0 7    /* lgamma(a0_d)                                                            (constant)   */
#define PYVB_ND_SXX 8        /* sum_n O_nd x_nd^2 over ALL rows (all ranks)                             (constant)   */
#define PYVB_ND_R 9          /* out: r_d = sum_n O_nd <(x_nd - w_d z_n - mu_d)^2>                                    */
#define PYVB_ND_EX 10        /* out: bound term of the X entries of column d                                         */
#define PYVB_ND_EB 11        /* out: bound term of the Gamma of column d                                             */
#define PYVB_ND_LEN 12

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
#define PYVB_ALGO_DMMA_K1 3  /* zstep: the tensor-core contraction alone (measurements, and the K1 of pyvb_zstep_known_f64);
                                the MZ rows are left as [qprec packed | eta] for pyvb_zsolve_f64 */

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
size_t pyvb_zsums_len(long long N, int q);             /* doubles to allocate: pyvb_zsums_blocks * pyvb_zsums_kw; 0 when K2 has no fast path for q */
int pyvb_zsums_blocks(long long N, int q);             /* partials the K2 kernel of q writes (at most 148) */

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
 * [<zz^T> packed | pad | zbar]; batched q x q SPD inverse / solve, q in {8,16,32,64}.  Sig may be NULL.  Only the packed
 * and zbar columns are written: the pad [P, Pp) and the columns past Pp + q are passed through (no reader of the rows uses them).
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

/* ---- per-dimension noise precisions (mode B, FP64; every Z-step path) ----
 * x_nd ~ N(w_d . z_n + mu_d, 1 / tau_d) with one Gamma posterior per data dimension (DiagonalGamma, nodes/nodes_todo.py:159-204).
 * nd: the block described at PYVB_ND_* (pyvb_nd_len(D) doubles, device).  The caller fills the constants once (qa_d needs the
 * global observed counts, sxx_d the global sums of squares) and tau_d / qb_d with the initial state, and keeps
 * gl[PYVB_GL_TAU] = 1: the per-dimension precisions then travel inside the Gw rows.
 *   pyvb_pack_gw_nd_f64   Gw rows [tau_d G_d | pad | tau_d <w_d> | <mu_d>]: pyvb_zstep_f64 (every algo), pyvb_zstep_i8_f64 and
 *                         pyvb_zstep_csr_f64 read them unchanged and compute qprec_n = P0 + sum_d O_nd tau_d G_d and
 *                         eta_n = h0 + sum_d O_nd tau_d (x_nd - mu_d) <w_d>
 *   pyvb_wupdate_nd_f64   pyvb_wupdate_f64 with tau_d in place of the shared tau
 *   pyvb_global_nd_f64    pyvb_global_f64 for this model: PYVB_OP_MU updates Mu with the current tau_d, PYVB_OP_BETA every
 *                         Gamma (qb_d, tau_d), PYVB_OP_BETA or PYVB_OP_ELBO write r_d and the per-d bound terms, PYVB_OP_ALPHA
 *                         is unchanged, PYVB_OP_ELBO adds everything up (fixed order: deterministic).  gl[PYVB_GL_RESID2]
 *                         receives sum_d r_d; gl[PYVB_GL_QA / QB / TAU] are not touched.  Mode B only (consts->mode_a = 0);
 *                         consts->a0 / b0 / psi_qa / lgam_qa / lgam_a0 are not read (nd carries them per d). */
size_t pyvb_nd_len(int D);
int pyvb_pack_gw_nd_f64(int D, int q, const double *Wbar, const double *Wvar, const double *mu, const double *nd,
                        double *Gw, int ldg, void *stream);
int pyvb_wupdate_nd_f64(int D, int q, int col_lo, int col_hi, const double *stats, const double *mu, const double *nd,
                        const double *gl, double *Wbar, double *Wvar, void *stream);
int pyvb_global_nd_f64(int D, int q, int ops, int col_lo, int col_hi, const double *stats, const double *Wbar,
                       const double *Wvar, double *mu, double *muvar, double *gl, double *nd, const double *P0,
                       const double *h0, const pyvb_consts *consts /* host */, double *elbo_out, void *stream);

/* ---- per-entry observation weights (mode B, FP64; the DMMA, generic and sparse paths) ----
 * x_nd ~ N(w_d . z_n + mu_d, 1 / (tau s_nd)) for every entry with x_nd not NaN and s_nd > 0, s_nd >= 0 a KNOWN weight (inverse
 * variances, repeat counts, confidences); s_nd = 0 is a missing entry, as a NaN is.  Lambda_n = tau diag(s_n) replaces
 * tau diag(mask_n) in every contraction:  qprec_n = P0 + tau sum_d s_nd G_d,  eta_n = h0 + tau sum_d s_nd (x_nd - mu_d) <w_d>,
 * T1 = (S.O)^T vec<zz^T>,  Bst = (S.O)^T Zbar,  Ast = (S.O.X)^T Zbar.  The weight of an entry whose x is NaN is never read.
 *   S       [N][lds] doubles, the layout of X (the DMMA path: lds even, S 16-byte aligned); a row range passes S + lo * lds
 *   weights the sparse paths: one double per stored entry, in the order of values (CSR) / vals (blocked CSC)
 * The statistics' X-only sums become cnt_d = sum_n s_nd, colsumX_d = sum_n s_nd x_nd, sum s x^2 -- but scal[PYVB_SC_NE] stays
 * the NUMBER of observed entries of positive weight: the caller's Gamma shape qa = a0 + nE / 2 (global) reads it.  xcache and
 * the sparse xcache hold the same weighted sums.
 *   pyvb_zstep_w_f64      pyvb_zstep_f64 with weights (algo generic or DMMA)
 *   pyvb_stats_w_f64      pyvb_stats_f64 with weights, mode B (no V / Xorig / qldX)
 *   pyvb_zstep_csr_w_f64, pyvb_stats_csr_w_f64   the CSR gathers with weights
 *   pyvb_global_w_f64     pyvb_global_f64 (nd = NULL) or pyvb_global_nd_f64 (nd != NULL) for weighted data: the X bound term
 *                         adds gl[PYVB_GL_LNS]; with nd, ncnt [D] (device) holds the NUMBER of observed entries of positive
 *                         weight of every column (global), which the per-dimension bound terms read in place of cnt_d.
 * pyvb_wupdate_f64 / pyvb_wupdate_nd_f64 / pyvb_pack_gw_*_f64 read only the statistics and the state: they serve both. */
int pyvb_zstep_w_f64(long long N, int D, int q, const double *X, long long ldx, const double *S, long long lds,
                     const double *Gw, int ldg, const double *P0, const double *h0, double *gl, double *Zbar, long long ldz,
                     double *M2, long long ldm, double *Sig, double *logdet, double *zsums, int algo, void *stream);
int pyvb_stats_w_f64(long long N, int D, int q, const double *X, long long ldx, const double *S, long long lds,
                     const double *Zbar, long long ldz, const double *M2, long long ldm, const double *logdet, double *stats,
                     void *ws, size_t ws_bytes, double *xcache, int xcache_valid, const double *zsums, int zsums_valid,
                     const pyvb_peers *peers /* host, nullable */, int algo, void *stream);
int pyvb_global_w_f64(int D, int q, int ops, int col_lo, int col_hi, const double *stats, const double *Wbar,
                      const double *Wvar, double *mu, double *muvar, double *gl, double *nd /* nullable */,
                      const double *ncnt /* nullable without nd */, const double *P0, const double *h0,
                      const pyvb_consts *consts /* host */, double *elbo_out, void *stream);

/* ---- row-wise W posterior (mode B, FP64, q in {8, 16, 32, 64}: the q of pyvb_zsolve_f64) ----
 * q(W) = prod_d N(w_d | wbar_d, Sigma_d), one full q x q covariance per data dimension, in place of the q column nodes with
 * diagonal covariances (pyvb_wupdate_f64).  The W step solves each row's block outright:
 *   Lambda_d = diag(<alpha>) + tau_d T1_d,   eta_d = tau_d (Ast_d - mu_d Bst_d),   Sigma_d = Lambda_d^-1,   wbar_d = Sigma_d eta_d
 * (tau_d = gl[PYVB_GL_TAU], or nd[PYVB_ND_TAU * D + d] with per-dimension noise; weighted statistics need nothing else).
 *   WM   [D][ldwm] scratch rows, ldwm = pyvb_mz_pitch(q), 16-byte aligned: the K2 row [Lambda_d packed | 0 | eta_d | 0] is
 *        assembled there and left as [<w_d w_d^T> packed | 0 | wbar_d | 0]
 *   Wcov [D][P]  packed Sigma_d (state: pyvb_pack_gw_rows_f64 and pyvb_global_rows_f64 read it)
 *   Wld  [D]     ln prod diag chol(Lambda_d) (= -1/2 ln det Sigma_d), the convention of the Z rows' logdet
 *   Wbar, Wvar [D][q]  wbar_d and diag Sigma_d (the ARD update and the bound's prior term read them)
 * A row whose Lambda_d is not positive definite is counted into gl[PYVB_GL_NONPD], as Z rows are.
 *   pyvb_wupdate_rows_f64   the W step above (every row; there is no column subset)
 *   pyvb_pack_gw_rows_f64   Gw rows with G_d = wbar_d wbar_d^T + Sigma_d (times tau_d with nd): every Z-step path reads them
 *   pyvb_global_rows_f64    pyvb_global_f64 / _nd_f64 / _w_f64 in one: nd and ncnt nullable as in pyvb_global_w_f64, weighted
 *                           != 0 adds gl[PYVB_GL_LNS] to the X term.  The residual contraction reads g = wbar_i wbar_j +
 *                           Sigma_d,ij; the W bound term keeps its prior part, sum_i [-D/2 ln 2pi + 1/2 ln det(alpha_i I) -
 *                           alpha_i/2 sum_d <w_di^2>], and takes the entropy of D row nodes with the reference's
 *                           q_ln_det = .5 / ln prod diag chol quirk per node: sum_d [q/2 ln 2pi + 1/2 (0.5 / Wld_d) + q/2]. */
int pyvb_wupdate_rows_f64(int D, int q, const double *stats, const double *mu, double *gl, const double *nd /* nullable */,
                          double *WM, int ldwm, double *Wbar, double *Wvar, double *Wcov, double *Wld, void *stream);
int pyvb_pack_gw_rows_f64(int D, int q, const double *Wbar, const double *Wcov, const double *mu,
                          const double *nd /* nullable */, double *Gw, int ldg, void *stream);
int pyvb_global_rows_f64(int D, int q, int ops, int col_lo, int col_hi, const double *stats, const double *Wbar,
                         const double *Wvar, const double *Wcov, const double *Wld, double *mu, double *muvar, double *gl,
                         double *nd /* nullable */, const double *ncnt /* nullable */, int weighted, const double *P0,
                         const double *h0, const pyvb_consts *consts /* host */, double *elbo_out, void *stream);

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
 * normalised data of BASELINE.json's configurations the bound sits at ~2^-50 and the guard never fires.
 * The digit planes are made from the packed G columns of Gw (which must be current), so Wbar / Wvar are not read. */
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
 * Same reference arithmetic as pyvb_zstep_f64's K1 (nodes/node.py:203-227).  D % 32 == 0; q in {16, 32, 64} for the
 * Z step (pyvb_f32_supported), q in {16, 32} for pyvb_stats_f32: it reads the column sums of the rows from K2's partials,
 * and K2 leaves none at q = 64 (pyvb_zsums_len_f32(N, 64) = 0).
 *   planes  bf16 [3][N][D]    mask | x_h | x_m  (x = x_h + x_m to 16 bits; zeros where not observed); static over sweeps
 *   GT      bf16 [3][NCP][D]  three-way split of [-mu_d <w_d> (q) | G_d packed (P) | pad]^T,  NCP = pyvb_f32_pitch(q)
 *   WT      bf16 [3][q][D]    three-way split of <W>^T
 *   MZ32    float [N][NCP]    out: [eta (q) | qprec packed (P) | pad]: the FP32 rows keep zbar / eta FIRST
 *                             (pyvb_f32_zoff(q) = 0, packed part at pyvb_f32_poff(q) = q) */
int pyvb_f32_pitch(int q);
int pyvb_f32_zoff(int q);
int pyvb_f32_poff(int q);
int pyvb_f32_supported(int D, int q);                 /* the Z step; the statistics also need q != 64 */
size_t pyvb_zsums_len_f32(long long N, int q);        /* K2 partials of the FP32 path (0 at q = 64) */
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
 * on X alone (xcache) and K2's column sums (zsums) must be valid: the FP32 path has no other source for them, hence
 * q in {16, 32} (PYVB_EINVAL at q = 64). */
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
/* the same with per-entry observation weights (see "per-entry observation weights" above): weights [nnz] in the order of
 * values, wts [nnz] in the order of vals; xcache then holds [sum s (D) | sum s x (D) | sum s x^2 | number of entries s > 0] */
int pyvb_zstep_csr_w_f64(long long N, int D, int q, const long long *indptr, const int *indices, const double *values,
                         const double *weights, const double *Gw, int ldg, const double *P0, const double *h0, double *gl,
                         double *MZ, long long ldmz, double *Sig, double *logdet, double *zsums, void *stream);
int pyvb_stats_csr_w_f64(long long N, int D, int q, int nblk, const long long *colptr, const int *rows, const double *vals,
                         const double *wts, const double *MZ, long long ldmz, const double *logdet, double *stats, void *ws,
                         size_t ws_bytes, const double *xcache, const double *zsums,
                         const pyvb_peers *peers /* host, nullable */, void *stream);

/* ---- known row covariates: known trailing latent dimensions (mode B, FP64, DESIGN.md 5f) ----
 * x_nd ~ N(w_d z_n + b_d c_n + mu_d, 1/tau) is the plate at q = q_free + k with z'_n = [z_n ; c_n] and W' = [W | B]: every
 * statistic, the W step, Mu, the Gammas and the bound run unchanged at q, with the priors P0' = blockdiag(P0, 0) and
 * h0' = [h0 ; 0].  Only the Z step changes: the Gaussian of z'_n conditioned on its known last k entries.
 *   C [N][ldc]   c_n, the k known entries of every row (ldc >= k); 1 <= k < q <= 64
 * pyvb_zknown_condition_f64: on MZ rows [qprec' packed | pad | eta'] (K1's output): eta_z -= qprec'_zc c, qprec'_zc = 0,
 *   qprec'_cc = I, eta'_c = c.  pyvb_zsolve_f64 then solves blockdiag(A_n, I): the free block is the conditioned posterior, the
 *   log-det is that of A_n (the identity pivots add ln 1 = 0).  Only the last k rows of the packed block and eta' are written.
 * pyvb_zknown_finish_f64: on K2's rows: <z'z'^T>_cc = c c^T and zbar'_c = c.  Only those entries are written.
 * The Z steps with covariates: K1 -> condition -> K2 -> finish on the DMMA path (S nullable: per-entry weights, as
 * pyvb_zstep_w_f64; algo PYVB_ALGO_GENERIC, or AUTO where the DMMA path does not run: the generic kernel with the
 * conditioning between its contraction and its factorisation, any q <= 64 and D), the INT8 path (K1-i8 -> condition -> K2 with the accuracy guard -> [K1-DMMA -> condition -> K2] as
 * conditional launches -> finish; gl[PYVB_GL_I8BAD] and gl[PYVB_GL_I8FALL] as pyvb_zstep_i8_f64) and the CSR path (weights
 * nullable).  The INT8 guard of a conditioned row compares against one scale, written to gmax [1] (device): the largest
 * fixed-point scale of the free columns of qprec', and of its zc columns times max(1, cmax), cmax >= max_n sum_j |c_nj| over
 * the rows of the call (the zc entries enter eta_z times c); the cc columns, which condition discards, do not count.
 * They leave no K2 partials: K2's column sums and maxima are wrong on the cc entries, so the statistics are called
 * with zsums = NULL and rebuild them from the finished rows.  Sig (nullable) receives Sigma'_n = blockdiag(Sigma_n, I). */
int pyvb_zknown_condition_f64(long long N, int q, int k, const double *C, long long ldc, double *MZ, long long ldmz,
                              void *stream);
int pyvb_zknown_finish_f64(long long N, int q, int k, const double *C, long long ldc, double *MZ, long long ldmz,
                           void *stream);
int pyvb_zstep_known_f64(long long N, int D, int q, int k, const double *C, long long ldc, const double *X, long long ldx,
                         const double *S /* nullable */, long long lds, const double *Gw, int ldg, const double *P0,
                         const double *h0, double *gl, double *MZ, long long ldmz, double *Sig, double *logdet, int algo,
                         void *stream);
int pyvb_zstep_i8_known_f64(long long N, int D, int q, int k, const double *C, long long ldc, double cmax, const double *X,
                            long long ldx, const void *mask, const double *Wbar, const double *Wvar, const double *Gw, int ldg,
                            const double *P0, const double *h0, double *gl, double *MZ, long long ldmz, void *GI,
                            double *gscale, double *gmax, double *Sig, double *logdet, void *stream);
int pyvb_zstep_csr_known_f64(long long N, int D, int q, int k, const double *C, long long ldc, const long long *indptr,
                             const int *indices, const double *values, const double *weights /* nullable */, const double *Gw,
                             int ldg, const double *P0, const double *h0, double *gl, double *MZ, long long ldmz, double *Sig,
                             double *logdet, void *stream);

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
