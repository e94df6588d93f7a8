// extern "C" boundary of libpyvb_b200.so -- see include/pyvb_b200.h for the contract.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "kernels.h"

using namespace pyvb;

static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, const char *detail) {
    snprintf(g_err, sizeof(g_err), fmt, detail);
    return code;
}
static int cuda_fail(cudaError_t e, const char *where) {
    snprintf(g_err, sizeof(g_err), "%s: %s", where, cudaGetErrorString(e));
    return PYVB_ECUDA;
}
#define ARG(cond, what)                                             \
    do {                                                            \
        if (!(cond)) return fail(PYVB_EINVAL, "bad argument: %s", what); \
    } while (0)

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

// Helper stream of the INT8 path: the FP64-tensor kernels on X (eta, Ast) are independent of the INT8 kernels on the mask and
// bound by different units, so they can run next to them (fork / join with two events around the pair).  Created on first
// use, one per device.  OFF unless PYVB_I8_OVERLAP=1: measured, the pairs do not overlap in practice (C2: 0.824 vs 0.838 ms for
// the K1 pair, the sweep unchanged) and the fork / join slows the chunked end-to-end path down.
struct AuxStream {
    cudaStream_t s = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
    int state = 0;   // 0 not tried, 1 ready, -1 unavailable
};
static AuxStream *aux_stream() {
    static AuxStream aux[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    AuxStream &a = aux[dev];
    if (a.state == 0) {
        const char *e = getenv("PYVB_I8_OVERLAP");
        a.state = -1;
        if ((e && e[0] == '1') && cudaStreamCreateWithFlags(&a.s, cudaStreamNonBlocking) == cudaSuccess &&
            cudaEventCreateWithFlags(&a.fork, cudaEventDisableTiming) == cudaSuccess &&
            cudaEventCreateWithFlags(&a.join, cudaEventDisableTiming) == cudaSuccess)
            a.state = 1;
    }
    return a.state == 1 ? &a : nullptr;
}

// Accuracy guard of the INT8 path (DESIGN.md 5a): relative accuracy (max norm, per row of qprec / per data dimension of T1)
// below which the fixed-point contraction is redone on the FP64 tensor cores.  PYVB_I8_GUARD=0 switches the guard off
// (measurement only), PYVB_I8_GUARD=force makes every call fall back (tests of the fall-back plumbing).
static const double I8_TOL = 3.637978807091713e-12;     // 2^-38
static int i8_guard_mode() {
    static int mode = -1;
    if (mode < 0) {
        const char *e = getenv("PYVB_I8_GUARD");
        mode = (e && e[0] == '0') ? 0 : (e && e[0] == 'f') ? 2 : 1;
    }
    return mode;
}

static int pick_algo(int algo, int D, int q) {
    if (algo == PYVB_ALGO_AUTO) return dmma_supported(D, q) ? PYVB_ALGO_DMMA : PYVB_ALGO_GENERIC;
    if (algo == PYVB_ALGO_DMMA_K1) return PYVB_ALGO_DMMA;
    return algo;
}

extern "C" {

int pyvb_version(void) { return 100; }
const char *pyvb_last_error(void) { return g_err; }

int pyvb_gw_pitch(int q) {
    // P + q + 1 used columns; pitch*8 bytes must be = 32 or 96 (mod 128) so that the four k-rows of a
    // DMMA B fragment fall into distinct shared-memory bank groups, and a multiple of 16 bytes for
    // bulk (TMA) copies.  => pitch = 4 (mod 8) ... choose the smallest such pitch >= P+q+1.
    const int used = gw_woff(q) + q + 1;
    int p = used;
    while ((p % 8) != 4) ++p;
    return p;
}

int pyvb_gw_woff(int q) { return gw_woff(q); }
int pyvb_mz_pitch(int q) { return pyvb_gw_pitch(q); }

size_t pyvb_stats_len(int D, int q) { return StatLayout(D, q).len; }

int pyvb_algo_supported(int algo, int D, int q) {
    if (q < 1 || q > PYVB_QMAX || D < 1) return 0;
    if (algo == PYVB_ALGO_GENERIC || algo == PYVB_ALGO_AUTO) return 1;
    if (algo == PYVB_ALGO_DMMA) return dmma_supported(D, q) ? 1 : 0;
    return 0;
}

size_t pyvb_stats_workspace_bytes(long long N, int D, int q, int algo) {
    const StatLayout L(D, q);
    if (N <= 0) return align256((L.len + PYVB_NSCAL) * sizeof(double));
    if (algo == PYVB_ALGO_F32) return align256((size_t)stats_f32_nchunks(N, D, q) * L.len * sizeof(double));
    int nch = stats_generic_nchunks(N);
    if (pick_algo(algo, D, q) == PYVB_ALGO_DMMA) {
        const int n2 = stats_dmma_nchunks(N, D, q);
        if (n2 > nch) nch = n2;
    }
    return align256((size_t)nch * L.len * sizeof(double)) +
           align256((size_t)rowscalars_nblk(N) * PYVB_NSCAL * sizeof(double));
}

size_t pyvb_zsums_len_f32(long long N, int q) {
    int nblk, kw;
    zsolve_partials_f32(N, q, nblk, kw);
    return (size_t)nblk * kw;
}

int pyvb_zsums_kw(int q) { return 2 * (gw_woff(q) + q) + PYVB_ZS_EXTRA; }

size_t pyvb_zsums_len(long long N, int q) {
    size_t len = 0;                                     // the largest over the K2 implementations (PYVB_K2 is read per call)
    for (int impl = 0; impl <= 5; ++impl) {
        int nblk, kw;
        zsolve_partials_of(impl, N, q, nblk, kw);
        if ((size_t)nblk * kw > len) len = (size_t)nblk * kw;
        // the Gauss-Jordan and blocked-sweep kernels run one CTA per SM at most, but how many rows a CTA takes depends on the
        // configuration picked by PYVB_GJ / PYVB_SWEEP, which is also read per call: size for the worst case
        if ((impl == 4 || impl == 5) && kw > 0) {
            const size_t worst = (size_t)(N < 148 ? (N < 1 ? 1 : N) : 148) * kw;
            if (worst > len) len = worst;
        }
    }
    return len;
}

int pyvb_zsums_blocks(long long N, int q) {
    int nblk, kw;
    zsolve_partials(N, q, nblk, kw);
    return nblk;
}

size_t pyvb_peer_bytes(size_t stats_len) { return peer_buffer_bytes(stats_len); }

int pyvb_peer_alloc(size_t bytes, void **dptr) {
    ARG(bytes > 0 && dptr, "bytes, dptr");
    cudaError_t e = cudaMalloc(dptr, bytes);
    if (e == cudaSuccess) e = cudaMemset(*dptr, 0, bytes);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "peer_alloc");
}
int pyvb_peer_free(void *dptr) {
    cudaError_t e = cudaFree(dptr);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "peer_free");
}
int pyvb_peer_export(void *dptr, unsigned char *handle64) {
    ARG(dptr && handle64, "null pointer");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, dptr);
    if (e != cudaSuccess) return cuda_fail(e, "peer_export");
    memcpy(handle64, &h, 64);
    return PYVB_OK;
}
int pyvb_peer_import(const unsigned char *handle64, void **dptr) {
    ARG(dptr && handle64, "null pointer");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    cudaError_t e = cudaIpcOpenMemHandle(dptr, h, cudaIpcMemLazyEnablePeerAccess);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "peer_import");
}
int pyvb_peer_close(void *dptr) {
    cudaError_t e = cudaIpcCloseMemHandle(dptr);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "peer_close");
}

int pyvb_pack_gw_f64(int D, int q, const double *Wbar, const double *Wvar, const double *mu, double *Gw, int ldg,
                     void *stream) {
    ARG(D >= 1 && q >= 1 && q <= PYVB_QMAX, "D, q");
    ARG(Wbar && Wvar && mu && Gw, "null pointer");
    ARG(ldg >= gw_woff(q) + q + 1, "ldg");
    cudaError_t e = launch_pack_gw(D, q, Wbar, Wvar, mu, Gw, ldg, (cudaStream_t)stream);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "pack_gw");
}

int pyvb_zstep_f64(long long N, int D, int q, const double *X, long long ldx, const double *Gw, int ldg,
                   const double *P0, const double *h0, double *gl, double *Zbar, long long ldz, double *M2,
                   long long ldm, double *Sig, double *logdet, double *zsums, int algo, void *stream) {
    ARG(N >= 0 && D >= 1 && q >= 1 && q <= PYVB_QMAX, "N, D, q");
    if (N == 0) return PYVB_OK;                      // an empty row block (e.g. an empty shard): nothing to update
    ARG(X && Gw && P0 && h0 && gl && Zbar && M2 && logdet, "null pointer");
    ARG(ldx >= D && ldz >= q && ldm >= q * (q + 1) / 2, "ldx, ldz, ldm");
    ARG(ldg >= gw_woff(q) + q + 1, "ldg");
    const int a = pick_algo(algo, D, q);
    cudaError_t e;
    if (a == PYVB_ALGO_DMMA) {
        if (!dmma_supported(D, q)) return fail(PYVB_ENOSUP, "%s", "DMMA path needs q in {8,16,32,64}, D % 16 == 0");
        ARG(ldg == pyvb_gw_pitch(q), "ldg must equal pyvb_gw_pitch(q) for the DMMA path");
        ARG((ldx % 2) == 0, "ldx must be even for the DMMA path");
        ARG(ldz == pyvb_mz_pitch(q) && ldm == ldz && Zbar == M2 + gw_woff(q),
            "the DMMA path needs the interleaved MZ layout (see pyvb_mz_pitch)");
        e = launch_zstep_dmma(N, D, q, X, ldx, Gw, ldg, P0, h0, gl, M2, Sig, logdet, zsums,
                              algo == PYVB_ALGO_DMMA_K1, (cudaStream_t)stream);
    } else if (a == PYVB_ALGO_GENERIC) {
        e = launch_zstep_generic(N, D, q, X, ldx, Gw, ldg, P0, h0, gl, Zbar, ldz, M2, ldm, Sig, logdet,
                                 (cudaStream_t)stream);
    } else {
        return fail(PYVB_EINVAL, "%s", "unknown algo");
    }
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "zstep");
}

int pyvb_zsolve_f64(long long N, int q, double *MZ, long long ldmz, double *Sig, double *logdet, double *gl,
                    double *zsums, void *stream) {
    ARG(N >= 0 && (q == 8 || q == 16 || q == 32 || q == 64), "N, q (8, 16, 32 or 64)");
    if (N == 0) return PYVB_OK;
    ARG(MZ && logdet && gl, "null pointer");
    ARG(ldmz == pyvb_mz_pitch(q), "ldmz must equal pyvb_mz_pitch(q)");
    cudaError_t e = launch_zsolve(N, q, MZ, Sig, logdet, gl, zsums, (cudaStream_t)stream);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "zsolve");
}

int pyvb_stats_f64(long long N, int D, int q, const double *X, long long ldx, const double *V,
                   const double *Xorig, const double *qldX, const double *Zbar, long long ldz, const double *M2,
                   long long ldm, const double *logdet, double *stats, void *ws, size_t ws_bytes, double *xcache,
                   int xcache_valid, const double *zsums, int zsums_valid, const pyvb_peers *peers, int algo,
                   void *stream) {
    ARG(N >= 0 && D >= 1 && q >= 1 && q <= PYVB_QMAX, "N, D, q");
    ARG(stats && ws, "null pointer");
    if (N == 0) {
        // an empty shard contributes zeros, but still takes part in the exchange
        ARG(ws_bytes >= (StatLayout(D, q).len + PYVB_NSCAL) * sizeof(double), "workspace too small");
        cudaError_t e0 = cudaMemsetAsync(ws, 0, (StatLayout(D, q).len + PYVB_NSCAL) * sizeof(double), (cudaStream_t)stream);
        if (e0 == cudaSuccess)
            e0 = launch_stats_reduce(D, q, (const double *)ws, 1, (const double *)ws + StatLayout(D, q).len, 1, stats,
                                     NULL, 0, NULL, 0, 0, peers ? peers->bufs : NULL, peers ? peers->world : 1,
                                     peers ? peers->rank : 0, peers ? peers->epoch : 0ULL, (cudaStream_t)stream);
        return e0 == cudaSuccess ? PYVB_OK : cuda_fail(e0, "stats (empty shard)");
    }
    ARG(X && Zbar && M2 && logdet, "null pointer");
    ARG(ldx >= D && ldz >= q && ldm >= q * (q + 1) / 2, "ldx, ldz, ldm");
    ARG((Xorig == NULL) || (V != NULL && qldX != NULL), "mode A needs V and qldX with Xorig");
    ARG(ws_bytes >= pyvb_stats_workspace_bytes(N, D, q, algo), "workspace too small");
    ARG(peers == NULL || (peers->bufs != NULL && peers->world >= 1 && peers->rank >= 0 && peers->rank < peers->world &&
                          peers->world <= 256 && peers->epoch >= 1),
        "peers");
    const StatLayout L(D, q);
    const int a = pick_algo(algo, D, q);
    cudaStream_t st = (cudaStream_t)stream;
    int nch, use_x = 0, nzblk = 0, zkw = 0;
    cudaError_t e;
    double *ws_main = (double *)ws;
    if (a == PYVB_ALGO_DMMA) {
        if (!dmma_supported(D, q)) return fail(PYVB_ENOSUP, "%s", "DMMA path needs q in {8,16,32,64}, D % 16 == 0");
        ARG((ldx % 2) == 0, "ldx must be even for the DMMA path");
        ARG(ldz == pyvb_mz_pitch(q) && ldm == ldz && Zbar == M2 + gw_woff(q),
            "the DMMA path needs the interleaved MZ layout (see pyvb_mz_pitch)");
        nch = stats_dmma_nchunks(N, D, q);
        use_x = (xcache != NULL && xcache_valid) ? 1 : 0;
        if (zsums != NULL && zsums_valid) zsolve_partials(N, q, nzblk, zkw);
        e = launch_stats_dmma(N, D, q, X, ldx, M2, ws_main, nch, st);
        if (e == cudaSuccess && nzblk == 0) e = launch_mzsums(N, D, q, Zbar, ldz, M2, ldm, ws_main, nch, st);
        if (e == cudaSuccess && !use_x) e = launch_colsums(N, D, q, X, ldx, ws_main, nch, st);
    } else if (a == PYVB_ALGO_GENERIC) {
        nch = stats_generic_nchunks(N);
        e = launch_stats_generic(N, D, q, X, ldx, Zbar, ldz, M2, ldm, ws_main, nch, st);
    } else {
        return fail(PYVB_EINVAL, "%s", "unknown algo");
    }
    if (e != cudaSuccess) return cuda_fail(e, "stats");
    double *ws_sc = (double *)((char *)ws + align256((size_t)nch * L.len * sizeof(double)));
    const int nblk = rowscalars_nblk(N);
    // mode B with cached X sums and K2's partials: nothing is left for the per-row scalar pass
    const int need_rows = !(use_x && Xorig == NULL && nzblk > 0);
    if (need_rows) {
        e = launch_rowscalars(N, D, X, ldx, V, Xorig, qldX, logdet, ws_sc, nblk, use_x && Xorig == NULL, st);
        if (e != cudaSuccess) return cuda_fail(e, "rowscalars");
    }
    e = launch_stats_reduce(D, q, ws_main, nch, need_rows ? ws_sc : NULL, nblk, stats, xcache, use_x,
                            nzblk > 0 ? zsums : NULL, nzblk, zkw, peers ? peers->bufs : NULL, peers ? peers->world : 1,
                            peers ? peers->rank : 0, peers ? peers->epoch : 0ULL, st);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "stats_reduce");
}

int pyvb_wupdate_f64(int D, int q, int col_lo, int col_hi, const double *stats, const double *mu, const double *gl,
                     double *Wbar, double *Wvar, void *stream) {
    ARG(D >= 1 && q >= 1 && q <= PYVB_QMAX, "D, q");
    ARG(0 <= col_lo && col_lo <= col_hi && col_hi <= q, "column range");
    ARG(stats && mu && gl && Wbar && Wvar, "null pointer");
    cudaError_t e = launch_wupdate(D, q, col_lo, col_hi, stats, mu, gl, Wbar, Wvar, (cudaStream_t)stream);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "wupdate");
}

int pyvb_global_f64(int D, int q, int ops, int col_lo, int col_hi, const double *stats, const double *Wbar, const double *Wvar, double *mu,
                    double *muvar, double *gl, const double *P0, const double *h0, const pyvb_consts *consts,
                    double *elbo_out, void *stream) {
    ARG(D >= 1 && q >= 1 && q <= PYVB_QMAX, "D, q");
    ARG(stats && Wbar && Wvar && mu && muvar && gl && P0 && h0 && consts, "null pointer");
    ARG(0 <= col_lo && col_lo <= col_hi && col_hi <= q, "column range");
    cudaError_t e =
        launch_global(D, q, ops, col_lo, col_hi, stats, Wbar, Wvar, mu, muvar, gl, P0, h0, *consts, elbo_out, (cudaStream_t)stream);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "global");
}

int pyvb_impute_f64(long long N, int D, int q, const double *Xorig, long long ldx, const double *Wbar,
                    const double *mu, const double *Zbar, long long ldz, const double *gl, double *Xhat, double *V,
                    double *qldX, void *stream) {
    ARG(N >= 0 && D >= 1 && q >= 1 && q <= PYVB_QMAX, "N, D, q");
    if (N == 0) return PYVB_OK;
    ARG(Xorig && Wbar && mu && Zbar && gl && Xhat && V && qldX, "null pointer");
    ARG(ldx >= D && ldz >= q, "ldx, ldz");
    cudaError_t e =
        launch_impute(N, D, q, Xorig, ldx, Wbar, mu, Zbar, ldz, gl, Xhat, V, qldX, (cudaStream_t)stream);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "impute");
}

int pyvb_i8_supported(int D, int q) { return (i8_supported(D, q) && dmma_supported(D, q)) ? 1 : 0; }
// digit planes of G, then (256-byte aligned) the compact [wbar | mu] array of the eta kernel
size_t pyvb_i8_digits_bytes(int D, int q) {
    return align256(i8_digits_bytes(D, q)) + align256((size_t)D * zstep_eta_pitch(q) * sizeof(double));
}
int pyvb_i8_ncols(int q) { return i8_ncols(q); }
size_t pyvb_i8_mask_bytes(long long N, int D) { return i8_mask_bytes(N, D); }

int pyvb_prepare_mask_i8(long long N, int D, const double *X, long long ldx, void *mask, void *stream) {
    ARG(N >= 0 && D >= 4 && (D % 4) == 0 && ldx >= D && (ldx % 2) == 0, "N, D (% 4), ldx (even)");
    if (N == 0) return PYVB_OK;
    ARG(X && mask, "null pointer");
    cudaError_t e = launch_prepare_mask_i8(N, D, X, ldx, mask, (cudaStream_t)stream);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "prepare_mask_i8");
}

int pyvb_zstep_i8_f64(long long N, int D, int q, const double *X, long long ldx, const void *mask, const double *Wbar,
                      const double *Wvar, const double *Gw, int ldg, const double *P0, const double *h0, double *gl,
                      double *MZ, long long ldmz, void *GI, double *gscale, double *Sig, double *logdet, double *zsums,
                      int k1_only, void *stream) {
    ARG(N >= 0 && D >= 1 && q >= 1 && q <= PYVB_QMAX, "N, D, q");
    if (!pyvb_i8_supported(D, q))
        return fail(PYVB_ENOSUP, "%s", "the INT8 path needs q in {16, 32, 64}, D % 64 == 0 and a mask block that fits shared memory");
    if (N == 0) return PYVB_OK;
    ARG(X && mask && Wbar && Wvar && Gw && P0 && h0 && gl && MZ && GI && gscale && logdet, "null pointer");
    ARG(ldx >= D && (ldx % 2) == 0, "ldx");
    ARG(ldg == pyvb_gw_pitch(q) && ldmz == pyvb_mz_pitch(q), "ldg / ldmz must equal pyvb_gw_pitch(q) / pyvb_mz_pitch(q)");
    cudaStream_t st = (cudaStream_t)stream;
    // k1_only: 0 whole Z step, 1 contraction only (INT8 qprec + DMMA eta), 2 INT8 part only, 3 eta part only
    cudaError_t e = cudaSuccess;
    AuxStream *aux = (k1_only < 2) ? aux_stream() : nullptr;     // both parts wanted: the eta kernel runs next to the INT8 kernel
    cudaStream_t st2 = st;
    if (aux) {
        e = cudaEventRecord(aux->fork, st);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(aux->s, aux->fork, 0);
        if (e != cudaSuccess) return cuda_fail(e, "zstep_i8 (fork)");
        st2 = aux->s;
    }
    if (k1_only != 3) {      // first: its CTAs take one slot per SM, the eta kernel's CTAs fill what is left
        e = launch_pack_g_i8(D, q, Wbar, Wvar, GI, gscale, gl, st);
        if (e == cudaSuccess) e = launch_zstep_i8(N, D, q, mask, GI, P0, gscale, gl, MZ, (int)ldmz, st);
    }
    if (e == cudaSuccess && k1_only != 2) {
        double *weta = (double *)((char *)GI + align256(i8_digits_bytes(D, q)));
        e = launch_zstep_eta_dmma(N, D, q, X, ldx, Gw, weta, P0, h0, gl, MZ, st2);
    }
    if (aux) {
        cudaError_t e2 = cudaEventRecord(aux->join, aux->s);
        if (e2 == cudaSuccess) e2 = cudaStreamWaitEvent(st, aux->join, 0);
        if (e == cudaSuccess) e = e2;
    }
    if (e == cudaSuccess && !k1_only) {
        // K2 checks every finished qprec row against the fixed-point bound of K1-i8 (kernels.h: I8Check); when a row fails,
        // the whole step is redone on the FP64 tensor cores by two conditional launches that exit at once otherwise
        const int guard = (k2_impl(q) == 0) ? 0 : i8_guard_mode();
        I8Check chk;
        if (guard) {
            chk.gscale = gscale;
            chk.ncols = q * (q + 1) / 2;
            chk.fac = (guard == 2) ? 1e300 : (double)D * 2.7755575615628914e-17 / I8_TOL;     // D * 2^-55 / tol
        }
        e = launch_zsolve(N, q, MZ, Sig, logdet, gl, zsums, st, nullptr, chk);
        if (e == cudaSuccess && guard)
            e = launch_zstep_dmma(N, D, q, X, ldx, Gw, ldg, P0, h0, gl, MZ, Sig, logdet, zsums, 0, st, gl + PYVB_GL_I8BAD);
    }
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "zstep_i8");
}

int pyvb_stats_i8_supported(int D, int q) { return (stats_i8_supported(D, q) && dmma_supported(D, q)) ? 1 : 0; }
long long pyvb_stats_i8_npad(long long N) { return stats_i8_npad(N); }
size_t pyvb_stats_i8_digits_bytes(long long N, int q) { return stats_i8_digits_bytes(N, q); }
int pyvb_stats_i8_fused(int D, int q) { return (pyvb_stats_i8_supported(D, q) && stats_i8_fused(D)) ? 1 : 0; }
size_t pyvb_stats_i8_maskt_bytes(long long N, int D) { return stats_i8_maskt_bytes(N, D); }
size_t pyvb_stats_i8_scratch_len(int q) { return stats_i8_scratch_len(q, pyvb_mz_pitch(q)); }
size_t pyvb_stats_i8_guard_offset(int q) {
    return (size_t)(stats_i8_guard((double *)0, q, pyvb_mz_pitch(q)) - (double *)0);
}
size_t pyvb_stats_i8_workspace_bytes(long long N, int D, int q) {
    const StatLayout L(D, q);
    if (N <= 0) return align256((L.len + PYVB_NSCAL) * sizeof(double));
    return align256((size_t)stats_i8_nchunks(N, D, q) * L.len * sizeof(double)) +
           align256((size_t)rowscalars_nblk(N) * PYVB_NSCAL * sizeof(double));
}

int pyvb_prepare_maskt_i8(long long N, int D, const double *X, long long ldx, void *maskT, void *stream) {
    ARG(N >= 0 && D >= 1 && ldx >= D, "N, D, ldx");
    if (N == 0) return PYVB_OK;
    ARG(X && maskT, "null pointer");
    cudaError_t e = launch_prepare_maskT_i8(N, D, X, ldx, maskT, (cudaStream_t)stream);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "prepare_maskT_i8");
}

int pyvb_stats_i8_f64(long long N, int D, int q, const double *X, long long ldx, const void *maskT, const double *MZ,
                      long long ldmz, const double *logdet, void *ZI, double *scratch, double *stats, void *ws,
                      size_t ws_bytes, const double *xcache, const double *zsums, const pyvb_peers *peers, void *stream) {
    ARG(N >= 0 && D >= 1 && q >= 1 && q <= PYVB_QMAX, "N, D, q");
    if (!pyvb_stats_i8_supported(D, q)) return fail(PYVB_ENOSUP, "%s", "the INT8 statistics need q in {16, 32, 64}, D % 16 == 0");
    ARG(stats && ws, "null pointer");
    ARG(peers == NULL || (peers->bufs != NULL && peers->world >= 1 && peers->rank >= 0 && peers->rank < peers->world &&
                          peers->world <= 256 && peers->epoch >= 1),
        "peers");
    cudaStream_t st = (cudaStream_t)stream;
    const StatLayout L(D, q);
    if (N == 0) {
        ARG(ws_bytes >= (L.len + PYVB_NSCAL) * sizeof(double), "workspace too small");
        cudaError_t e0 = cudaMemsetAsync(ws, 0, (L.len + PYVB_NSCAL) * sizeof(double), st);
        if (e0 == cudaSuccess)
            e0 = launch_stats_reduce(D, q, (const double *)ws, 1, (const double *)ws + L.len, 1, stats, NULL, 0, NULL, 0, 0,
                                     peers ? peers->bufs : NULL, peers ? peers->world : 1, peers ? peers->rank : 0,
                                     peers ? peers->epoch : 0ULL, st);
        return e0 == cudaSuccess ? PYVB_OK : cuda_fail(e0, "stats_i8 (empty shard)");
    }
    ARG(X && maskT && MZ && scratch && xcache, "null pointer (xcache is required)");
    ARG(ZI || stats_i8_fused(D), "ZI is required where pyvb_stats_i8_fused(D, q) is 0");
    ARG(zsums || logdet, "zsums or logdet");
    ARG(logdet || k2_impl(q) >= 1, "logdet is needed when the K2 partials carry no column maxima");
    ARG(ldx >= D && (ldx % 2) == 0 && ldmz == pyvb_mz_pitch(q), "ldx, ldmz");
    ARG(ws_bytes >= pyvb_stats_i8_workspace_bytes(N, D, q), "workspace too small");
    int nzblk = 0, zkw = 0;
    if (zsums) zsolve_partials(N, q, nzblk, zkw);
    const int nch = stats_i8_nchunks(N, D, q);
    // the default K2 kernels leave bounds on the column maxima behind their column sums: [sums OROW | 4 | maxima OROW]
    const bool kmax = nzblk > 0 && k2_impl(q) >= 1;
    AuxStream *aux = aux_stream();                              // Ast (FP64 tensor cores on X) next to digitize + the INT8 kernel
    cudaStream_t st2 = st;
    cudaError_t e = cudaSuccess;
    if (aux) {
        e = cudaEventRecord(aux->fork, st);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(aux->s, aux->fork, 0);
        if (e != cudaSuccess) return cuda_fail(e, "stats_i8 (fork)");
        st2 = aux->s;
    }
    // K2's partials when they carry the maxima, else one pass over the MZ rows builds the same partials in `scratch`
    const double *zs = NULL;
    int zn = 0, zk = 0;
    e = launch_stats_i8(N, D, q, maskT, MZ, (int)ldmz, ZI, scratch, (double *)ws, nch, zsums, nzblk, zkw, kmax ? 1 : 0, logdet,
                        &zs, &zn, &zk, st);
    if (e == cudaSuccess) e = launch_stats_x_dmma(N, D, q, X, ldx, MZ, (double *)ws, nch, st2);
    if (aux) {
        cudaError_t e2 = cudaEventRecord(aux->join, aux->s);
        if (e2 == cudaSuccess) e2 = cudaStreamWaitEvent(st, aux->join, 0);
        if (e == cudaSuccess) e = e2;
    }
    if (e != cudaSuccess) return cuda_fail(e, "stats_i8");
    if (i8_guard_mode()) {
        // the same guard for T1 / Bst: a data dimension whose sums are not accurate to I8_TOL sends the whole pass to the
        // FP64 tensor cores (one conditional launch that exits at once otherwise); both before the exchange
        double *guard = stats_i8_guard(scratch, q, (int)ldmz);
        e = launch_stats_i8_check(D, q, (const double *)ws, nch, xcache, scratch, (int)ldmz,
                                  i8_guard_mode() == 2 ? 0.0 : I8_TOL, st);      // (tol = 0: every observed dimension fails)
        if (e == cudaSuccess) e = launch_stats_dmma(N, D, q, X, ldx, MZ, (double *)ws, nch, st, guard);
        if (e != cudaSuccess) return cuda_fail(e, "stats_i8 (guard)");
    }
    e = launch_stats_reduce(D, q, (const double *)ws, nch, NULL, 0, stats, const_cast<double *>(xcache), 1, zs, zn, zk,
                            peers ? peers->bufs : NULL, peers ? peers->world : 1, peers ? peers->rank : 0,
                            peers ? peers->epoch : 0ULL, st);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "stats_reduce");
}

int pyvb_csr_supported(int D, int q) { return (D >= 1 && csr_supported(q)) ? 1 : 0; }
int pyvb_csr_stats_blocks(long long N, int D, int q) { return csr_stats_nblocks(N, D, q); }
long long pyvb_csr_block_rows(long long N, int D, int q) { return csr_block_rows(N, D, q); }
size_t pyvb_stats_csr_workspace_bytes(long long N, int D, int q, int nblk) {
    const StatLayout L(D, q);
    if (N <= 0) return align256((L.len + PYVB_NSCAL) * sizeof(double));
    return align256((size_t)(nblk < 1 ? 1 : nblk) * L.len * sizeof(double)) +
           align256((size_t)rowscalars_nblk(N) * PYVB_NSCAL * sizeof(double));
}

int pyvb_zstep_csr_f64(long long N, int D, int q, const long long *indptr, const int *indices, const double *values,
                       const double *Gw, int ldg, const double *P0, const double *h0, double *gl, double *MZ,
                       long long ldmz, double *Sig, double *logdet, double *zsums, void *stream) {
    ARG(N >= 0 && D >= 1, "N, D");
    if (!csr_supported(q)) return fail(PYVB_ENOSUP, "%s", "the CSR path needs q in {8, 16, 32, 64}");
    if (N == 0) return PYVB_OK;
    ARG(indptr && indices && values && Gw && P0 && h0 && gl && MZ && logdet, "null pointer");
    ARG(ldg == pyvb_gw_pitch(q) && ldmz == pyvb_mz_pitch(q), "ldg / ldmz must equal pyvb_gw_pitch(q) / pyvb_mz_pitch(q)");
    ARG((reinterpret_cast<uintptr_t>(Gw) & 15) == 0 && (reinterpret_cast<uintptr_t>(MZ) & 15) == 0,
        "Gw and MZ must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = launch_zstep_csr(N, q, indptr, indices, values, Gw, ldg, P0, h0, gl, MZ, (int)ldmz, st);
    if (e == cudaSuccess) e = launch_zsolve(N, q, MZ, Sig, logdet, gl, zsums, st);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "zstep_csr");
}

int pyvb_stats_csr_f64(long long N, int D, int q, int nblk, const long long *colptr, const int *rows, const double *vals,
                       const double *MZ, long long ldmz, const double *logdet, double *stats, void *ws, size_t ws_bytes,
                       const double *xcache, const double *zsums, const pyvb_peers *peers, void *stream) {
    ARG(N >= 0 && D >= 1, "N, D");
    if (!csr_supported(q)) return fail(PYVB_ENOSUP, "%s", "the CSR path needs q in {8, 16, 32, 64}");
    ARG(stats && ws, "null pointer");
    ARG(peers == NULL || (peers->bufs != NULL && peers->world >= 1 && peers->rank >= 0 && peers->rank < peers->world &&
                          peers->world <= 256 && peers->epoch >= 1),
        "peers");
    const StatLayout L(D, q);
    cudaStream_t st = (cudaStream_t)stream;
    if (N == 0) {
        // an empty shard contributes zeros, but still takes part in the exchange
        ARG(ws_bytes >= (L.len + PYVB_NSCAL) * sizeof(double), "workspace too small");
        cudaError_t e0 = cudaMemsetAsync(ws, 0, (L.len + PYVB_NSCAL) * sizeof(double), st);
        if (e0 == cudaSuccess)
            e0 = launch_stats_reduce(D, q, (const double *)ws, 1, (const double *)ws + L.len, 1, stats, NULL, 0, NULL, 0, 0,
                                     peers ? peers->bufs : NULL, peers ? peers->world : 1, peers ? peers->rank : 0,
                                     peers ? peers->epoch : 0ULL, st);
        return e0 == cudaSuccess ? PYVB_OK : cuda_fail(e0, "stats_csr (empty shard)");
    }
    ARG(nblk >= 1 && colptr && rows && vals && MZ && xcache, "nblk, null pointer (xcache is required)");
    ARG(zsums || logdet, "zsums or logdet");
    ARG(ldmz == pyvb_mz_pitch(q) && (reinterpret_cast<uintptr_t>(MZ) & 15) == 0, "ldmz must equal pyvb_mz_pitch(q), MZ 16-byte aligned");
    ARG(ws_bytes >= pyvb_stats_csr_workspace_bytes(N, D, q, nblk), "workspace too small");
    double *ws_main = (double *)ws;
    cudaError_t e = launch_stats_csc(D, q, nblk, colptr, rows, vals, MZ, (int)ldmz, ws_main, st);
    if (e != cudaSuccess) return cuda_fail(e, "stats_csr");
    int nzblk = 0, zkw = 0;
    if (zsums) zsolve_partials(N, q, nzblk, zkw);
    // without K2's partials: S, zsum from one pass over the MZ rows, the log-det scalars from the per-row pass (which reads
    // no X with skip_x set)
    double *ws_sc = NULL;
    const int nsc = rowscalars_nblk(N);
    if (nzblk == 0) {
        ws_sc = (double *)((char *)ws + align256((size_t)nblk * L.len * sizeof(double)));
        const int gz = gw_woff(q);
        e = launch_mzsums(N, D, q, MZ + gz, ldmz, MZ, ldmz, ws_main, nblk, st);
        if (e == cudaSuccess) e = launch_rowscalars(N, D, NULL, D, NULL, NULL, NULL, logdet, ws_sc, nsc, 1, st);
        if (e != cudaSuccess) return cuda_fail(e, "stats_csr (row sums)");
    }
    e = launch_stats_reduce(D, q, ws_main, nblk, ws_sc, nsc, stats, const_cast<double *>(xcache), 1,
                            nzblk > 0 ? zsums : NULL, nzblk, zkw, peers ? peers->bufs : NULL, peers ? peers->world : 1,
                            peers ? peers->rank : 0, peers ? peers->epoch : 0ULL, st);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "stats_reduce");
}

int pyvb_f32_pitch(int q) { return f32_ncp(q); }
int pyvb_f32_zoff(int q) { return f32_zoff(q); }
int pyvb_f32_poff(int q) { return f32_poff(q); }
int pyvb_f32_supported(int D, int q) { return f32_supported(D, q) ? 1 : 0; }

int pyvb_prepare_x_f32(long long N, int D, const double *X, long long ldx, void *planes, void *stream) {
    ARG(N >= 0 && D >= 1 && ldx >= D, "N, D, ldx");
    if (N == 0) return PYVB_OK;
    ARG(X && planes, "null pointer");
    cudaError_t e = launch_prepare_x_f32(N, D, X, ldx, planes, (cudaStream_t)stream);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "prepare_x_f32");
}

int pyvb_pack_gw_f32(int D, int q, const double *Wbar, const double *Wvar, const double *mu, void *GT, void *WT,
                     void *stream) {
    ARG(f32_supported(D, q), "the FP32 path needs q in {16, 32, 64} and D % 32 == 0");
    ARG(Wbar && Wvar && mu && GT && WT, "null pointer");
    cudaError_t e = launch_pack_gw_f32(D, q, Wbar, Wvar, mu, GT, WT, (cudaStream_t)stream);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "pack_gw_f32");
}

int pyvb_zstep_k1_f32(long long N, int D, int q, const void *planes, const void *GT, const void *WT, const double *P0,
                      const double *h0, const double *gl, float *MZ32, void *stream) {
    ARG(N >= 0 && f32_supported(D, q), "the FP32 path needs q in {16, 32, 64} and D % 32 == 0");
    ARG(planes && GT && WT && P0 && h0 && gl && MZ32, "null pointer");
    cudaError_t e = launch_zstep_f32(N, N, D, q, planes, GT, WT, P0, h0, gl, MZ32, (cudaStream_t)stream);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "zstep_k1_f32");
}

int pyvb_zstep_f32(long long N, long long nalloc, int D, int q, const void *planes, const void *GT, const void *WT,
                   const double *P0, const double *h0, double *gl, float *MZ32, void *MP, double *Sig, double *logdet,
                   double *zsums, void *stream) {
    ARG(N >= 0 && nalloc >= N && f32_supported(D, q), "the FP32 path needs q in {16, 32, 64} and D % 32 == 0");
    if (N == 0) return PYVB_OK;
    ARG(planes && GT && WT && P0 && h0 && gl && MZ32 && MP && logdet, "null pointer");
    cudaError_t e = launch_zstep_f32(N, nalloc, D, q, planes, GT, WT, P0, h0, gl, MZ32, (cudaStream_t)stream);
    if (e == cudaSuccess) e = launch_zsolve_f32(N, q, MZ32, MP, Sig, logdet, gl, zsums, (cudaStream_t)stream);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "zstep_f32");
}

int pyvb_stats_f32(long long N, long long nalloc, int D, int q, const void *planes, const void *MP, double *stats,
                   void *ws, size_t ws_bytes, double *xcache, const double *zsums, const pyvb_peers *peers,
                   void *stream) {
    ARG(N >= 0 && nalloc >= N && f32_supported(D, q), "the FP32 path needs q in {16, 32, 64} and D % 32 == 0");
    ARG(stats && ws, "null pointer");
    if (N == 0) {
        ARG(ws_bytes >= (StatLayout(D, q).len + PYVB_NSCAL) * sizeof(double), "workspace too small");
        cudaError_t e0 = cudaMemsetAsync(ws, 0, (StatLayout(D, q).len + PYVB_NSCAL) * sizeof(double), (cudaStream_t)stream);
        if (e0 == cudaSuccess)
            e0 = launch_stats_reduce(D, q, (const double *)ws, 1, (const double *)ws + StatLayout(D, q).len, 1, stats,
                                     NULL, 0, NULL, 0, 0, peers ? peers->bufs : NULL, peers ? peers->world : 1,
                                     peers ? peers->rank : 0, peers ? peers->epoch : 0ULL, (cudaStream_t)stream);
        return e0 == cudaSuccess ? PYVB_OK : cuda_fail(e0, "stats_f32 (empty shard)");
    }
    ARG(planes && MP && xcache && zsums, "null pointer (xcache and zsums are required)");
    ARG(ws_bytes >= pyvb_stats_workspace_bytes(N, D, q, PYVB_ALGO_F32), "workspace too small");
    ARG(peers == NULL || (peers->bufs != NULL && peers->world >= 1 && peers->rank >= 0 && peers->rank < peers->world &&
                          peers->world <= 256 && peers->epoch >= 1),
        "peers");
    int nzblk = 0, zkw = 0;
    zsolve_partials_f32(N, q, nzblk, zkw);
    ARG(nzblk > 0, "no K2 column sums for this q in the FP32 path");
    const int nch = stats_f32_nchunks(N, D, q);
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = launch_stats_f32(N, nalloc, D, q, planes, MP, (double *)ws, nch, st);
    if (e != cudaSuccess) return cuda_fail(e, "stats_f32");
    e = launch_stats_reduce(D, q, (const double *)ws, nch, NULL, 0, stats, xcache, 1, zsums, nzblk, zkw,
                            peers ? peers->bufs : NULL, peers ? peers->world : 1, peers ? peers->rank : 0,
                            peers ? peers->epoch : 0ULL, st);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "stats_reduce");
}

int pyvb_lds_max_len(void) {
    int T = 16;
    while (lds_smem_bytes(T + 1, 8) <= 227 * 1024) ++T;
    return T;
}

int pyvb_lds_iterate_f64(int B, int T, int q, int d, const double *Y, double *X, double *Xcov3, double *A, double *Avar,
                         double *C, double *Cvar, double *Qa, double *Qb, double *Ra, double *Rb, double alpha0,
                         double a0, double b0, int niters, double *status, void *stream) {
    ARG(B >= 0 && q >= 1 && q <= 8 && d >= 1 && d <= 8 && niters >= 0, "B, q (<= 8), d (<= 8), niters");
    ARG(T >= 3 && T <= pyvb_lds_max_len(), "T (3 .. pyvb_lds_max_len())");
    if (B == 0) return PYVB_OK;
    ARG(Y && X && Xcov3 && A && Avar && C && Cvar && Qa && Qb && Ra && Rb && status, "null pointer");
    cudaError_t e = launch_lds_iterate(B, T, q, d, Y, X, Xcov3, A, Avar, C, Cvar, Qa, Qb, Ra, Rb, alpha0, a0, b0, niters,
                                       status, (cudaStream_t)stream);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "lds_iterate");
}

int pyvb_lds_iterate_known_f64(int B, int T, int q, int d, const double *Y, double *X, double *Xcov3, double *A, double *Avar,
                               double *C, double *Cvar, double *Qa, double *Qb, double *Ra, double *Rb, const double *Aknown,
                               double alpha0, double a0, double b0, int niters, double *status, void *stream) {
    ARG(B >= 0 && q >= 1 && q <= 8 && d >= 1 && d <= 8 && niters >= 0, "B, q (<= 8), d (<= 8), niters");
    ARG(T >= 3 && T <= pyvb_lds_max_len(), "T (3 .. pyvb_lds_max_len())");
    if (B == 0) return PYVB_OK;
    ARG(Y && X && Xcov3 && A && Avar && C && Cvar && Qa && Qb && Ra && Rb && status, "null pointer");
    cudaError_t e = launch_lds_iterate(B, T, q, d, Y, X, Xcov3, A, Avar, C, Cvar, Qa, Qb, Ra, Rb, alpha0, a0, b0, niters,
                                       status, (cudaStream_t)stream, Aknown);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "lds_iterate");
}

int pyvb_bench_umma(int blocks, int iters, int n, int kind, int mode, const void *src, long long *clk_out, void *stream) {
    ARG(blocks >= 1 && blocks <= 148 && iters >= 1 && n >= 16 && n <= 256 && (n % 16) == 0 && (kind == 0 || kind == 1) && clk_out,
        "arguments");
    ARG(!(mode & 4) || src, "mode 4 needs a source buffer of blocks MiB");
    cudaError_t e = launch_bench_umma(blocks, iters, n, kind, mode, src, clk_out, (cudaStream_t)stream);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "bench_umma");
}

int pyvb_bench_dmma_f64(int blocks, int iters, double *scratch, void *stream) {
    ARG(blocks >= 1 && iters >= 1 && scratch, "blocks, iters, scratch");
    cudaError_t e = launch_bench_dmma(blocks, iters, scratch, (cudaStream_t)stream);
    return e == cudaSuccess ? PYVB_OK : cuda_fail(e, "bench_dmma");
}

}  // extern "C"
