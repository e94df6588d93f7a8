// K2 at q = 64 as a BLOCKED symmetric sweep: 8 x 8 pivot tiles factored by scalar elimination, everything else on the FP64 tensor
// cores, in place in shared memory on a tile-swizzled copy of the packed rows.
//
// Replaces cho_factor / cho_solve(., I) / dot(qcov, .) / q_ln_det of Gaussian.update (nodes/gaussian.py:117-123).
//
// The Gauss-Jordan kernel (kernels_k2g.cu) is FP64-ISSUE bound: q^3 DFMA per matrix, one issue slot per 32 of them, and half of
// them redundant (it cannot use the symmetry).  Here the matrix is swept 8 pivots (one tile column K) at a time with the
// symmetric sweep operator
//
//   M_KK <- -inv(M_KK),    M_IK <- M_IK inv(M_KK),    M_IJ <- M_IJ - M_IK inv(M_KK) M_KJ     (I, J != K),
//
// which keeps the state symmetric, so that only the lower tiles exist, every intermediate overwrites the tile it replaces, and
// after q / 8 sweeps the tiles hold -Sigma.  inv(M_KK) is only ever applied in FACTORED form, M_KK = L D L^T, X = L^-1:
//
//   pivot   the 8 x 8 pivot tiles of the warp's MPW matrices together, lane (m, r) = row r of matrix m's tile: elimination without
//           pivoting on [M_KK | I] gives D and X (one published column entry per lane and pivot, the pivot lane's row of X);
//   panel   W_J = old_J X^T  and the new panel  M_JK <- (W_J D^-1) X;   pivot tile  M_KK <- -X^T D^-1 X;
//   update  M_IJ -= (W_I D^-1) W_J^T  for the lower tiles outside row / column K
//
// -- all DMMA.8x8x4 (256 FMA per issue slot).  This is block Cholesky (||W D^-1/2||^2 <= ||M||): as stable as the unblocked
// elimination.  (The first version applied the explicit inverse of the pivot tile, T_J = old_J inv(M_KK), M_IJ -= T_I old_J^T:
// block LU, 4 - 22 x the error of the Cholesky route at q = 32 and cond 1e4 - 1e6, 1e-8 on a rank-deficient q = 64 case; a
// recursive Schur-complement version with explicit 16 x 16 / 32 x 32 inverses was 400 x worse.  Both were found and measured in
// the lane-level restatement, oracle/sweep_oracle.py, before / beside the GPU runs.)
//
// Working layout: once its bulk copy has landed, every matrix is re-laid-out in place: lower tile (I, J) -> 64 doubles at
// (I (I + 1) / 2 + J) 64, element (r, c) at the swizzled offset of the blocked Cholesky kernel,
// r 8 + (((c >> 2) ^ ((r >> 1) & 1)) << 2) + (c & 3): accumulator-layout accesses are conflict-free 128-bit, A and B fragments
// conflict-free 64-bit, and the diagonal tiles are kept whole (no mirror reads).  (The sweep used to run on the packed rows as they
// lie in HBM; it was bound by shared-memory bandwidth, 45 % of its wavefronts bank conflicts of the packed triangle --
// profiles/r02_k2_ncu.md, DESIGN.md 5.)  zbar = Sigma eta runs on the tensor core too (eta in column 0 of the B fragment), and the
// <zz^T> pass puts the rows back into the packed order for the bulk store.
//
// ln prod diag chol = 1/2 sum ln(pivots): the pivots are those of the unblocked elimination.  Column sums / maxima bounds / log-det
// scalars per CTA as in the other K2 kernels (partial layout of the blocked kernel).
#include "common.cuh"
#include "kernels.h"
#include "ptx.cuh"

namespace pyvb {

namespace {

__host__ __device__ constexpr int s_tri(int i) { return i * (i + 1) / 2; }
__host__ __device__ constexpr int s_pitch(int q) {          // == pyvb_mz_pitch(q)
    int p = ((s_tri(q) + 7) & ~7) + q + 1;
    while ((p % 8) != 4) ++p;
    return p;
}

// 1 / d to the last bit or so: MUFU.RCP64H seed + two Newton steps (as kernels_k2g.cu)
__device__ __forceinline__ double s_rcp(double d) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    double e = fma(-d, r, 1.0);
    r = fma(r, e, r);
    e = fma(-d, r, 1.0);
    return fma(r, e, r);
}

__host__ __device__ constexpr int s_sw(int r, int c) { return r * 8 + ((((c >> 2) ^ ((r >> 1) & 1))) << 2) + (c & 3); }
__host__ __device__ constexpr int s_toff(int I, int J) { return (s_tri(I) + J) * 64; }

template <int Q, int MPW_, int WARPS_, int STAGES_, int UM_> struct SBT {
    static constexpr int MPW = MPW_, WARPS = WARPS_, STAGES = STAGES_, UM = UM_;
    static constexpr int NBT = Q / 8, NT = s_tri(NBT);
    static constexpr int P = s_tri(Q), PP = (P + 7) & ~7, OROW = PP + Q, PITCH = s_pitch(Q);
    static constexpr int KW = 2 * OROW + PYVB_ZS_EXTRA;
    static constexpr int EOFF = NT * 64;                       // eta / zbar behind the tiles
    static constexpr int TS = EOFF + Q;                        // stage slot of one matrix (the packed row lands in its first PITCH doubles)
    static constexpr int STAGE_D = MPW * TS;
    static constexpr int BC_D = 2 * MPW * 16;
    static constexpr int WARP_D = STAGES * STAGE_D + BC_D + OROW + 4 + 2 * Q + 2;
    static constexpr size_t SMEM = (size_t)WARPS * WARP_D * 8;
    static_assert(MPW == 1 || MPW == 2 || MPW == 4, "the diagonal sweep spreads MPW x 8 tile rows over the lanes");
    static_assert(TS >= PITCH && (TS % 2) == 0 && (OROW % 2) == 0 && (WARP_D % 2) == 0, "slot size, 16-byte alignment");
    static_assert(STAGES == 1 || STAGES == 2, "one or two stages");
};

struct SwzLane {             // the lane's offsets inside a tile
    int a[2];                // A fragment (gid, 4h + qd)
    int b[2];                // B fragment / transposed A fragment (4h + qd, gid)
    int c;                   // accumulator pair (gid, 2qd), (gid, 2qd + 1): adjacent
    int ct[2];               // transposed accumulator element (2qd + e, gid)
};

template <int K, typename T>
__device__ __forceinline__ void t_pivot_tile(double *stg, double *bc, int lane, double &pr, bool &pos) {
    const int m = (lane >> 3) % T::MPW, r = lane & 7;
    double *tl = stg + m * T::TS + s_toff(K, K) + r * 8;
    const int s4 = ((r >> 1) & 1) << 2;
    double a[8], x[8];
#pragma unroll
    for (int g = 0; g < 2; ++g)
#pragma unroll
        for (int p = 0; p < 2; ++p) {
            const double2 v = *reinterpret_cast<const double2 *>(tl + ((g << 2) ^ s4) + 2 * p);
            a[4 * g + 2 * p] = v.x;
            a[4 * g + 2 * p + 1] = v.y;
        }
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] = 0.0;
    double dinv = 1.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        double *b = bc + (k & 1) * (T::MPW * 16) + m * 16;      // [column k of the reduced tile (8) | row k of X (8)]
        b[r] = a[k];
        if (r == k) {
#pragma unroll
            for (int j = 0; j < k; ++j) b[8 + j] = x[j];
        }
        __syncwarp();
        double B[8], XK[8];
#pragma unroll
        for (int j2 = k / 2; j2 < 4; ++j2) {
            const double2 v = *reinterpret_cast<const double2 *>(b + 2 * j2);
            B[2 * j2] = v.x;
            B[2 * j2 + 1] = v.y;
        }
#pragma unroll
        for (int j2 = 0; j2 < (k + 1) / 2; ++j2) {
            const double2 v = *reinterpret_cast<const double2 *>(b + 8 + 2 * j2);
            XK[2 * j2] = v.x;
            XK[2 * j2 + 1] = v.y;
        }
        const double rc = s_rcp(B[k]);
        dinv = (r == k) ? rc : dinv;
        const double l = (r > k) ? a[k] * rc : 0.0;
#pragma unroll
        for (int j = k + 1; j < 8; ++j) a[j] = fma(-l, B[j], a[j]);
#pragma unroll
        for (int j = 0; j < k; ++j) x[j] = fma(-l, XK[j], x[j]);
        x[k] = -l;
    }
    if ((lane >> 3) < T::MPW) {
        pr *= dinv;
        pos = pos && (dinv > 0.0);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j)
        if (j < r) tl[((j & 4) ^ s4) + (j & 3)] = x[j];
    tl[((r & 4) ^ s4) + (r & 3)] = dinv;
    __syncwarp();
}

// block (I, K), I != K, of the symmetric state: A fragment of half h / store of accumulator-layout values
template <int I, int K>
__device__ __forceinline__ double t_afrag(const double *st, const SwzLane &sw, int h) {
    return (I > K) ? st[s_toff(I, K) + sw.a[h]] : st[s_toff(K, I) + sw.b[h]];
}
template <int J, int K>
__device__ __forceinline__ void t_cstore(double *st, const SwzLane &sw, double v0, double v1) {
    if (J > K) {
        *reinterpret_cast<double2 *>(st + s_toff(J, K) + sw.c) = make_double2(v0, v1);
    } else {
        st[s_toff(K, J) + sw.ct[0]] = v0;
        st[s_toff(K, J) + sw.ct[1]] = v1;
    }
}

template <int K, int J, typename T>
struct TSteps {       // compile-time loops over the tile index J (the tile offsets are template arguments)
    static __device__ __forceinline__ void load_panel(const double *st, const SwzLane &sw, double (&f)[T::NBT][2]) {
        if constexpr (J < T::NBT) {
            if constexpr (J != K) {
                f[J][0] = t_afrag<J, K>(st, sw, 0);
                f[J][1] = t_afrag<J, K>(st, sw, 1);
            }
            TSteps<K, J + 1, T>::load_panel(st, sw, f);
        }
    }
    static __device__ __forceinline__ void store_panel(double *st, const SwzLane &sw, const double (&w)[T::NBT][2]) {
        if constexpr (J < T::NBT) {
            if constexpr (J != K) t_cstore<J, K>(st, sw, w[J][0], w[J][1]);
            TSteps<K, J + 1, T>::store_panel(st, sw, w);
        }
    }
    static __device__ __forceinline__ void new_panel(double *st, const SwzLane &sw, const double (&wd)[T::NBT][2], const double (&xb)[2]) {
        if constexpr (J < T::NBT) {
            if constexpr (J != K) {
                double t0 = 0.0, t1 = 0.0;
                dmma884(t0, t1, wd[J][0], xb[0]);
                dmma884(t0, t1, wd[J][1], xb[1]);
                t_cstore<J, K>(st, sw, t0, t1);
            }
            TSteps<K, J + 1, T>::new_panel(st, sw, wd, xb);
        }
    }
};

template <int K, typename T>
__device__ __forceinline__ void t_sweep_tile(double *stg, double *bc, int lane, const SwzLane &sw, double &pr, bool &pos) {
    constexpr int NBT = T::NBT;
    const int gid = lane >> 2, qd = lane & 3;
    t_pivot_tile<K, T>(stg, bc, lane, pr, pos);
#pragma unroll(T::UM)
    for (int m = 0; m < T::MPW; ++m) {
        double *st = stg + m * T::TS;
        const double *pt = st + s_toff(K, K);
        double of[NBT][2];
        TSteps<K, 0, T>::load_panel(st, sw, of);
        double xa[2], xb[2], dk[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const double va = pt[sw.a[h]], vb = pt[sw.b[h]];
            xa[h] = (gid > 4 * h + qd) ? va : ((gid == 4 * h + qd) ? 1.0 : 0.0);
            xb[h] = (4 * h + qd > gid) ? vb : ((gid == 4 * h + qd) ? 1.0 : 0.0);
            dk[h] = pt[s_sw(4 * h + qd, 4 * h + qd)];
        }
        double wt[NBT][2];
#pragma unroll
        for (int J = 0; J < NBT; ++J) {
            if (J == K) continue;
            wt[J][0] = wt[J][1] = 0.0;
            dmma884(wt[J][0], wt[J][1], of[J][0], xa[0]);
            dmma884(wt[J][0], wt[J][1], of[J][1], xa[1]);
        }
        double pv0 = 0.0, pv1 = 0.0;
        dmma884(pv0, pv1, xb[0], xb[0] * dk[0]);
        dmma884(pv0, pv1, xb[1], xb[1] * dk[1]);
        __syncwarp();                                           // every lane has read the old panel and X
        *reinterpret_cast<double2 *>(st + s_toff(K, K) + sw.c) = make_double2(-pv0, -pv1);
        TSteps<K, 0, T>::store_panel(st, sw, wt);
        __syncwarp();
        double wa[NBT][2], wd[NBT][2];
        TSteps<K, 0, T>::load_panel(st, sw, wa);
#pragma unroll
        for (int I = 0; I < NBT; ++I)
#pragma unroll
            for (int h = 0; h < 2; ++h)
                if (I != K) wd[I][h] = wa[I][h] * dk[h];
        __syncwarp();                                           // every lane has read W
        TSteps<K, 0, T>::new_panel(st, sw, wd, xb);
#pragma unroll
        for (int I = 0; I < NBT; ++I) {
            if (I == K) continue;
            const double na0 = -wd[I][0], na1 = -wd[I][1];
#pragma unroll
            for (int J = 0; J <= I; ++J) {
                if (J == K) continue;
                double2 *o = reinterpret_cast<double2 *>(st + s_toff(I, J) + sw.c);
                double2 c = *o;
                dmma884(c.x, c.y, na0, wa[J][0]);
                dmma884(c.x, c.y, na1, wa[J][1]);
                *o = c;
            }
        }
    }
    __syncwarp();
}

template <int K, typename T>
__device__ __forceinline__ void t_sweep_all(double *stg, double *bc, int lane, const SwzLane &sw, double &pr, bool &pos) {
    if constexpr (K < T::NBT) {
        t_sweep_tile<K, T>(stg, bc, lane, sw, pr, pos);
        t_sweep_all<K + 1, T>(stg, bc, lane, sw, pr, pos);
    }
}

template <int Q, int MPW_, int WARPS_, int STAGES_, int UM_>
__global__ void __launch_bounds__(32 * WARPS_, 1)
zsolve_tsweep_kernel(long long N, double *__restrict__ MZ, double *__restrict__ Sig, double *__restrict__ logdet, double *gl,
                     double *__restrict__ zsums, const double *__restrict__ cond, const I8Check chk) {
    using T = SBT<Q, MPW_, WARPS_, STAGES_, UM_>;
    constexpr int MPW = T::MPW, P = T::P, PP = T::PP, PITCH = T::PITCH, NBT = T::NBT, TS = T::TS, EOFF = T::EOFF;
    constexpr int NE = (Q + 31) / 32;                            // eta / zbar entries per lane
    if (cond != nullptr && !(*cond > 0.0)) return;               // conditional (fall-back) launch: nothing to redo
    __shared__ double s_chk[T::WARPS + 1];
    extern __shared__ __align__(16) double smem_sb[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int gid = lane >> 2, qd = lane & 3;
    SwzLane sw;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        sw.a[h] = s_sw(gid, 4 * h + qd);
        sw.b[h] = s_sw(4 * h + qd, gid);
        sw.ct[h] = s_sw(2 * qd + h, gid);
    }
    sw.c = s_sw(gid, 2 * qd);
    double *stage = smem_sb + (size_t)warp * T::WARP_D;
    double *bc = stage + T::STAGES * T::STAGE_D;
    double *csum = bc + T::BC_D;                                  // [OROW]
    double *wsc = csum + T::OROW;                                 // [4]
    double *wmx = wsc + 4;                                        // [2 Q]: max_n <z_i z_i>, max_n |<z_i>| of this warp's rows
    uint64_t *bar = reinterpret_cast<uint64_t *>(wmx + 2 * Q);

    for (int c = lane; c < T::OROW; c += 32) csum[c] = 0.0;
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_init(bar + 1, 1);
    }
    if (chk.gscale != nullptr) {                                 // INT8 guard (kernels.h: I8Check), kernel-uniform
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

    // the lanes with qd == 0 track rows 8 I + gid: max <z_i z_i>, max |z_i|
    double dmx[NBT], zmx[NBT], s_qld = 0.0, s_ld = 0.0, s_n = 0.0;
#pragma unroll
    for (int I = 0; I < NBT; ++I) dmx[I] = zmx[I] = 0.0;

    const long long nwarps = (long long)gridDim.x * T::WARPS;
    const long long ngroups = (N + MPW - 1) / MPW;
    long long g = (long long)blockIdx.x * T::WARPS + warp;
    auto load_group = [&](long long grp, double *dst, uint64_t *b) {      // lane 0: one bulk copy per row into its slot
        const long long left = N - grp * MPW;
        const int nv = (int)(left < MPW ? left : MPW);
        mbar_arrive_expect_tx(b, (uint32_t)(nv * PITCH * 8));
        for (int m = 0; m < nv; ++m) bulk_g2s(dst + m * TS, MZ + (grp * MPW + m) * PITCH, (uint32_t)(PITCH * 8), b);
    };
    if (g < ngroups && lane == 0) load_group(g, stage, bar);
    for (int it = 0; g < ngroups; g += nwarps, ++it) {
        const int sidx = (T::STAGES == 2) ? (it & 1) : 0;
        double *stg = stage + sidx * T::STAGE_D;
        const long long n0 = g * MPW;
        const int nval = (N - n0 < MPW) ? (int)(N - n0) : MPW;
        const long long gn = g + nwarps;
        if (T::STAGES == 2) {
            if (lane == 0 && gn < ngroups) {
                bulk_wait_read_all();
                load_group(gn, stage + (sidx ^ 1) * T::STAGE_D, bar + (sidx ^ 1));
            }
            mbar_wait(bar + sidx, (uint32_t)((it >> 1) & 1));
        } else {
            mbar_wait(bar, (uint32_t)(it & 1));
        }

        // ---- packed rows -> swizzled tiles, in place: everything is read before anything is written
#pragma unroll 1
        for (int m = 0; m < MPW; ++m) {
            double *st = stg + m * TS;
            double v[T::NT][2], e[NE];
#pragma unroll
            for (int I = 0; I < NBT; ++I)
#pragma unroll
                for (int J = 0; J <= I; ++J)
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int row = 8 * I + gid, col = 8 * J + 2 * qd + h;
                        v[s_tri(I) + J][h] = (I > J || col <= row) ? st[s_tri(row) + col] : st[s_tri(col) + row];
                    }
#pragma unroll
            for (int k = 0; k < NE; ++k) e[k] = (32 * k + lane < Q) ? st[PP + 32 * k + lane] : 0.0;
            __syncwarp();
#pragma unroll
            for (int t = 0; t < T::NT; ++t) *reinterpret_cast<double2 *>(st + t * 64 + sw.c) = make_double2(v[t][0], v[t][1]);
#pragma unroll
            for (int k = 0; k < NE; ++k)
                if (32 * k + lane < Q) st[EOFF + 32 * k + lane] = e[k];
        }
        __syncwarp();

        {   // ---- the sweep; it leaves -Sigma in the tiles.  Lane (m8, r8) = pivot-tile row r8 of matrix m8 (with MPW < 4: shadows)
            const int m8 = lane >> 3, r8 = lane & 7;
            if (thr >= 0.0) {                                    // INT8 guard: largest diagonal entry of qprec (kernel-uniform branch)
                const double *st = stg + (m8 % MPW) * TS;
                double dm = 0.0;
#pragma unroll
                for (int t = 0; t < NBT; ++t) dm = fmax(dm, st[s_toff(t, t) + s_sw(r8, r8)]);
#pragma unroll
                for (int o = 4; o > 0; o >>= 1) dm = fmax(dm, __shfl_xor_sync(0xffffffffu, dm, o));
                if (r8 == 0 && m8 < nval && m8 < MPW && thr > dm) atomicAdd(&gl[PYVB_GL_I8BAD], 1.0);
            }
            double pr = 1.0;
            bool pos = true;
            t_sweep_all<0, T>(stg, bc, lane, sw, pr, pos);
            double lg = pos ? log(pr) : __longlong_as_double(0x7ff8000000000000LL);
#pragma unroll
            for (int o = 4; o > 0; o >>= 1) lg += __shfl_xor_sync(0xffffffffu, lg, o);
            const double ldsum = -0.5 * lg;
            if (r8 == 0 && m8 < nval && m8 < MPW) {
                logdet[n0 + m8] = ldsum;
                s_qld += 0.5 / ldsum;
                s_ld += ldsum;
                s_n += 1.0;
                if (!(ldsum - ldsum == 0.0)) atomicAdd(&gl[PYVB_GL_NONPD], 1.0);   // NaN / inf <=> a pivot was <= 0
            }
        }

        // ---- per matrix: zbar = Sigma eta on the tensor core, <zz^T> = Sigma + zbar zbar^T, back into the packed order
#pragma unroll 1
        for (int m = 0; m < MPW; ++m) {
            double *st = stg + m * TS;
            double z[NBT];                                       // lanes with qd == 0: z[8 I + gid]
#pragma unroll
            for (int I = 0; I < NBT; ++I) {
                double z0 = 0.0, z1 = 0.0;
#pragma unroll
                for (int J = 0; J < NBT; ++J)
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const double a = (I >= J) ? st[s_toff(I, J) + sw.a[h]] : st[s_toff(J, I) + sw.b[h]];
                        const double ev = st[EOFF + 8 * J + 4 * h + qd];
                        dmma884(z0, z1, a, gid == 0 ? ev : 0.0);
                    }
                z[I] = -z0;
            }
            __syncwarp();                                        // every lane has read eta
            if (qd == 0) {
#pragma unroll
                for (int I = 0; I < NBT; ++I) st[EOFF + 8 * I + gid] = z[I];
            }
            __syncwarp();
            double out[T::NT][2], zb[NE];
            double *sg = (Sig != nullptr && m < nval) ? Sig + (n0 + m) * P : nullptr;
#pragma unroll
            for (int I = 0; I < NBT; ++I) {
                const double zi = st[EOFF + 8 * I + gid];
#pragma unroll
                for (int J = 0; J <= I; ++J) {
                    const double2 c = *reinterpret_cast<const double2 *>(st + s_toff(I, J) + sw.c);
                    const double2 zj = *reinterpret_cast<const double2 *>(st + EOFF + 8 * J + 2 * qd);
                    out[s_tri(I) + J][0] = fma(zi, zj.x, -c.x);
                    out[s_tri(I) + J][1] = fma(zi, zj.y, -c.y);
                    if (sg != nullptr) {                         // (uncoalesced; the Sigma output is optional)
                        const int row = 8 * I + gid, col = 8 * J + 2 * qd;
                        if (col <= row) sg[s_tri(row) + col] = -c.x;
                        if (col + 1 <= row) sg[s_tri(row) + col + 1] = -c.y;
                    }
                }
                if (qd == 0 && m < nval) {                       // the diagonal entry <z_i z_i> exactly as it is stored
                    const double d = st[s_toff(I, I) + s_sw(gid, gid)];
                    dmx[I] = fmax(dmx[I], fma(zi, zi, -d));
                    zmx[I] = fmax(zmx[I], fabs(zi));
                }
            }
#pragma unroll
            for (int k = 0; k < NE; ++k) zb[k] = (32 * k + lane < Q) ? st[EOFF + 32 * k + lane] : 0.0;
            __syncwarp();                                        // the tiles have been read: the packed row takes their place
#pragma unroll
            for (int I = 0; I < NBT; ++I)
#pragma unroll
                for (int J = 0; J <= I; ++J)
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int row = 8 * I + gid, col = 8 * J + 2 * qd + h;
                        if (I > J || col <= row) st[s_tri(row) + col] = out[s_tri(I) + J][h];
                    }
#pragma unroll
            for (int k = 0; k < NE; ++k)
                if (32 * k + lane < Q) st[PP + 32 * k + lane] = zb[k];
        }
        fence_async_smem();
        __syncwarp();
        // ---- rows back to HBM (one bulk store per row), column sums of the finished rows, next group in
        if (lane == 0) {
            for (int m = 0; m < nval; ++m) bulk_s2g(MZ + (n0 + m) * PITCH, stg + m * TS, (uint32_t)(PITCH * 8));
            bulk_commit();
        }
        if (zsums != nullptr) {                                  // kernel-uniform
            for (int c = lane; c < T::OROW; c += 32) {
                double v = 0.0;
#pragma unroll
                for (int mm = 0; mm < MPW; ++mm)
                    if (mm < nval) v += stg[mm * TS + c];
                csum[c] += v;
            }
        }
        __syncwarp();
        if (T::STAGES == 1 && lane == 0 && gn < ngroups) {       // one stage: the store has to have read it first
            bulk_wait_read_all();
            load_group(gn, stage, bar);
        }
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
    if (qd == 0) {
#pragma unroll
        for (int I = 0; I < NBT; ++I) {
            wmx[8 * I + gid] = dmx[I];
            wmx[Q + 8 * I + gid] = zmx[I];
        }
    }
    __syncthreads();
    double *outp = zsums + (size_t)blockIdx.x * T::KW;
    const double *w0 = smem_sb + T::STAGES * T::STAGE_D + T::BC_D;    // csum of warp 0
    for (int c = tid; c < T::OROW + 4; c += 32 * T::WARPS) {
        double v = 0.0;
        for (int w = 0; w < T::WARPS; ++w) v += w0[(size_t)w * T::WARP_D + c];   // [csum OROW | scalars 4] is contiguous
        outp[c] = v;
    }
    const double *m0 = w0 + T::OROW + 4;
    double *fm = smem_sb;                                        // warp 0's stage is free now: [2 Q] folded maxima
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
        outp[T::OROW + 4 + c] = v;
    }
}

// The configuration (matrices per warp and stage, warps per CTA, stages, matrices unrolled together).  Measured per launch (B200,
// q = 64, 400k rows): (2, 4, 1, 1) 11.4 ms, (1, 6, 1, 1) 12.0 (profiles/r02_k2_sweep_v3_timings.txt)
using SW64 = SBT<64, 2, 4, 1, 1>;

}  // namespace

int zsolve_sweep_blocks(long long N, int q) {
    if (q != 64) return 0;
    long long b = (N + (long long)SW64::MPW * SW64::WARPS - 1) / ((long long)SW64::MPW * SW64::WARPS);
    if (b > 148) b = 148;
    if (b < 1) b = 1;
    return (int)b;
}

int zsolve_sweep_kw(int q) { return q == 64 ? SW64::KW : 0; }

cudaError_t launch_zsolve_sweep(long long N, int q, double *MZ, double *Sig, double *logdet, double *gl, double *zsums,
                                cudaStream_t st, const double *cond, I8Check chk) {
    if (N <= 0) return cudaSuccess;
    if (q != 64) return cudaErrorNotSupported;
    static_assert(SW64::SMEM <= 232448 - 1024, "shared memory of one CTA");
    auto kernel = zsolve_tsweep_kernel<64, SW64::MPW, SW64::WARPS, SW64::STAGES, SW64::UM>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SW64::SMEM);
    if (e != cudaSuccess) return e;
    kernel<<<zsolve_sweep_blocks(N, q), 32 * SW64::WARPS, SW64::SMEM, st>>>(N, MZ, Sig, logdet, gl, zsums, cond, chk);
    return cudaGetLastError();
}

}  // namespace pyvb
