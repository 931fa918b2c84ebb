// K3 (blocked, look-ahead): batched block-banded FP64 Cholesky + MVN draw for the V columns.
//
// Replaces sample_mvn_from_precision + CHOLMOD (fast_mvn.py:33-74) and the kron / SpGEMM assembly of
// factor.py:396-408: right-looking block-banded Cholesky with KB x KB blocks (block half-bandwidth Q = order + 1)
// in a shift-free circular shared-memory window, the per-column statistics prefetched from global memory, the
// factor spilled by block columns for the backward solve.  Organised around the one chain that cannot be
// parallelised - the KB sequential pivots of every diagonal block:
//   * the diagonal block of step t+1 is factorised by warp 0 WHILE the other warps finish the
//     trailing update of step t, spill block column t and assemble the entering block row
//     (statistics prefetched into registers before the tensor-pipe work);
//   * warp 0 also inverts the KB x KB triangular factor, so the Q blocks below the diagonal become
//     L_ut = A_ut L_tt^-T = A_ut Linv^T on the tensor pipe (no per-row substitution chains), the
//     right-hand side y_t = Linv b_t, and every backward step two small matrix-vector products
//     (x_t = Linv^T (w_t - sum_u L_ut^T x_{t+u})) instead of a KB-step shuffle chain;
//   * the backward sweep streams [Linv_t | L_1t .. L_Qt | y_t] through a cp.async double buffer
//     and an otherwise idle warp draws the normals of the next step.
// Critical path per block column: one tensor-pipe solve, one KB x KB syrk tile row, one potrf.
// Measured per column (K = 16, T = 64, one CTA per SM): see DESIGN.md K3.
#include <cstdio>
#include <type_traits>
#include "kernels.h"

namespace btf {

namespace {

__device__ __forceinline__ void la_cp_async16(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void la_cp_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N>
__device__ __forceinline__ void la_cp_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

__device__ __forceinline__ void la_dmma(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// 1/d for the pivot chain: hardware seed (relative error < 2^-20) and ONE third-order step
// y0 (1 + e + e^2), e = 1 - d y0  ->  relative error ~2^-60 plus rounding: three dependent FP64
// operations instead of the five of an IEEE division (every FP64 operation on this chain costs
// its full pipeline latency).  d is positive and finite here.
__device__ __forceinline__ double la_rcp_pos(double d) {
    double y0;
    asm("rcp.approx.ftz.f64 %0, %1;\n" : "=d"(y0) : "d"(d));
    const double e = fma(-d, y0, 1.0);
    const double e2 = fma(e, e, e);
    return fma(e2, y0, y0);
}

template <int KB, int Q>
struct LaGeom {
    static constexpr int KS = KB + 4;                      // padded row stride of a block in shared memory
    static constexpr int BLK = KB * KS;
    static constexpr int NBLK = (Q + 1) * (Q + 2) / 2;
    static constexpr int KK = KB * KB;                     // unpadded block (global layout)
    static constexpr int TB = KB / 8;
    static constexpr int NW = KB > 16 ? 8 : 4;             // warp 0: potrf; warps 1..: workers
    static constexpr int NT = 32 * NW;
    static constexpr int NWK = NW - 1, NWT = 32 * NWK;
    static constexpr int MINB = KB > 16 ? 1 : 4;
    static constexpr int COLE = (Q + 1) * KK;              // global block column: Linv_t | L_1t .. L_Qt
    static constexpr int BWD = COLE + KB;                  // + y_t : one backward stage
    static constexpr int NST = 3;                          // backward stages: the block column of step t-2 is in flight during step t
    static constexpr int WREG = NBLK * BLK > NST * BWD ? NBLK * BLK : NST * BWD;
    static constexpr int NSW = TB <= 2 ? TB : 1;           // 8-row strips a worker warp runs together (independent tensor-pipe chains)
    static constexpr int PF = (KB * (KB + 1) / 2 + NWT - 1) / NWT;   // prefetched statistics per worker thread
    __host__ __device__ static constexpr int base(int d) { return d * (Q + 1) - d * (d - 1) / 2; }
    __device__ static __forceinline__ int slot(int a, int d) { return base(d) + a % (Q + 1 - d); }
    static size_t smem_doubles(int T, int RD) {
        return (size_t)WREG + 2 * BLK + (Q + 1) * KB + KB + 2 * (Q + 1) * KB + 2 * KB + 2 * KB + (size_t)T * (Q + 1) +
               RD + 48 + 96 + (KB * (KB + 1) / 2 + 3) / 4;
    }
};

}  // namespace

template <int KB, int Q>
__global__ void __launch_bounds__(LaGeom<KB, Q>::NT, LaGeom<KB, Q>::MINB) band_lookahead_kernel(BandSolveArgs a) {
    using G = LaGeom<KB, Q>;
    constexpr int KS = G::KS, BLK = G::BLK, NT = G::NT, KK = G::KK, TB = G::TB, NW = G::NW, NWK = G::NWK, NWT = G::NWT;
    constexpr int COLE = G::COLE, BWD = G::BWD, PF = G::PF;
    extern __shared__ __align__(16) double sm[];
    const int Kr = a.K;                                  // true embedding size (<= KB)
    const int L = Kr * (Kr + 1) / 2, nco = L + Kr, kd = Q * Kr, LS = kd + 1;
    const int T = a.T, n = T * Kr;
    const int lane = threadIdx.x & 31;
    const int warp = (int)(threadIdx.x >> 5);
    const int tid = warp * 32 + lane;
    const int jl = blockIdx.x, jg = a.col_begin + jl;
    const unsigned full = 0xffffffffu;

    double* Wb = sm;                                   // [NBLK][BLK] window  (backward: NST stages of BWD)
    double* Li = Wb + G::WREG;                         // [2][BLK]   inverse of the diagonal factor (padded rows)
    double* bw = Li + 2 * BLK;                         // [Q+1][KB]  right-hand-side window
    double* ycur = bw + (Q + 1) * KB;                  // [KB]
    double* xw = ycur + KB;                            // [2][Q+1][KB] backward solution window
    double* rb = xw + 2 * (Q + 1) * KB;                // [2][KB]    backward right-hand sides
    double* zb = rb + 2 * KB;                          // [2][KB]    normals of the current / next backward step
    double* Pband = zb + 2 * KB;                       // [T][Q+1]
    double* linv = Pband + (size_t)T * (Q + 1);        // [RD]
    double* red = linv + a.RD;                         // [40]
    double* colb = red + 48;                           // [2][32] pivot column of the potrf warp
    double* dbuf = colb + 64;                          // [32]    pivots d_j, then 1/sqrt(d_j)
    unsigned short* pairtab = reinterpret_cast<unsigned short*>(dbuf + 32);   // [L] packed index -> (i << 8 | c)
    __shared__ int fail_flag;

    const double scale = a.homoskedastic ? 1.0 / a.scal->nu2 : 1.0;
    const double lam2 = a.scal->lam2;
    for (int r = tid; r < a.RD; r += NT) {
        double pv = 1.0 / (lam2 * a.Tau2[(size_t)jg * a.RD + r]);
        if (a.prior_clip > 0.0) pv = fmin(fmax(pv, a.prior_clip), 1.0 / a.prior_clip);
        linv[r] = pv;
    }
    if (tid == 0) fail_flag = 0;
    for (int e = tid; e < Kr * Kr; e += NT) {
        const int i = e / Kr, c = e % Kr;
        if (c <= i) pairtab[tri(i, c)] = (unsigned short)((i << 8) | c);
    }
    __syncthreads();
    for (int e = tid; e < T * (Q + 1); e += NT) {
        double s = 0.0;
        for (int x = a.pm_ptr[e]; x < a.pm_ptr[e + 1]; ++x) s += a.pm_coef[x] * linv[a.pm_row[x]];
        Pband[e] = s;
    }
    __syncthreads();

    // global workspace of this column: block columns [T][Linv | L_1t..L_Qt] (unpadded KB x KB), y [T KB]
    double* Lg = a.work_L + (size_t)jl * a.work_L_stride;
    double* yg = a.work_y + (size_t)jl * a.work_y_stride;
    const bool have_stats = a.stats != nullptr;
    const double* stats0 = have_stats ? a.stats + (size_t)jg * T * nco : nullptr;

#ifdef BTF_BAND_PROFILE
    long long pc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    long long wp[4] = {0, 0, 0, 0};
    long long wq[4] = {0, 0, 0, 0};
    long long pc0 = clock64(), pc1;
#define LAPROF(i) do { pc1 = clock64(); pc[i] += pc1 - pc0; pc0 = pc1; } while (0)
#else
#define LAPROF(i)
#endif
    double jitter = 0.0, eps = a.eps;
    int attempt = 0;
    bool failed = false;

    // everything of block row `arow` except the statistics: prior band, padding, off-diagonal blocks
    auto init_rest = [&](int arow, int t0, int nthreads) {
        double* D = Wb + G::slot(arow, 0) * BLK;
        for (int e = t0; e < (KB - Kr) * KB; e += nthreads) {          // padding rows Kr..KB-1: identity
            const int i = Kr + e / KB, c = e % KB;
            if (c <= i) D[i * KS + c] = (c == i) ? 1.0 : 0.0;
        }
#pragma unroll
        for (int d = 1; d <= Q; ++d) {                                 // (arow, arow - d) = P[arow][arow-d] * I
            if (arow - d >= 0) {
                double* B = Wb + G::slot(arow, d) * BLK;
                const double pv = Pband[(arow - d) * (Q + 1) + d];
                for (int e = t0; e < KB * KB; e += nthreads) {
                    const int i = e / KB, c = e % KB;
                    B[i * KS + c] = (i == c && i < Kr) ? pv : 0.0;
                }
                if (a.diag_band)
                    for (int e = t0; e < Kr; e += nthreads)
                        a.diag_band[((size_t)jl * n + arow * Kr + e) * LS + kd - d * Kr] = pv;
            }
        }
    };
    // one packed lower-triangle entry of the diagonal block
    auto put_diag = [&](int arow, int e, double sv) {
        const int i = pairtab[e] >> 8, c = pairtab[e] & 0xff;
        double v = sv * scale;
        if (c == i) v += Pband[arow * (Q + 1)] + jitter;
        if (a.diag_band) a.diag_band[((size_t)jl * n + arow * Kr + i) * LS + kd - (i - c)] = v;
        Wb[G::slot(arow, 0) * BLK + i * KS + c] = v;
    };
    auto stat_sum = [&](const double* p) {
        double sv = p[0];
        for (int s = 1; s < a.nsplit; ++s) sv += p[s * a.split_stride];
        return sv;
    };
    // assemble a whole block row with direct loads (initial window)
    auto init_row = [&](int arow, int t0, int nthreads) {
        const double* sb = have_stats ? stats0 + (size_t)arow * nco : nullptr;
        for (int e = t0; e < L; e += nthreads) put_diag(arow, e, have_stats ? stat_sum(sb + e) : 0.0);
        for (int e = t0; e < KB; e += nthreads)
            bw[(arow % (Q + 1)) * KB + e] = (have_stats && e < Kr) ? stat_sum(sb + L + e) * scale : 0.0;
        init_rest(arow, t0, nthreads);
    };

    // warp 0: Cholesky of the diagonal block of step t in registers (lane = row) and its inverse into
    // Li[t & 1].  KB <= 16: lanes KB..2KB-1 carry the rows of the identity through the same column
    // operations, which leaves I L^-T = Linv^T in them at no cost to the pivot chain.  KB = 32 has
    // no idle lanes: the inverse is a second pass (row `lane` of Linv from x L = e_lane).
    auto potrf_inv = [&](int t) {
        constexpr bool AUG = 2 * KB <= 32;
        double* D = Wb + G::slot(t, 0) * BLK;
        double* Lv = Li + (t & 1) * BLK;
        double ar[KB];
#pragma unroll
        for (int c = 0; c < KB; ++c) {
            double v = 0.0;
            if (lane < KB) v = D[lane * KS + c];
            else if (AUG && lane - KB == c) v = 1.0;
            ar[c] = v;
        }
        // The pivot chain runs on the UNSCALED columns (L D L^T form): with q_j = 1/d_j,
        //   a_ik <- a_ik - (a_ij q_j) a_kj,   d_{j+1} = a_{j+1,j+1} - a_{j+1,j}^2 q_j  (own lane, no exchange).
        // The loop is issue bound, so it is kept short: the pivot column goes through shared memory
        // once (one store, broadcast reads) instead of one 64-bit shuffle pair per entry, the update
        // is unconditional (entries above the diagonal are never read), and the square roots that turn
        // column j into L_ij = a_ij / sqrt(d_j) are taken once, one per lane, after the loop.
        bool ok = true;
        double d = __shfl_sync(full, ar[0], 0);
        if (!(d > 0.0) || isinf(d)) ok = false;
#pragma unroll
        for (int j = 0; j < KB; ++j) {
            const double dj = ok ? d : 1.0;
            const double aj = ar[j];
            double* cb = colb + (j & 1) * 32;
            cb[lane] = aj;
            if (lane == 0) dbuf[j] = dj;
            const double q = la_rcp_pos(dj);
            if (j + 1 < KB) {
                const double dloc = fma(-(aj * aj), q, ar[j + 1]);      // what lane j+1 is about to hold
                d = __shfl_sync(full, dloc, j + 1);
                if (!(d > 0.0) || isinf(d)) ok = false;
            }
            __syncwarp();
            const double tq = -(aj * q);
#pragma unroll
            for (int k = 0; k < KB; ++k)
                if (k > j) ar[k] = fma(tq, cb[k], ar[k]);   // rectangular loop + constant predicate: fully unrollable
        }
        __syncwarp();
        const double mydinv = rsqrt(dbuf[lane < KB ? lane : 0]);
        __syncwarp();
        if (lane < KB) dbuf[lane] = mydinv;
        __syncwarp();
#pragma unroll
        for (int c = 0; c < KB; ++c) ar[c] *= dbuf[c];
        if (!ok && lane == 0) fail_flag = 1;
        if (lane < KB) {
#pragma unroll
            for (int c = 0; c < KB; ++c) D[lane * KS + c] = (c <= lane) ? ar[c] : 0.0;
        }
        if (AUG) {
            // lane KB + i holds row i of L^-T = column i of Linv
            if (lane >= KB && lane < 2 * KB) {
#pragma unroll
                for (int c = 0; c < KB; ++c) Lv[c * KS + (lane - KB)] = ar[c];
            }
        } else {
            __syncwarp();
            double x[KB];
#pragma unroll
            for (int k = KB - 1; k >= 0; --k) {
                double acc = (k == lane) ? -1.0 : 0.0;
#pragma unroll
                for (int m = KB - 1; m >= 0; --m)
                    if (m > k) acc += x[m] * D[m * KS + k];         // the newest x (m = k + 1) enters last
                const double dk = __shfl_sync(full, mydinv, k);
                x[k] = -acc * dk;
            }
            if (lane < KB) {
#pragma unroll
                for (int c = 0; c < KB; ++c) Lv[lane * KS + c] = x[c];
            }
        }
    };

    // C[8 rows of strip tm][all KB columns] -= A[strip tm] B^T  (SUB) or  = A[strip tm] Linv^T in place (!SUB):
    // one warp, TB independent accumulator chains on the tensor pipe
    // NS consecutive 8-row strips starting at strip tm0, all KB columns:  C -= A B^T  (strip_sub)  or
    // A <- A Linv^T in place (strip_solve).  One warp; every tile has two accumulator chains (even / odd
    // k-steps) and all NS * TB tiles are in flight together, because one FP64 mma costs far more latency
    // than issue.
    auto strip_sub = [&](auto ns_tag, double* C, const double* A, const double* B, int tm0) {
        constexpr int NS = decltype(ns_tag)::value;
        double af[NS][KB / 4];
        double cc[NS][TB][2][2];
#pragma unroll
        for (int sidx = 0; sidx < NS; ++sidx) {
            const double* ap = A + ((tm0 + sidx) * 8 + (lane >> 2)) * KS + (lane & 3);
#pragma unroll
            for (int ks = 0; ks < KB / 4; ++ks) af[sidx][ks] = -ap[ks * 4];
            const double* cp = C + ((tm0 + sidx) * 8 + (lane >> 2)) * KS + (lane & 3) * 2;
#pragma unroll
            for (int tn = 0; tn < TB; ++tn) {
                const double2 c2 = *reinterpret_cast<const double2*>(cp + tn * 8);
                cc[sidx][tn][0][0] = c2.x; cc[sidx][tn][0][1] = c2.y; cc[sidx][tn][1][0] = 0.0; cc[sidx][tn][1][1] = 0.0;
            }
        }
#pragma unroll
        for (int ks = 0; ks < KB / 4; ++ks)
#pragma unroll
            for (int tn = 0; tn < TB; ++tn) {
                const double bv = B[(tn * 8 + (lane >> 2)) * KS + (lane & 3) + ks * 4];
#pragma unroll
                for (int sidx = 0; sidx < NS; ++sidx) la_dmma(cc[sidx][tn][ks & 1][0], cc[sidx][tn][ks & 1][1], af[sidx][ks], bv);
            }
#pragma unroll
        for (int sidx = 0; sidx < NS; ++sidx) {
            double* cp = C + ((tm0 + sidx) * 8 + (lane >> 2)) * KS + (lane & 3) * 2;
#pragma unroll
            for (int tn = 0; tn < TB; ++tn)
                *reinterpret_cast<double2*>(cp + tn * 8) =
                    make_double2(cc[sidx][tn][0][0] + cc[sidx][tn][1][0], cc[sidx][tn][0][1] + cc[sidx][tn][1][1]);
        }
    };
    auto strip_solve = [&](auto ns_tag, double* A, const double* Lv, int tm0) {
        constexpr int NS = decltype(ns_tag)::value;
        double af[NS][KB / 4];
        double cc[NS][TB][2][2];
#pragma unroll
        for (int sidx = 0; sidx < NS; ++sidx) {
            const double* ap = A + ((tm0 + sidx) * 8 + (lane >> 2)) * KS + (lane & 3);
#pragma unroll
            for (int ks = 0; ks < KB / 4; ++ks) af[sidx][ks] = ap[ks * 4];
#pragma unroll
            for (int tn = 0; tn < TB; ++tn) cc[sidx][tn][0][0] = cc[sidx][tn][0][1] = cc[sidx][tn][1][0] = cc[sidx][tn][1][1] = 0.0;
        }
#pragma unroll
        for (int ks = 0; ks < KB / 4; ++ks)
#pragma unroll
            for (int tn = 0; tn < TB; ++tn)
                if (ks < 2 * (tn + 1)) {        // Linv is lower triangular
                    const double bv = Lv[(tn * 8 + (lane >> 2)) * KS + (lane & 3) + ks * 4];
#pragma unroll
                    for (int sidx = 0; sidx < NS; ++sidx) la_dmma(cc[sidx][tn][ks & 1][0], cc[sidx][tn][ks & 1][1], af[sidx][ks], bv);
                }
        __syncwarp();
#pragma unroll
        for (int sidx = 0; sidx < NS; ++sidx) {
            double* cp = A + ((tm0 + sidx) * 8 + (lane >> 2)) * KS + (lane & 3) * 2;
#pragma unroll
            for (int tn = 0; tn < TB; ++tn)
                *reinterpret_cast<double2*>(cp + tn * 8) =
                    make_double2(cc[sidx][tn][0][0] + cc[sidx][tn][1][0], cc[sidx][tn][0][1] + cc[sidx][tn][1][1]);
        }
    };
    constexpr std::integral_constant<int, 1> one_strip{};
    constexpr std::integral_constant<int, G::NSW> worker_strips{};
    // b_{t+u} -= L_ut y_t for the rows of block u: thread e of `nthreads`
    auto rhs_update = [&](int t, int u, int e) {
        if (e < KB && t + u < T) {
            const double* Lr = Wb + G::slot(t + u, u) * BLK + e * KS;
            double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
            for (int c = 0; c < KB; c += 4) {
                s0 += Lr[c] * ycur[c]; s1 += Lr[c + 1] * ycur[c + 1];
                s2 += Lr[c + 2] * ycur[c + 2]; s3 += Lr[c + 3] * ycur[c + 3];
            }
            bw[((t + u) % (Q + 1)) * KB + e] -= (s0 + s1) + (s2 + s3);
        }
    };

    while (true) {
        // ---- initial window: block rows 0..Q, then the first diagonal factor
        for (int r = 0; r <= Q && r < T; ++r) init_row(r, tid, NT);
        __syncthreads();
        if (warp == 0) potrf_inv(0);
        __syncthreads();
        LAPROF(0);
        bool broke = fail_flag != 0;
        for (int t = 0; t < T && !broke; ++t) {
            const double* Lv = Li + (t & 1) * BLK;
            // ================= B (critical): L_{t+1,t} = A_{t+1,t} Linv^T on the tensor pipe, y_t = Linv b_t
            if (t + 1 < T) {
                double* A = Wb + G::slot(t + 1, 1) * BLK;
#pragma unroll
                for (int tm = 0; tm < TB; ++tm)
                    if ((tm % NW) == warp) strip_solve(one_strip, A, Lv, tm);
            }
            if (warp == NW - 1 && lane < KB) {
                const double* bt = bw + (t % (Q + 1)) * KB;
                double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
#pragma unroll
                for (int k = 0; k < KB; k += 4) {
                    s0 += Lv[lane * KS + k] * bt[k]; s1 += Lv[lane * KS + k + 1] * bt[k + 1];
                    s2 += Lv[lane * KS + k + 2] * bt[k + 2]; s3 += Lv[lane * KS + k + 3] * bt[k + 3];
                }
                const double y = (s0 + s1) + (s2 + s3);
                ycur[lane] = y;
                yg[t * KB + lane] = y;
            }
            __syncthreads();
            LAPROF(1);

            // ================= C1 (critical): D_{t+1} -= L_{t+1,t} L_{t+1,t}^T, b_{t+1} -= L_{t+1,t} y_t
            if (t + 1 < T) {
                const double* A = Wb + G::slot(t + 1, 1) * BLK;
                double* C = Wb + G::slot(t + 1, 0) * BLK;
#pragma unroll
                for (int tm = 0; tm < TB; ++tm)
                    if ((tm % NW) == warp) strip_sub(one_strip, C, A, A, tm);
            }
            if (warp == NW - 1) rhs_update(t, 1, lane);
            __syncthreads();
            LAPROF(2);

            // ================= C2: potrf of step t+1 (warp 0)  ||  everything else of step t (workers)
            if (warp == 0) {
                // its share of the spill first (Linv_t and L_{t+1,t} are final since phase B), signalled to the
                // workers, who recycle these slots for the entering row; then the look-ahead factorisation
                double* dstg = Lg + (size_t)t * COLE;
#pragma unroll
                for (int ub = 0; ub <= (Q < 1 ? Q : 1); ++ub) {
                    if (ub > 0 && t + ub >= T) continue;
                    const double* srcb = ub == 0 ? Li + (t & 1) * BLK : Wb + G::slot(t + ub, ub) * BLK;
                    double2* dst2 = reinterpret_cast<double2*>(dstg + ub * KK);
                    for (int e = lane; e < KK / 2; e += 32) {
                        const int i = e / (KB / 2), c2 = e % (KB / 2);
                        dst2[e] = *reinterpret_cast<const double2*>(srcb + i * KS + 2 * c2);
                    }
                }
                asm volatile("bar.arrive 1, %0;\n" ::"n"(NT));
                if (t + 1 < T) potrf_inv(t + 1);
            } else {
                const int wk = warp - 1, wt = tid - 32;
                const int arow = t + 1 + Q;
                const bool enter = arow < T;
                // (a) statistics of the entering block row: loads in flight during the tensor-pipe work
                double pf[PF][2], pfb[2] = {0.0, 0.0};
#pragma unroll
                for (int i = 0; i < PF; ++i) pf[i][0] = pf[i][1] = 0.0;
                if (enter && have_stats) {
                    const double* sb = stats0 + (size_t)arow * nco;
                    const bool two = a.nsplit > 1;
#pragma unroll
                    for (int i = 0; i < PF; ++i) {
                        const int e = wt + i * NWT;
                        if (e < L) { pf[i][0] = sb[e]; if (two) pf[i][1] = sb[a.split_stride + e]; }
                    }
                    if (wt < Kr) { pfb[0] = sb[L + wt]; if (two) pfb[1] = sb[a.split_stride + L + wt]; }
                    if (a.nsplit > 2) {                       // deeper split-K: sum the rest now
#pragma unroll
                        for (int i = 0; i < PF; ++i) {
                            const int e = wt + i * NWT;
                            if (e < L) for (int sp = 2; sp < a.nsplit; ++sp) pf[i][1] += sb[sp * a.split_stride + e];
                        }
                        if (wt < Kr) for (int sp = 2; sp < a.nsplit; ++sp) pfb[1] += sb[sp * a.split_stride + L + wt];
                    }
                }
#ifdef BTF_BAND_PROFILE
                long long v0 = clock64(); wq[0] += v0 - pc0;
#endif
                // (a') the blocks further down: L_ut = A_ut Linv^T, u >= 2; then their right-hand sides
                if (Q > 1) {
                    int job = 0;
#pragma unroll
                    for (int u = 2; u <= Q; ++u) {
#pragma unroll
                        for (int tm = 0; tm < TB; tm += G::NSW) {
                            if ((job++ % NWK) != wk) continue;
                            if (t + u < T) strip_solve(worker_strips, Wb + G::slot(t + u, u) * BLK, Lv, tm);
                        }
                    }
#ifdef BTF_BAND_PROFILE
                    long long v1 = clock64(); wq[1] += v1 - v0; v0 = v1;
#endif
                    asm volatile("bar.sync 2, %0;\n" ::"n"(NWT));
#ifdef BTF_BAND_PROFILE
                    v1 = clock64(); wq[2] += v1 - v0; v0 = v1;
#endif
                }
                // (b) the trailing pairs that do not touch the diagonal block of step t+1, by 8-row strips
                {
                    int job = 0;
#pragma unroll
                    for (int uu = 2; uu <= Q; ++uu) {
#pragma unroll
                        for (int vv = 1; vv <= uu; ++vv) {
#pragma unroll
                            for (int tm = 0; tm < TB; tm += G::NSW) {
                                if ((job++ % NWK) != wk) continue;
                                if (t + uu >= T) continue;
                                strip_sub(worker_strips, Wb + G::slot(t + uu, uu - vv) * BLK, Wb + G::slot(t + uu, uu) * BLK,
                                          Wb + G::slot(t + vv, vv) * BLK, tm);
                            }
                        }
                    }
#ifdef BTF_BAND_PROFILE
                    { long long v1 = clock64(); wq[3] += v1 - v0; }
#endif
#pragma unroll
                    for (int u = 2; u <= Q; ++u)
                        if (((u - 2) % NWK) == wk) rhs_update(t, u, lane);
                }
#ifdef BTF_BAND_PROFILE
                long long w0 = clock64(); wp[0] += w0 - pc0;
#endif
                // (c) block column t -> global: Linv_t | L_1t .. L_Qt (unpadded), 16-byte stores
                {
                    double* dstg = Lg + (size_t)t * COLE;
#pragma unroll
                    for (int ub = 2; ub <= Q; ++ub) {
                        if (t + ub >= T) continue;
                        const double* srcb = Wb + G::slot(t + ub, ub) * BLK;
                        double2* dst2 = reinterpret_cast<double2*>(dstg + ub * KK);
                        for (int e = wt; e < KK / 2; e += NWT) {
                            const int i = e / (KB / 2), c2 = e % (KB / 2);
                            dst2[e] = *reinterpret_cast<const double2*>(srcb + i * KS + 2 * c2);
                        }
                    }
                    if (a.diag_chol) {
#pragma unroll
                        for (int ub = 0; ub <= Q; ++ub) {
                            if (t + ub >= T) continue;
                            const double* srcb = Wb + G::slot(t + ub, ub) * BLK;
                            for (int e = wt; e < KK; e += NWT) {
                                const int i = e / KB, c = e % KB, dist = ub * Kr + i - c;
                                if (i < Kr && c < Kr && dist >= 0 && dist <= kd)
                                    a.diag_chol[((size_t)jl * n + (t + ub) * Kr + i) * LS + kd - dist] = srcb[i * KS + c];
                            }
                        }
                    }
                }
#ifdef BTF_BAND_PROFILE
                long long w1 = clock64(); wp[1] += w1 - w0;
#endif
                // (d) the entering row reuses the slots of block column t: wait for every worker and for warp 0's spill
                asm volatile("bar.sync 1, %0;\n" ::"n"(NT));
#ifdef BTF_BAND_PROFILE
                long long w2 = clock64(); wp[2] += w2 - w1;
#endif
                if (enter) {
#pragma unroll
                    for (int i = 0; i < PF; ++i) {
                        const int e = wt + i * NWT;
                        if (e < L) put_diag(arow, e, pf[i][0] + pf[i][1]);
                    }
                    if (wt < KB) bw[(arow % (Q + 1)) * KB + wt] = (pfb[0] + pfb[1]) * scale;
                    init_rest(arow, wt, NWT);
                }
            }
#ifdef BTF_BAND_PROFILE
            { long long q0 = clock64(); pc[6] += q0 - pc0; }   // own work in C2 before the barrier
#endif
            __syncthreads();
            LAPROF(3);
            if (fail_flag) broke = true;
        }
        if (!broke) break;
        __syncthreads();
        if (tid == 0) fail_flag = 0;
        if (a.force_psd && attempt < a.attempts) {
            jitter += eps; eps *= 10.0; ++attempt;
            __syncthreads();
            continue;
        }
        failed = true;
        break;
    }
    if (tid == 0) {
        if (a.diag_retries) a.diag_retries[jl] = attempt;
        if (attempt) atomicAdd(&a.scal->retries_v, attempt);
        if (failed) atomicAdd(&a.scal->info_v, 1);
    }
    if (failed) {
        if (a.resid_partials && tid == 0) a.resid_partials[jl] = 0.0;
        return;
    }
    __syncthreads();

    // ---- backward substitution by block columns: x_t = Linv_t^T (w_t - sum_u L_ut^T x_{t+u})
    // warp 0: the draw (w = y + z); warp 1: the conditional mean (w = y), only when asked for;
    // warp 2: the normals of the next step
    double* Lc = Wb;                                   // [NST][BWD]
    constexpr int NST = G::NST;
    const unsigned long long sweep = a.scal->sweep;
    double* Vout = a.V + (size_t)jg * n;
    const bool want_mean = a.diag_mean != nullptr;
    auto fetch = [&](int t, int buf) {
        const double* src = Lg + (size_t)t * COLE;
        double* dst = Lc + buf * BWD;
        for (int e = tid; e < COLE / 2; e += NT) la_cp_async16(dst + 2 * e, src + 2 * e);
        if (tid < KB / 2) la_cp_async16(dst + COLE + 2 * tid, yg + (size_t)t * KB + 2 * tid);
    };
    auto zgen = [&](int t) {
        if (lane < KB) {
            double z = 0.0;
            if (lane < Kr) {
                if (a.z_inject) z = a.z_inject[(size_t)jg * n + t * Kr + lane];
                else { Rng rng(a.seed, STREAM_V, sweep, (uint64_t)jg * n + t * Kr + lane); z = rng.normal(); }
            }
            zb[(t & 1) * KB + lane] = z;
        }
    };
    // prefetch distance NST - 1 = 2 steps: one step is shorter than the latency of the factor coming back from HBM
    fetch(T - 1, (T - 1) % NST);
    la_cp_commit();
    if (T > 1) fetch(T - 2, (T - 2) % NST);
    la_cp_commit();
    if (warp == 2) zgen(T - 1);
    for (int t = T - 1; t >= 0; --t) {
        if (t > 1) fetch(t - 2, (t - 2) % NST);
        la_cp_commit();
        la_cp_wait<2>();
        __syncthreads();
        const double* Lt = Lc + (t % NST) * BWD;
        if (warp < 2 && (warp == 0 || want_mean)) {
            const int rhs = warp, k = lane < KB ? lane : 0;
            double r = Lt[COLE + k] + (rhs == 0 ? zb[(t & 1) * KB + k] : 0.0);
            // many short accumulator chains: every dependent FP64 operation costs its full latency
            double sa[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) sa[q] = 0.0;
#pragma unroll
            for (int ub = 1; ub <= Q; ++ub) {
                if (t + ub < T) {
                    const double* Lu = Lt + ub * KK;
                    const double* xv = xw + (rhs * (Q + 1) + (t + ub) % (Q + 1)) * KB;
#pragma unroll
                    for (int i = 0; i < KB; ++i) sa[i & 7] += Lu[i * KB + k] * xv[i];
                }
            }
            r -= ((sa[0] + sa[1]) + (sa[2] + sa[3])) + ((sa[4] + sa[5]) + (sa[6] + sa[7]));
            if (lane < KB) rb[rhs * KB + k] = r;
            __syncwarp();
            const double* rv = rb + rhs * KB;
            double xa[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) xa[q] = 0.0;
#pragma unroll
            for (int j = 0; j < KB; ++j) xa[j & 7] += Lt[j * KB + k] * rv[j];      // column k of Linv (zero above the diagonal)
            const double x0 = xa[0] + xa[1], x1 = xa[2] + xa[3], x2 = xa[4] + xa[5], x3 = xa[6] + xa[7];
            const double xk = (x0 + x1) + (x2 + x3);
            if (lane < KB) {
                xw[(rhs * (Q + 1) + t % (Q + 1)) * KB + k] = xk;
                if (k < Kr) {
                    if (rhs == 0) Vout[t * Kr + k] = xk;
                    else a.diag_mean[(size_t)jg * n + t * Kr + k] = xk;
                }
            }
        } else if (warp == 2 && t > 0) {
            zgen(t - 1);
        }
        __syncthreads();
    }
    la_cp_wait<0>();
    __syncthreads();
    LAPROF(4);

    // ---- nu2 by-product: sum_t v_t^T A_t v_t - 2 v_t . b_t with the UNSCALED statistics
    if (a.resid_partials && have_stats) {
        double accum = 0.0;
        for (int c = tid; c < nco; c += NT) {
            int k1 = 0, k2 = 0;
            double wgt = -2.0;
            if (c < L) {
                k1 = pairtab[c] >> 8; k2 = pairtab[c] & 0xff;
                wgt = k1 == k2 ? 1.0 : 2.0;
            } else {
                k1 = c - L;
            }
            const bool quad = c < L;
            const double* sb = stats0 + c;
            double p[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) p[q] = 0.0;
            int t = 0;
            // eight independent load chains per thread (the statistics come from L2 / HBM)
            for (; t + 8 <= T; t += 8) {
                double sv[8];
#pragma unroll
                for (int q = 0; q < 8; ++q) sv[q] = sb[(size_t)(t + q) * nco];
                for (int sp = 1; sp < a.nsplit; ++sp) {
                    const double* sq = sb + sp * a.split_stride + (size_t)t * nco;
#pragma unroll
                    for (int q = 0; q < 8; ++q) sv[q] += sq[(size_t)q * nco];
                }
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    const double* vt = Vout + (size_t)(t + q) * Kr;
                    p[q] += sv[q] * vt[k1] * (quad ? vt[k2] : 1.0);
                }
            }
            for (; t < T; ++t) {
                const double* vt = Vout + (size_t)t * Kr;
                p[0] += stat_sum(sb + (size_t)t * nco) * vt[k1] * (quad ? vt[k2] : 1.0);
            }
            accum += wgt * (((p[0] + p[1]) + (p[2] + p[3])) + ((p[4] + p[5]) + (p[6] + p[7])));
        }
        double tot = block_sum(accum, red);
        if (threadIdx.x == 0) a.resid_partials[jl] = tot;
    }
    LAPROF(5);
#ifdef BTF_BAND_PROFILE
    if ((tid == 0 || tid == 32) && jl == 0)
        printf("la T %d K %d tid %d: init %lld | B %lld | C1 %lld | C2 %lld (own %lld: prefetch %lld solve %lld bar2 %lld pairs %lld all-to-spill %lld spill %lld bar %lld) | backward %lld | resid %lld cycles\n",
               T, Kr, tid, pc[0], pc[1], pc[2], pc[3], pc[6], wq[0], wq[1], wq[2], wq[3], wp[0], wp[1], wp[2], pc[4], pc[5]);
    if ((tid == 64 || tid == 96) && jl == 0)
        printf("la tid %d: prefetch %lld solve %lld bar2 %lld pairs %lld all-to-spill %lld spill %lld bar %lld own %lld\n",
               tid, wq[0], wq[1], wq[2], wq[3], wp[0], wp[1], wp[2], pc[6]);
#endif
}

template <int KB, int Q>
static void launch_lookahead_t(const BandSolveArgs& a, cudaStream_t st) {
    using G = LaGeom<KB, Q>;
    const size_t smem = G::smem_doubles(a.T, a.RD) * sizeof(double);
    auto kern = band_lookahead_kernel<KB, Q>;
    static PerDeviceMax max_set;
    if (smem > 48 * 1024 && max_set.raise(smem)) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    kern<<<a.ncols_loc, G::NT, smem, st>>>(a);
}

bool launch_band_solve_lookahead(const BandSolveArgs& a, cudaStream_t st) {
    const int Q = a.order + 1;
#define BTF_LA(KB_)                                                     \
    do {                                                                \
        switch (Q) {                                                    \
            case 1: launch_lookahead_t<KB_, 1>(a, st); return true;     \
            case 2: launch_lookahead_t<KB_, 2>(a, st); return true;     \
            case 3: launch_lookahead_t<KB_, 3>(a, st); return true;     \
            case 4: launch_lookahead_t<KB_, 4>(a, st); return true;     \
            default: return false;                                      \
        }                                                               \
    } while (0)
    if (a.K <= 8) BTF_LA(8);
    if (a.K <= 16) BTF_LA(16);
    if (a.K <= 32) BTF_LA(32);
#undef BTF_LA
    return false;
}

}  // namespace btf
