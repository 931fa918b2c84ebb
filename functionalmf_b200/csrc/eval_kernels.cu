// Held-out evaluation of the chain on the device (SURVEY.md 8f row 3).
//
// The reference scripts keep every saved (W, V) sample on the host, rebuild
// Mu = einsum('znk,zmtk->znmt') there and score it with numpy:
//   politics/benchmark.py:163-180   per-sample RMSE / MAE / Poisson log-likelihood of the NB mean
//                                   R P / (1 - P), P = ilogit(clip(psi, -10, 10)) (155-156),
//                                   split into in-sample and held-out cells, averaged over samples;
//   flutrends/benchmark.py:129-143  RMSE / MAE of the posterior-mean surface and coverage of the
//                                   posterior-predictive band (68-75);
//   examples/poisson_tensor_filtering.py:20-23, 165-173  coverage of a truth by the central
//                                   percentile band of the samples (np.percentile, linear).
// Here one pass per saved sample (eval_update_kernel) recomputes the cell means from the resident
// factors and updates (a) per-sample per-class error sums and (b) an O(1) per-cell state from which
// the percentile-band membership of the target is decided EXACTLY without storing or sorting the
// samples: with c_lt = #{x_s < y}, c_le = #{x_s <= y}, lo = max{x_s < y}, hi = min{x_s > y}, the two
// order statistics that bracket any percentile position are known whenever the target lies between
// them, and in every other case the comparison is decided by the counts alone.
//
// HBM traffic per saved sample: target 8 B + class 1 B per cell, + 2 x 40 B of per-cell state when
// it is kept; the K-term dot product per cell is free next to that.
#include <algorithm>
#include "kernels.h"

namespace btf {

namespace {

__device__ __forceinline__ double eval_transform(const EvalArgs& a, double psi, int il, int p) {
    if (a.transform == EVAL_IDENTITY) return psi;
    const double pc = clampd(psi, -10.0, 10.0);
    if (a.transform == EVAL_ILOGIT) return 1.0 / (1.0 + exp(-psi));
    // EVAL_NB_MEAN: R P / (1 - P) = R exp(clip(psi)) (politics/benchmark.py:155-156)
    const int j = p / a.T, t = p - j * a.T;
    const int g = ((a.Rn > 1 ? a.row_begin + il : 0) * a.Rm + (a.Rm > 1 ? j : 0)) * a.Rt + (a.Rt > 1 ? t : 0);
    const double P = 1.0 / (1.0 + exp(-pc));
    return a.Rdisp[g] * P / (1.0 - P);
}

__device__ __forceinline__ double eval_loglik(int kind, double y, double mu, double nu2) {
    if (kind == EVAL_LL_POISSON)   // scipy.stats.poisson.logpmf = xlogy(y, mu) - lgamma(y + 1) - mu
        return (y == 0.0 ? 0.0 : y * log(mu)) - lgamma(y + 1.0) - mu;
    if (kind == EVAL_LL_GAUSSIAN) {
        const double d = y - mu;
        return -0.5 * (log(6.283185307179586477 * nu2) + d * d / nu2);
    }
    return 0.0;
}

// numpy's _lerp (numpy/lib/_function_base_impl.py): a + (b-a) t, from the far end when t >= 0.5
__device__ __forceinline__ double np_lerp(double a, double b, double t) {
    const double d = b - a;
    double r = t >= 0.5 ? b - d * (1.0 - t) : a + d * t;
    if (d == 0.0) r = a;
    return r;
}

}  // namespace

// 64 rows x 256 cells per block: thread = one (column, depth) cell position p with its V row in
// registers, walking the block's rows in batches whose loads are all issued before any is used
// (one load round trip per batch instead of per cell: the pass is latency bound otherwise).
template <int KMAX, bool STATE>
__global__ void __launch_bounds__(256, KMAX <= 16 ? 2 : 1) eval_update_kernel(EvalArgs a) {
    constexpr int B = STATE ? 4 : 8;
    __shared__ double ws[64 * KMAX];
    __shared__ double red[8][EVAL_MAX_CLASSES * 4];
    const int K = a.K;
    const int p = blockIdx.x * 256 + threadIdx.x;
    const int i0 = blockIdx.y * 64;
    const int nr = min(64, a.nloc - i0);
    for (int e = threadIdx.x; e < nr * K; e += 256) ws[e] = a.W[(long long)i0 * K + e];
    double v[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) v[k] = (k < K && p < a.P) ? a.V[(long long)p * K + k] : 0.0;
    __syncthreads();
    const double nu2 = a.scal->nu2;
    const double inv_sd = rsqrt(nu2), inv_nu2 = 1.0 / nu2, lognorm = log(6.283185307179586477 * nu2);
    const double inv_count = 1.0 / a.count;
    const bool live = p < a.P;
    double acc[EVAL_MAX_CLASSES][4];
    unsigned ncell[EVAL_MAX_CLASSES];
#pragma unroll
    for (int c = 0; c < EVAL_MAX_CLASSES; ++c) {
        ncell[c] = 0u;
#pragma unroll
        for (int m = 0; m < 4; ++m) acc[c][m] = 0.0;
    }
    for (int r0 = 0; r0 < nr; r0 += B) {
        double yv[B], nv[B];
        int cv[B];
        double mv[B], bv[B], av[B], fv[B];
        unsigned ltv[B], lev[B];
#pragma unroll
        for (int u = 0; u < B; ++u) {
            const bool ok = live && r0 + u < nr;
            const long long o = (long long)(i0 + r0 + u) * a.P + p;
            yv[u] = ok ? a.target[o] : NAN;
            cv[u] = ok ? (a.cls ? (int)a.cls[o] : 0) : 255;
            nv[u] = (ok && a.nu2c) ? a.nu2c[o] : nu2;
        }
        if (STATE) {
#pragma unroll
            for (int u = 0; u < B; ++u) {
                const long long o = (long long)(i0 + r0 + u) * a.P + p;
                const bool on = yv[u] == yv[u] && cv[u] < a.ncls;
                mv[u] = on ? a.mean[o] : 0.0;
                bv[u] = on ? a.below[o] : 0.0;
                av[u] = on ? a.above[o] : 0.0;
                ltv[u] = on ? a.c_lt[o] : 0u;
                lev[u] = on ? a.c_le[o] : 0u;
                fv[u] = (on && a.cdf) ? a.cdf[o] : 0.0;
            }
        }
#pragma unroll
        for (int u = 0; u < B; ++u) {
            const double y = yv[u];
            const int cl = cv[u];
            if (y != y || cl >= a.ncls) continue;
            const int r = r0 + u;
            const long long o = (long long)(i0 + r) * a.P + p;
            double psi = 0.0;
#pragma unroll
            for (int k = 0; k < KMAX; ++k)
                if (k < K) psi += ws[r * K + k] * v[k];
            const double mu = eval_transform(a, psi, i0 + r, p);
            const double d = y - mu;
            double ln = lognorm, inu = inv_nu2, isd = inv_sd;
            if (a.nu2c) { ln = log(6.283185307179586477 * nv[u]); inu = 1.0 / nv[u]; isd = rsqrt(nv[u]); }
            double ll = 0.0;
            if (a.loglik == EVAL_LL_GAUSSIAN) ll = -0.5 * (ln + d * d * inu);
            else if (a.loglik == EVAL_LL_POISSON) ll = eval_loglik(EVAL_LL_POISSON, y, mu, nu2);
#pragma unroll
            for (int c = 0; c < EVAL_MAX_CLASSES; ++c) {
                const bool on = cl == c;
                ncell[c] += on ? 1u : 0u;
                acc[c][1] += on ? d * d : 0.0;
                acc[c][2] += on ? fabs(d) : 0.0;
                acc[c][3] += on ? ll : 0.0;
            }
            if (STATE) {
                a.mean[o] = mv[u] + (mu - mv[u]) * inv_count;
                if (mu < y) {
                    a.c_lt[o] = ltv[u] + 1; a.c_le[o] = lev[u] + 1;
                    if (mu > bv[u]) a.below[o] = mu;
                } else if (mu == y) a.c_le[o] = lev[u] + 1;
                else if (mu < av[u]) a.above[o] = mu;
                if (a.cdf) a.cdf[o] = fv[u] + 0.5 * erfc(-(d * isd) * 0.70710678118654752440);
            }
        }
    }
    // fixed-order block reduction: warp shuffles, then the 8 warp partials in order
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int c = 0; c < EVAL_MAX_CLASSES; ++c)
#pragma unroll
        for (int m = 0; m < 4; ++m) {
            const double sw = warp_sum(m == 0 ? (double)ncell[c] : acc[c][m]);
            if (lane == 0) red[w][c * 4 + m] = sw;
        }
    __syncthreads();
    if (threadIdx.x < a.ncls * 4) {
        double sum = 0.0;
        for (int ww = 0; ww < 8; ++ww) sum += red[ww][threadIdx.x];
        a.partial[((long long)blockIdx.y * gridDim.x + blockIdx.x) * (a.ncls * 4) + threadIdx.x] = sum;
    }
}

// out[v] = sum_b partial[b][v] in a fixed order; one block per output value
__global__ void __launch_bounds__(256) eval_reduce_kernel(const double* __restrict__ partial, int nblocks, int nvals,
                                                          double* __restrict__ out) {
    __shared__ double red[32];
    const int v = blockIdx.x;
    double s = 0.0;
    for (int b = threadIdx.x; b < nblocks; b += 256) s += partial[(long long)b * nvals + v];
    s = block_sum(s, red);
    if (threadIdx.x == 0) out[v] = s;
}

void launch_eval_update(const EvalArgs& a, double* sample_out, cudaStream_t st) {
    dim3 grid((a.P + 255) / 256, (a.nloc + 63) / 64);
    if (a.mean) {
        if (a.K <= 8) eval_update_kernel<8, true><<<grid, 256, 0, st>>>(a);
        else if (a.K <= 16) eval_update_kernel<16, true><<<grid, 256, 0, st>>>(a);
        else eval_update_kernel<32, true><<<grid, 256, 0, st>>>(a);
    } else {
        if (a.K <= 8) eval_update_kernel<8, false><<<grid, 256, 0, st>>>(a);
        else if (a.K <= 16) eval_update_kernel<16, false><<<grid, 256, 0, st>>>(a);
        else eval_update_kernel<32, false><<<grid, 256, 0, st>>>(a);
    }
    eval_reduce_kernel<<<a.ncls * 4, 256, 0, st>>>(a.partial, (int)(grid.x * grid.y), a.ncls * 4, sample_out);
}
long long eval_partial_elems(int nloc, int P, int ncls) {
    return (long long)((P + 255) / 256) * ((nloc + 63) / 64) * ncls * 4;
}

// initial per-cell state: below = -inf, above = +inf, everything else 0
__global__ void eval_init_kernel(double* below, double* above, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { below[i] = -INFINITY; above[i] = INFINITY; }
}
void launch_eval_init(double* below, double* above, long long n, cudaStream_t st) {
    eval_init_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(below, above, n);
}

// Scores of the posterior-mean surface and band membership per class:
// out[c] = {n, sum (y - mean)^2, sum |y - mean|, sum loglik(y | mean), #covered by the
//           [lo_pct, hi_pct] percentile band of the samples, #with lo_frac <= mean cdf <= hi_frac}
__global__ void __launch_bounds__(256) eval_summary_kernel(EvalArgs a, double lo_pct, double hi_pct, double lo_frac,
                                                           double hi_frac, double* __restrict__ partial) {
    __shared__ double red[32];
    const long long cells = (long long)a.nloc * a.P;
    const double S = a.count;
    // numpy: virtual index = (n - 1) * (q / 100)
    const double h_lo = (S - 1.0) * (lo_pct / 100.0), h_hi = (S - 1.0) * (hi_pct / 100.0);
    const double j_lo = floor(h_lo), g_lo = h_lo - j_lo, j_hi = floor(h_hi), g_hi = h_hi - j_hi;
    const double nu2 = a.scal->nu2;
    double acc[EVAL_MAX_CLASSES][6];
#pragma unroll
    for (int c = 0; c < EVAL_MAX_CLASSES; ++c)
#pragma unroll
        for (int m = 0; m < 6; ++m) acc[c][m] = 0.0;
    for (long long o = (long long)blockIdx.x * 256 + threadIdx.x; o < cells; o += (long long)gridDim.x * 256) {
        const double y = a.target[o];
        if (y != y) continue;
        const int cl = a.cls ? (int)a.cls[o] : 0;
        if (cl >= a.ncls) continue;
        const double mean = a.mean[o];
        const double d = y - mean;
        const double ll = eval_loglik(a.loglik, y, mean, a.nu2c ? a.nu2c[o] : nu2);
        const double c_lt = (double)a.c_lt[o], c_le = (double)a.c_le[o];
        const bool tie = c_le > c_lt;
        // lower end: y >= Q(lo)
        bool ok_lo;
        if (c_le >= j_lo + 2.0) ok_lo = true;
        else if (c_le <= j_lo) ok_lo = false;
        else if (j_lo + 1.0 > S - 1.0) ok_lo = true;
        else ok_lo = y >= np_lerp(tie ? y : a.below[o], a.above[o], g_lo);
        // upper end: y <= Q(hi)
        bool ok_hi;
        if (c_lt <= j_hi) ok_hi = true;
        else if (c_lt >= j_hi + 2.0 || j_hi + 1.0 > S - 1.0) ok_hi = false;
        else ok_hi = y <= np_lerp(a.below[o], tie ? y : a.above[o], g_hi);
        const double F = a.cdf ? a.cdf[o] / S : 0.0;
        const bool ok_pred = a.cdf && F >= lo_frac && F <= hi_frac;
#pragma unroll
        for (int c = 0; c < EVAL_MAX_CLASSES; ++c) {
            const bool on = cl == c;
            acc[c][0] += on ? 1.0 : 0.0;
            acc[c][1] += on ? d * d : 0.0;
            acc[c][2] += on ? fabs(d) : 0.0;
            acc[c][3] += on ? ll : 0.0;
            acc[c][4] += (on && ok_lo && ok_hi) ? 1.0 : 0.0;
            acc[c][5] += (on && ok_pred) ? 1.0 : 0.0;
        }
    }
    for (int c = 0; c < a.ncls; ++c)
#pragma unroll
        for (int m = 0; m < 6; ++m) {
            double val = 0.0;
#pragma unroll
            for (int cc = 0; cc < EVAL_MAX_CLASSES; ++cc) val = cc == c ? acc[cc][m] : val;
            const double s = block_sum(val, red);
            if (threadIdx.x == 0) partial[(long long)blockIdx.x * (a.ncls * 6) + c * 6 + m] = s;
        }
}

int eval_summary_blocks(int nloc, int P) {
    const long long cells = (long long)nloc * P;
    return (int)std::min<long long>((cells + 255) / 256, 148 * 8);
}
void launch_eval_summary(const EvalArgs& a, double lo_pct, double hi_pct, double lo_frac, double hi_frac,
                         double* partial, double* out, cudaStream_t st) {
    const int nb = eval_summary_blocks(a.nloc, a.P);
    eval_summary_kernel<<<nb, 256, 0, st>>>(a, lo_pct, hi_pct, lo_frac, hi_frac, partial);
    eval_reduce_kernel<<<a.ncls * 6, 256, 0, st>>>(partial, nb, a.ncls * 6, out);
}

}  // namespace btf
