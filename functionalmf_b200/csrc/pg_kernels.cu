// K4a: on-device Polya-Gamma sampler (replaces pypolyagamma's pgdrawv, factor.py:431-432, 459)
// K4c: negative-binomial dispersion update by random-walk MH (factor.py:513-554)
//
// PG(1, z): Devroye's exact alternating-series sampler (Polson, Scott & Windle 2013,
// Alg. 1; truncation t = 0.64).  PG(b, z): floor(b) such draws + truncated
// sum-of-gammas for the fractional part (tail replaced by its moment-matched normal); b > 170: the
// moment-matched normal approximation (the rule of the hybrid sampler the
// reference's third-party dependency implements).  All randomness is Philox,
// keyed by (seed, sweep, global cell index).
#include <cstdlib>
#include "kernels.h"

namespace btf {

#define PG_TRUNC 0.64
#define PG_PI 3.14159265358979323846
#define PG_NORMAL_B 170.0
#define PG_SERIES 32

__device__ __forceinline__ double log_phi(double x) {
    if (x > -5.0) return log(0.5 * erfc(-x * 0.70710678118654752440));
    double u = -x * 0.70710678118654752440;
    return log(0.5 * erfcx(u)) - u * u;
}

// 1/d for a positive, finite, normal d: hardware seed (relative error < 2^-20) and one third-order step
// y0 (1 + e + e^2), e = 1 - d y0  ->  relative error ~2^-60 plus rounding.  No special-case branch: the IEEE division
// the compiler emits carries a slow path that is never taken here but costs instruction-cache and issue slots.
__device__ __forceinline__ double pg_rcp_pos(double d) {
    double y0;
    asm("rcp.approx.ftz.f64 %0, %1;\n" : "=d"(y0) : "d"(d));
    const double e = fma(-d, y0, 1.0);
    const double e2 = fma(e, e, e);
    return fma(e2, y0, y0);
}

struct PgTilt { double Z, inv_fz, inv_p, inv_qp; };   // per cell; reused by every draw of the cell

__device__ __forceinline__ PgTilt pg_setup(double z) {
    PgTilt c;
    c.Z = 0.5 * fabs(z);
    const double fz = PG_PI * PG_PI / 8.0 + 0.5 * c.Z * c.Z;
    const double rt = 1.25;   // sqrt(1 / 0.64)
    double b = rt * (PG_TRUNC * c.Z - 1.0), a = -rt * (PG_TRUNC * c.Z + 1.0);
    double qdivp;   // q / p: mass of the truncated inverse-Gaussian part over the mass of the exponential tail
    if (c.Z < 12.0) {
        // fz exp(fz t) [exp(-Z) Phi(b) + exp(Z) Phi(a)] without logarithms or divisions (no overflow for |z| < 24)
        const double pb = 0.5 * erfc(-b * 0.70710678118654752440), pa = 0.5 * erfc(-a * 0.70710678118654752440);
        const double x0 = fz * PG_TRUNC;
        qdivp = 4.0 / PG_PI * fz * (exp(x0 - c.Z) * pb + exp(x0 + c.Z) * pa);
    } else {
        const double x0 = log(fz) + fz * PG_TRUNC;
        qdivp = 4.0 / PG_PI * (exp(x0 - c.Z + log_phi(b)) + exp(x0 + c.Z + log_phi(a)));
    }
    // q / p grows like exp(0.32 Z^2): it overflows to inf for |z| > ~97, and past 2^1022 its hardware reciprocal
    // flushes to zero; (up - 1) * inv_qp would then be NaN (inf * 0) or 0 instead of a uniform, and the
    // inverse-Gaussian proposal would never take its mu^2 / X root.  From 2^900 on the exponential tail's probability
    // 1 / (1 + q/p) is below 2^-900, far under the 2^-53 resolution of u1, so every draw takes the inverse-Gaussian
    // branch; with q/p capped at that power of two, up = u1 2^900 and (up - 1) 2^-900 round to exactly u1, the
    // proper U(0,1) of the branch.
    if (!(qdivp < 0x1p900)) qdivp = 0x1p900;
    c.inv_fz = pg_rcp_pos(fz);
    c.inv_p = 1.0 + qdivp;                               // 1 / P(exponential tail)
    c.inv_qp = qdivp > 1e-300 ? pg_rcp_pos(qdivp) : 0.0;  // (u1 / p - 1) / (q / p) is U(0,1) given the inverse-Gaussian branch
    return c;
}

__device__ __forceinline__ double pg_acoef(int n, double x) {
    const double k = (n + 0.5) * PG_PI;
    if (x > PG_TRUNC) return k * exp(-0.5 * k * k * x);
    return exp(-1.5 * (log(0.5 * PG_PI) + log(x)) + log(k) - 2.0 * (n + 0.5) * (n + 0.5) / x);
}

// Accept/reject DECISIONS  u <= exp(x)  are taken in FP32 when they are not borderline and
// re-evaluated in FP64 otherwise, so every decision equals the FP64 one while most FP64
// exponentials disappear; all VALUES that reach the output are computed in FP64.
__device__ __forceinline__ bool leq_exp(double u, double x) {
    const float ef = __expf((float)x), uf = (float)u;
    if (uf < ef * 0.9999f - 1e-30f) return true;
    if (uf > ef * 1.0001f + 1e-30f) return false;
    return u <= exp(x);
}

// A decision uniform is consumed 32 bits at a time: its leading word decides everything but a borderline
// (probability ~1e-4) case, for which 32 more bits are drawn - the comparison is the one a 64-bit uniform gives,
// at half a Philox call per decision.
__device__ __forceinline__ double refine_uniform(Rng& rng, uint32_t hi) {
    const uint4 q = rng.next4();
    return ((double)(((unsigned long long)hi << 32) | q.x) + 0.5) * (1.0 / 18446744073709551616.0);
}
__device__ __forceinline__ bool leq_exp32(Rng& rng, uint32_t hi, double x) {
    const float ef = __expf((float)x), uf = ((float)hi + 0.5f) * 2.3283064365386963e-10f;
    if (uf < ef * 0.9999f - 1e-30f) return true;
    if (uf > ef * 1.0001f + 1e-30f) return false;
    return refine_uniform(rng, hi) <= exp(x);
}

// Truncated inverse-Gaussian(1/Z, 1) on (0, t].  `u0` is a spare value uniform and `a_hi` a spare 32-bit decision
// word the caller already holds, so the common path costs no Philox call of its own.
//
// mu = 1/Z > t: Polson-Scott-Windle propose X = t / (1 + t E)^2 with E accepted from Exp(1) with probability
// exp(-t E^2 / 2), i.e. E ~ N(-1/t, 1/t) truncated to E > 0.  With Y = sqrt(t) (E + 1/t) that is X = 1 / Y^2 for a
// standard normal Y truncated to Y > 1/sqrt(t) - the Levy law cut at t - so the inner rejection loop (acceptance
// 0.69 per lane: a warp iterated until its slowest lane got through, ~4 rounds of Philox + log + exp each) is
// replaced by ONE inversion Y = Phi^-1(U Phi(-1/sqrt(t))): same distribution, no loop, no divergence.
__device__ double pg_rtigauss(Rng& rng, double Z, double u0, uint32_t a_hi, double& inv_x) {
    const double t = PG_TRUNC;
    bool first = true;
    if (!(Z > 1.0 / t)) {   // mu = 1/Z > t (including Z == 0)
        const double QT = 0.10564977366685535;      // Phi(-1.25), 1/sqrt(0.64) = 1.25
        const double hz2 = -0.5 * Z * Z;
        for (int it = 0; it < 10000; ++it) {
            double uv;
            uint32_t ah;
            if (first) { uv = u0; ah = a_hi; first = false; }
            else { const uint4 r = rng.next4(); uv = Rng::to_unit(r.x, r.y); ah = r.z; }
            const double Y = normcdfinv(fmax(uv, 1e-300) * QT);   // < -1.25
            const double Y2 = Y * Y;
            const double X = pg_rcp_pos(Y2);                        // <= t
            if (leq_exp32(rng, ah, hz2 * X)) { inv_x = Y2; return X; }
        }
        inv_x = 1.0 / t;
        return t;
    }
    const double mu = pg_rcp_pos(Z);
    for (int it = 0; it < 10000; ++it) {
        double2 nu = rng.normal2();
        double ua = first ? u0 : rng.uniform();
        first = false;
        double Y = nu.x * nu.x;
        double X = mu + 0.5 * mu * mu * Y - 0.5 * mu * sqrt(4.0 * mu * Y + (mu * Y) * (mu * Y));
        if (ua > mu / (mu + X)) X = mu * mu / X;
        if (X <= t) { inv_x = 1.0 / X; return X; }
    }
    inv_x = 1.0 / t;
    return t;
}

// One PG(1, z) draw (Devroye / Polson-Scott-Windle alternating series): ONE Philox call on the common path - 53
// bits for the proposal's value, 32 bits for each of the two decisions (refined when borderline).  The first
// acceptance test  U a_0 <= a_0 - a_1  only needs the ratio a_1 / a_0 = 3 exp(-4/x) (x <= t)
// or 3 exp(-pi^2 x) (x > t); the full coefficients are evaluated only on the rare (< 0.6 %)
// continuation of the series.
__device__ double pg_one(Rng& rng, const PgTilt& c) {
    for (int it = 0; it < 10000; ++it) {
        const uint4 r = rng.next4();
        const double u1 = Rng::to_unit(r.x, r.y);
        double X, arg;
        const double up = u1 * c.inv_p;                                   // u1 / P(tail): < 1 selects the exponential tail
        if (up < 1.0) {
            X = PG_TRUNC - log(up) * c.inv_fz;                            // up is U(0,1) given the branch; X > t
            arg = -PG_PI * PG_PI * X;
        } else {
            double inv_x;
            X = pg_rtigauss(rng, c.Z, (up - 1.0) * c.inv_qp, r.z, inv_x);  // X <= t, inv_x = 1 / X without a division
            arg = -4.0 * inv_x;
        }
        // u2 <= 1 - 3 exp(arg): FP32 screen (the threshold is within 2e-2 of 1), full precision when borderline
        const float thr = 1.0f - 3.0f * __expf((float)arg);
        const float u2f = ((float)r.w + 0.5f) * 2.3283064365386963e-10f;
        if (u2f < thr - 2e-6f) return 0.25 * X;
        const double u2 = refine_uniform(rng, r.w);
        if (u2f <= thr + 2e-6f && u2 <= 1.0 - 3.0 * exp(arg)) return 0.25 * X;
        // continue the series from n = 2 with explicit coefficients
        double S = pg_acoef(0, X);
        const double Y = u2 * S;
        S -= pg_acoef(1, X);
        if (Y <= S) return 0.25 * X;               // (the screen above is a bound on the same test)
        for (int n = 2; n < 400; ++n) {
            if (n & 1) { S -= pg_acoef(n, X); if (Y <= S) return 0.25 * X; }
            else { S += pg_acoef(n, X); if (Y > S) break; }
        }
    }
    return 0.25 * PG_TRUNC;
}

__device__ __forceinline__ double pg_mean(double b, double z) {
    z = fabs(z);
    if (z < 1e-6) return b * 0.25 * (1.0 - z * z / 12.0);
    return b * tanh(0.5 * z) / (2.0 * z);
}
__device__ __forceinline__ double pg_var(double b, double z) {
    z = fabs(z);
    if (z < 1e-3) return b * (1.0 / 24.0) * (1.0 - z * z * 0.2);
    // (sinh z - z) / cosh^2(z/2) = 2 tanh(z/2) - z sech^2(z/2): finite for every z, where the quotient is
    // inf / inf = NaN past z = 710
    const double sech = 1.0 / cosh(0.5 * z);
    return b * (2.0 * tanh(0.5 * z) - z * sech * sech) / (4.0 * z * z * z);
}

__device__ double pg_draw(Rng& rng, double b, double z) {
    if (!(b > 0.0) || isinf(b) || !(z == z) || isinf(z)) return 0.0;
    if (b > PG_NORMAL_B) {
        double v = pg_mean(b, z) + sqrt(pg_var(b, z)) * rng.normal();
        return v > 0.0 ? v : pg_mean(b, z);
    }
    const PgTilt c = pg_setup(z);
    const int bi = (int)floor(b);
    const double bf = b - bi;
    double acc = 0.0;
    for (int k = 0; k < bi; ++k) acc += pg_one(rng, c);
    if (bf > 1e-12) {
        // fractional part: PG(bf, z) = 2 sum_k g_k / d_k, g_k ~ Gamma(bf, 1), d_k = 4 pi^2 (k-1/2)^2 + z^2.
        // The first PG_SERIES terms are drawn; the remainder (about 1 % of the mass, a sum of many
        // small independent terms) is replaced by a normal with its exact mean and variance.
        double s = 0.0, d1 = 0.0, d2 = 0.0;
        for (int k = 1; k <= PG_SERIES; ++k) {
            const double km = k - 0.5;
            const double d = 4.0 * PG_PI * PG_PI * km * km + z * z;
            const double di = 1.0 / d;
            s += rng.gamma(bf) * di;
            d1 += di;
            d2 += di * di;
        }
        const double tail_mean = pg_mean(bf, z) - 2.0 * bf * d1;
        const double tail_var = fmax(pg_var(bf, z) - 4.0 * bf * d2, 0.0);
        acc += 2.0 * s + fmax(tail_mean + sqrt(tail_var) * rng.normal(), 0.0);
    }
    return acc;
}

// ---------------------------------------------------------------- omega ~ PG(ntr, w.v)
template <int KMAX, int MINB>
__global__ void __launch_bounds__(256, MINB) pg_draw_kernel(PgArgs a) {
    __shared__ double ws[32 * KMAX];
    const int K = a.K;
    const int p = blockIdx.x * 256 + threadIdx.x;
    const int i0 = blockIdx.y * 32;
    for (int e = threadIdx.x; e < 32 * K; e += 256) ws[e] = a.W[(size_t)i0 * K + e];
    double v[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) v[k] = (k < K && p < a.Ppad) ? a.V[(size_t)p * K + k] : 0.0;
    __syncthreads();
    if (p >= a.P) return;
    const unsigned long long sweep = a.scal->sweep;
    // the observed flag and the trial count of row r + 1 are loaded while row r is sampled (the loads were 10 % of the
    // stall samples: every row started with a dependent global load)
    const int nrow = min(32, a.nloc - i0);
    unsigned char ob_n = 0; double nt_n = 0.0;
    if (nrow > 0) { const size_t o0 = (size_t)i0 * a.ld + p; ob_n = a.obs[o0]; nt_n = a.ntr[o0]; }
    for (int r = 0; r < nrow; ++r) {
        const int il = i0 + r;
        const size_t o = (size_t)il * a.ld + p;
        const unsigned char ob = ob_n; const double nt = nt_n;
        if (r + 1 < nrow) { ob_n = a.obs[o + a.ld]; nt_n = a.ntr[o + a.ld]; }
        double om = 0.0;
        if (ob) {
            double psi = 0.0;
#pragma unroll
            for (int k = 0; k < KMAX; ++k)
                if (k < K) psi += ws[r * K + k] * v[k];
            Rng rng(a.seed, STREAM_PG, sweep, (uint64_t)(a.row_begin + il) * a.P + p);
            om = pg_draw(rng, nt, psi);
        }
        a.omega[o] = om;
    }
}

// Small tensors (fewer cells than the GPU has thread slots): G lanes share one cell.  A PG(b, z)
// draw is a sum of floor(b) independent PG(1, z) draws plus a fractional term, each a long chain
// of FP64 transcendentals, so the sum is split over the lanes (lane l takes draws l, l+G, ... and the
// series terms k = l+1, l+1+G, ... of the fractional part, on its own Philox stream) and added up
// with shuffles.  Same distribution as pg_draw; the streams differ from the one-thread-per-cell kernel.
template <int G>
__global__ void __launch_bounds__(256) pg_draw_group_kernel(PgArgs a) {
    const long long gt = (long long)blockIdx.x * 256 + threadIdx.x;
    const long long cell = gt / G;
    const int l = (int)(gt % G);
    const long long cells = (long long)a.nloc * a.P;
    const bool in = cell < cells;
    const int il = in ? (int)(cell / a.P) : 0, p = in ? (int)(cell - (long long)il * a.P) : 0;
    const size_t o = (size_t)il * a.ld + p;
    const bool obs = in && a.obs[o];
    double acc = 0.0;
    double b = 0.0, z = 0.0;
    bool series = false;
    double s = 0.0, d1 = 0.0, d2 = 0.0, bf = 0.0;
    if (obs) {
        const double* w = a.W + (size_t)il * a.K;
        const double* v = a.V + (size_t)p * a.K;
        for (int k = 0; k < a.K; ++k) z += w[k] * v[k];
        b = a.ntr[o];
        const bool bad = !(b > 0.0) || isinf(b) || !(z == z) || isinf(z);
        Rng rng(a.seed, STREAM_PG + 16u * (uint32_t)(l + 1), a.scal->sweep, (uint64_t)(a.row_begin + il) * a.P + p);
        if (bad) {
            b = 0.0;
        } else if (b > PG_NORMAL_B) {
            if (l == 0) {
                const double m = pg_mean(b, z);
                const double vv = m + sqrt(pg_var(b, z)) * rng.normal();
                acc = vv > 0.0 ? vv : m;
            }
        } else {
            const PgTilt c = pg_setup(z);
            const int bi = (int)floor(b);
            bf = b - bi;
            for (int k = l; k < bi; k += G) acc += pg_one(rng, c);
            if (bf > 1e-12) {
                series = true;
                for (int k = 1 + l; k <= PG_SERIES; k += G) {
                    const double km = k - 0.5;
                    const double d = 4.0 * PG_PI * PG_PI * km * km + z * z;
                    const double di = 1.0 / d;
                    s += rng.gamma(bf) * di;
                    d1 += di;
                    d2 += di * di;
                }
            }
        }
    }
    // fixed-order sums inside the lane group (groups are aligned inside the warp)
#pragma unroll
    for (int off = G / 2; off > 0; off >>= 1) {
        acc += __shfl_xor_sync(0xffffffffu, acc, off);
        s += __shfl_xor_sync(0xffffffffu, s, off);
        d1 += __shfl_xor_sync(0xffffffffu, d1, off);
        d2 += __shfl_xor_sync(0xffffffffu, d2, off);
    }
    if (in && l == 0) {
        if (series) {
            Rng rng(a.seed, STREAM_PG, a.scal->sweep, (uint64_t)(a.row_begin + il) * a.P + p);
            const double tail_mean = pg_mean(bf, z) - 2.0 * bf * d1;
            const double tail_var = fmax(pg_var(bf, z) - 4.0 * bf * d2, 0.0);
            acc += 2.0 * s + fmax(tail_mean + sqrt(tail_var) * rng.normal(), 0.0);
        }
        a.omega[o] = obs ? acc : 0.0;
    }
}

void launch_pg_draw(const PgArgs& a, cudaStream_t st) {
    const long long cells = (long long)a.nloc * a.P;
    // lane groups while the one-thread-per-cell kernel would leave most of the 148 x 2048 thread slots empty
    int G = 1;
    while (G < 8 && cells * (2 * G) <= (1ll << 20)) G *= 2;
    if (G > 1) {
        const unsigned nb = (unsigned)((cells * G + 255) / 256);
        if (G == 2) pg_draw_group_kernel<2><<<nb, 256, 0, st>>>(a);
        else if (G == 4) pg_draw_group_kernel<4><<<nb, 256, 0, st>>>(a);
        else pg_draw_group_kernel<8><<<nb, 256, 0, st>>>(a);
        return;
    }
    dim3 grid((a.P + 255) / 256, (a.nloc + 31) / 32);
    // 80 registers / three CTAs per SM instead of 126 / two (the sampler is a chain of dependent FP64 operations: more
    // resident warps hide more of its latency, at the price of a few spilled values): 11.4 -> 10.4 ms at C3
    if (a.K <= 8) pg_draw_kernel<8, 3><<<grid, 256, 0, st>>>(a);
    else if (a.K <= 16) pg_draw_kernel<16, 3><<<grid, 256, 0, st>>>(a);
    else pg_draw_kernel<32, 2><<<grid, 256, 0, st>>>(a);
}

__global__ void pg_sample_kernel(const double* b, const double* z, double* out, long long n, uint64_t seed,
                                 unsigned long long sweep) {
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    Rng rng(seed, STREAM_PG, sweep, (uint64_t)e);
    out[e] = pg_draw(rng, b[e], z[e]);
}
void launch_pg_sample(const double* b, const double* z, double* out, long long n, uint64_t seed,
                      unsigned long long sweep, cudaStream_t st) {
    pg_sample_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(b, z, out, n, seed, sweep);
}

// raw variates of the device generator, for moment tests: kind 0 normal, 1 gamma(param),
// 2 exponential, 3 uniform
__global__ void rng_sample_kernel(int kind, double param, double* out, long long n, uint64_t seed) {
    long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    Rng rng(seed, 99u, 1ull, (uint64_t)e);
    double v;
    if (kind == 0) v = rng.normal();
    else if (kind == 1) v = rng.gamma(param);
    else if (kind == 2) v = rng.exponential();
    else v = rng.uniform();
    out[e] = v;
}
void launch_rng_sample(int kind, double param, double* out, long long n, uint64_t seed, cudaStream_t st) {
    rng_sample_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(kind, param, out, n, seed);
}

// ---------------------------------------------------------------- negative-binomial R
// atomicAdd with warp aggregation: lanes that target the same group are summed by a leader
// (with rdims = (0,1,2) there is ONE group, and per-lane atomics on one address serialise)
__device__ __forceinline__ void group_add(double* base, int g, double v, bool active) {
    const unsigned mask = __ballot_sync(0xffffffffu, active);
    if (!active) return;
    const unsigned peers = __match_any_sync(mask, g);
    const int leader = __ffs(peers) - 1;
    double sum = 0.0;
    // fixed-order sum over the peer lanes
    for (unsigned m = peers; m; m &= m - 1) {
        const int src = __ffs(m) - 1;
        sum += __shfl_sync(peers, v, src);
    }
    if ((int)(threadIdx.x & 31) == leader) atomicAdd(base + g, sum);
}

// work layout (Rs = number of R entries):
//   logR[Rs] cand[Rs] candlog[Rs] lg_cur[Rs] lg_cand[Rs] slog[Rs] ng[Rs]
__device__ __forceinline__ int nb_group(const NbArgs& a, int i, int j, int t) {
    return ((a.Rn > 1 ? i : 0) * a.Rm + (a.Rm > 1 ? j : 0)) * a.Rt + (a.Rt > 1 ? t : 0);
}

// per cell: psi -> log(1-P); accumulate slog_g, n_g and lg_cur_g = sum lgamma(y + R_g)
__global__ void nb_prepare_kernel(NbArgs a) {
    const int Rs = a.Rn * a.Rm * a.Rt;
    double *lg_cur = a.work + 3 * Rs, *slog = a.work + 5 * Rs, *ng = a.work + 6 * Rs;
    const long long cells = (long long)a.nloc * a.P;
    // block-uniform trip count: every lane reaches the warp-collective group_add
    for (long long eb = (long long)blockIdx.x * blockDim.x; eb < cells; eb += (long long)gridDim.x * blockDim.x) {
        const long long e = eb + threadIdx.x;
        const bool in = e < cells;
        int g = 0, c = 0;
        double lg = 0.0, sl = 0.0;
        if (in) {
            const int il = (int)(e / a.P), p = (int)(e - (long long)il * a.P);
            const int j = p / a.T, t = p - j * a.T;
            g = nb_group(a, a.row_begin + il, j, t);
            const double* y = a.Yraw + e * a.R;
            const double Rg = a.Rdisp[g];
            for (int r = 0; r < a.R; ++r) {
                double v = y[r];
                if (v == v) { ++c; if (!a.hist) lg += lgamma(v + Rg); }
            }
            if (c) {
                double psi = 0.0;
                for (int k = 0; k < a.K; ++k) psi += a.W[(size_t)il * a.K + k] * a.V[(size_t)p * a.K + k];
                psi = clampd(psi, -10.0, 10.0);
                const double Pr = 1.0 / (1.0 + exp(-psi));      // ilogit as in utils.py:106-107
                sl = c * log(1.0 - Pr);
            }
        }
        const bool act = in && c > 0;
        group_add(slog, g, sl, act);
        group_add(ng, g, (double)c, act);
        if (!a.hist) group_add(lg_cur, g, lg, act);
    }
}

__global__ void nb_init_kernel(NbArgs a) {
    const int Rs = a.Rn * a.Rm * a.Rt;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= Rs) return;
    a.work[g] = log(a.Rdisp[g]);
    a.work[3 * Rs + g] = 0.0; a.work[4 * Rs + g] = 0.0; a.work[5 * Rs + g] = 0.0; a.work[6 * Rs + g] = 0.0;
}

// accept/reject the pending proposal of step `step-1` (if any), then propose for `step`
__global__ void nb_mh_kernel(NbArgs a, int step) {
    const int Rs = a.Rn * a.Rm * a.Rt;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= Rs) return;
    double *logR = a.work, *cand = a.work + Rs, *candlog = a.work + 2 * Rs, *lg_cur = a.work + 3 * Rs,
           *lg_cand = a.work + 4 * Rs, *slog = a.work + 5 * Rs, *ng = a.work + 6 * Rs;
    const unsigned long long sweep = a.scal->sweep;
    if (step > 0) {
        const int s = step - 1;
        const double R = a.Rdisp[g], Rc = cand[g], l = logR[g], lc = candlog[g];
        const double dprior = -(lc * lc - l * l) / (2.0 * a.rstdev * a.rstdev);
        const double ll = lg_cand[g] - lg_cur[g] - ng[g] * (lgamma(Rc) - lgamma(R)) + (Rc - R) * slog[g];
        const double prob = exp(clampd(dprior + ll, -10.0, 1.0));
        double u;
        if (a.u_inject) u = a.u_inject[(size_t)s * Rs + g];
        else { Rng rng(a.seed, STREAM_R, sweep, (uint64_t)(2 * s + 1) * Rs + g); u = rng.uniform(); }
        if (u <= prob && Rc > 1.0) { a.Rdisp[g] = Rc; logR[g] = lc; lg_cur[g] = lg_cand[g]; }
    }
    if (step < a.nmh) {
        double z;
        if (a.z_inject) z = a.z_inject[(size_t)step * Rs + g];
        else { Rng rng(a.seed, STREAM_R, sweep, (uint64_t)(2 * step) * Rs + g); z = rng.normal(); }
        const double lc = logR[g] + a.rpropstdev * z;
        candlog[g] = lc;
        cand[g] = exp(lc);
        lg_cand[g] = 0.0;
    }
}

__global__ void nb_lgamma_kernel(NbArgs a) {
    const int Rs = a.Rn * a.Rm * a.Rt;
    const double* cand = a.work + Rs;
    double* lg_cand = a.work + 4 * Rs;
    const long long cells = (long long)a.nloc * a.P;
    for (long long eb = (long long)blockIdx.x * blockDim.x; eb < cells; eb += (long long)gridDim.x * blockDim.x) {
        const long long e = eb + threadIdx.x;
        const bool in = e < cells;
        int g = 0;
        double lg = 0.0;
        bool any = false;
        if (in) {
            const int il = (int)(e / a.P), p = (int)(e - (long long)il * a.P);
            const int j = p / a.T, t = p - j * a.T;
            g = nb_group(a, a.row_begin + il, j, t);
            const double* y = a.Yraw + e * a.R;
            const double Rc = cand[g];
            for (int r = 0; r < a.R; ++r) { double v = y[r]; if (v == v) { lg += lgamma(v + Rc); any = true; } }
        }
        group_add(lg_cand, g, lg, in && any);
    }
}

// pseudo-counts of the PG step: N = sum_obs (y + R), kappa = sum_obs y - N/2 (factor.py:553, 507-508, 439)
__global__ void nb_counts_kernel(NbArgs a) {
    const long long cells = (long long)a.nloc * a.P;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < cells; e += (long long)gridDim.x * blockDim.x) {
        const int il = (int)(e / a.P), p = (int)(e - (long long)il * a.P);
        const int j = p / a.T, t = p - j * a.T;
        const double Rg = a.Rdisp[nb_group(a, a.row_begin + il, j, t)];
        const double* y = a.Yraw + e * a.R;
        double ys = 0.0, ns = 0.0;
        int c = 0;
        for (int r = 0; r < a.R; ++r) { double v = y[r]; if (v == v) { ys += v; ns += v + Rg; ++c; } }
        const size_t o = (size_t)il * a.ld + p;
        a.obs[o] = c ? 1 : 0;
        a.ntr[o] = c ? ns : 0.0;
        a.kappa[o] = c ? ys - 0.5 * ns : 0.0;
    }
}

// ---- count-histogram form of the MH loop: sum_e lgamma(y_e + r) = sum_v hist_g[v] lgamma(v + r)
// (the counts are small non-negative integers and do not change between sweeps), so the whole
// nmh-step chain of a group runs in ONE block without touching the data tensor again.
__global__ void nb_scan_kernel(const double* __restrict__ Y, long long n, unsigned long long* out) {
    // out[0] = max value (as integer), out[1] = 1 if any observed entry is negative / non-integer / huge
    unsigned long long mx = 0, bad = 0;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const double v = Y[e];
        if (v == v) {
            if (v < 0.0 || v > 1e9 || v != floor(v)) bad = 1;
            else mx = max(mx, (unsigned long long)v);
        }
    }
    atomicMax(&out[0], mx);
    if (bad) atomicMax(&out[1], 1ull);
}

void launch_nb_scan(const double* Y, long long n, unsigned long long* out, cudaStream_t st) {
    int nb = (int)((n + 255) / 256);
    if (nb > 148 * 8) nb = 148 * 8;
    if (nb < 1) nb = 1;
    nb_scan_kernel<<<nb, 256, 0, st>>>(Y, n, out);
}

__global__ void nb_hist_kernel(NbArgs a, int vstride) {
    const long long cells = (long long)a.nloc * a.P;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < cells; e += (long long)gridDim.x * blockDim.x) {
        const int il = (int)(e / a.P), p = (int)(e - (long long)il * a.P);
        const int j = p / a.T, t = p - j * a.T;
        const int g = nb_group(a, a.row_begin + il, j, t);
        const double* y = a.Yraw + e * a.R;
        for (int r = 0; r < a.R; ++r) {
            const double v = y[r];
            if (v == v) atomicAdd(&a.hist[(size_t)g * vstride + (int)v], 1.0);
        }
    }
}

void launch_nb_hist(const NbArgs& a, int vstride, cudaStream_t st) {
    const long long cells = (long long)a.nloc * a.P;
    int nb = (int)((cells + 255) / 256);
    if (nb > 148 * 8) nb = 148 * 8;
    if (nb < 1) nb = 1;
    nb_hist_kernel<<<nb, 256, 0, st>>>(a, vstride);
}

// All nmh random-walk steps of one R group in one block.  The step chain is kept as short as the
// algorithm allows (FP64 transcendentals cost thousands of cycles of dependent latency): the
// proposal normals and acceptance uniforms are drawn up front, one per thread; the group term
// -n_g lgamma(r) rides along in the block sum of the histogram terms (so one lgamma deep per
// step when the histogram fits the block); the current value's sum is carried across steps.
__global__ void __launch_bounds__(256) nb_mh_hist_kernel(NbArgs a, int vstride) {
    constexpr int MAXS = 256;
    __shared__ double sh[40];
    __shared__ double zs[MAXS], us[MAXS];
    const int Rs = a.Rn * a.Rm * a.Rt;
    const int g = blockIdx.x;
    const double* hist = a.hist + (size_t)g * vstride;
    const double slog = a.work[5 * Rs + g], ng = a.work[6 * Rs + g];
    const unsigned long long sweep = a.scal->sweep;
    auto draw_z = [&](int s) -> double {
        if (a.z_inject) return a.z_inject[(size_t)s * Rs + g];
        Rng rng(a.seed, STREAM_R, sweep, (uint64_t)(2 * s) * Rs + g);
        return rng.normal();
    };
    auto draw_u = [&](int s) -> double {
        if (a.u_inject) return a.u_inject[(size_t)s * Rs + g];
        Rng rng(a.seed, STREAM_R, sweep, (uint64_t)(2 * s + 1) * Rs + g);
        return rng.uniform();
    };
    const bool pre = a.nmh <= MAXS;
    if (pre) {
        for (int s = threadIdx.x; s < a.nmh; s += blockDim.x) { zs[s] = draw_z(s); us[s] = draw_u(s); }
    }
    // sum_v hist[v] lgamma(v + r) - n_g lgamma(r)
    auto lgsum = [&](double r) -> double {
        double acc = 0.0;
        for (int v = threadIdx.x; v < vstride; v += blockDim.x) {
            const double h = hist[v];
            if (h != 0.0) acc += h * lgamma((double)v + r);
        }
        if (threadIdx.x == blockDim.x - 1) acc -= ng * lgamma(r);
        acc = block_sum(acc, sh);
        if (threadIdx.x == 0) sh[36] = acc;
        __syncthreads();
        return sh[36];
    };
    double R = a.Rdisp[g], logR = log(R);
    double lg_cur = lgsum(R);
    for (int s = 0; s < a.nmh; ++s) {
        const double z = pre ? zs[s] : draw_z(s);
        const double lc = logR + a.rpropstdev * z, Rc = exp(lc);
        const double lg_cand = lgsum(Rc);
        const double dprior = -(lc * lc - logR * logR) / (2.0 * a.rstdev * a.rstdev);
        const double ll = lg_cand - lg_cur + (Rc - R) * slog;
        const double prob = exp(clampd(dprior + ll, -10.0, 1.0));
        const double u = pre ? us[s] : draw_u(s);
        if (u <= prob && Rc > 1.0) { R = Rc; logR = lc; lg_cur = lg_cand; }     // block-uniform
    }
    if (threadIdx.x == 0) a.Rdisp[g] = R;
}

void launch_nb_update(const NbArgs& a, cudaStream_t st) {
    const int Rs = a.Rn * a.Rm * a.Rt;
    const long long cells = (long long)a.nloc * a.P;
    int nb = (int)((cells + 255) / 256);
    if (nb > 148 * 8) nb = 148 * 8;
    if (nb < 1) nb = 1;
    const int gb = (Rs + 127) / 128;
    if (a.nmh > 0 && a.hist) {
        nb_init_kernel<<<gb, 128, 0, st>>>(a);
        nb_prepare_kernel<<<nb, 256, 0, st>>>(a);
        nb_mh_hist_kernel<<<Rs, 256, 0, st>>>(a, a.hist_stride);
    } else if (a.nmh > 0) {
        nb_init_kernel<<<gb, 128, 0, st>>>(a);
        nb_prepare_kernel<<<nb, 256, 0, st>>>(a);
        for (int s = 0; s < a.nmh; ++s) {
            nb_mh_kernel<<<gb, 128, 0, st>>>(a, s);
            nb_lgamma_kernel<<<nb, 256, 0, st>>>(a);
        }
        nb_mh_kernel<<<gb, 128, 0, st>>>(a, a.nmh);
    }
    nb_counts_kernel<<<nb, 256, 0, st>>>(a);
}

}  // namespace btf
