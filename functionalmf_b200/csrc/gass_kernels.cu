// GASS: generalized analytic slice sampling of the constrained model's W rows and V columns under a built-in
// likelihood, Poisson, Binomial or Gaussian (functionalmf_b200/gass.py, factor.py:665-892).  One CTA per row or column:
//   1. the constraint products a = A(x - mu), b = A v, c = C - A mu of every constraint row, without the Kronecker
//      matrix (rows: coefficients sum_t A[c,t] V[j,t,:]; columns: A[c,t] W[i,:]);
//   2. the feasible grid of gass.feasible_angles: "outside" intervals are removed as index ranges through a difference
//      array, the "inside" ones intersected into [lo, hi]; no active constraint selects the coarse grid;
//   3. thinning by a partial Fisher-Yates over the ascending feasible index list;
//   4. the log-likelihood of every candidate (FP64, fixed-order block reductions) and the uniform pick among those
//      at or above the slice height.  The kernels are instantiated per likelihood: a cell type loads what a cell of
//      the data holds and evaluates its log-likelihood at a candidate's rate or probability.
// Every random choice is a function of ngrid + 2 uniforms per row / column (slice, thinning, pick): Philox keyed by
// (seed, sweep, stream, row or column), or injected.
#include "kernels.h"

namespace btf {

constexpr int GASS_THREADS = 256;
constexpr int GASS_CHUNK = 8;                 // candidates evaluated per pass over the cells
constexpr double GASS_EDGE_EPS = 1e-6;        // gass.EDGE_EPS
constexpr double LOG_SQRT_2PI = 0.91893853320467274178;

// exact IEEE products and sums (no FMA contraction): the discriminant and the outside test decide which grid points
// survive, and numpy evaluates them without fused operations
__device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }

// deterministic block reductions of an int / a double (max, min); result broadcast to every thread
__device__ int block_sum_int(int v, int* sh) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) sh[w] = v;
    __syncthreads();
    int r = 0;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) r += sh[i];
    __syncthreads();
    return r;
}
template <bool MAX>
__device__ double block_ext(double v, double* sh) {
    for (int o = 16; o > 0; o >>= 1) {
        const double u = __shfl_xor_sync(0xffffffffu, v, o);
        v = MAX ? fmax(v, u) : fmin(v, u);
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) sh[w] = v;
    __syncthreads();
    double r = sh[0];
    for (int i = 1; i < (int)(blockDim.x >> 5); ++i) r = MAX ? fmax(r, sh[i]) : fmin(r, sh[i]);
    __syncthreads();
    return r;
}
// exclusive prefix sum over the block (thread order); *total receives the sum
__device__ int block_scan_int(int v, int* sh, int* total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
    int x = v;
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    __syncthreads();
    if (lane == 31) sh[w] = x;
    __syncthreads();
    int off = 0, tot = 0;
    for (int i = 0; i < nw; ++i) { if (i < w) off += sh[i]; tot += sh[i]; }
    __syncthreads();
    *total = tot;
    return off + x - v;
}

// first index with g[idx] > x (g ascending)
__device__ __forceinline__ int upper_index(const double* g, int n, double x) {
    int lo = 0, hi = n;
    while (lo < hi) { const int m = (lo + hi) >> 1; if (g[m] > x) hi = m; else lo = m + 1; }
    return lo;
}
// first index with g[idx] >= x
__device__ __forceinline__ int lower_index(const double* g, int n, double x) {
    int lo = 0, hi = n;
    while (lo < hi) { const int m = (lo + hi) >> 1; if (g[m] >= x) hi = m; else lo = m + 1; }
    return lo;
}

// scipy.stats.poisson.logpmf summed over the observed replicates of a cell (n of them, sum s, lg = sum lgamma(y + 1))
// and dropped by nansum where it is NaN: lam > 0 -> s log lam - n lam - lg; lam = 0 -> 0 or -inf; lam < 0 (NaN in
// scipy) -> 0.  The constant lg does not cancel in ll >= height: a cell drops out of the sum with it wherever lam < 0.
__device__ __forceinline__ double poisson_cell(double lam, int n, double s, double lg) {
    if (n == 0) return 0.0;
    if (lam > 0.0) return s * log(lam) - n * lam - lg;
    if (lam == 0.0) return s > 0.0 ? -INFINITY : 0.0;
    return 0.0;
}
// scipy.stats.binom.logpmf(y, n, p) of one observed cell, dropped by nansum where it is NaN (scipy 1.18's _logpmf:
// combiln + xlogy(y, p) + xlog1py(n - y, -p), combiln = lgamma(n + 1) - (lgamma(y + 1) + lgamma(n - y + 1)) = lc):
// 0 < p < 1 -> lc + y log p + (n - y) log1p(-p), a zero count contributing exactly 0; p = 0 -> 0 if y = 0, else -inf;
// p = 1 -> 0 if y = n, else -inf; p outside [0, 1] (NaN in scipy) -> 0, with lc; n = 0 -> 0.  Evaluated without fused
// operations, in scipy's order.
__device__ __forceinline__ double binomial_cell(double p, double y, double n, double lc) {
    if (n == 0.0) return 0.0;
    if (p > 0.0 && p < 1.0) {
        const double ty = y > 0.0 ? mul(y, log(p)) : 0.0;
        const double tn = n > y ? mul(n - y, log1p(-p)) : 0.0;
        return add(add(lc, ty), tn);
    }
    if (p == 0.0) return y > 0.0 ? -INFINITY : 0.0;
    if (p == 1.0) return y < n ? -INFINITY : 0.0;
    return 0.0;
}

// The cell likelihoods gass_body is instantiated for: load() reads what the data keep for a cell, ll() is its
// log-likelihood at the rate / probability lam of a candidate.
struct PoissonLik {
    struct Cell { int n; double s, lg; };
    static __device__ __forceinline__ Cell load(const GassArgs& a, size_t cell) {
        Cell c;
        c.n = a.cnt[cell];
        c.s = a.S[cell]; c.lg = a.lgy[cell];
        return c;
    }
    static __device__ __forceinline__ double ll(double lam, const Cell& c) { return poisson_cell(lam, c.n, c.s, c.lg); }
};
struct BinomialLik {
    struct Cell { bool obs; double y, n, lc; };
    static __device__ __forceinline__ Cell load(const GassArgs& a, size_t cell) {
        Cell c;
        c.obs = a.cnt[cell] != 0;
        c.n = a.ntr[cell];
        c.y = a.S[cell] + 0.5 * c.n;       // kappa = y - n/2: exact for integer counts
        c.lc = a.lgy[cell];
        return c;
    }
    static __device__ __forceinline__ double ll(double p, const Cell& c) { return c.obs ? binomial_cell(p, c.y, c.n, c.lc) : 0.0; }
};
// scipy.stats.norm.logpdf(y, tau, sigma) summed over the n observed replicates of a cell, in the centred form
// -n log sigma - n log sqrt(2 pi) - (ss + n (ybar - tau)^2) / (2 sigma^2) with ss = sum (y - ybar)^2: expanding the
// square instead (sum y^2 - 2 tau sum y + n tau^2) cancels badly when |y| is large against the noise, and which
// candidates clear the slice depends on the value.  The variance is the scalar nu2 or the cell's known variance; a cell
// with n = 0 or an infinite variance (missing) contributes 0.  Evaluated without fused operations.
struct GaussianLik {
    struct Cell { double n, ybar, ss, c0, tv; };    // n = 0: not observed; c0 = -n (log sigma + log sqrt(2 pi)), tv = 2 sigma^2
    static __device__ __forceinline__ Cell load(const GassArgs& a, size_t cell) {
        Cell c;
        const int n = a.cnt[cell];
        const double var = a.nu2c ? a.nu2c[cell] : a.scal->nu2;
        c.n = n > 0 && var < INFINITY ? (double)n : 0.0;
        c.ybar = n > 0 ? a.S[cell] / n : 0.0;
        c.ss = a.lgy[cell];
        c.c0 = -mul(c.n, add(0.5 * log(var), LOG_SQRT_2PI));
        c.tv = 2.0 * var;
        return c;
    }
    static __device__ __forceinline__ double ll(double tau, const Cell& c) {
        if (c.n == 0.0) return 0.0;
        const double d = add(c.ybar, -tau);
        return add(c.c0, -(add(c.ss, mul(c.n, mul(d, d))) / c.tv));
    }
};

// scipy.stats.norm.logpdf(lam, mu, sigma)
__device__ __forceinline__ double norm_logpdf(double lam, double mu, double sg) {
    const double z = (lam - mu) / sg;
    return -(z * z) / 2.0 - LOG_SQRT_2PI - log(sg);
}

__device__ __forceinline__ double gass_uniform(const GassArgs& a, int item, int slot) {
    const size_t stride = (size_t)a.ngrid + 2;
    if (a.u_inject) return a.u_inject[(size_t)item * stride + slot];
    Rng rng(a.seed, a.col ? STREAM_GASS_V : STREAM_GASS_W, a.scal->sweep, (uint64_t)item * stride + slot);
    return rng.uniform();
}

// Dynamic shared memory: x, mu, v [D] | work [max(nfine + 1 ints, ngrid doubles)] | idx [nfine] u16
__host__ __device__ inline size_t gass_work_bytes(int nfine, int ngrid) {
    const size_t d = (size_t)(nfine + 1) * sizeof(int), l = (size_t)ngrid * sizeof(double);
    return d > l ? d : l;
}
size_t gass_smem_bytes(int D, int nfine, int ngrid) {
    return (size_t)3 * D * sizeof(double) + ((gass_work_bytes(nfine, ngrid) + 15) & ~(size_t)15) + (size_t)nfine * sizeof(uint16_t);
}

// One row (col = false: W row i, D = min(K, i + 1) entries) or one column (col = true: V[j], D = T K, t-major).
template <class Lik>
__device__ void gass_body(const GassArgs& a, bool col) {
    extern __shared__ __align__(16) unsigned char gsm[];
    __shared__ double shd[32];
    __shared__ int shi[32];
    __shared__ double s_theta;
    const int tid = threadIdx.x, NT = blockDim.x;
    const int item = blockIdx.x;
    const int K = a.K, T = a.T;
    const int D = col ? T * K : min(K, item + 1);
    const int nfine = a.nfine;
    double* x = (double*)gsm;
    double* mu = x + D;
    double* v = mu + D;
    unsigned char* wbase = (unsigned char*)(v + D);
    int* diff = (int*)wbase;                  // difference array of the removed ranges, later the candidates' ll
    double* cll = (double*)wbase;
    const size_t work = gass_work_bytes(nfine, a.ngrid);
    uint16_t* idx = (uint16_t*)(wbase + ((work + 15) & ~(size_t)15));

    // ---- the state, the ellipse's centre and its proposal direction
    const double* xs = col ? a.Vold + (size_t)item * D : a.Wold + (size_t)item * K;
    const double* dr = col ? a.Vnew + (size_t)item * D : a.Wnew + (size_t)item * K;
    const double* mn = col ? a.Vmean : a.Wmean;
    for (int k = tid; k < D; k += NT) {
        const double m = mn ? mn[(size_t)item * (col ? D : K) + k] : 0.0;
        x[k] = xs[k];
        mu[k] = m;
        v[k] = dr[k] - m;
    }
    for (int k = tid; k <= nfine; k += NT) diff[k] = 0;
    __syncthreads();

    // ---- constraints: row i: (j, c) for all j, c, then the row constraints; column j: (i, c) for all i, c
    const int J = a.J;
    const int ncons = col ? a.N * J : a.M * J + a.nrc;
    int n_active = 0, n_inside = 0, n_bad = 0;
    double lo_max = -INFINITY, hi_min = INFINITY;
    for (int r = tid; r < ncons; r += NT) {
        double ax = 0.0, aa = 0.0, ab = 0.0, am = 0.0, cr;
        if (!col && r >= a.M * J) {
            const double* rc = a.rowcons + (size_t)(r - a.M * J) * (K + 1);
            for (int k = 0; k < D; ++k) { ax += rc[k] * x[k]; aa += rc[k] * (x[k] - mu[k]); ab += rc[k] * v[k]; am += rc[k] * mu[k]; }
            cr = rc[K];
        } else {
            const int o = r / J, c = r % J;          // o = column j (row step) or row i (column step)
            const double* Ac = a.A + (size_t)c * T;
            cr = a.C[c];
            if (!col) {
                const double* Vj = a.Vcur + (size_t)o * T * K;
                for (int k = 0; k < D; ++k) {
                    double coef = 0.0;
                    for (int t = 0; t < T; ++t) if (Ac[t] != 0.0) coef += Ac[t] * Vj[(size_t)t * K + k];
                    ax += coef * x[k]; aa += coef * (x[k] - mu[k]); ab += coef * v[k]; am += coef * mu[k];
                }
            } else {
                const double* Wi = a.Wcur + (size_t)o * K;
                for (int t = 0; t < T; ++t) {
                    if (Ac[t] == 0.0) continue;
                    for (int k = 0; k < K; ++k) {
                        const double coef = Ac[t] * Wi[k];
                        const int e = t * K + k;
                        ax += coef * x[e]; aa += coef * (x[e] - mu[e]); ab += coef * v[e]; am += coef * mu[e];
                    }
                }
            }
        }
        if (ax < cr) ++n_bad;
        if (a.check_only) continue;
        const double cc = cr - am;
        const double disc = add(add(mul(aa, aa), mul(ab, ab)), -mul(cc, cc));
        if (!(disc >= 0.0) || aa == -cc) continue;
        ++n_active;
        const double root = sqrt(disc), denom = aa + cc;
        const double t1 = 2.0 * atan((ab + root) / denom), t2 = 2.0 * atan((ab - root) / denom);
        const double tmin = fmin(t1, t2), tmax = fmax(t1, t2);
        if (mul(aa, aa) < mul(cc, cc)) {
            // outside: the grid points strictly between the roots go
            const int i0 = upper_index(a.grid_fine, nfine, tmin), i1 = lower_index(a.grid_fine, nfine, tmax);
            if (i0 < i1) { atomicAdd(&diff[i0], 1); atomicAdd(&diff[i1], -1); }
        } else {
            ++n_inside;
            lo_max = fmax(lo_max, tmin);
            hi_min = fmin(hi_min, tmax);
        }
    }
    n_bad = block_sum_int(n_bad, shi);
    if (a.check_only) {
        if (tid == 0 && n_bad > 0) atomicAdd(a.nbad, 1);
        return;
    }
    n_active = block_sum_int(n_active, shi);
    n_inside = block_sum_int(n_inside, shi);
    lo_max = block_ext<true>(lo_max, shd);
    hi_min = block_ext<false>(hi_min, shd);
    __syncthreads();

    // ---- the feasible grid as an ascending index list
    const double* grid = a.grid_fine;
    int F = 0;
    if (n_active == 0) {
        grid = a.grid_coarse;
        F = a.ngrid;
        for (int k = tid; k < F; k += NT) idx[k] = (uint16_t)k;
    } else {
        const double lo = n_inside ? lo_max + GASS_EDGE_EPS : -INFINITY;
        const double hi = n_inside ? hi_min - GASS_EDGE_EPS : INFINITY;
        const int per = (nfine + NT - 1) / NT, b0 = min(nfine, tid * per), b1 = min(nfine, b0 + per);
        int dsum = 0;
        for (int g = b0; g < b1; ++g) dsum += diff[g];
        int tot = 0;
        int cover = block_scan_int(dsum, shi, &tot);
        int cnt = 0;
        {
            int cv = cover;
            for (int g = b0; g < b1; ++g) {
                cv += diff[g];
                if (cv == 0 && grid[g] >= lo && grid[g] <= hi) ++cnt;
            }
        }
        int pos = block_scan_int(cnt, shi, &F);
        __syncthreads();            // every diff read is done before idx (a separate region) is written
        for (int g = b0; g < b1; ++g) {
            cover += diff[g];
            if (cover == 0 && grid[g] >= lo && grid[g] <= hi) idx[pos++] = (uint16_t)g;
        }
    }
    __syncthreads();

    // ---- slice height, thinning
    const int ncand = min(F, a.ngrid);
    if (tid == 0 && F > a.ngrid) {
        for (int k = 0; k < a.ngrid; ++k) {
            const double u = gass_uniform(a, item, 1 + k);
            int r = k + (int)floor(u * (double)(F - k));
            r = min(max(r, k), F - 1);
            const uint16_t tmp = idx[k]; idx[k] = idx[r]; idx[r] = tmp;
        }
    }
    __syncthreads();

    // ---- log-likelihoods: the current state (chunk 0, candidate -1), then the candidates in chunks
    const int P = a.P;
    const int ncells = col ? a.N * T : P;
    double cur_ll = 0.0;
    for (int c0 = -1; c0 < ncand; c0 += (c0 < 0 ? 1 : GASS_CHUNK)) {
        const int nc = c0 < 0 ? 1 : min(GASS_CHUNK, ncand - c0);
        double cs[GASS_CHUNK], sn[GASS_CHUNK], acc[GASS_CHUNK];
#pragma unroll
        for (int q = 0; q < GASS_CHUNK; ++q) {
            acc[q] = 0.0; cs[q] = 1.0; sn[q] = 0.0;
            if (c0 >= 0 && q < nc) sincos(grid[idx[c0 + q]], &sn[q], &cs[q]);
        }
        for (int e = tid; e < ncells; e += NT) {
            size_t cell;
            if (col) {
                const int i = e / T, t = e % T;
                const double* f = a.Wcur + (size_t)i * K;
                cell = (size_t)i * a.ld + (size_t)item * T + t;
                double tx = 0.0, t0 = 0.0, tv = 0.0, tm = 0.0;
                for (int k = 0; k < K; ++k) {
                    const double fk = f[k], xk = x[t * K + k], mk = mu[t * K + k];
                    tx += fk * xk; t0 += fk * (xk - mk); tv += fk * v[t * K + k]; tm += fk * mk;
                }
                const typename Lik::Cell cd = Lik::load(a, cell);
                const bool ep = a.ep_mu != nullptr;
                const double em = ep ? a.ep_mu[cell] : 0.0, es = ep ? a.ep_sig[cell] : 1.0;
#pragma unroll
                for (int q = 0; q < GASS_CHUNK; ++q) {
                    if (q >= nc) continue;
                    const double lam = c0 < 0 ? tx : t0 * cs[q] + tv * sn[q] + tm;
                    acc[q] += Lik::ll(lam, cd);
                    if (ep) acc[q] -= norm_logpdf(lam, em, es);
                }
            } else {
                const double* f = a.Vcur + (size_t)e * K;
                cell = (size_t)item * a.ld + e;
                double tx = 0.0, t0 = 0.0, tv = 0.0, tm = 0.0;
                for (int k = 0; k < D; ++k) {
                    const double fk = f[k];
                    tx += fk * x[k]; t0 += fk * (x[k] - mu[k]); tv += fk * v[k]; tm += fk * mu[k];
                }
                const typename Lik::Cell cd = Lik::load(a, cell);
                const bool ep = a.ep_mu != nullptr;
                const double em = ep ? a.ep_mu[cell] : 0.0, es = ep ? a.ep_sig[cell] : 1.0;
#pragma unroll
                for (int q = 0; q < GASS_CHUNK; ++q) {
                    if (q >= nc) continue;
                    const double lam = c0 < 0 ? tx : t0 * cs[q] + tv * sn[q] + tm;
                    acc[q] += Lik::ll(lam, cd);
                    if (ep) acc[q] -= norm_logpdf(lam, em, es);
                }
            }
        }
#pragma unroll
        for (int q = 0; q < GASS_CHUNK; ++q) {
            if (q < nc) {           // (nc is the same in every thread)
                const double r = block_sum(acc[q], shd);
                if (tid == 0) { if (c0 < 0) cur_ll = r; else cll[c0 + q] = r; }
            }
        }
        __syncthreads();
    }

    // ---- the pick among the candidates at or above the slice height, in candidate order
    if (tid == 0) {
        double theta = 0.0;
        int G = 0;
        if (F > 0) {
            const double height = cur_ll + log(gass_uniform(a, item, 0));
            for (int k = 0; k < ncand; ++k) G += cll[k] >= height;
            if (G > 0) {
                int pick = (int)floor(gass_uniform(a, item, a.ngrid + 1) * (double)G);
                pick = min(max(pick, 0), G - 1);
                for (int k = 0; k < ncand; ++k) {
                    if (cll[k] >= height) {
                        if (pick == 0) { theta = grid[idx[k]]; break; }
                        --pick;
                    }
                }
            }
        }
        s_theta = theta;
        if (a.diag) { a.diag[(size_t)item * 3] = F; a.diag[(size_t)item * 3 + 1] = G; a.diag[(size_t)item * 3 + 2] = theta; }
    }
    __syncthreads();
    // ---- (x - mu) cos + v sin + mu, evaluated as numpy does (no fused operations); theta = 0 keeps x exactly
    const double theta = s_theta;
    double* out = col ? a.Vnew + (size_t)item * D : a.Wnew + (size_t)item * K;
    if (theta == 0.0) {
        for (int k = tid; k < D; k += NT) out[k] = x[k];
    } else {
        double s, c;
        sincos(theta, &s, &c);
        for (int k = tid; k < D; k += NT) out[k] = add(add(mul(add(x[k], -mu[k]), c), mul(v[k], s)), mu[k]);
    }
}

template <class Lik>
__global__ void __launch_bounds__(GASS_THREADS) gass_row_kernel(GassArgs a) { gass_body<Lik>(a, false); }
template <class Lik>
__global__ void __launch_bounds__(GASS_THREADS) gass_col_kernel(GassArgs a) { gass_body<Lik>(a, true); }

template <class Lik>
static void launch_gass_lik(const GassArgs& a, cudaStream_t st) {
    static PerDeviceMax attr_row, attr_col;
    const int D = a.col ? a.T * a.K : a.K;
    const size_t smem = gass_smem_bytes(D, a.nfine, a.ngrid);
    if (a.col) {
        if (attr_col.raise(smem)) cudaFuncSetAttribute(gass_col_kernel<Lik>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        gass_col_kernel<Lik><<<a.M, GASS_THREADS, smem, st>>>(a);
    } else {
        if (attr_row.raise(smem)) cudaFuncSetAttribute(gass_row_kernel<Lik>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        gass_row_kernel<Lik><<<a.N, GASS_THREADS, smem, st>>>(a);
    }
}

void launch_gass(const GassArgs& a, cudaStream_t st) {
    if (a.gaussian) launch_gass_lik<GaussianLik>(a, st);
    else if (a.binomial) launch_gass_lik<BinomialLik>(a, st);
    else launch_gass_lik<PoissonLik>(a, st);
}

}  // namespace btf
