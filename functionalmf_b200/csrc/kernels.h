// Host-side launchers of the BTF kernels (one translation unit per kernel family).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "common.cuh"

namespace btf {
// cudaFuncSetAttribute belongs to a device's context: "already done" bookkeeping is kept per device, so that a process
// that drives several GPUs (or creates engines on different devices one after the other) configures each of them.
struct PerDeviceOnce {
    unsigned long long mask = 0;
    bool first() {
        int d = 0;
        cudaGetDevice(&d);
        const unsigned long long b = 1ull << (d & 63);
        if (mask & b) return false;
        mask |= b;
        return true;
    }
};
struct PerDeviceMax {
    size_t v[64] = {};
    bool raise(size_t s) {
        int d = 0;
        cudaGetDevice(&d);
        if (s <= v[d & 63]) return false;
        v[d & 63] = s;
        return true;
    }
};


// ---------------------------------------------------------------- K0 prereduce
// Y chunk [rows][P][R] (NaN = missing) -> cnt u8, S f64 at pitch `ld`; per-block
// partial (sum of squares, #observed) appended to `partials` [2*nblocks].
void launch_prereduce_gaussian(const double* Y, int rows, int P, int R, uint8_t* cnt, double* S,
                               long long ld, double* partials, int* nblocks_out, cudaStream_t st);
// Binomial: (Ysucc, Ntrials) [rows][P] -> obs u8, kappa = y - n/2, ntr = n (0 where missing)
void launch_prereduce_binomial(const double* Y, const double* Nt, int rows, int P, uint8_t* obs,
                               double* kappa, double* ntr, long long ld, cudaStream_t st);
// Known per-cell noise variances nu2 [rows][P] at pitch `lds` -> f64 weights w = cnt / nu2 and s = S / nu2 at pitch `ld`
// (0 where cnt = 0 or nu2 = +inf); `keep` (optional) receives nu2 at pitch `ld`; *nbad += # observed cells whose
// variance is NaN or <= 0.
void launch_nu2_weights(const double* nu2, long long lds, int rows, int P, const uint8_t* cnt, const double* S,
                        long long ld, double* keep, double* w, double* s, unsigned long long* nbad, cudaStream_t st);
// dst[0] += sum(src[0..n) step stride) in a fixed order (single block)
void launch_reduce_add(const double* src, int n, int stride, double* dst, cudaStream_t st);

// ---------------------------------------------------------------- K1 statistics
struct StatsPlan {
    int cfg;          // 0: BM=128 (K<=16), 1: BM=32 (K<=32), 2: BM=128 small (K<=8)
    int K, L, nct_z, nct_f, zw;
    int BM, KC;
    int mtiles, nchunks, nsplit, chunks_per_split;
    int overlap;      // 1: Z generation overlapped with the DMMA loop (K = 32, f64 weights)
    int zpre, zwg;    // 1: right operand pre-generated in global memory with row pitch zwg (stats_zpre.cu)
    size_t smem_bytes;
    size_t out_elems_per_split;   // m_valid * (L+K)
};
// trans=false: row statistics (m = local row, contraction over p = (j,t));
// trans=true : column statistics (m = p, contraction over local rows).
// weights_f64: weight operand is double (omega) instead of uint8 counts.
bool plan_stats(StatsPlan* plan, int K, bool trans, bool weights_f64, int mdim_pad, int kdim_pad,
                int m_valid, int nsplit_request, int sm_count);
// frows: rows of F the contraction runs over (padded); zscratch: frows * plan.zwg doubles when plan.zpre
void launch_stats(const StatsPlan& plan, bool trans, bool weights_f64, const void* wt, const double* sv,
                  const double* F, long long frows, long long ld, int m_valid, double* out, double* zscratch,
                  cudaStream_t st);
// count weights at K = 16 / 32
bool plan_stats_zpre(StatsPlan* p, bool trans, int mdim_pad, int kdim_pad, int nsplit_request, int sm_count);
void launch_stats_zpre(const StatsPlan& p, bool trans, const void* wt, const double* sv, const double* F,
                       long long frows, long long ld, int m_valid, double* out, double* Zg, cudaStream_t st);

// ---------------------------------------------------------------- K1 on the integer tensor cores (stats_i8.cu, i8gemm2.cu)
// Fixed-point form of a column of Z: q = rint(Z 2^(54 - e_c)), |q| <= 2^54, in 7 signed base-256 digits d_s in [-128, 127].
// The digit planes are stored tile-major for the 2-CTA GEMM: a tile = 36 product columns x 7 planes = 252 rows, plane-major.
constexpr int I8_NPLANES = 7, I8_FIXBITS = 54, I8_COLS_PER_TILE = 36;
__host__ __device__ inline int i8_plane_row(int c, int s) {
    return (c / I8_COLS_PER_TILE) * (I8_COLS_PER_TILE * I8_NPLANES) + s * I8_COLS_PER_TILE + (c % I8_COLS_PER_TILE);
}
inline int i8_plane_rows(int L) { return ((L + I8_COLS_PER_TILE - 1) / I8_COLS_PER_TILE) * (I8_COLS_PER_TILE * I8_NPLANES); }
struct StatsI8Sizes { size_t planes_bytes, d_elems, cntT_bytes, bpart_elems; int nsplit_b_row, L; };
struct StatsI8Buffers {
    int8_t* planes;                 // [i8_plane_rows(L)][kdim_pad] signed base-256 digits of Z, tile-major (i8_plane_row)
    unsigned long long* colmax;     // [L] max |Z| per column (bit pattern)
    int* expo;                      // [L] column exponents
    int32_t* D;                     // [i8_plane_rows(L)][m_pad] exact digit-plane contractions (split-K route only)
    double* bpart;                  // [nsplit][m][K] partial sums of the linear block
    int nsplit_b_row;
};
// K in {8, 16, 32}, int32 accumulators that cannot overflow, and the 2-CTA GEMM can run on the current device (its
// shared-memory attribute is set there)
bool stats_i8_supported(int K, int nreps, long long kdim_row, long long kdim_col);
// nall_pad: padded GLOBAL row count (contraction length of the column side), ploc: columns (j,t) owned by this rank
void stats_i8_sizes(int K, int nloc_pad, int Ppad, int nloc, int P, int nall_pad, int ploc, StatsI8Sizes* s);
void launch_transpose_u8(const uint8_t* src, long long lds, int rows, int cols, uint8_t* dst, long long ldd, cudaStream_t st);
// element-wise guard of the fixed-point product block, see below
struct I8Guard {
    const unsigned* cntsum;     // [m] sum of the counts of row m (stats_i8_count_rows, once per data set)
    unsigned char* flags;       // [m] zero except for flagged rows
    int* nflag;                 // rows recomputed by the last stats_i8_fallback
    double tol;
};
// the four stages of the integer path (engine: tensor-core contraction and HBM-bound linear block on separate streams)
void stats_i8_digits(const StatsI8Buffers& w, int K, const double* F, int f_rows, int kdim_pad, cudaStream_t st);
// route of the product block on the 2-CTA GEMM: its fused epilogue wrote `out` (>= 48 tiles of 256 x 256, or a contraction
// too short to split), or split-K left int32 planes in w.D for stats_i8_combine
enum I8Route { I8_ROUTE_FUSED = 2, I8_ROUTE_SPLITK = 3 };
// returns the I8Route taken, 0 when the launch failed
int stats_i8_product(const StatsI8Buffers& w, int K, const uint8_t* B, long long ldb, int kdim_pad, int m_valid, int m_pad,
                     double* out, const I8Guard* guard, cudaStream_t st);
int stats_i8_linear(const StatsI8Buffers& w, bool trans, int K, const double* S, long long lds, const double* F,
                    int kdim_pad, int m_valid, int max_split, double* out, cudaStream_t st);     // returns the split count of `out`
void stats_i8_combine(const StatsI8Buffers& w, int K, int m_valid, int m_pad, bool product_done,
                      const double* bpart, int nsplit_b, long long bpart_m0, long long bpart_rows, double* out,
                      const I8Guard* guard, cudaStream_t st);
// element-wise guard of the fixed-point product block (see stats_i8.cu): the kernels that produce the block flag the rows
// whose diagonal entries cannot be guaranteed to `tol` relative (2^(e_c - 55) sum_k cnt[m][k] > tol out[m][(k,k)]);
// stats_i8_fallback recomputes the flagged rows in FP64, clears the flags and counts them in *nflag.
void stats_i8_count_rows(const uint8_t* B, long long ldb, int m_valid, int kdim_pad, unsigned* cntsum, cudaStream_t st);
void stats_i8_fallback(int K, const uint8_t* B, long long ldb, const double* F, int f_rows, int m_valid, double* out,
                       const I8Guard& g, cudaStream_t st);

// ---------------------------------------------------------------- residual (nu2)
// resid_partials[b] = sum over the block's cells of cnt*Mu^2 - 2*Mu*S
void launch_residual(const uint8_t* cnt, const double* S, long long ld, const double* W, const double* V,
                     int nrows_pad, int Ppad, int K, double* partials, int* nblocks_out, cudaStream_t st);

// running posterior mean / M2 of Mu = W V^T over the local cells (Welford), count = samples so far
void launch_mu_moments(const double* W, const double* V, int K, int nloc, int P, double* mean, double* m2,
                       double count, cudaStream_t st);

// ---------------------------------------------------------------- held-out evaluation (eval_kernels.cu)
enum { EVAL_IDENTITY = 0, EVAL_ILOGIT = 1, EVAL_NB_MEAN = 2 };
enum { EVAL_LL_NONE = 0, EVAL_LL_GAUSSIAN = 1, EVAL_LL_POISSON = 2 };
constexpr int EVAL_MAX_CLASSES = 4;
struct EvalArgs {
    const double* W; const double* V;      // W already offset to the local row block
    int K, nloc, P, T, row_begin;
    const double* target;                  // [nloc][P], NaN = not scored
    const uint8_t* cls; int ncls;          // class per cell (>= ncls: not scored) or nullptr (all class 0)
    int transform, loglik;
    const double* Rdisp; int Rn, Rm, Rt;   // NB dispersion (EVAL_NB_MEAN)
    const Scalars* scal;                   // nu2 of the current sample (Gaussian log-likelihood / predictive cdf)
    const double* nu2c;                    // [nloc][P] known per-cell variances used instead of scal->nu2, or nullptr
    double count;                          // samples seen including this one
    double *mean, *below, *above, *cdf;    // per-cell state, all nullptr when not kept (cdf optional)
    unsigned *c_lt, *c_le;
    double* partial;                       // per-block partial sums
};
long long eval_partial_elems(int nloc, int P, int ncls);
// one saved sample: sample_out[c][4] = {n, sum (y-mu)^2, sum |y-mu|, sum loglik}; 2 launches
void launch_eval_update(const EvalArgs& a, double* sample_out, cudaStream_t st);
void launch_eval_init(double* below, double* above, long long n, cudaStream_t st);
int eval_summary_blocks(int nloc, int P);
void launch_eval_summary(const EvalArgs& a, double lo_pct, double hi_pct, double lo_frac, double hi_frac,
                         double* partial, double* out, cudaStream_t st);

// ---------------------------------------------------------------- K2 row solve
struct RowSolveArgs {
    const double* stats;   // [nsplit][nloc][L+K]
    int nsplit; size_t split_stride;
    int nloc, row_begin, K;
    const double* scale_from_nu2;   // Scalars* (uses 1/nu2) or nullptr (weights already scaled)
    Scalars* scal;
    double* W;             // global [N][K]
    const double* z_inject;   // [N][K] or nullptr
    uint64_t seed;
    double *diag_Q, *diag_L, *diag_mean, *diag_b;   // optional [N][K][K], [N][K]
};
void launch_row_solve(const RowSolveArgs& a, int* nblocks_out, cudaStream_t st);

// ---------------------------------------------------------------- K3 band solve
struct BandSolveArgs {
    const double* stats;   // [nsplit][P][L+K] (column statistics, unscaled)
    int nsplit; size_t split_stride;
    int col_begin, ncols_loc, T, K, order, RD;
    int homoskedastic;     // 1: scale statistics by 1/nu2
    double prior_clip;     // > 0: clip 1/(lam2 tau2) to [prior_clip, 1/prior_clip] (factor.py:767)
    Scalars* scal;
    const double* Tau2;    // [M][RD]
    const int* pm_ptr; const int* pm_row; const double* pm_coef;   // CSR of Delta^T diag Delta band
    double* V;             // [M][T][K]
    const double* z_inject;   // [M][T][K] or nullptr
    uint64_t seed;
    double* work_L;        // [ncols_loc][n][kd+K+1]  (scalar kernel uses the first n*(kd+1) of each)
    double* work_y;        // [ncols_loc][work_y_stride]  y | 1/diag(L)
    size_t work_L_stride, work_y_stride;   // per-column strides (sized for the padded block size)
    int force_psd, attempts; double eps;
    int force_scalar;      // 1: the scalar kernel even where the look-ahead kernel applies (BTF_BAND_SCALAR)
    double *diag_band, *diag_chol, *diag_mean; int* diag_retries;
    double* resid_partials;   // [ncols_loc]: sum_t v^T A v - 2 v.b   (nu2 by-product)
};
void launch_band_solve(const BandSolveArgs& a, cudaStream_t st);
// look-ahead variant (band_lookahead.cu): potrf of step t+1 overlapped with the trailing update of step t
bool launch_band_solve_lookahead(const BandSolveArgs& a, cudaStream_t st);

// ---------------------------------------------------------------- K5 hyper-parameters
struct HyperArgs {
    Scalars* scal;
    const double* V; int M, T, K, RD;
    const int* d_start; const int* d_width; const double* d_coef; int d_maxw;   // Delta stencils
    double *Tau2, *Tau2_a, *Tau2_b, *Tau2_c;
    double stability;
    const double* g_inject;   // [M][4][RD] or nullptr
    uint64_t seed;
    double* lam_partials;     // [M]: 0.5 * sum_{r,k} delta^2 / tau2   (new tau2)
    int col_begin, col_end;
};
void launch_tau2(const HyperArgs& a, cudaStream_t st);
struct ScalarStepArgs {
    Scalars* scal; uint64_t seed;
    double prior_a, prior_b;
    const double* g_inject;   // standard gamma(s) or nullptr
};
// nu2 | rest : uses scal->resid, scal->n_obs
void launch_nu2(const ScalarStepArgs& a, cudaStream_t st);
// sigma2 | rest : uses scal->w_sumsq and n_free
void launch_sigma2(const ScalarStepArgs& a, double n_free, cudaStream_t st);
// lam2, lam2_a | rest
void launch_lam2(const ScalarStepArgs& a, const double* lam_partials, int M, int ref_compat, double shape,
                 cudaStream_t st);
void launch_w_sumsq(const double* W, int N, int K, Scalars* scal, double* partials /* >= 296 */, cudaStream_t st);
void launch_bump_sweep(Scalars* scal, cudaStream_t st);
void launch_clear_info(Scalars* scal, cudaStream_t st);
void launch_set_resid(Scalars* scal, const double* partials, int n, cudaStream_t st);   // resid = ss_total + sum

void launch_init_scalars(Scalars* s, uint64_t seed, int mask, double sigma2_a, double sigma2_b, double nu2_a,
                         double nu2_b, cudaStream_t st);
void launch_init_tau2(double* Tau2, double* Ta, double* Tb, double* Tc, size_t n, uint64_t seed, cudaStream_t st);
void launch_init_W(double* W, int N, int K, const Scalars* s, uint64_t seed, cudaStream_t st);
void launch_clip(double* x, size_t n, double lo, double hi, cudaStream_t st);

// ---------------------------------------------------------------- K4 Polya-Gamma / negative binomial
struct PgArgs {
    const uint8_t* obs; const double* ntr; double* omega; long long ld;
    const double* W; const double* V;     // W local rows [nloc_pad][K], V [Ppad][K]
    int nloc, nrows_pad, P, Ppad, K, row_begin;
    Scalars* scal; uint64_t seed;
};
// omega[i,p] ~ PG(ntr[i,p], w_i . v_p) for observed cells, 0 elsewhere (factor.py:447-460)
void launch_pg_draw(const PgArgs& a, cudaStream_t st);
// standalone sampler for moment tests: out[e] ~ PG(b[e], z[e])
void launch_pg_sample(const double* b, const double* z, double* out, long long n, uint64_t seed,
                      unsigned long long sweep, cudaStream_t st);

void launch_rng_sample(int kind, double param, double* out, long long n, uint64_t seed, cudaStream_t st);

struct NbArgs {
    const double* Yraw;      // [nloc][P][R] raw counts (NaN = missing), contiguous
    int nloc, P, R, M, T, K, row_begin, nrows_global;
    long long ld;
    const double* W; const double* V;
    double* Rdisp;           // dispersion, broadcast shape [Rn, Rm, Rt] (1 where shared)
    int Rn, Rm, Rt;          // extents of R (1 or the dim)
    int nmh; double rpropstdev, rstdev;
    const double* z_inject; const double* u_inject;   // [nmh][Rsize] or nullptr
    Scalars* scal; uint64_t seed;
    double* work;            // scratch [>= 4 * Rsize + nblocks * Rsize ...]
    uint8_t* obs; double* kappa; double* ntr;         // outputs of the pseudo-count refresh
    double* hist; int hist_stride;                    // per-group count histogram [Rs][hist_stride] or nullptr
};
void launch_nb_scan(const double* Y, long long n, unsigned long long* out, cudaStream_t st);
void launch_nb_hist(const NbArgs& a, int vstride, cudaStream_t st);
// R | rest by nmh random-walk MH steps on log R, then N = sum_r (y + R), kappa = sum_r y - N/2
// (factor.py:513-554, 494-511)
void launch_nb_update(const NbArgs& a, cudaStream_t st);

// ---------------------------------------------------------------- GASS steps of the constrained Poisson, Binomial and
// Gaussian models (gass_kernels.cu)
struct GassArgs {
    bool col;                                   // false: one CTA per W row (gass_row_kernel), true: per V column (gass_col_kernel)
    int N, M, T, K, P; long long ld;
    const uint8_t* cnt; const double* S;        // Poisson, Gaussian: observed replicates and their sum; Binomial: observed
                                                // flag and kappa = y - n/2, [N][ld]
    const double* lgy;                          // Poisson: sum of lgamma(y + 1) over the observed replicates; Binomial: the
                                                // log binomial coefficient lgamma(n + 1) - (lgamma(y + 1) + lgamma(n - y + 1));
                                                // Gaussian: sum (y - ybar)^2 over the observed replicates, [N][ld]
    const double *ep_mu, *ep_sig;               // EP approximation [N][ld], or nullptr
    const double* A; const double* C; int J;    // constraints A[c] . Mu[i, j, :] >= C[c], A [J][T]
    const double* rowcons; int nrc;             // row constraints [nrc][K + 1] (W rows only)
    const double* grid_fine; int nfine;         // ascending angle grids of the feasible set
    const double* grid_coarse; int ngrid;
    const double *Wold, *Vold;                  // the state x before the step
    double *Wnew, *Vnew;                        // in: the Gaussian draw mu + v; out: the new state
    const double *Wmean, *Vmean;                // the centre mu (nullptr: 0)
    const double *Wcur, *Vcur;                  // the other factor (column step: W, row step: V)
    const double* u_inject;                     // [rows or cols][ngrid + 2] uniforms, or nullptr (Philox)
    const Scalars* scal; uint64_t seed;
    double* diag;                               // [rows or cols][3] = (F, G, theta), or nullptr
    int check_only; int* nbad;                  // 1: only count the rows / columns whose state violates a constraint
    // (appended, so that the Poisson kernels read every field above at the offsets they always had)
    const double* ntr;                          // Binomial: trials n, [N][ld]
    bool binomial;                              // the cell likelihood: false Poisson, true Binomial
    const double* nu2c;                         // Gaussian: known per-cell variances [N][ld], or nullptr (the scalar nu2)
    bool gaussian;                              // the cell likelihood is Gaussian (then binomial is false)
};
size_t gass_smem_bytes(int D, int nfine, int ngrid);
void launch_gass(const GassArgs& a, cudaStream_t st);

}  // namespace btf
