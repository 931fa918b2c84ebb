/*
 * btf_b200.h -- C ABI of the B200-native Gibbs-sweep engine for Bayesian Tensor
 * Filtering (drop-in for the sampler loop of tansey/functionalmf).
 *
 * The reference has no FFI: its boundary is the Python class API
 * (functionalmf/factor.py:23-563, functionalmf/genlasso.py:37-66).  Every entry
 * point below is what a ctypes binding for that path binds; the citation names
 * the reference code it replaces.  Plain pointers and sizes only; all host
 * arrays are C-order float64 unless stated.  All functions return 0 on success
 * and a negative BTF_E* code on failure (message via btf_last_error()).
 *
 * One engine = one GPU = one host thread.  Multi-GPU: one engine per rank, rows
 * of the data sharded by [row_begin,row_end), columns of the V update by
 * [col_begin,col_end); the exchange steps run over NCCL (btf_nccl_*).
 */
#ifndef BTF_B200_H
#define BTF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BTF_OK            0
#define BTF_EINVAL       -1   /* bad argument / shape */
#define BTF_ECUDA        -2   /* CUDA runtime error */
#define BTF_ENOTPD       -3   /* a Cholesky factorisation failed (after retries) */
#define BTF_ESTATE       -4   /* call order / missing data */
#define BTF_ENCCL        -5   /* NCCL error */

/* BTF_POISSON, BTF_CBINOMIAL and BTF_CGAUSSIAN: the constrained model's built-in likelihoods, whose W and V steps are
 * GASS transitions (Poisson counts; Binomial successes out of trials with the identity link p = W V^T; Gaussian
 * observations with mean W V^T and a noise variance nu2 that is sampled, fixed, or known per cell) */
enum { BTF_GAUSSIAN = 0, BTF_BINOMIAL = 1, BTF_NEGBINOMIAL = 2, BTF_POISSON = 3, BTF_CBINOMIAL = 4, BTF_CGAUSSIAN = 5 };

/* sample_mask bits: which variables resample() updates (factor.py:112-128, 306-311) */
enum {
    BTF_SAMPLE_NU2 = 1, BTF_SAMPLE_SIGMA2 = 2, BTF_SAMPLE_TAU2 = 4, BTF_SAMPLE_LAM2 = 8,
    BTF_SAMPLE_W = 16, BTF_SAMPLE_V = 32, BTF_SAMPLE_R = 64, BTF_SAMPLE_ALL = 127
};

typedef struct btf_engine btf_engine;

/* Constructor arguments of *BayesianTensorFiltering (factor.py:24-36, 287-289,
 * 426-427, 464-471).  Zero-initialise, then btf_config_default(). */
typedef struct btf_config {
    int32_t nrows, ncols, ndepth;      /* global N, M, T */
    int32_t nembeds, tf_order;         /* K, p */
    int32_t likelihood;                /* BTF_GAUSSIAN / BINOMIAL / NEGBINOMIAL / POISSON / CBINOMIAL / CGAUSSIAN */
    double  sigma2_a, sigma2_b;        /* factor.py:27 */
    double  nu2_a, nu2_b;              /* factor.py:289 */
    double  stability;                 /* factor.py:32 */
    int32_t force_psd, force_psd_attempts;   /* factor.py:33-35 */
    double  force_psd_eps;
    int32_t ref_compat_lam2;           /* 1: factor.py:150 as written (last column only) */
    int32_t sample_mask;               /* BTF_SAMPLE_* */
    uint64_t seed;                     /* Philox key */
    int32_t device;                    /* CUDA device ordinal */
    /* negative-binomial dispersion update (factor.py:464-471) */
    int32_t nmetropolis;
    double  rpropstdev, rstdev;
    int32_t rdims_mask;                /* bit d set: R is shared along dim d (0=rows,1=cols,2=depth) */
    /* sharding (single GPU: 0,nrows,0,ncols,1,0) */
    int32_t row_begin, row_end, col_begin, col_end;
    int32_t world_size, rank;
    /* tuning / debugging */
    int32_t resid_direct;              /* 1: always recompute the nu2 residual by a full pass */
    int32_t use_graph;                 /* 1: replay the sweep as a CUDA graph when possible */
    int32_t stats_splits_row, stats_splits_col;  /* 0 = auto */
    int32_t clip_prior_precision;      /* 1: 1/(lam2 Tau2) clipped to [stability, 1/stability] (factor.py:767) */
} btf_config;

void btf_config_default(btf_config* cfg);

int  btf_create(const btf_config* cfg, btf_engine** out);
void btf_destroy(btf_engine* e);
const char* btf_last_error(void);

/* ---- data (factor.py:316-330, 437-445, 494-508).  `Y` holds the LOCAL rows
 * [row_end-row_begin, M, T, nreps]; NaN = missing.  Host or device pointers are
 * both accepted (detected with cudaPointerGetAttributes).  1 <= nreps <= 255: the
 * compact form keeps the number of observed replicates of a cell in one byte (the
 * reference has no such limit; BTF_EINVAL otherwise).  Ordinary (pageable) host memory
 * is copied through pinned bounce buffers by several host threads (DESIGN.md section 2). */
int btf_set_data_gaussian(btf_engine* e, const double* Y, int32_t nreps);
/* streaming form: rows [row0, row0+nrows) of the local shard; reset != 0 on the first piece.  BTF_ESTATE on a
 * BTF_CGAUSSIAN engine, which takes its data whole through btf_set_data_gaussian. */
int btf_set_data_gaussian_rows(btf_engine* e, const double* Y, int32_t row0, int32_t nrows, int32_t nreps,
                               int32_t reset);
/* Successes and trials [Nloc, M, T] each (a cell is missing where either is NaN).  BTF_BINOMIAL (Polya-Gamma) or
 * BTF_CBINOMIAL (see the constrained models below; there every observed cell must hold non-negative integers y <= n,
 * else BTF_EINVAL giving the number of such cells, and nothing changes). */
int btf_set_data_binomial(btf_engine* e, const double* Ysucc, const double* Ntrials);
int btf_set_data_negbin(btf_engine* e, const double* Y, int32_t nreps);
/* Known per-cell noise variances of a Gaussian or constrained Gaussian model: the reference's heteroskedastic branch, nu2 an
 * [N, M, T] array (factor.py:345-346, 390-391; SURVEY.md 3.2).  `nu2` holds the LOCAL rows [Nloc, M, T] in
 * C order, host or device memory; NULL returns to the scalar nu2.  The W and V conditionals then weight
 * cell (i,j,t) by cnt / nu2[i,j,t] with right-hand side S / nu2[i,j,t]; nu2 = +inf makes an observed cell
 * count as missing, and at missing cells any value is accepted.  The weights are formed again after every
 * btf_set_data_gaussian*; the variances are kept on the device (24 B per cell with the two weight buffers).
 * BTF_ESTATE on an engine that is neither BTF_GAUSSIAN nor BTF_CGAUSSIAN, BTF_EINVAL on a sharded one
 * (world_size > 1) and when observed cells have a variance that is NaN or <= 0 (the message gives their
 * number; the engine stays in scalar mode).  While the variances are set, btf_sweep / btf_run* refuse
 * BTF_SAMPLE_NU2 with BTF_ESTATE: the reference holds an array nu2 fixed.  On a BTF_CGAUSSIAN engine no
 * weights are formed (the GASS steps read the variances; its weight buffers hold the EP approximation's):
 * the variances are checked and kept, 8 B per cell. */
int btf_set_nu2_cells(btf_engine* e, const double* nu2);

/* ---- the constrained Poisson, Binomial and Gaussian models (ConstrainedNonconjugateBayesianTensorFiltering with the
 * Poisson likelihood of examples/poisson_tensor_filtering.py, a Binomial or a Gaussian one; factor.py:894-1017).  A
 * BTF_POISSON, BTF_CBINOMIAL or BTF_CGAUSSIAN engine runs the whole sweep on the device: sigma2, Tau2, lam2, then for W and for V the Gaussian centre
 * and proposal (the f64-weight statistics of an EP approximation, or the prior alone) followed by one GASS transition
 * per row / column (gass.py:13-130) under ll = nansum of the cells' log-likelihoods at lambda = W V^T, minus
 * sum_cells norm.logpdf(lambda; mu_ep, sigma_ep) with EP:
 *   Poisson: scipy.stats.poisson.logpmf(y, lambda) over the observed replicates (a cell with lambda < 0 is NaN there and
 *     drops out, lambda = 0 with y > 0 gives -inf);
 *   Binomial: scipy.stats.binom.logpmf(y, n, p = lambda) (p outside [0, 1] is NaN there and drops out; p = 0 with y > 0
 *     and p = 1 with y < n give -inf; n = 0 gives 0).  The data come through btf_set_data_binomial and take 25 B / cell
 *     (observed flag, kappa = y - n/2, n and the log binomial coefficient); btf_set_data_poisson refuses this engine
 *     with BTF_ESTATE, as btf_set_data_binomial refuses a Poisson one.
 *   Gaussian: scipy.stats.norm.logpdf(y, lambda, sqrt(nu2)) over the observed replicates, evaluated per cell in the
 *     centred form -n log sqrt(2 pi nu2) - (ss + n (ybar - lambda)^2) / (2 nu2), ss = sum_r (y_r - ybar)^2.  nu2 is the
 *     scalar state "nu2" or, after btf_set_nu2_cells, the cell's known variance (+inf: the cell is missing).  With
 *     BTF_SAMPLE_NU2 every sweep starts with the Gaussian model's conjugate nu2 step on the residual of the current
 *     (W, V), recomputed by a direct pass each sweep.  The data come through btf_set_data_gaussian (btf_set_data_gaussian_rows
 *     refuses this engine) and take 17 B / cell (count, sum and ss); observed values that are +-inf give BTF_EINVAL with
 *     their number, and nothing changes.  btf_set_data_poisson and btf_set_data_binomial refuse this engine with
 *     BTF_ESTATE, as btf_set_data_gaussian refuses the other two.
 * Single GPU: btf_create refuses world_size > 1 for these likelihoods.
 *
 * Counts Y [Nloc, M, T, nreps] (NaN = missing, host or device memory), kept in the Gaussian data's compact form
 * plus sum_r lgamma(y_r + 1) per cell (17 B / cell).  BTF_EINVAL when observed values are negative or not integers (the message gives their number). */
int btf_set_data_poisson(btf_engine* e, const double* Y, int32_t nreps);
/* Constraints and angle grids (host memory).  A [J, T], C [J]: every cell's depth profile tau = Mu[i, j, :] must satisfy
 * A tau >= C (the Kronecker form of factor.py:711-721, 847-853 is never built); rowcons [nrowcons, K + 1] (may be NULL when
 * nrowcons = 0): row i of W satisfies rowcons[:, :nd] w >= rowcons[:, K], nd = min(K, i + 1).  grid_fine (ascending,
 * ngrid_fine <= 65535 points; gass.py uses linspace(-pi, pi, 10000)) is the grid the feasible angles are taken from;
 * grid_coarse (ngrid points) is used instead when no constraint is active.  ngrid candidates at most are evaluated:
 * 1 <= ngrid <= ngrid_fine.  Every btf_sweep / btf_run* first checks that the state satisfies the constraints
 * ('Invalid starting point!' in the reference) and fails with BTF_ESTATE, giving the number of rows and columns in
 * violation, before anything changes. */
int btf_set_gass(btf_engine* e, const double* A, const double* C, int32_t J, const double* rowcons, int32_t nrowcons,
                 const double* grid_fine, int32_t ngrid_fine, const double* grid_coarse, int32_t ngrid);
/* EP approximation (host memory, [Nloc, M, T] each; NULL: none) of any of these models.  The W / V centres come from the weights 1 / sigma^2 and
 * the right-hand side mu / sigma^2; every candidate's ll subtracts sum norm.logpdf(lambda; mu, sigma) over ALL cells of the
 * row / column.  BTF_EINVAL when a mean is not finite or a scale is not finite and > 0 (with their number). 32 B / cell. */
int btf_set_ep(btf_engine* e, const double* mu, const double* sigma);

/* ---- state: names "W" [N,K] (global), "V" [M,T,K], "Tau2","Tau2_a","Tau2_b",
 * "Tau2_c" [M,R_D], "lam2","lam2_a","sigma2","nu2" [1], "omega" [Nloc,M,T]
 * (Binomial/NB: 1/nu2), "R" [R shape], "Ntrials" [Nloc,M,T] (read-only on BTF_CBINOMIAL engines), "Delta" [R_D,T]
 * (read-only, utils.py:56-98).  `n` = number of doubles in `host`. */
int btf_set_state(btf_engine* e, const char* name, const double* host, size_t n);
int btf_get_state(btf_engine* e, const char* name, double* host, size_t n);
int btf_delta_rows(const btf_engine* e);      /* R_D = Delta.shape[0] */
/* the sample_* flags of the reference are mutable attributes (examples/poisson_tensor_filtering.py:58-81) */
int btf_set_sample_mask(btf_engine* e, int32_t mask);

/* ---- sampling.  btf_sweep = nsweeps x resample(data) (factor.py:306-311,
 * 112-128, 494-511).  btf_run = run_gibbs (genlasso.py:37-66): nburn + nthin *
 * nsamples sweeps, state saved after burn-in every nthin-th sweep into the
 * caller's arrays (any may be NULL): W [S,N,K], V [S,M,T,K], Tau2 [S,M,R_D],
 * scalars [S,4] = (sigma2, lam2, nu2, lam2_a), R [S,*R.shape]. */
int btf_sweep(btf_engine* e, int32_t nsweeps);
int btf_run(btf_engine* e, int32_t nburn, int32_t nthin, int32_t nsamples,
            double* W_out, double* V_out, double* Tau2_out, double* scalars_out,
            double* R_out, double* omega_out);
/* a segment of a chain: exactly nsweeps sweeps; the state after local sweeps first_save,
 * first_save+nthin, ... goes to sample slots sample_offset, sample_offset+1, ... */
int btf_run_segment(btf_engine* e, int32_t nsweeps, int32_t first_save, int32_t nthin, int64_t sample_offset,
                    double* W_out, double* V_out, double* Tau2_out, double* scalars_out,
                    double* R_out, double* omega_out);
int btf_synchronize(btf_engine* e);
/* Running posterior mean / variance of Mu = einsum('nk,mtk->nmt', W, V) on the device, updated at
 * every saved sample (SURVEY.md 8f row 2; the reference keeps all samples on the host,
 * genlasso.py:51-65).  mean_out / var_out: [Nloc, M, T], either may be NULL. */
int btf_mu_stats_track(btf_engine* e, int32_t track);
int btf_mu_stats_get(btf_engine* e, double* mean_out, double* var_out, int64_t* count_out);
/* Held-out evaluation on the device (SURVEY.md 8f row 3).  Replaces the numpy scoring of the saved
 * samples in politics/benchmark.py:163-180 (per-sample RMSE / MAE / Poisson log-likelihood of the NB
 * mean, in-sample vs held-out), flutrends/benchmark.py:129-143 (RMSE / MAE of the posterior mean,
 * coverage of the predictive band, 68-75) and examples/poisson_tensor_filtering.py:20-23
 * (coverage_at: truth inside the central np.percentile band of the samples).
 *   target [Nloc, M, T]  value to score against, NaN = not scored
 *   cls    [Nloc, M, T]  class of every cell (0 .. nclasses-1; anything else = not scored), NULL = all 0
 *   transform  0 identity, 1 ilogit(psi), 2 NB mean R P / (1 - P) with P = ilogit(clip(psi, -10, 10))
 *   loglik     0 none, 1 Gaussian with the sample's nu2, 2 Poisson
 *   cell_state 0 per-sample sums only; 1 + per-cell running mean and percentile-band state (40 B/cell);
 *              2 + mixture cdf for the Gaussian posterior-predictive band
 *   auto_update != 0: every sample saved by btf_run / btf_run_segment is scored
 * Up to 4 evaluators (slots 0..3) per engine.  Sums are over the LOCAL rows; ranks add them up. */
int btf_eval_set(btf_engine* e, int32_t slot, const double* target, const uint8_t* cls, int32_t nclasses,
                 int32_t transform, int32_t loglik, int32_t cell_state, int32_t auto_update, int64_t max_samples);
/* Per-cell variances [Nloc, M, T] of the slot's cells (host or device memory; NULL: back to the sample's
 * scalar nu2): the Gaussian log-likelihood per sample and of the posterior mean, and the predictive band,
 * then use nu2[cell], as the reference's heteroskedastic branch scores a model fitted with known
 * variances (see btf_set_nu2_cells).  Call after btf_eval_set, which clears them. */
int btf_eval_set_nu2(btf_engine* e, int32_t slot, const double* nu2);
int btf_eval_clear(btf_engine* e, int32_t slot);
int btf_eval_update(btf_engine* e, int32_t slot);
/* out [count, nclasses, 4] = {n, sum (y-mu)^2, sum |y-mu|, sum loglik} per scored sample */
int btf_eval_samples(btf_engine* e, int32_t slot, double* out, int64_t* count_out);
/* out [nclasses, 6] = {n, sum (y-mean)^2, sum |y-mean|, sum loglik(y|mean), # targets inside the
 * [lo_pct, hi_pct] percentile band of the samples, # targets with pred_lo <= predictive cdf <= pred_hi};
 * mean_out (optional) [Nloc, M, T] posterior mean of the transformed surface */
int btf_eval_summary(btf_engine* e, int32_t slot, double lo_pct, double hi_pct, double pred_lo, double pred_hi,
                     double* out, double* mean_out);
/* Constructor draws from the priors on the device (factor.py:230-253, 293-304, 560-563;
 * utils.py:115-124).  init_mask bits: 1 sigma2, 2 lam2, 4 nu2, 8 Tau2, 16 W, 32 V, 64 R. */
int btf_init_state(btf_engine* e, int32_t init_mask);
/* pinned host memory for result arrays (so sample collection overlaps the next sweep) */
void* btf_host_alloc(size_t bytes);
void  btf_host_free(void* p);
int   btf_host_register(void* p, size_t bytes);     /* page-lock an existing allocation in place */
int   btf_host_unregister(void* p);
/* nsweeps sweeps bracketed by CUDA events on the engine's stream; *ms_out = elapsed ms */
int btf_sweep_timed(btf_engine* e, int32_t nsweeps, double* ms_out);

/* ---- parity hooks.  Inject the noise the NEXT sweep consumes instead of the
 * Philox stream (cleared after that sweep): "z_W" [N,K], "z_V" [M,T,K] t-major,
 * "g_tau" [M,4,R_D], "g_lam" [2], "g_sigma2" [1], "g_nu2" [1] (standard gammas),
 * "omega" [Nloc,M,T], "z_R"/"u_R" [nmetropolis,*R.shape],
 * "gass_u_W" [N, ngrid+2], "gass_u_V" [M, ngrid+2] (GASS models: per row / column the slice uniform, ngrid thinning
 * uniforms -- candidate k swaps position k with k + floor(u_k (F - k)) of the ascending feasible list when F > ngrid --
 * and the pick uniform: candidate floor(u G) of the G at or above the slice). */
int btf_inject_noise(btf_engine* e, const char* name, const double* host, size_t n);
/* Diagnostics of the LAST sweep (enable with btf_enable_diag before it):
 * "W_Q","W_L" [N,K,K], "W_mean" [N,K], "W_b" [N,K], "V_mean" [M,T,K],
 * "V_band","V_chol" [Mloc,T*K,(p+1)K+1] (column j of the band / factor in row j),
 * "V_retries" [Mloc], "row_stats" [Nloc,L+K], "col_stats" [M*T,L+K],
 * "nu2_rate" [3] = (a_post,b_post,n_obs), "lam2_rate" [2],
 * "i8_route" [2] = route of the last row / column product block of the integer
 * statistics path: 0 none yet, 2 2-CTA kernel with the fused epilogue, 3 2-CTA
 * kernel in split-K mode (recorded without btf_enable_diag),
 * "gass_W" [N,3], "gass_V" [M,3] = (# feasible grid angles F, # candidates at or above the slice G, chosen angle;
 * 0 when the state is kept). */
int btf_enable_diag(btf_engine* e, int32_t on);
int btf_get_diag(btf_engine* e, const char* name, double* host, size_t n);

/* ---- counters / measurement */
int64_t btf_kernel_launches(const btf_engine* e);   /* kernels launched by this engine so far */
int  btf_time_phases(btf_engine* e, int32_t nsweeps, double* ms_out, int32_t nphases); /* per-phase ms */
/* FP64 throughput micro-benchmarks (roofline denominators):
 * mode 0 = DFMA chains, 1 = mma.sync m8n8k4 f64 (DMMA).  Returns TFLOP/s. */
double btf_fp64_peak(int32_t device, int32_t mode, int32_t iters);
double btf_hbm_copy_gbs(int32_t device, size_t bytes, int32_t iters);
/* int8 tensor-core throughput (tcgen05.mma.kind::i8, operands resident in shared memory, every SM busy):
 * the measured denominator of the int8 GEMM's roofline.  Returns Top/s (2 x MAC). */
double btf_i8_peak(int32_t device, int32_t iters);

/* ---- sampler test hooks: out[e] ~ PG(b[e], z[e]) (replaces pypolyagamma pgdrawv, factor.py:459);
 * raw variates of the device generator: kind 0 normal, 1 gamma(param), 2 exponential, 3 uniform */
int btf_pg_sample(int32_t device, const double* b, const double* z, double* out, int64_t n, uint64_t seed);
int btf_rng_sample(int32_t device, int32_t kind, double param, double* out, int64_t n, uint64_t seed);

/* ---- NCCL plumbing for the sharded sweep (SURVEY.md section 8e) */
int btf_nccl_unique_id(char* id128);                    /* 128-byte ncclUniqueId */
int btf_nccl_init(btf_engine* e, const char* id128);    /* uses cfg.world_size / cfg.rank */

#ifdef __cplusplus
}
#endif
#endif /* BTF_B200_H */
