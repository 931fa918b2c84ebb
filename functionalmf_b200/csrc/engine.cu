// C ABI of the BTF Gibbs-sweep engine (include/btf_b200.h): device-resident state,
// sweep scheduling (eager or CUDA-graph replay), sample collection, parity hooks.
#include "../../include/btf_b200.h"
#include "kernels.h"
#include "nccl_shard.h"

#include <nvtx3/nvToolsExt.h>
#include <sched.h>
#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <map>
#include <string>
#include <thread>
#include <vector>

using namespace btf;

static thread_local char g_err[512] = "";
static int set_err(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CK(call)                                                                              \
    do {                                                                                      \
        cudaError_t _e = (call);                                                              \
        if (_e != cudaSuccess)                                                                \
            return set_err(BTF_ECUDA, "%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
    } while (0)

struct DevBuf {
    double* p = nullptr;
    size_t n = 0;
};

// Environment switches (INTEGRATION.md §1), read once per engine by read_env(); the kernel files get the values as arguments.
struct EnvSwitches {
    bool no_i8 = false, force_i8 = false;   // BTF_STATS_NO_I8, BTF_STATS_FORCE_I8
    bool i8_guard = true;                   // BTF_I8_NO_GUARD
    double i8_guard_tol = 1e-12;            // BTF_I8_GUARD_TOL
    bool scol = true;                       // BTF_NO_SCOL
    bool upload_bounce = true;              // BTF_UPLOAD_BOUNCE
    int upload_threads = 0;                 // BTF_UPLOAD_THREADS (0: the cores this process may use, at most 16)
    bool nvtx = false;                      // BTF_NVTX
    bool band_scalar = false;               // BTF_BAND_SCALAR
    bool nb_hist = true;                    // BTF_NB_NO_HIST
};

enum Phase { PH_NU2 = 0, PH_SIGMA2, PH_TAU2, PH_LAM2, PH_ROW_STATS, PH_ROW_SOLVE, PH_COL_STATS, PH_BAND_SOLVE, PH_COMM, PH_COUNT };

// one held-out evaluator (eval_kernels.cu)
struct EvalSlot {
    bool active = false, auto_update = false;
    int ncls = 1, transform = 0, loglik = 0;
    double* target = nullptr; uint8_t* cls = nullptr;
    double *mean = nullptr, *below = nullptr, *above = nullptr, *cdf = nullptr;
    unsigned *c_lt = nullptr, *c_le = nullptr;
    double *partial = nullptr, *samples = nullptr, *summary = nullptr;
    double* nu2 = nullptr;       // [nloc][P] known per-cell variances of the scored cells (btf_eval_set_nu2)
    long long count = 0, max_samples = 0;
};
constexpr int EVAL_SLOTS = 4;

struct btf_engine {
    btf_config cfg;
    int N, M, T, K, order, q, kd, RD, L, nco, P, Ppad, nloc, nloc_pad, n;
    int Mloc;
    int Nall_pad;                // global row count padded to 128: contraction length of the column-sharded product block
    int p0, Ploc;                // this rank's (j,t) range: [p0, p0 + Ploc) = [col_begin T, col_end T)
    int Kp;                      // K rounded up to the band solver's block size (8, 16, 32)
    size_t wL_stride, wy_stride; // per-column workspace strides of the band solver
    int sm_count;
    cudaStream_t stream = nullptr, copy_stream = nullptr;
    cudaStream_t side[2] = {nullptr, nullptr};   // forked inside a sweep: tensor-core product block | HBM-bound linear block
    cudaEvent_t ev_fork = nullptr, ev_join[2] = {nullptr, nullptr};
    EnvSwitches env;
    // state
    double *W = nullptr, *V = nullptr, *Tau2 = nullptr, *Tau2_a = nullptr, *Tau2_b = nullptr, *Tau2_c = nullptr;
    Scalars* scal = nullptr;
    // data
    uint8_t* cnt = nullptr;      // Gaussian: # observed replicates; PG paths: observed flag
    double* S = nullptr;         // Gaussian: replicate sum; PG paths: kappa = y - n/2
    double* ntr = nullptr;       // PG paths: number of trials b
    double* omega = nullptr;     // PG paths: Polya-Gamma draws
    double* Yraw = nullptr;      // NB: raw counts [nloc][P][R]
    // Gaussian with known per-cell noise variances (btf_set_nu2_cells; single GPU): the statistics take the f64 weights
    // wc = cnt / nu2 and sc = S / nu2, formed from the kept variances nu2c whenever data or variances change
    bool nu2_cells = false, nu2_dirty = false;
    unsigned long long nu2_bad = 0;                            // observed cells whose variance is NaN or <= 0
    double *nu2c = nullptr, *wc = nullptr, *sc = nullptr;      // [nloc_pad][Ppad], allocated on first use
    unsigned long long* nu2_nbad = nullptr;
    StatsPlan plan_row_w{}, plan_col_w{};                      // statistics plans for those f64 weights
    // Constrained Poisson, Binomial and Gaussian models (GASS steps, gass_kernels.cu; single GPU).  With an EP
    // approximation the W / V centres come from the f64-weight statistics of wc = 1 / sigma^2 and sc = mu / sigma^2 (the
    // buffers of the per-cell nu2 mode; a constrained Gaussian engine keeps its known variances in nu2c alone)
    bool gass_set = false, ep_on = false;
    int gJ = 0, gnrc = 0, gnfine = 0, gngrid = 0;
    double *gA = nullptr, *gC = nullptr, *growc = nullptr, *ggrid_f = nullptr, *ggrid_c = nullptr;
    double *Wold = nullptr, *Vold = nullptr, *gmeanW = nullptr, *gmeanV = nullptr;   // the state before the step, the centres
    double *ep_mu = nullptr, *ep_sig = nullptr;                // [nloc_pad][Ppad]
    double* lgy = nullptr;                                     // [nloc_pad][Ppad] Poisson: sum of lgamma(y + 1) over the observed
                                                               // replicates; Binomial: the log binomial coefficient;
                                                               // Gaussian: sum (y - ybar)^2 over the observed replicates
    int* gass_nbad = nullptr;                                  // [2] rows / columns whose starting point violates a constraint
    int nreps = 1;
    bool has_data = false, data_reduced = false;
    double* staging[2] = {nullptr, nullptr};   // upload staging (kept for the engine's lifetime: no malloc/free per call, no leak on error paths)
    size_t staging_bytes = 0;
    cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_k0[2] = {nullptr, nullptr};
    double* hstage[2] = {nullptr, nullptr};    // pinned bounce buffers for uploads from ordinary (pageable) host memory
    size_t hstage_bytes = 0;
    // NB dispersion
    double* Rdisp = nullptr; int Rn = 1, Rm = 1, Rt = 1; double* nb_work = nullptr;
    double* nb_hist = nullptr; int nb_hist_stride = 0;   // count histograms per R group (integer counts)
    // penalty
    std::vector<double> delta;   // dense [RD][T]
    int *d_start = nullptr, *d_width = nullptr; double* d_coef = nullptr; int d_maxw = 0;
    int *pm_ptr = nullptr, *pm_row = nullptr; double* pm_coef = nullptr;
    // statistics
    StatsPlan plan_row, plan_col;
    double *row_stats = nullptr, *col_stats = nullptr;
    bool col_collapsed = false;  // split 0 of col_stats already holds the sum over splits
    // K1 on the integer tensor cores (stats_i8.cu): decided per data set, buffers allocated on first use
    bool i8_on = false, i8_decided = false;
    StatsI8Buffers i8{};
    int i8_route[2] = {0, 0};    // I8Route of the last row / column product block (0: none yet)
    unsigned *cnt_rowsum = nullptr, *cnt_colsum = nullptr;   // sum of the counts of every local row / owned (j,t): guard of the fixed-point block
    int* guard_n = nullptr;                                  // [2] rows / (j,t) recomputed in FP64 by the last W / V step
    unsigned char* guard_flags = nullptr;                    // [nloc + Ploc] flags set by the kernels that produce the block
    double* Scol = nullptr;      // sharded engines, when it fits: S of this rank's (j,t) over ALL rows, [Nall_pad][Ploc_pad] -> the
                                 // linear block of the V step needs no reduce-scatter
    int Ploc_pad = 0;
    uint8_t* cntT = nullptr;     // [Ploc][Nall_pad] counts of this rank's columns over ALL rows (right operand of the column contraction)
    double *mu_mean = nullptr, *mu_m2 = nullptr; long long mu_count = 0; bool mu_track = false;   // posterior moments of Mu
    double* zbuf = nullptr;      // pre-generated right operand of the statistics GEMMs (plan.zpre)
    EvalSlot eval[EVAL_SLOTS];
    // workspaces
    double *work_L = nullptr, *work_y = nullptr, *partials = nullptr, *lam_partials = nullptr, *resid_partials = nullptr;
    size_t partials_n = 0;
    // snapshots for async sample collection
    double *snapW = nullptr, *snapV = nullptr, *snapTau2 = nullptr, *snapScal = nullptr, *snapR = nullptr;
    cudaEvent_t ev_snap = nullptr, ev_copied = nullptr;
    double* pinned_scal = nullptr;
    // parity hooks
    std::map<std::string, DevBuf> inject;
    bool diag = false;
    std::map<std::string, DevBuf> diagbuf;
    int* diag_retries = nullptr;
    // scheduling
    bool resid_valid = false;
    bool tau_sharded = false;    // Tau2 chain updated for own columns (+ the last column) only; gathered at API boundaries
    bool tau_stale = false;
    int64_t eager_sweeps = 0;    // sharded engines run their first sweep eagerly (NCCL sets up its channels on first use)
    cudaGraphExec_t graph_exec = nullptr;
    int graph_launches = 0;
    int64_t launches = 0;
    // phase timing
    bool time_phases = false;
    cudaEvent_t ph_ev[PH_COUNT + 1] = {nullptr};
    cudaEvent_t i8_ev[2][3] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};   // [row|col][before gemm, after gemm, after linear]
    double ph_ms[PH_COUNT] = {0};
    // multi GPU
    NcclShard* shard = nullptr;
};

static int round_up(int x, int m) { return (x + m - 1) / m * m; }

// the likelihoods whose W and V steps are GASS transitions (gass_kernels.cu)
static bool gass_likelihood(int lik) { return lik == BTF_POISSON || lik == BTF_CBINOMIAL || lik == BTF_CGAUSSIAN; }
static const char* gass_name(int lik) { return lik == BTF_POISSON ? "Poisson" : lik == BTF_CBINOMIAL ? "Binomial" : "Gaussian"; }

void btf_config_default(btf_config* c) {
    memset(c, 0, sizeof(*c));
    c->nembeds = 5; c->tf_order = 2;
    c->sigma2_a = c->sigma2_b = 0.1; c->nu2_a = c->nu2_b = 0.1;
    c->stability = 1e-6;
    c->force_psd = 1; c->force_psd_eps = 1e-6; c->force_psd_attempts = 4;
    c->ref_compat_lam2 = 1;
    c->sample_mask = BTF_SAMPLE_ALL;
    c->seed = 42;
    c->nmetropolis = 30; c->rpropstdev = 0.1; c->rstdev = 1.0; c->rdims_mask = 7;
    c->world_size = 1;
    c->use_graph = 1;
}

const char* btf_last_error(void) { return g_err; }

// ---- trend-filtering penalty (utils.py:56-98), dense on the host
static std::vector<double> build_delta(int T, int order, int* RD_out) {
    auto matmul = [](const std::vector<double>& A, int ar, int ac, const std::vector<double>& B, int bc) {
        std::vector<double> C((size_t)ar * bc, 0.0);
        for (int i = 0; i < ar; ++i)
            for (int k = 0; k < ac; ++k) {
                double a = A[(size_t)i * ac + k];
                if (a == 0.0) continue;
                for (int j = 0; j < bc; ++j) C[(size_t)i * bc + j] += a * B[(size_t)k * bc + j];
            }
        return C;
    };
    std::vector<double> D((size_t)(T - 1) * T, 0.0), Dt((size_t)T * (T - 1), 0.0);
    for (int i = 0; i < T - 1; ++i) {
        D[(size_t)i * T + i] = -1.0; D[(size_t)i * T + i + 1] = 1.0;
        Dt[(size_t)i * (T - 1) + i] = -1.0; Dt[(size_t)(i + 1) * (T - 1) + i] = 1.0;
    }
    std::vector<double> out(T, 0.0);
    out[0] = 1.0;   // anchor row e_0
    int rows = 1;
    for (int k = 0; k <= order; ++k) {
        std::vector<double> cur = D;
        int cr = T - 1;
        for (int i = 0; i < k; ++i) {
            if (i % 2 == 0) { cur = matmul(Dt, T, T - 1, cur, T); cr = T; }
            else { cur = matmul(D, T - 1, T, cur, T); cr = T - 1; }
        }
        out.insert(out.end(), cur.begin(), cur.end());
        rows += cr;
    }
    *RD_out = rows;
    return out;
}

template <typename Tp>
static cudaError_t dev_alloc(Tp** p, size_t n, bool zero = true) {
    // cudaMemset of device memory returns before the fill has run, and the fill is ordered on the LEGACY stream, which
    // the engine's non-blocking streams do not wait for: without the synchronize a kernel enqueued right after the
    // allocation can have its output zeroed underneath it (seen as a half-zeroed column count matrix at C2 sizes).
    cudaError_t e = cudaMalloc((void**)p, std::max<size_t>(n, 1) * sizeof(Tp));
    if (e == cudaSuccess && zero) {
        e = cudaMemsetAsync(*p, 0, std::max<size_t>(n, 1) * sizeof(Tp), cudaStreamLegacy);
        if (e == cudaSuccess) e = cudaStreamSynchronize(cudaStreamLegacy);
    }
    return e;
}

// Blocking host-to-device copy that has LANDED when it returns: cudaMemcpy from pageable memory may return once the bytes
// are staged, the transfer itself being ordered on the legacy stream only - which the engine's non-blocking streams do
// not wait for.
static cudaError_t h2d(void* dst, const void* src, size_t bytes) {
    cudaError_t e = cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaStreamSynchronize(cudaStreamLegacy);
    return e;
}

static bool is_device_ptr(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

// The environment switches of INTEGRATION.md §1, read when an engine is created.
static EnvSwitches read_env() {
    auto on = [](const char* nm) { return getenv(nm) != nullptr; };
    EnvSwitches s;
    s.no_i8 = on("BTF_STATS_NO_I8");
    s.force_i8 = on("BTF_STATS_FORCE_I8");
    s.i8_guard = !on("BTF_I8_NO_GUARD");
    if (const char* t = getenv("BTF_I8_GUARD_TOL")) s.i8_guard_tol = atof(t);
    s.scol = !on("BTF_NO_SCOL");
    if (const char* b = getenv("BTF_UPLOAD_BOUNCE")) s.upload_bounce = b[0] != '0';
    if (const char* n = getenv("BTF_UPLOAD_THREADS")) s.upload_threads = std::max(1, atoi(n));
    s.nvtx = on("BTF_NVTX");
    s.band_scalar = on("BTF_BAND_SCALAR");
    s.nb_hist = !on("BTF_NB_NO_HIST");
    return s;
}

void btf_destroy(btf_engine* e);

int btf_create(const btf_config* c, btf_engine** out) {
    if (!c || !out) return set_err(BTF_EINVAL, "null argument");
    if (c->nrows < 1 || c->ncols < 1 || c->ndepth < 2) return set_err(BTF_EINVAL, "bad shape");
    if (c->nembeds < 1 || c->nembeds > 32) return set_err(BTF_EINVAL, "nembeds must be in [1, 32]");
    if (c->tf_order < 0 || c->tf_order > 3) return set_err(BTF_EINVAL, "tf_order must be in [0, 3]");
    if (c->ndepth < c->tf_order + 2) return set_err(BTF_EINVAL, "ndepth must be >= tf_order + 2");
    if (c->likelihood < BTF_GAUSSIAN || c->likelihood > BTF_CGAUSSIAN) return set_err(BTF_EINVAL, "unknown likelihood %d", c->likelihood);
    if (gass_likelihood(c->likelihood) && c->world_size > 1)
        return set_err(BTF_EINVAL, "the constrained %s model is single-GPU", gass_name(c->likelihood));
    btf_engine* e = new btf_engine();
    // every early return below releases what has been created so far (streams, events, device buffers)
    struct Guard { btf_engine* e; ~Guard() { if (e) btf_destroy(e); } } guard{e};
    e->cfg = *c;
    if (e->cfg.world_size <= 1) {
        e->cfg.world_size = 1; e->cfg.rank = 0;
        e->cfg.row_begin = 0; e->cfg.row_end = c->nrows; e->cfg.col_begin = 0; e->cfg.col_end = c->ncols;
    }
    e->N = c->nrows; e->M = c->ncols; e->T = c->ndepth; e->K = c->nembeds; e->order = c->tf_order;
    e->q = e->order + 1; e->kd = e->q * e->K; e->n = e->T * e->K;
    e->L = e->K * (e->K + 1) / 2; e->nco = e->L + e->K;
    e->P = e->M * e->T; e->Ppad = round_up(e->P, 256);
    e->nloc = e->cfg.row_end - e->cfg.row_begin;
    e->nloc_pad = round_up(std::max(e->nloc, 1), 128);
    e->Mloc = e->cfg.col_end - e->cfg.col_begin;
    if (e->nloc < 0 || e->Mloc < 0) { return set_err(BTF_EINVAL, "bad shard"); }
    e->Nall_pad = e->cfg.world_size > 1 ? round_up(e->N, 128) : e->nloc_pad;
    e->p0 = e->cfg.col_begin * e->T; e->Ploc = e->Mloc * e->T;
    e->env = read_env();
    CK(cudaSetDevice(c->device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, c->device));
    e->sm_count = prop.multiProcessorCount;
    {
        // the main stream carries the latency-bound kernels (band solve, row solve): highest priority, so that their CTAs
        // are placed ahead of the queued tiles of the throughput kernels on the side streams
        int lo = 0, hi = 0;
        CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        CK(cudaStreamCreateWithPriority(&e->stream, cudaStreamNonBlocking, hi));
    }
    CK(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        // side[0] (tensor-core product block) above side[1] (linear block): when both have CTAs pending, the GEMM's persistent
        // CTA pairs are placed first and the linear block fills what is left of every SM
        { int lo = 0, hi = 0; CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));
          CK(cudaStreamCreateWithPriority(&e->side[i], cudaStreamNonBlocking, i == 0 ? std::min(lo, hi + 1) : lo)); }
        CK(cudaEventCreateWithFlags(&e->ev_join[i], cudaEventDisableTiming));
    }
    CK(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&e->ev_snap, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&e->ev_copied, cudaEventDisableTiming));
    for (int i = 0; i <= PH_COUNT; ++i) CK(cudaEventCreate(&e->ph_ev[i]));
    for (int i = 0; i < 6; ++i) CK(cudaEventCreate(&e->i8_ev[i / 3][i % 3]));

    e->delta = build_delta(e->T, e->order, &e->RD);
    const int RD = e->RD, T = e->T, q = e->q;
    // stencils
    std::vector<int> hs(RD), hw(RD);
    int maxw = 1;
    for (int r = 0; r < RD; ++r) {
        int a = -1, b = -1;
        for (int t = 0; t < T; ++t) if (e->delta[(size_t)r * T + t] != 0.0) { if (a < 0) a = t; b = t; }
        hs[r] = a < 0 ? 0 : a; hw[r] = a < 0 ? 0 : b - a + 1;
        maxw = std::max(maxw, hw[r]);
    }
    e->d_maxw = maxw;
    std::vector<double> hc((size_t)RD * maxw, 0.0);
    for (int r = 0; r < RD; ++r)
        for (int x = 0; x < hw[r]; ++x) hc[(size_t)r * maxw + x] = e->delta[(size_t)r * T + hs[r] + x];
    // CSR of the band of Delta^T diag(.) Delta : entry (t, m) -> P[t+m, t]
    std::vector<int> pp(1, 0), pr;
    std::vector<double> pc;
    for (int t = 0; t < T; ++t)
        for (int m = 0; m <= q; ++m) {
            if (t + m < T)
                for (int r = 0; r < RD; ++r) {
                    double a = e->delta[(size_t)r * T + t], b = e->delta[(size_t)r * T + t + m];
                    if (a != 0.0 && b != 0.0) { pr.push_back(r); pc.push_back(a * b); }
                }
            pp.push_back((int)pr.size());
        }
    CK(dev_alloc(&e->d_start, RD)); CK(dev_alloc(&e->d_width, RD)); CK(dev_alloc(&e->d_coef, hc.size()));
    CK(dev_alloc(&e->pm_ptr, pp.size())); CK(dev_alloc(&e->pm_row, pr.size())); CK(dev_alloc(&e->pm_coef, pc.size()));
    CK(h2d(e->d_start, hs.data(), RD * sizeof(int)));
    CK(h2d(e->d_width, hw.data(), RD * sizeof(int)));
    CK(h2d(e->d_coef, hc.data(), hc.size() * sizeof(double)));
    CK(h2d(e->pm_ptr, pp.data(), pp.size() * sizeof(int)));
    if (!pr.empty()) {
        CK(h2d(e->pm_row, pr.data(), pr.size() * sizeof(int)));
        CK(h2d(e->pm_coef, pc.data(), pc.size() * sizeof(double)));
    }

    // state (W and V padded with zero rows so the statistics tiles may over-read)
    const size_t Wn = ((size_t)round_up(e->N, 128) + 256) * e->K;
    CK(dev_alloc(&e->W, Wn));
    CK(dev_alloc(&e->V, (size_t)e->Ppad * e->K + 64));
    const size_t tn = (size_t)e->M * RD;
    CK(dev_alloc(&e->Tau2, tn)); CK(dev_alloc(&e->Tau2_a, tn)); CK(dev_alloc(&e->Tau2_b, tn)); CK(dev_alloc(&e->Tau2_c, tn));
    CK(dev_alloc(&e->scal, 1));
    Scalars h;
    memset(&h, 0, sizeof(h));
    h.nu2 = 1.0; h.sigma2 = 1.0; h.lam2 = 1.0; h.lam2_a = 1.0;
    CK(h2d(e->scal, &h, sizeof(h)));
    // one-time fills so a forgotten set_state cannot divide by zero
    {
        std::vector<double> ones(tn, 1.0);
        for (double* p : {e->Tau2, e->Tau2_a, e->Tau2_b, e->Tau2_c})
            CK(h2d(p, ones.data(), tn * sizeof(double)));
    }

    // data
    const size_t cells = (size_t)e->nloc_pad * e->Ppad;
    CK(dev_alloc(&e->cnt, cells));
    CK(dev_alloc(&e->S, cells));
    const bool pg = c->likelihood != BTF_GAUSSIAN;      // f64 weights in the statistics (GASS models: the EP weights)
    if (c->likelihood == BTF_BINOMIAL || c->likelihood == BTF_NEGBINOMIAL) { CK(dev_alloc(&e->ntr, cells)); CK(dev_alloc(&e->omega, cells)); }
    if (c->likelihood == BTF_CBINOMIAL) CK(dev_alloc(&e->ntr, cells));
    if (c->likelihood == BTF_NEGBINOMIAL) {
        e->Rn = (c->rdims_mask & 1) ? 1 : e->N;
        e->Rm = (c->rdims_mask & 2) ? 1 : e->M;
        e->Rt = (c->rdims_mask & 4) ? 1 : e->T;
        CK(dev_alloc(&e->Rdisp, (size_t)e->Rn * e->Rm * e->Rt));
    }

    // statistics plans and buffers
    if (!plan_stats(&e->plan_row, e->K, false, pg, e->nloc_pad, e->Ppad, e->nloc, c->stats_splits_row, e->sm_count))
        { return set_err(BTF_EINVAL, "no row-statistics plan for K=%d", c->nembeds); }
    if (!plan_stats(&e->plan_col, e->K, true, pg, e->Ppad, e->nloc_pad, e->P, c->stats_splits_col, e->sm_count))
        { return set_err(BTF_EINVAL, "no column-statistics plan for K=%d", c->nembeds); }
    CK(dev_alloc(&e->row_stats, e->plan_row.nsplit * e->plan_row.out_elems_per_split));
    CK(dev_alloc(&e->col_stats, e->plan_col.nsplit * e->plan_col.out_elems_per_split));
    {
        size_t zr = e->plan_row.zpre ? (size_t)e->Ppad * e->plan_row.zwg : 0;
        size_t zc = e->plan_col.zpre ? (size_t)e->nloc_pad * e->plan_col.zwg : 0;
        if (std::max(zr, zc)) CK(dev_alloc(&e->zbuf, std::max(zr, zc)));
    }

    // workspaces (the blocked band solver works on K padded to 8 / 16 / 32)
    e->Kp = e->K <= 8 ? 8 : (e->K <= 16 ? 16 : 32);
    e->wL_stride = std::max((size_t)e->T * (e->q + 1) * e->Kp * e->Kp, (size_t)e->n * (e->kd + 1));
    e->wy_stride = (size_t)2 * e->T * e->Kp;
    CK(dev_alloc(&e->work_L, (size_t)std::max(e->Mloc, 1) * e->wL_stride));
    CK(dev_alloc(&e->work_y, (size_t)std::max(e->Mloc, 1) * e->wy_stride));
    e->partials_n = std::max<size_t>((size_t)(e->Ppad / 256) * (e->nloc_pad / 64), (size_t)2 * 148 * 16) + 64;
    CK(dev_alloc(&e->partials, e->partials_n));
    CK(dev_alloc(&e->lam_partials, e->M + 512));     // [M] lam2 partials + scratch for the W sum of squares
    CK(dev_alloc(&e->resid_partials, e->M));
    CK(dev_alloc(&e->snapW, (size_t)e->N * e->K));
    CK(dev_alloc(&e->snapV, (size_t)e->P * e->K));
    CK(dev_alloc(&e->snapTau2, tn));
    CK(dev_alloc(&e->snapScal, 8));
    if (e->Rdisp) CK(dev_alloc(&e->snapR, (size_t)e->Rn * e->Rm * e->Rt));
    CK(cudaMallocHost((void**)&e->pinned_scal, 64 * sizeof(double)));
    CK(dev_alloc(&e->diag_retries, std::max(e->Mloc, 1)));
    // shared-memory needs that grow with the depth (tau2_kernel stages V[j] = T K doubles; the band kernels keep T (q + 1)
    // + RD doubles of per-column tables): refuse shapes that cannot launch instead of failing inside a sweep
    {
        // tau2_kernel stages V[j] (T K doubles); the band kernels keep T (q + 1) + RD doubles of per-column tables next to their window
        const size_t blk = (size_t)e->Kp * (e->Kp + 4), nblk = (size_t)(e->q + 1) * (e->q + 2) / 2;
        const size_t need = std::max((size_t)e->T * e->K, (size_t)e->T * (e->q + 1) + e->RD + (nblk + 2) * blk + 1024) * sizeof(double);
        if (need > (size_t)prop.sharedMemPerBlockOptin)
            return set_err(BTF_EINVAL, "ndepth = %d needs %zu bytes of shared memory per block, the device offers %zu", e->T, need,
                           (size_t)prop.sharedMemPerBlockOptin);
    }
    guard.e = nullptr;
    *out = e;
    return BTF_OK;
}

// the statistics plan of the rows (col = false) or columns: count weights, or f64 weights with per-cell variances
static const StatsPlan& stats_plan(const btf_engine* e, bool col) {
    // (a constrained Gaussian engine's variances do not enter the statistics: its f64 weights are the EP approximation's)
    if (e->nu2_cells && e->cfg.likelihood == BTF_GAUSSIAN) return col ? e->plan_col_w : e->plan_row_w;
    return col ? e->plan_col : e->plan_row;
}

static void free_graph(btf_engine* e) {
    if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
}

static void eval_free(EvalSlot& s) {
    void* ptrs[] = {s.target, s.cls, s.mean, s.below, s.above, s.cdf, s.c_lt, s.c_le, s.partial, s.samples, s.summary, s.nu2};
    for (void* p : ptrs) if (p) cudaFree(p);
    s = EvalSlot();
}

void btf_destroy(btf_engine* e) {
    if (!e) return;
    cudaSetDevice(e->cfg.device);
    cudaDeviceSynchronize();
    free_graph(e);
    if (e->shard) nccl_shard_destroy(e->shard);
    void* ptrs[] = {e->W, e->V, e->Tau2, e->Tau2_a, e->Tau2_b, e->Tau2_c, e->scal, e->cnt, e->S, e->ntr, e->omega,
                    e->Yraw, e->Rdisp, e->nb_work, e->nb_hist, e->d_start, e->d_width, e->d_coef, e->pm_ptr, e->pm_row, e->pm_coef,
                    e->row_stats, e->col_stats, e->zbuf, e->mu_mean, e->mu_m2, e->work_L, e->work_y, e->partials, e->lam_partials, e->resid_partials,
                    e->snapW, e->snapV, e->snapTau2, e->snapScal, e->snapR, e->diag_retries, e->nu2c, e->wc, e->sc, e->nu2_nbad,
                    e->gA, e->gC, e->growc, e->ggrid_f, e->ggrid_c, e->Wold, e->Vold, e->gmeanW, e->gmeanV, e->ep_mu, e->ep_sig,
                    e->gass_nbad, e->lgy};
    for (void* p : ptrs) if (p) cudaFree(p);
    {
        void* i8p[] = {e->i8.planes, e->i8.colmax, e->i8.expo, e->i8.D, e->i8.bpart, e->cntT, e->cnt_rowsum, e->cnt_colsum, e->guard_n, e->guard_flags, e->Scol};
        for (void* q : i8p) if (q) cudaFree(q);
    }
    for (int i = 0; i < EVAL_SLOTS; ++i) eval_free(e->eval[i]);
    for (auto& kv : e->inject) if (kv.second.p) cudaFree(kv.second.p);
    for (auto& kv : e->diagbuf) if (kv.second.p) cudaFree(kv.second.p);
    if (e->pinned_scal) cudaFreeHost(e->pinned_scal);
    if (e->ev_snap) cudaEventDestroy(e->ev_snap);
    if (e->ev_copied) cudaEventDestroy(e->ev_copied);
    for (int i = 0; i <= PH_COUNT; ++i) if (e->ph_ev[i]) cudaEventDestroy(e->ph_ev[i]);
    for (int i = 0; i < 6; ++i) if (e->i8_ev[i / 3][i % 3]) cudaEventDestroy(e->i8_ev[i / 3][i % 3]);
    for (int i = 0; i < 2; ++i) {
        if (e->staging[i]) cudaFree(e->staging[i]);
        if (e->hstage[i]) cudaFreeHost(e->hstage[i]);
        if (e->ev_h2d[i]) cudaEventDestroy(e->ev_h2d[i]);
        if (e->ev_k0[i]) cudaEventDestroy(e->ev_k0[i]);
        if (e->side[i]) cudaStreamDestroy(e->side[i]);
        if (e->ev_join[i]) cudaEventDestroy(e->ev_join[i]);
    }
    if (e->ev_fork) cudaEventDestroy(e->ev_fork);
    if (e->stream) cudaStreamDestroy(e->stream);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    delete e;
}

int btf_delta_rows(const btf_engine* e) { return e ? e->RD : 0; }
int btf_set_sample_mask(btf_engine* e, int32_t mask) {
    if (!e) return set_err(BTF_EINVAL, "null engine");
    if (mask != e->cfg.sample_mask) {
        cudaStreamSynchronize(e->stream);
        if (e->graph_exec) { cudaGraphExecDestroy(e->graph_exec); e->graph_exec = nullptr; }
        e->cfg.sample_mask = mask;
        e->resid_valid = false;
    }
    return BTF_OK;
}
int64_t btf_kernel_launches(const btf_engine* e) { return e ? e->launches : 0; }

// ------------------------------------------------------------------ data
static int upload_rows(btf_engine* e, const double* src, size_t row_elems, int row0, int rows, double* staging) {
    // src is a host pointer to the first of `rows` rows of row_elems doubles
    CK(cudaMemcpyAsync(staging, src + (size_t)row0 * row_elems, (size_t)rows * row_elems * sizeof(double),
                       cudaMemcpyHostToDevice, e->stream));
    return BTF_OK;
}

// Is `p` ordinary host memory (neither page-locked by CUDA nor device / managed memory)?
static bool is_pageable_host_ptr(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return at.type == cudaMemoryTypeUnregistered;
}

// memcpy with several host threads: one thread copies ~10 GB/s, which is also all a cudaMemcpy from pageable memory
// reaches (it goes through the driver's own single-threaded bounce buffer)
static void parallel_memcpy(void* dst, const void* src, size_t bytes, int threads) {
    // threads: the cores this process may run on, at most 16 (C2 on the bench box: 8 threads 36.6 GB/s, 16 threads 40.6 GB/s,
    // pinned source 55 GB/s), and at least 4 MB each
    unsigned hw = std::thread::hardware_concurrency();
    cpu_set_t cs;
    if (sched_getaffinity(0, sizeof(cs), &cs) == 0 && CPU_COUNT(&cs) > 0) hw = (unsigned)CPU_COUNT(&cs);
    int nt = (int)std::min<size_t>(std::min<unsigned>(hw ? hw : 4, 16), std::max<size_t>(1, bytes >> 22));
    if (threads > 0) nt = threads;
    if (nt <= 1) { memcpy(dst, src, bytes); return; }
    std::vector<std::thread> th;
    const size_t per = ((bytes + nt - 1) / nt + 4095) & ~(size_t)4095;
    for (int i = 0; i < nt; ++i) {
        const size_t o = (size_t)i * per;
        if (o >= bytes) break;
        const size_t n = std::min(per, bytes - o);
        th.emplace_back([=]() { memcpy((char*)dst + o, (const char*)src + o, n); });
    }
    for (auto& t : th) t.join();
}

// Pre-reduce `nrows` local rows starting at local row `row0` (streaming form for shards that
// are generated or loaded piecewise; reset != 0 clears the running totals first).
static int set_data_compact(btf_engine* e, const double* Y, int32_t row0, int32_t nrows, int32_t nreps, int32_t reset);

int btf_set_data_gaussian_rows(btf_engine* e, const double* Y, int32_t row0, int32_t nrows, int32_t nreps,
                               int32_t reset) {
    if (!e || !Y || nreps < 1 || nreps > 255) return set_err(BTF_EINVAL, "bad arguments (1 <= nreps <= 255)");
    if (e->cfg.likelihood == BTF_CGAUSSIAN)
        return set_err(BTF_ESTATE, "a constrained Gaussian engine takes its data whole: use btf_set_data_gaussian");
    if (e->cfg.likelihood != BTF_GAUSSIAN) return set_err(BTF_ESTATE, "engine is not Gaussian");
    return set_data_compact(e, Y, row0, nrows, nreps, reset);
}

// the compact form of replicated observations (K0): # observed replicates (u8) and their sum per cell
static int set_data_compact(btf_engine* e, const double* Y, int32_t row0, int32_t nrows, int32_t nreps, int32_t reset) {
    if (row0 < 0 || nrows < 0 || row0 + nrows > e->nloc) return set_err(BTF_EINVAL, "row range outside the shard");
    if (!reset && e->shard && e->data_reduced)
        return set_err(BTF_ESTATE, "a sharded engine that has already run holds all-reduced totals: restart the upload with reset = 1");
    CK(cudaSetDevice(e->cfg.device));
    free_graph(e);
    e->nreps = nreps;
    const size_t row_elems = (size_t)e->P * nreps;
    if (reset) CK(cudaMemsetAsync(&e->scal->ss_total, 0, 2 * sizeof(double), e->stream));   // ss_total, n_obs
    const bool on_dev = is_device_ptr(Y);
    // Ordinary numpy memory: a cudaMemcpy from it runs at ~10 GB/s, and page-locking it in place for one upload costs
    // more than that copy (cudaHostRegister ~5-8 GB/s; tools/upload_timing.py) - so it is copied by several host threads
    // into two pinned bounce buffers, from which the asynchronous copies run at link speed.  BTF_UPLOAD_BOUNCE=0: plain copy.
    const bool bounce = !on_dev && is_pageable_host_ptr(Y) && e->env.upload_bounce;
    int chunk = nrows;
    if (!on_dev) {
        // two staging buffers: the copy of piece i + 1 (copy stream) runs under the pre-reduction of piece i
        const size_t piece_bytes = bounce ? ((size_t)64 << 20) : ((size_t)256 << 20);
        chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)std::max(nrows, 1), piece_bytes / (row_elems * 8)));
        const size_t need = (size_t)chunk * row_elems * sizeof(double);
        if (bounce && need > e->hstage_bytes) {
            for (int b = 0; b < 2; ++b) { if (e->hstage[b]) cudaFreeHost(e->hstage[b]); e->hstage[b] = nullptr; }
            e->hstage_bytes = 0;
            for (int b = 0; b < 2; ++b) CK(cudaMallocHost((void**)&e->hstage[b], need));
            e->hstage_bytes = need;
        }
        if (need > e->staging_bytes) {
            for (int b = 0; b < 2; ++b) { if (e->staging[b]) cudaFree(e->staging[b]); e->staging[b] = nullptr; }
            e->staging_bytes = 0;
            for (int b = 0; b < 2; ++b) CK(cudaMalloc((void**)&e->staging[b], need));
            e->staging_bytes = need;
        }
        for (int b = 0; b < 2; ++b) {
            if (!e->ev_h2d[b]) CK(cudaEventCreateWithFlags(&e->ev_h2d[b], cudaEventDisableTiming));
            if (!e->ev_k0[b]) CK(cudaEventCreateWithFlags(&e->ev_k0[b], cudaEventDisableTiming));
        }
        CK(cudaStreamSynchronize(e->stream));
    }
    int piece = 0;
    for (int r0 = 0; r0 < nrows; r0 += chunk, ++piece) {
        int rows = std::min(chunk, nrows - r0);
        const int b = piece & 1;
        const double* src = on_dev ? Y + (size_t)r0 * row_elems : e->staging[b];
        if (!on_dev) {
            const double* hsrc = Y + (size_t)r0 * row_elems;
            if (bounce) {
                if (piece >= 2) CK(cudaEventSynchronize(e->ev_h2d[b]));                    // the bounce buffer's previous copy has left it
                parallel_memcpy(e->hstage[b], hsrc, (size_t)rows * row_elems * sizeof(double), e->env.upload_threads);
                hsrc = e->hstage[b];
            }
            if (piece >= 2) CK(cudaStreamWaitEvent(e->copy_stream, e->ev_k0[b], 0));       // the buffer's previous pre-reduction is done
            CK(cudaMemcpyAsync(e->staging[b], hsrc, (size_t)rows * row_elems * sizeof(double),
                               cudaMemcpyHostToDevice, e->copy_stream));
            CK(cudaEventRecord(e->ev_h2d[b], e->copy_stream));
            CK(cudaStreamWaitEvent(e->stream, e->ev_h2d[b], 0));
        }
        int nb = 0;
        const size_t o = (size_t)(row0 + r0) * e->Ppad;
        launch_prereduce_gaussian(src, rows, e->P, nreps, e->cnt + o, e->S + o, e->Ppad, e->partials, &nb, e->stream);
        launch_reduce_add(e->partials, nb, 2, &e->scal->ss_total, e->stream);
        launch_reduce_add(e->partials + 1, nb, 2, &e->scal->n_obs, e->stream);
        if (!on_dev) CK(cudaEventRecord(e->ev_k0[b], e->stream));
        e->launches += 3;
    }
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaGetLastError());
    e->has_data = true; e->data_reduced = false; e->resid_valid = false; e->i8_decided = false;
    e->nu2_dirty = true;
    return BTF_OK;
}

static int copy_pitched(btf_engine* e, double* dev, double* host, bool to_host);

// The constrained Gaussian model: observations [Nloc, M, T, nreps] in the compact form, plus the within-cell sum of
// squared deviations ss = sum_r (y_r - ybar)^2 per cell, so that the GASS steps evaluate the log-likelihood in its
// centred form.  Every observed value must be finite.
static int set_data_cgaussian(btf_engine* e, const double* Y, int32_t nreps) {
    if (!Y || nreps < 1 || nreps > 255) return set_err(BTF_EINVAL, "bad arguments (1 <= nreps <= 255)");
    CK(cudaSetDevice(e->cfg.device));
    const size_t cells = (size_t)e->nloc * e->P, total = cells * nreps;
    std::vector<double> hcopy;
    const double* hy = Y;
    if (is_device_ptr(Y)) {
        hcopy.resize(total);
        CK(cudaMemcpy(hcopy.data(), Y, total * sizeof(double), cudaMemcpyDeviceToHost));
        hy = hcopy.data();
    }
    unsigned long long nbad = 0;
    std::vector<double> ss(cells, 0.0);
    for (size_t c = 0; c < cells; ++c) {
        const double* y = hy + c * nreps;
        int n = 0;
        double sum = 0.0;
        for (int r = 0; r < nreps; ++r) {
            if (std::isnan(y[r])) continue;
            if (!std::isfinite(y[r])) { ++nbad; continue; }
            ++n; sum += y[r];
        }
        if (n < 2) continue;
        const double ybar = sum / n;
        double q = 0.0;
        for (int r = 0; r < nreps; ++r)
            if (std::isfinite(y[r])) q += (y[r] - ybar) * (y[r] - ybar);
        ss[c] = q;
    }
    if (nbad) return set_err(BTF_EINVAL, "%llu observed value(s) are not finite", nbad);
    if (!e->lgy) CK(dev_alloc(&e->lgy, (size_t)e->nloc_pad * e->Ppad));
    CK(cudaStreamSynchronize(e->stream));
    { int rc = copy_pitched(e, e->lgy, ss.data(), false); if (rc) return rc; }
    return set_data_compact(e, Y, 0, e->nloc, nreps, 1);
}

int btf_set_data_gaussian(btf_engine* e, const double* Y, int32_t nreps) {
    if (!e) return set_err(BTF_EINVAL, "null engine");
    if (e->cfg.likelihood == BTF_CGAUSSIAN) return set_data_cgaussian(e, Y, nreps);
    return btf_set_data_gaussian_rows(e, Y, 0, e->nloc, nreps, 1);
}

// Poisson counts [Nloc, M, T, nreps] in the compact form of the Gaussian data, plus sum_r lgamma(y_r + 1) per cell
// (scipy's logpmf keeps it, and a cell whose rate is negative drops out of the log-likelihood together with it).
// Every observed value must be a non-negative integer.
int btf_set_data_poisson(btf_engine* e, const double* Y, int32_t nreps) {
    if (!e || !Y || nreps < 1 || nreps > 255) return set_err(BTF_EINVAL, "bad arguments (1 <= nreps <= 255)");
    if (e->cfg.likelihood != BTF_POISSON) return set_err(BTF_ESTATE, "engine is not Poisson");
    CK(cudaSetDevice(e->cfg.device));
    const size_t cells = (size_t)e->nloc * e->P, total = cells * nreps;
    std::vector<double> hcopy;
    const double* hy = Y;
    if (is_device_ptr(Y)) {
        hcopy.resize(total);
        CK(cudaMemcpy(hcopy.data(), Y, total * sizeof(double), cudaMemcpyDeviceToHost));
        hy = hcopy.data();
    }
    unsigned long long nbad = 0;
    std::vector<double> lg(cells, 0.0);
    for (size_t c = 0; c < cells; ++c)
        for (int r = 0; r < nreps; ++r) {
            const double y = hy[c * nreps + r];
            if (std::isnan(y)) continue;
            if (!(y >= 0.0 && std::isfinite(y) && y == std::floor(y))) ++nbad;
            else lg[c] += std::lgamma(y + 1.0);
        }
    if (nbad) return set_err(BTF_EINVAL, "%llu observed value(s) are not non-negative integer counts", nbad);
    if (!e->lgy) CK(dev_alloc(&e->lgy, (size_t)e->nloc_pad * e->Ppad));
    CK(cudaStreamSynchronize(e->stream));
    { int rc = copy_pitched(e, e->lgy, lg.data(), false); if (rc) return rc; }
    return set_data_compact(e, Y, 0, e->nloc, nreps, 1);
}

// The constrained Binomial model: every observed cell (y and n not NaN) must hold non-negative integers with y <= n.
// The log binomial coefficient lgamma(n + 1) - (lgamma(y + 1) + lgamma(n - y + 1)) of each observed cell goes to `lc`:
// scipy's logpmf keeps it, and a cell whose probability leaves [0, 1] drops out of the log-likelihood together with it.
static int binomial_coefficients(btf_engine* e, const double* Ys, const double* Nt, std::vector<double>* lc) {
    const size_t cells = (size_t)e->nloc * e->P;
    std::vector<double> hy, hn;
    if (is_device_ptr(Ys)) { hy.resize(cells); CK(cudaMemcpy(hy.data(), Ys, cells * sizeof(double), cudaMemcpyDeviceToHost)); Ys = hy.data(); }
    if (is_device_ptr(Nt)) { hn.resize(cells); CK(cudaMemcpy(hn.data(), Nt, cells * sizeof(double), cudaMemcpyDeviceToHost)); Nt = hn.data(); }
    lc->assign(cells, 0.0);
    unsigned long long nbad = 0;
    for (size_t c = 0; c < cells; ++c) {
        const double y = Ys[c], n = Nt[c];
        if (std::isnan(y) || std::isnan(n)) continue;
        const bool count_y = y >= 0.0 && std::isfinite(y) && y == std::floor(y);
        const bool count_n = n >= 0.0 && std::isfinite(n) && n == std::floor(n);
        if (!(count_y && count_n && y <= n)) { ++nbad; continue; }
        (*lc)[c] = std::lgamma(n + 1.0) - (std::lgamma(y + 1.0) + std::lgamma(n - y + 1.0));
    }
    if (nbad)
        return set_err(BTF_EINVAL, "%llu observed cell(s) do not hold non-negative integer counts y <= n (successes, trials)", nbad);
    return BTF_OK;
}

int btf_set_data_binomial(btf_engine* e, const double* Ys, const double* Nt) {
    if (!e || !Ys || !Nt) return set_err(BTF_EINVAL, "null argument");
    if (e->cfg.likelihood != BTF_BINOMIAL && e->cfg.likelihood != BTF_CBINOMIAL) return set_err(BTF_ESTATE, "engine is not Binomial");
    CK(cudaSetDevice(e->cfg.device));
    std::vector<double> lc;
    if (e->cfg.likelihood == BTF_CBINOMIAL) {
        int rc = binomial_coefficients(e, Ys, Nt, &lc);
        if (rc) return rc;
        if (!e->lgy) CK(dev_alloc(&e->lgy, (size_t)e->nloc_pad * e->Ppad));
    }
    free_graph(e);
    const size_t row_elems = (size_t)e->P;
    const bool on_dev = is_device_ptr(Ys) && is_device_ptr(Nt);
    double *sy = nullptr, *sn = nullptr;
    int chunk = e->nloc;
    if (!on_dev) {
        chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)std::max(e->nloc, 1), ((size_t)128 << 20) / (row_elems * 8)));
        const size_t need = (size_t)chunk * row_elems * sizeof(double);
        if (need > e->staging_bytes) {                 // engine-lifetime staging buffers (freed by btf_destroy)
            for (int b = 0; b < 2; ++b) { if (e->staging[b]) cudaFree(e->staging[b]); e->staging[b] = nullptr; }
            e->staging_bytes = 0;
            for (int b = 0; b < 2; ++b) CK(cudaMalloc((void**)&e->staging[b], need));
            e->staging_bytes = need;
        }
        sy = e->staging[0]; sn = e->staging[1];
    }
    for (int r0 = 0; r0 < e->nloc; r0 += chunk) {
        int rows = std::min(chunk, e->nloc - r0);
        const double *py = Ys + (size_t)r0 * row_elems, *pn = Nt + (size_t)r0 * row_elems;
        if (!on_dev) {
            int rc = upload_rows(e, Ys, row_elems, r0, rows, sy); if (rc) return rc;
            rc = upload_rows(e, Nt, row_elems, r0, rows, sn); if (rc) return rc;
            py = sy; pn = sn;
        }
        launch_prereduce_binomial(py, pn, rows, e->P, e->cnt + (size_t)r0 * e->Ppad, e->S + (size_t)r0 * e->Ppad,
                                  e->ntr + (size_t)r0 * e->Ppad, e->Ppad, e->stream);
        e->launches += 1;
    }
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaGetLastError());
    if (!lc.empty()) { int rc = copy_pitched(e, e->lgy, lc.data(), false); if (rc) return rc; }
    e->has_data = true; e->data_reduced = true; e->i8_decided = false;
    return BTF_OK;
}

int btf_set_data_negbin(btf_engine* e, const double* Y, int32_t nreps) {
    if (!e || !Y || nreps < 1) return set_err(BTF_EINVAL, "bad arguments");
    if (e->cfg.likelihood != BTF_NEGBINOMIAL) return set_err(BTF_ESTATE, "engine is not NegativeBinomial");
    if (e->cfg.world_size > 1) return set_err(BTF_EINVAL, "negative-binomial path is single-GPU");
    CK(cudaSetDevice(e->cfg.device));
    free_graph(e);
    e->nreps = nreps;
    const size_t total = (size_t)e->nloc * e->P * nreps;
    if (e->Yraw) { CK(cudaFree(e->Yraw)); e->Yraw = nullptr; }
    CK(cudaMalloc((void**)&e->Yraw, total * sizeof(double)));
    CK(cudaMemcpy(e->Yraw, Y, total * sizeof(double), is_device_ptr(Y) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice));
    CK(cudaStreamSynchronize(cudaStreamLegacy));
    if (e->nb_work) { CK(cudaFree(e->nb_work)); e->nb_work = nullptr; }
    const size_t rsize = (size_t)e->Rn * e->Rm * e->Rt;
    CK(dev_alloc(&e->nb_work, 8 * rsize + 64));
    // count histograms for the fused MH chain (integer counts of moderate range only)
    if (e->nb_hist) { CK(cudaFree(e->nb_hist)); e->nb_hist = nullptr; }
    e->nb_hist_stride = 0;
    {
        unsigned long long* scan = nullptr;
        CK(dev_alloc(&scan, 2));
        launch_nb_scan(e->Yraw, (long long)total, scan, e->stream);
        unsigned long long h[2];
        CK(cudaMemcpyAsync(h, scan, sizeof(h), cudaMemcpyDeviceToHost, e->stream));
        CK(cudaStreamSynchronize(e->stream));
        CK(cudaFree(scan));
        const size_t vstride = (size_t)h[0] + 1;
        if (!h[1] && vstride * rsize <= ((size_t)1 << 24) && e->env.nb_hist) {
            CK(dev_alloc(&e->nb_hist, vstride * rsize));
            e->nb_hist_stride = (int)vstride;
            NbArgs nb;
            memset(&nb, 0, sizeof(nb));
            nb.Yraw = e->Yraw; nb.nloc = e->nloc; nb.P = e->P; nb.R = nreps; nb.M = e->M; nb.T = e->T; nb.K = e->K;
            nb.row_begin = e->cfg.row_begin; nb.Rn = e->Rn; nb.Rm = e->Rm; nb.Rt = e->Rt; nb.hist = e->nb_hist;
            launch_nb_hist(nb, (int)vstride, e->stream);
            CK(cudaStreamSynchronize(e->stream));
            e->launches += 2;
        }
    }
    e->has_data = true; e->data_reduced = true; e->i8_decided = false;
    return BTF_OK;
}

// Known per-cell noise variances (the reference's heteroskedastic Gaussian branch: nu2 an [N, M, T] array).
// First use: the statistics plans for f64 weights (their split buffers may be larger) and the cell buffers.
static int ensure_nu2_buffers(btf_engine* e) {
    if (e->cfg.likelihood == BTF_CGAUSSIAN) {
        // the GASS steps read the variances themselves; wc / sc belong to the EP approximation
        if (!e->nu2c) { CK(dev_alloc(&e->nu2_nbad, 1)); CK(dev_alloc(&e->nu2c, (size_t)e->nloc_pad * e->Ppad)); }
        return BTF_OK;
    }
    if (e->wc) return BTF_OK;
    if (!plan_stats(&e->plan_row_w, e->K, false, true, e->nloc_pad, e->Ppad, e->nloc, e->cfg.stats_splits_row, e->sm_count) ||
        !plan_stats(&e->plan_col_w, e->K, true, true, e->Ppad, e->nloc_pad, e->P, e->cfg.stats_splits_col, e->sm_count))
        return set_err(BTF_EINVAL, "no statistics plan for per-cell weights at K=%d", e->K);
    auto grow = [](double** buf, const StatsPlan& have, const StatsPlan& want) -> cudaError_t {
        const size_t nh = have.nsplit * have.out_elems_per_split, nw = want.nsplit * want.out_elems_per_split;
        if (nw <= nh) return cudaSuccess;
        cudaFree(*buf); *buf = nullptr;
        return dev_alloc(buf, nw);
    };
    CK(grow(&e->row_stats, e->plan_row, e->plan_row_w));
    CK(grow(&e->col_stats, e->plan_col, e->plan_col_w));
    const size_t cells = (size_t)e->nloc_pad * e->Ppad;
    CK(dev_alloc(&e->nu2_nbad, 1));
    CK(dev_alloc(&e->nu2c, cells));
    CK(dev_alloc(&e->sc, cells));
    CK(dev_alloc(&e->wc, cells));
    return BTF_OK;
}

// Weights from `rows` rows of variances at pitch lds (starting at local row row0); keep != 0: store the variances too.
// A constrained Gaussian engine forms no weights (its wc / sc hold the EP approximation's): it only checks and keeps.
static void enqueue_nu2_weights(btf_engine* e, const double* nu2, long long lds, int row0, int rows, bool keep) {
    const size_t o = (size_t)row0 * e->Ppad;
    const bool weights = e->cfg.likelihood == BTF_GAUSSIAN;
    launch_nu2_weights(nu2, lds, rows, e->P, e->cnt + o, e->S + o, e->Ppad, keep ? e->nu2c + o : nullptr,
                       weights ? e->wc + o : nullptr, weights ? e->sc + o : nullptr, e->nu2_nbad, e->stream);
    e->launches++;
}

static int read_nu2_bad(btf_engine* e) {
    CK(cudaMemcpyAsync(e->pinned_scal, e->nu2_nbad, sizeof(unsigned long long), cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaGetLastError());
    memcpy(&e->nu2_bad, e->pinned_scal, sizeof(unsigned long long));
    return BTF_OK;
}

static int nu2_bad_error(btf_engine* e) {
    return set_err(BTF_EINVAL, "%llu observed cell(s) have a noise variance that is NaN or <= 0 (+inf marks a cell as missing)",
                   e->nu2_bad);
}

int btf_set_nu2_cells(btf_engine* e, const double* nu2) {
    if (!e) return set_err(BTF_EINVAL, "null engine");
    if (e->cfg.likelihood != BTF_GAUSSIAN && e->cfg.likelihood != BTF_CGAUSSIAN)
        return set_err(BTF_ESTATE, "per-cell noise variances need a Gaussian or constrained Gaussian engine");
    if (e->cfg.world_size > 1) return set_err(BTF_EINVAL, "per-cell noise variances are single-GPU");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    // the sweep changes route (and the integer statistics path is decided again): drop the captured graph
    free_graph(e);
    e->i8_decided = false;
    e->resid_valid = false;
    e->nu2_cells = false;         // scalar mode until the variances are accepted
    if (!nu2) return BTF_OK;
    { int rc = ensure_nu2_buffers(e); if (rc) return rc; }
    CK(cudaMemsetAsync(e->nu2_nbad, 0, sizeof(unsigned long long), e->stream));
    const size_t row_elems = (size_t)e->P;
    if (is_device_ptr(nu2)) {
        enqueue_nu2_weights(e, nu2, e->P, 0, e->nloc, true);
    } else {
        const int chunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)std::max(e->nloc, 1), ((size_t)128 << 20) / (row_elems * 8)));
        const size_t need = (size_t)chunk * row_elems * sizeof(double);
        if (need > e->staging_bytes) {                 // engine-lifetime staging buffers (freed by btf_destroy)
            for (int b = 0; b < 2; ++b) { if (e->staging[b]) cudaFree(e->staging[b]); e->staging[b] = nullptr; }
            e->staging_bytes = 0;
            for (int b = 0; b < 2; ++b) CK(cudaMalloc((void**)&e->staging[b], need));
            e->staging_bytes = need;
        }
        int piece = 0;
        for (int r0 = 0; r0 < e->nloc; r0 += chunk, ++piece) {
            const int rows = std::min(chunk, e->nloc - r0);
            double* buf = e->staging[piece & 1];
            int rc = upload_rows(e, nu2, row_elems, r0, rows, buf); if (rc) return rc;
            enqueue_nu2_weights(e, buf, e->P, r0, rows, true);
        }
    }
    { int rc = read_nu2_bad(e); if (rc) return rc; }
    e->nu2_dirty = false;
    if (e->nu2_bad) return nu2_bad_error(e);
    e->nu2_cells = true;
    return BTF_OK;
}

// pitched [nloc][P] <-> dense copies for omega / Ntrials / the EP approximation
static int copy_pitched(btf_engine* e, double* dev, double* host, bool to_host) {
    if (to_host)
        CK(cudaMemcpy2D(host, (size_t)e->P * 8, dev, (size_t)e->Ppad * 8, (size_t)e->P * 8, e->nloc, cudaMemcpyDeviceToHost));
    else
        CK(cudaMemcpy2D(dev, (size_t)e->Ppad * 8, host, (size_t)e->P * 8, (size_t)e->P * 8, e->nloc, cudaMemcpyHostToDevice));
    return BTF_OK;
}

// ------------------------------------------------------------------ constrained Poisson, Binomial and Gaussian models (GASS steps)
static cudaError_t upload_copy(double** dst, const double* src, size_t n) {
    if (*dst) { cudaFree(*dst); *dst = nullptr; }
    cudaError_t ce = dev_alloc(dst, std::max<size_t>(n, 1), false);
    if (ce == cudaSuccess && n) ce = h2d(*dst, src, n * sizeof(double));
    return ce;
}

int btf_set_gass(btf_engine* e, const double* A, const double* C, int32_t J, const double* rowcons, int32_t nrowcons,
                 const double* grid_fine, int32_t ngrid_fine, const double* grid_coarse, int32_t ngrid) {
    if (!e) return set_err(BTF_EINVAL, "null engine");
    if (!gass_likelihood(e->cfg.likelihood)) return set_err(BTF_ESTATE, "GASS steps need a constrained Poisson, Binomial or Gaussian engine");
    if (J < 0 || nrowcons < 0 || (J > 0 && (!A || !C)) || (nrowcons > 0 && !rowcons))
        return set_err(BTF_EINVAL, "constraints: J >= 0 rows of A [J, T] and C [J], nrowcons >= 0 rows of [K + 1]");
    if (!grid_fine || !grid_coarse || ngrid < 1 || ngrid > ngrid_fine || ngrid_fine > 65535)
        return set_err(BTF_EINVAL, "grids: 1 <= ngrid <= ngrid_fine <= 65535 (got ngrid = %d, ngrid_fine = %d)", ngrid, ngrid_fine);
    size_t nonfinite = 0;
    for (size_t i = 0; i < (size_t)J * e->T; ++i) nonfinite += !std::isfinite(A[i]);
    for (int i = 0; i < J; ++i) nonfinite += !std::isfinite(C[i]);
    for (size_t i = 0; i < (size_t)nrowcons * (e->K + 1); ++i) nonfinite += !std::isfinite(rowcons[i]);
    if (nonfinite) return set_err(BTF_EINVAL, "%zu constraint coefficient(s) are not finite", nonfinite);
    for (int i = 0; i < ngrid_fine; ++i)
        if (!std::isfinite(grid_fine[i]) || (i && !(grid_fine[i] >= grid_fine[i - 1]))) return set_err(BTF_EINVAL, "the fine grid must be finite and ascending");
    for (int i = 0; i < ngrid; ++i)
        if (!std::isfinite(grid_coarse[i])) return set_err(BTF_EINVAL, "the coarse grid must be finite");
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, e->cfg.device));
    const size_t smem = gass_smem_bytes(e->T * e->K, ngrid_fine, ngrid) + 1024;
    if (smem > (size_t)prop.sharedMemPerBlockOptin)
        return set_err(BTF_EINVAL, "GASS steps at T K = %d with %d grid points need %zu bytes of shared memory per block, the device offers %zu",
                       e->T * e->K, ngrid_fine, smem, (size_t)prop.sharedMemPerBlockOptin);
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    free_graph(e);
    e->gass_set = false;
    CK(upload_copy(&e->gA, A, (size_t)J * e->T));
    CK(upload_copy(&e->gC, C, (size_t)J));
    CK(upload_copy(&e->growc, rowcons, (size_t)nrowcons * (e->K + 1)));
    CK(upload_copy(&e->ggrid_f, grid_fine, (size_t)ngrid_fine));
    CK(upload_copy(&e->ggrid_c, grid_coarse, (size_t)ngrid));
    if (!e->Wold) {
        CK(dev_alloc(&e->Wold, (size_t)e->N * e->K));
        CK(dev_alloc(&e->Vold, (size_t)e->P * e->K));
        CK(dev_alloc(&e->gmeanW, (size_t)e->N * e->K));
        CK(dev_alloc(&e->gmeanV, (size_t)e->P * e->K));
        CK(dev_alloc(&e->gass_nbad, 2));
    }
    e->gJ = J; e->gnrc = nrowcons; e->gnfine = ngrid_fine; e->gngrid = ngrid;
    e->gass_set = true;
    return BTF_OK;
}

// EP approximation N(mu, sigma^2) per cell (host memory, [Nloc, M, T]); NULL: none
int btf_set_ep(btf_engine* e, const double* mu, const double* sigma) {
    if (!e) return set_err(BTF_EINVAL, "null engine");
    if (!gass_likelihood(e->cfg.likelihood)) return set_err(BTF_ESTATE, "an EP approximation needs a constrained Poisson, Binomial or Gaussian engine");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    if (!mu || !sigma) {
        if (e->ep_on) free_graph(e);
        e->ep_on = false;
        return BTF_OK;
    }
    const size_t n = (size_t)e->nloc * e->P;
    size_t nbad = 0;
    for (size_t i = 0; i < n; ++i) nbad += !(std::isfinite(mu[i]) && std::isfinite(sigma[i]) && sigma[i] > 0.0);
    if (nbad) return set_err(BTF_EINVAL, "%zu cell(s) of the EP approximation have a mean that is not finite or a scale that is not finite and > 0", nbad);
    free_graph(e);
    e->ep_on = false;
    const size_t cells = (size_t)e->nloc_pad * e->Ppad;
    if (!e->ep_mu) {
        CK(dev_alloc(&e->ep_mu, cells)); CK(dev_alloc(&e->ep_sig, cells));
        CK(dev_alloc(&e->wc, cells)); CK(dev_alloc(&e->sc, cells));
    }
    // the statistics' weights as numpy forms them: w = 1 / sigma**2, s = mu * w
    std::vector<double> w(n), s(n);
    for (size_t i = 0; i < n; ++i) { w[i] = 1.0 / (sigma[i] * sigma[i]); s[i] = mu[i] * w[i]; }
    { int rc = copy_pitched(e, e->ep_mu, const_cast<double*>(mu), false); if (rc) return rc; }
    { int rc = copy_pitched(e, e->ep_sig, const_cast<double*>(sigma), false); if (rc) return rc; }
    { int rc = copy_pitched(e, e->wc, w.data(), false); if (rc) return rc; }
    { int rc = copy_pitched(e, e->sc, s.data(), false); if (rc) return rc; }
    CK(cudaStreamSynchronize(cudaStreamLegacy));
    e->ep_on = true;
    return BTF_OK;
}

// ------------------------------------------------------------------ state
struct StateRef { double* p; size_t n; bool scalar_field; };

static bool state_ref(btf_engine* e, const std::string& nm, StateRef* r) {
    const size_t tn = (size_t)e->M * e->RD;
    r->scalar_field = false;
    if (nm == "W") { r->p = e->W; r->n = (size_t)e->N * e->K; return true; }
    if (nm == "V") { r->p = e->V; r->n = (size_t)e->P * e->K; return true; }
    if (nm == "Tau2") { r->p = e->Tau2; r->n = tn; return true; }
    if (nm == "Tau2_a") { r->p = e->Tau2_a; r->n = tn; return true; }
    if (nm == "Tau2_b") { r->p = e->Tau2_b; r->n = tn; return true; }
    if (nm == "Tau2_c") { r->p = e->Tau2_c; r->n = tn; return true; }
    if (nm == "R" && e->Rdisp) { r->p = e->Rdisp; r->n = (size_t)e->Rn * e->Rm * e->Rt; return true; }
    r->scalar_field = true; r->n = 1;
    if (nm == "nu2") { r->p = &e->scal->nu2; return true; }
    if (nm == "sigma2") { r->p = &e->scal->sigma2; return true; }
    if (nm == "lam2") { r->p = &e->scal->lam2; return true; }
    if (nm == "lam2_a") { r->p = &e->scal->lam2_a; return true; }
    if (nm == "resid") { r->p = &e->scal->resid; return true; }
    if (nm == "ss_total") { r->p = &e->scal->ss_total; return true; }
    if (nm == "n_obs") { r->p = &e->scal->n_obs; return true; }
    return false;
}

int btf_set_state(btf_engine* e, const char* name, const double* host, size_t n) {
    if (!e || !name || !host) return set_err(BTF_EINVAL, "null argument");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    std::string nm(name);
    if (nm == "sweep") {
        // the sweep counter is a Philox counter word: restoring it (with the seed and the state arrays) resumes a chain
        // on exactly the random stream it would have continued with
        if (n != 1 || !(host[0] >= 0.0) || host[0] > 9007199254740992.0) return set_err(BTF_EINVAL, "sweep: one non-negative integer below 2^53");
        const unsigned long long v = (unsigned long long)host[0];
        CK(h2d(&e->scal->sweep, &v, sizeof(v)));
        e->resid_valid = false;
        return BTF_OK;
    }
    if (nm == "Ntrials" && e->cfg.likelihood == BTF_CBINOMIAL)
        return set_err(BTF_ESTATE, "the trials of a constrained Binomial engine come with its data: use btf_set_data_binomial");
    if ((nm == "omega" && e->omega) || (nm == "Ntrials" && e->ntr)) {
        if (n != (size_t)e->nloc * e->P) return set_err(BTF_EINVAL, "%s: expected %zu values", name, (size_t)e->nloc * e->P);
        return copy_pitched(e, nm == "omega" ? e->omega : e->ntr, const_cast<double*>(host), false);
    }
    StateRef r;
    if (!state_ref(e, nm, &r)) return set_err(BTF_EINVAL, "unknown state '%s'", name);
    if (n != r.n) return set_err(BTF_EINVAL, "%s: expected %zu values, got %zu", name, r.n, n);
    CK(h2d(r.p, host, n * sizeof(double)));
    if (nm == "W" || nm == "V") e->resid_valid = false;
    // restoring a checkpoint: the residual sum that belongs to the (W, V) just set, so that the next nu2 step uses the same
    // number the interrupted chain would have used (set it AFTER W and V)
    if (nm == "resid" && e->cfg.likelihood == BTF_GAUSSIAN && e->has_data && !e->nu2_cells) e->resid_valid = true;
    return BTF_OK;
}

int btf_get_state(btf_engine* e, const char* name, double* host, size_t n) {
    if (!e || !name || !host) return set_err(BTF_EINVAL, "null argument");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    std::string nm(name);
    if (nm == "sweep") {
        if (n != 1) return set_err(BTF_EINVAL, "sweep: 1 value");
        unsigned long long v = 0;
        CK(cudaMemcpy(&v, &e->scal->sweep, sizeof(v), cudaMemcpyDeviceToHost));
        host[0] = (double)v;
        return BTF_OK;
    }
    if (nm == "Delta") {
        if (n != e->delta.size()) return set_err(BTF_EINVAL, "Delta: expected %zu values", e->delta.size());
        memcpy(host, e->delta.data(), n * sizeof(double));
        return BTF_OK;
    }
    if ((nm == "omega" && e->omega) || (nm == "Ntrials" && e->ntr) || (nm == "kappa" && e->S)) {
        if (n != (size_t)e->nloc * e->P) return set_err(BTF_EINVAL, "%s: expected %zu values", name, (size_t)e->nloc * e->P);
        return copy_pitched(e, nm == "omega" ? e->omega : (nm == "kappa" ? e->S : e->ntr), host, true);
    }
    StateRef r;
    if (!state_ref(e, nm, &r)) return set_err(BTF_EINVAL, "unknown state '%s'", name);
    if (n != r.n) return set_err(BTF_EINVAL, "%s: expected %zu values, got %zu", name, r.n, n);
    CK(cudaMemcpy(host, r.p, n * sizeof(double), cudaMemcpyDeviceToHost));
    return BTF_OK;
}

// ------------------------------------------------------------------ parity hooks
int btf_inject_noise(btf_engine* e, const char* name, const double* host, size_t n) {
    if (!e || !name || !host) return set_err(BTF_EINVAL, "null argument");
    CK(cudaSetDevice(e->cfg.device));
    std::string nm(name);
    size_t want = 0;
    const size_t rsize = (size_t)e->Rn * e->Rm * e->Rt;
    if (nm == "z_W") want = (size_t)e->N * e->K;
    else if (nm == "z_V") want = (size_t)e->P * e->K;
    else if (nm == "g_tau") want = (size_t)e->M * 4 * e->RD;
    else if (nm == "g_lam") want = 2;
    else if (nm == "g_sigma2" || nm == "g_nu2") want = 1;
    else if (nm == "omega") want = (size_t)e->nloc * e->P;
    else if (nm == "z_R" || nm == "u_R") want = (size_t)e->cfg.nmetropolis * rsize;
    else if (nm == "gass_u_W" || nm == "gass_u_V") {
        if (!e->gass_set) return set_err(BTF_ESTATE, "%s: call btf_set_gass first", name);
        want = (size_t)(nm == "gass_u_W" ? e->N : e->M) * (e->gngrid + 2);
    }
    else return set_err(BTF_EINVAL, "unknown noise '%s'", name);
    if (n != want) return set_err(BTF_EINVAL, "%s: expected %zu values, got %zu", name, want, n);
    DevBuf& b = e->inject[nm];
    if (b.p && b.n != n) { cudaFree(b.p); b.p = nullptr; }
    if (!b.p) { CK(cudaMalloc((void**)&b.p, n * sizeof(double))); b.n = n; }
    CK(cudaStreamSynchronize(e->stream));
    CK(h2d(b.p, host, n * sizeof(double)));
    return BTF_OK;
}

static const double* inj(btf_engine* e, const char* nm) {
    auto it = e->inject.find(nm);
    return it == e->inject.end() ? nullptr : it->second.p;
}

static void clear_inject(btf_engine* e) {
    for (auto& kv : e->inject) if (kv.second.p) cudaFree(kv.second.p);
    e->inject.clear();
}

static double* diag_get(btf_engine* e, const char* nm, size_t n) {
    if (!e->diag) return nullptr;
    DevBuf& b = e->diagbuf[nm];
    if (!b.p || b.n != n) {
        if (b.p) cudaFree(b.p);
        b.p = nullptr;
        if (cudaMalloc((void**)&b.p, std::max<size_t>(n, 1) * sizeof(double)) != cudaSuccess) { b.p = nullptr; return nullptr; }
        b.n = n;
    }
    cudaMemsetAsync(b.p, 0, n * sizeof(double), e->stream);
    return b.p;
}

int btf_enable_diag(btf_engine* e, int32_t on) {
    if (!e) return set_err(BTF_EINVAL, "null engine");
    e->diag = on != 0;
    if (!e->diag) {
        for (auto& kv : e->diagbuf) if (kv.second.p) cudaFree(kv.second.p);
        e->diagbuf.clear();
    }
    return BTF_OK;
}

int btf_get_diag(btf_engine* e, const char* name, double* host, size_t n) {
    if (!e || !name || !host) return set_err(BTF_EINVAL, "null argument");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    std::string nm(name);
    if (nm == "nu2_rate" || nm == "lam2_rate" || nm == "info") {
        Scalars h;
        CK(cudaMemcpy(&h, e->scal, sizeof(h), cudaMemcpyDeviceToHost));
        if (nm == "nu2_rate") { if (n != 3) return set_err(BTF_EINVAL, "nu2_rate: 3 values"); host[0] = h.nu2_a_post; host[1] = h.nu2_b_post; host[2] = h.n_obs; }
        else if (nm == "lam2_rate") { if (n != 2) return set_err(BTF_EINVAL, "lam2_rate: 2 values"); host[0] = h.lam2_rate; host[1] = h.lam2_shape; }
        else { if (n != 3) return set_err(BTF_EINVAL, "info: 3 values"); host[0] = h.info_w; host[1] = h.info_v; host[2] = h.retries_v; }
        return BTF_OK;
    }
    if (nm == "row_stats" || nm == "col_stats") {
        // sum of the split partials, in split order
        const StatsPlan& pl = stats_plan(e, nm == "col_stats");
        const double* src = nm == "row_stats" ? e->row_stats : e->col_stats;
        if (n != pl.out_elems_per_split) return set_err(BTF_EINVAL, "%s: expected %zu values", name, pl.out_elems_per_split);
        std::vector<double> tmp(n);
        std::fill(host, host + n, 0.0);
        const int ns = (e->i8_on || (nm == "col_stats" && e->col_collapsed)) ? 1 : pl.nsplit;
        for (int s = 0; s < ns; ++s) {
            CK(cudaMemcpy(tmp.data(), src + (size_t)s * n, n * sizeof(double), cudaMemcpyDeviceToHost));
            for (size_t i = 0; i < n; ++i) host[i] += tmp[i];
        }
        return BTF_OK;
    }
    if (nm == "i8_guard") {
        if (n != 2) return set_err(BTF_EINVAL, "i8_guard: 2 values");
        host[0] = host[1] = 0.0;
        if (e->guard_n) { int h[2]; CK(cudaMemcpy(h, e->guard_n, sizeof(h), cudaMemcpyDeviceToHost)); host[0] = h[0]; host[1] = h[1]; }
        return BTF_OK;
    }
    if (nm == "i8_route") {
        if (n != 2) return set_err(BTF_EINVAL, "i8_route: 2 values");
        host[0] = e->i8_route[0]; host[1] = e->i8_route[1];
        return BTF_OK;
    }
    if (nm == "V_retries") {
        if (n != (size_t)e->Mloc) return set_err(BTF_EINVAL, "V_retries: expected %d values", e->Mloc);
        std::vector<int> tmp(e->Mloc);
        CK(cudaMemcpy(tmp.data(), e->diag_retries, e->Mloc * sizeof(int), cudaMemcpyDeviceToHost));
        for (int i = 0; i < e->Mloc; ++i) host[i] = tmp[i];
        return BTF_OK;
    }
    auto it = e->diagbuf.find(nm);
    if (it == e->diagbuf.end() || !it->second.p) return set_err(BTF_ESTATE, "diagnostic '%s' not recorded (btf_enable_diag before the sweep)", name);
    if (n != it->second.n) return set_err(BTF_EINVAL, "%s: expected %zu values, got %zu", name, it->second.n, n);
    CK(cudaMemcpy(host, it->second.p, n * sizeof(double), cudaMemcpyDeviceToHost));
    return BTF_OK;
}

// ------------------------------------------------------------------ the sweep
// Phase boundaries: CUDA events for btf_time_phases, and NVTX ranges (BTF_NVTX=1) so that a timeline tool shows
// nu2 / sigma2 / tau2 / lam2 / row_stats / row_solve / col_stats / band_solve / comm around the launches of a sweep.
static const char* const kPhaseNames[] = {"btf:nu2_or_pg", "btf:sigma2", "btf:tau2", "btf:lam2", "btf:row_stats", "btf:row_solve",
                                          "btf:col_stats", "btf:band_solve", "btf:comm"};
static inline void phase_mark(btf_engine* e, int idx) {
    if (e->time_phases) cudaEventRecord(e->ph_ev[idx], e->stream);
    if (e->env.nvtx) {
        if (idx > 0) nvtxRangePop();
        if (idx < PH_COUNT) nvtxRangePushA(kPhaseNames[idx]);
    }
}

// ---- K1 on the integer tensor cores, staged over the engine's streams (stats_i8.cu).
// begin_*: digits + tensor-core product block on side[0], FP64 linear block on side[1] (or everything on the main
// stream when `fork` is false); finish_*: join, exchange of the linear block (sharded columns), recombination.
struct I8Pending { int product = 0, nsplit = 1; };

static void fork_side(btf_engine* e, bool fork) {
    if (!fork) return;
    cudaEventRecord(e->ev_fork, e->stream);
    cudaStreamWaitEvent(e->side[0], e->ev_fork, 0);
    cudaStreamWaitEvent(e->side[1], e->ev_fork, 0);
}
static void join_side(btf_engine* e, bool fork) {
    if (!fork) return;
    for (int i = 0; i < 2; ++i) {
        cudaEventRecord(e->ev_join[i], e->side[i]);
        cudaStreamWaitEvent(e->stream, e->ev_join[i], 0);
    }
}

static int begin_row_stats_i8(btf_engine* e, bool fork, int timer, I8Pending* pd) {
    cudaStream_t sa = fork ? e->side[0] : e->stream, sb = fork ? e->side[1] : e->stream;
    cudaEvent_t* ev = (e->time_phases && timer >= 0) ? e->i8_ev[timer] : nullptr;
    fork_side(e, fork);
    stats_i8_digits(e->i8, e->K, e->V, e->P, e->Ppad, sa);
    if (ev) cudaEventRecord(ev[0], sa);
    const I8Guard gr{e->cnt_rowsum, e->guard_flags, e->guard_n, e->env.i8_guard_tol};
    pd->product = stats_i8_product(e->i8, e->K, e->cnt, e->Ppad, e->Ppad, e->nloc, e->nloc_pad, e->row_stats,
                                   e->env.i8_guard ? &gr : nullptr, sa);
    if (!pd->product) return set_err(BTF_ECUDA, "integer row statistics failed to launch");
    e->i8_route[0] = pd->product;
    if (ev) cudaEventRecord(ev[1], sa);
    pd->nsplit = stats_i8_linear(e->i8, false, e->K, e->S, e->Ppad, e->V, e->Ppad, e->nloc, e->i8.nsplit_b_row, e->i8.bpart, sb);
    if (ev) cudaEventRecord(ev[2], sb);
    e->launches += 4;
    return BTF_OK;
}
static int finish_row_stats_i8(btf_engine* e, bool fork, const I8Pending& pd) {
    join_side(e, fork);
    const I8Guard gr{e->cnt_rowsum, e->guard_flags, e->guard_n, e->env.i8_guard_tol};
    stats_i8_combine(e->i8, e->K, e->nloc, e->nloc_pad, pd.product == I8_ROUTE_FUSED, e->i8.bpart, pd.nsplit, 0, e->nloc,
                     e->row_stats, e->env.i8_guard ? &gr : nullptr, e->stream);
    e->launches += 1;
    if (e->env.i8_guard) {
        stats_i8_fallback(e->K, e->cnt, e->Ppad, e->V, e->P, e->nloc, e->row_stats, gr, e->stream);
        e->launches += 1;
    }
    return cudaGetLastError() == cudaSuccess ? BTF_OK : set_err(BTF_ECUDA, "integer row statistics failed");
}

// Columns: every rank contracts ITS columns over ALL rows (column-sharded copy of the counts, digit planes of the
// all-gathered W), so the product block needs no exchange; the linear block is a partial sum over the local rows
// for all columns (S stays row-sharded: it is read once either way) and is reduce-scattered (M T K doubles), unless
// the rank holds the column-sharded copy of S.  Then the recombination, the guard's fallback and the band solve.
// band: launches the band solve of all local columns on the main stream
template <typename BandFn>
static int col_step_i8(btf_engine* e, bool fork, int timer, BandFn band) {
    cudaStream_t st = e->stream;
    cudaStream_t sa = fork ? e->side[0] : st, sb = fork ? e->side[1] : st;
    cudaEvent_t* ev = (e->time_phases && timer >= 0) ? e->i8_ev[timer] : nullptr;
    const int np = e->Ploc;
    const int ldd = round_up(std::max(np, 1), 256);
    const double* Wloc = e->W + (size_t)e->cfg.row_begin * e->K;
    fork_side(e, fork);
    if (np > 0) { stats_i8_digits(e->i8, e->K, e->W, e->N, e->Nall_pad, sa); e->launches += 2; }
    if (ev) cudaEventRecord(ev[0], sa);
    // linear block: sharded engines need the partial sums of ALL columns before the exchange -> one launch
    // (on the side stream when forked; in the serial mode it is issued after the product block, see below)
    const bool scol = e->shard != nullptr && e->Scol != nullptr;     // own columns over all rows: nothing to exchange
    int lin_split = 1;
    auto linear = [&]() -> int {
        if (scol) {
            // (few row tiles per rank: split the contraction so that the launch still fills the GPU; the partials fit in the
            //  2 P K doubles of the buffer because P_loc <= P / world ... and at least P / 2 for two ranks)
            const int max_split = std::max(1, std::min(8, (int)((2ll * e->P) / std::max(np, 1))));
            if (np > 0) { lin_split = stats_i8_linear(e->i8, true, e->K, e->Scol, e->Ploc_pad, e->W, e->Nall_pad, np, max_split, e->i8.bpart, sb); e->launches++; }
        } else if (e->nloc > 0) {
            // one GPU: the contraction may be split (the partial sums fit in the buffer that also serves the row step);
            // a row-sharded engine reduce-scatters ONE set of partial sums
            const size_t cap = std::max((size_t)e->i8.nsplit_b_row * e->nloc * e->K, (size_t)2 * e->P * e->K) / ((size_t)e->P * e->K);
            const int max_split = e->shard ? 1 : (int)std::min<size_t>(4, std::max<size_t>(cap, 1));
            lin_split = stats_i8_linear(e->i8, true, e->K, e->S, e->Ppad, Wloc, e->nloc_pad, e->P, max_split, e->i8.bpart, sb); e->launches++;
        } else {
            cudaMemsetAsync(e->i8.bpart, 0, (size_t)e->P * e->K * sizeof(double), sb);
        }
        if (fork) { cudaEventRecord(e->ev_join[1], sb); cudaStreamWaitEvent(st, e->ev_join[1], 0); }
        if (e->shard && !scol && nccl_reduce_scatter_cols(e->shard, e->i8.bpart, (size_t)e->T * e->K, st))
            return set_err(BTF_ENCCL, "reduce-scatter(linear block) failed: %s", nccl_shard_error());
        return BTF_OK;
    };
    if (fork) { int rc = linear(); if (rc) return rc; }
    int product = 0;
    double* out = e->col_stats + (size_t)e->p0 * e->nco;
    const I8Guard gc{e->cnt_colsum, e->guard_flags + std::max(e->nloc, 1), e->guard_n + 1, e->env.i8_guard_tol};
    const I8Guard* gp = e->env.i8_guard ? &gc : nullptr;
    if (np > 0) {
        product = stats_i8_product(e->i8, e->K, e->cntT, e->Nall_pad, e->Nall_pad, np, ldd, out, gp, sa);
        if (!product) return set_err(BTF_ECUDA, "integer column statistics failed to launch");
        e->i8_route[1] = product;
        e->launches++;
    }
    if (fork) { cudaEventRecord(e->ev_join[0], sa); cudaStreamWaitEvent(st, e->ev_join[0], 0); }
    if (ev) cudaEventRecord(ev[1], sa);
    if (!fork) { int rc = linear(); if (rc) return rc; }
    if (ev) cudaEventRecord(ev[2], sb);
    if (np > 0) {
        stats_i8_combine(e->i8, e->K, np, ldd, product == I8_ROUTE_FUSED, e->i8.bpart, lin_split, scol ? 0 : e->p0,
                         scol ? np : e->P, out, gp, st);
        e->launches++;
        if (gp) {
            stats_i8_fallback(e->K, e->cntT, e->Nall_pad, e->W, e->N, np, out, gc, st);
            e->launches += 1;
        }
    }
    phase_mark(e, PH_BAND_SOLVE);
    if (e->Mloc > 0) band();
    return cudaGetLastError() == cudaSuccess ? BTF_OK : set_err(BTF_ECUDA, "integer column statistics failed");
}

// The integer-tensor-core statistics path: Gaussian data (count weights), K in {8, 16, 32}, accumulators
// that cannot overflow, a device that runs the 2-CTA GEMM, and a tensor large enough for the digit planes to pay (BTF_STATS_FORCE_I8=1
// forces it for any size, BTF_STATS_NO_I8=1 disables it).  The decision only uses global quantities, so
// every rank of a sharded engine takes the same path (the two paths exchange different things).
static int ensure_i8(btf_engine* e) {
    if (e->i8_decided) return BTF_OK;
    e->i8_decided = true;
    e->i8_on = false;
    // (per-cell variances make the weights cnt / nu2 non-integer)
    if (e->cfg.likelihood != BTF_GAUSSIAN || !e->has_data || e->env.no_i8 || e->nu2_cells) return BTF_OK;
    const long long cells = (long long)e->N * e->P / std::max(1, e->cfg.world_size);
    if (!stats_i8_supported(e->K, e->nreps, e->Ppad, e->Nall_pad)) return BTF_OK;
    if (e->cfg.world_size > 1 && !e->shard) return BTF_OK;       // a shard without a communicator cannot build its column copy
    if (!e->env.force_i8 && cells < (1ll << 24)) return BTF_OK;
    cudaStream_t st = e->stream;
    if (!e->i8.planes) {
        StatsI8Sizes z;
        stats_i8_sizes(e->K, e->nloc_pad, e->Ppad, e->nloc, e->P, e->Nall_pad, e->Ploc, &z);
        CK(cudaMalloc((void**)&e->i8.planes, z.planes_bytes));
        CK(cudaMemsetAsync(e->i8.planes, 0, z.planes_bytes, st));
        CK(dev_alloc(&e->i8.colmax, (size_t)z.L));
        CK(dev_alloc(&e->i8.expo, (size_t)z.L));
        CK(dev_alloc(&e->i8.D, z.d_elems, false));
        CK(dev_alloc(&e->i8.bpart, z.bpart_elems));
        CK(dev_alloc(&e->cntT, z.cntT_bytes));
        CK(dev_alloc(&e->cnt_rowsum, (size_t)std::max(e->nloc, 1)));
        CK(dev_alloc(&e->cnt_colsum, (size_t)std::max(e->Ploc, 1)));
        CK(dev_alloc(&e->guard_n, 2));
        CK(dev_alloc(&e->guard_flags, (size_t)std::max(e->nloc, 1) + std::max(e->Ploc, 1)));
        e->i8.nsplit_b_row = z.nsplit_b_row;
    }
    if (!e->shard) {
        launch_transpose_u8(e->cnt, e->Ppad, e->nloc, e->P, e->cntT, e->Nall_pad, st);
        e->launches++;
    } else {
        // transpose the local row block, then exchange: every rank keeps the counts of ITS columns over all rows
        uint8_t *tT = nullptr, *tmp = nullptr;
        const size_t tbytes = (size_t)e->P * e->nloc_pad;
        const size_t rbytes = (size_t)std::max(e->Ploc, 1) * round_up(std::max(nccl_shard_max_rows(e->shard), 1), 128);
        CK(cudaMalloc((void**)&tT, std::max<size_t>(tbytes, 1)));
        if (cudaMalloc((void**)&tmp, rbytes) != cudaSuccess) { cudaFree(tT); return set_err(BTF_ECUDA, "out of memory for the count exchange"); }
        cudaMemsetAsync(tT, 0, std::max<size_t>(tbytes, 1), st);
        cudaMemsetAsync(e->cntT, 0, (size_t)std::max(e->Ploc, 1) * e->Nall_pad, st);
        if (e->nloc > 0) { launch_transpose_u8(e->cnt, e->Ppad, e->nloc, e->P, tT, e->nloc_pad, st); e->launches++; }
        const int rc = nccl_exchange_counts(e->shard, tT, e->nloc_pad, e->T, e->cntT, e->Nall_pad, tmp, st);
        cudaError_t ce = cudaStreamSynchronize(st);
        cudaFree(tT); cudaFree(tmp);
        if (rc) return set_err(BTF_ENCCL, "exchange of the count blocks failed: %s", nccl_shard_error());
        if (ce != cudaSuccess) return set_err(BTF_ECUDA, "exchange of the count blocks: %s", cudaGetErrorString(ce));
        // Column-sharded copy of S as well when it is cheap (a quarter of the free memory at most; every rank must agree,
        // so the decision uses the largest shard): the linear block of the V step then covers the rank's own columns over
        // all rows and the M T K reduce-scatter disappears from the critical path (C2 on 8 GPUs: 0.06 of 0.77 ms).
        e->Ploc_pad = round_up(std::max(e->Ploc, 1), 256);
        if (e->Scol) { cudaFree(e->Scol); e->Scol = nullptr; }
        if (e->env.scol) {
            const size_t max_rows = (size_t)std::max(nccl_shard_max_rows(e->shard), 1);
            const size_t max_pl = (size_t)round_up(std::max(nccl_shard_max_cols(e->shard), 1) * e->T, 256);
            const size_t need = ((size_t)e->Nall_pad + 32) * max_pl * 8 + 2 * max_rows * max_pl * 8;
            size_t free_b = 0, total_b = 0;
            cudaMemGetInfo(&free_b, &total_b);
            double fits = need <= free_b / 4 ? 1.0 : 0.0, *dflag = nullptr;
            CK(cudaMalloc((void**)&dflag, 8));
            CK(h2d(dflag, &fits, 8));
            if (nccl_allreduce_sum(e->shard, dflag, 1, st)) { cudaFree(dflag); return set_err(BTF_ENCCL, "all-reduce failed: %s", nccl_shard_error()); }
            CK(cudaMemcpyAsync(&fits, dflag, 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            cudaFree(dflag);
            if (fits >= (double)e->cfg.world_size - 0.5) {
                double *ts = nullptr, *tr = nullptr;
                const size_t sc_elems = ((size_t)e->Nall_pad + 32) * e->Ploc_pad;
                if (cudaMalloc((void**)&e->Scol, sc_elems * 8) != cudaSuccess || cudaMalloc((void**)&ts, max_rows * max_pl * 8) != cudaSuccess ||
                    cudaMalloc((void**)&tr, max_rows * max_pl * 8) != cudaSuccess) {
                    cudaGetLastError();
                    if (ts) cudaFree(ts);
                    if (tr) cudaFree(tr);
                    if (e->Scol) { cudaFree(e->Scol); e->Scol = nullptr; }
                    return set_err(BTF_ECUDA, "out of memory for the column-sharded data copy");
                }
                cudaMemsetAsync(e->Scol, 0, sc_elems * 8, st);
                const int rc2 = nccl_exchange_rows_f64(e->shard, e->S, e->Ppad, e->T, e->Scol, e->Ploc_pad, ts, tr, st);
                ce = cudaStreamSynchronize(st);
                cudaFree(ts); cudaFree(tr);
                if (rc2) return set_err(BTF_ENCCL, "exchange of the data blocks failed: %s", nccl_shard_error());
                if (ce != cudaSuccess) return set_err(BTF_ECUDA, "exchange of the data blocks: %s", cudaGetErrorString(ce));
            }
        }
    }
    // count sums of every local row and every owned (j, t): the error bound of the fixed-point block is 2^(e_c - 55) n_m
    stats_i8_count_rows(e->cnt, e->Ppad, e->nloc, e->Ppad, e->cnt_rowsum, st);
    stats_i8_count_rows(e->cntT, e->Nall_pad, e->Ploc, e->Nall_pad, e->cnt_colsum, st);
    e->launches += 2;
    // one eager pass so that every kernel attribute is set before a graph capture
    e->i8_on = true;
    I8Pending pd;
    if (e->nloc > 0) {
        int rc = begin_row_stats_i8(e, false, -1, &pd); if (rc) { e->i8_on = false; return rc; }
        rc = finish_row_stats_i8(e, false, pd); if (rc) { e->i8_on = false; return rc; }
    }
    { int rc = col_step_i8(e, false, -1, []() {}); if (rc) { e->i8_on = false; return rc; } }
    CK(cudaStreamSynchronize(st));
    free_graph(e);
    return BTF_OK;
}

static int ensure_data_reduced(btf_engine* e) {
    { int rc = ensure_i8(e); if (rc) return rc; }
    if (e->data_reduced) return BTF_OK;
    if (e->shard) {
        int rc = nccl_allreduce_sum(e->shard, &e->scal->ss_total, 2, e->stream);   // ss_total, n_obs adjacent
        if (rc) return set_err(BTF_ENCCL, "all-reduce of data totals failed");
    }
    e->data_reduced = true;
    return BTF_OK;
}

// The GASS step of the W rows (col = false) or V columns after their Gaussian draw (the old state is in Wold / Vold)
static GassArgs gass_args(btf_engine* e, bool col) {
    GassArgs g;
    memset(&g, 0, sizeof(g));
    g.col = col;
    g.N = e->N; g.M = e->M; g.T = e->T; g.K = e->K; g.P = e->P; g.ld = e->Ppad;
    g.cnt = e->cnt; g.S = e->S; g.lgy = e->lgy; g.ntr = e->ntr;
    g.binomial = e->cfg.likelihood == BTF_CBINOMIAL;
    g.gaussian = e->cfg.likelihood == BTF_CGAUSSIAN;
    g.nu2c = e->nu2_cells ? e->nu2c : nullptr;
    g.ep_mu = e->ep_on ? e->ep_mu : nullptr; g.ep_sig = e->ep_on ? e->ep_sig : nullptr;
    g.A = e->gA; g.C = e->gC; g.J = e->gJ; g.rowcons = e->growc; g.nrc = e->gnrc;
    g.grid_fine = e->ggrid_f; g.nfine = e->gnfine; g.grid_coarse = e->ggrid_c; g.ngrid = e->gngrid;
    g.Wold = e->Wold; g.Vold = e->Vold; g.Wnew = e->W; g.Vnew = e->V;
    g.Wcur = e->W; g.Vcur = e->V;
    g.u_inject = inj(e, col ? "gass_u_V" : "gass_u_W");
    g.scal = e->scal; g.seed = e->cfg.seed;
    g.diag = diag_get(e, col ? "gass_V" : "gass_W", (size_t)(col ? e->M : e->N) * 3);
    return g;
}

// The reference asserts that every GASS step starts from a feasible point ('Invalid starting point!'): count the rows and
// columns whose current state violates a constraint before a sweep changes anything
static int gass_check_start(btf_engine* e) {
    const int mask = e->cfg.sample_mask;
    if (!(mask & (BTF_SAMPLE_W | BTF_SAMPLE_V))) return BTF_OK;
    cudaStream_t st = e->stream;
    CK(cudaMemsetAsync(e->gass_nbad, 0, 2 * sizeof(int), st));
    for (int col = 0; col < 2; ++col) {
        if (!(mask & (col ? BTF_SAMPLE_V : BTF_SAMPLE_W))) continue;
        GassArgs g = gass_args(e, col != 0);
        g.Wold = e->W; g.Vold = e->V; g.u_inject = nullptr; g.diag = nullptr;
        g.check_only = 1; g.nbad = e->gass_nbad + col;
        launch_gass(g, st); e->launches++;
    }
    int h[2] = {0, 0};
    CK(cudaMemcpyAsync(h, e->gass_nbad, sizeof(h), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    if (h[0] || h[1])
        return set_err(BTF_ESTATE, "invalid starting point: the state violates a constraint in %d row(s) and %d column(s)", h[0], h[1]);
    return BTF_OK;
}

// Enqueue one resample(data) on e->stream.  Order: factor.py:306-311 (nu2 / omega),
// then 112-128 (sigma2, Tau2, lam2, W, V); NB adds the R update first (494-511).
static int enqueue_sweep(btf_engine* e) {
    const btf_config& c = e->cfg;
    cudaStream_t st = e->stream;
    const bool gauss = c.likelihood == BTF_GAUSSIAN;
    const bool cgauss = c.likelihood == BTF_CGAUSSIAN;
    // known per-cell variances: the PG models' f64-weight route, with weights cnt / nu2 and right-hand side S / nu2
    const bool percell = gauss && e->nu2_cells;
    const bool homo = gauss && !percell;      // one scalar nu2 scales the statistics
    const int mask = c.sample_mask;
    launch_bump_sweep(e->scal, st); e->launches++;
    phase_mark(e, PH_NU2);
    // Integer statistics path: the row statistics only read V and the data, so they start now on the side streams
    // (tensor-core product block | HBM-bound linear block) while the hyper-parameter steps run on the main stream.
    const bool doW = (mask & BTF_SAMPLE_W) && e->nloc > 0;
    const bool fork = e->i8_on && !e->time_phases;
    I8Pending pend_row;
    if (fork && doW) { int rc = begin_row_stats_i8(e, true, 0, &pend_row); if (rc) return rc; }

    if (c.likelihood == BTF_NEGBINOMIAL) {
        NbArgs nb;
        nb.Yraw = e->Yraw; nb.nloc = e->nloc; nb.P = e->P; nb.R = e->nreps; nb.M = e->M; nb.T = e->T; nb.K = e->K;
        nb.row_begin = c.row_begin; nb.nrows_global = e->N; nb.ld = e->Ppad;
        nb.W = e->W + (size_t)c.row_begin * e->K; nb.V = e->V; nb.Rdisp = e->Rdisp; nb.Rn = e->Rn; nb.Rm = e->Rm; nb.Rt = e->Rt;
        nb.nmh = (mask & BTF_SAMPLE_R) ? c.nmetropolis : 0; nb.rpropstdev = c.rpropstdev; nb.rstdev = c.rstdev;
        nb.z_inject = inj(e, "z_R"); nb.u_inject = inj(e, "u_R");
        nb.scal = e->scal; nb.seed = c.seed; nb.work = e->nb_work;
        nb.obs = e->cnt; nb.kappa = e->S; nb.ntr = e->ntr;
        nb.hist = e->nb_hist; nb.hist_stride = e->nb_hist_stride;
        launch_nb_update(nb, st); e->launches += nb.nmh > 0 ? (nb.hist ? 4 : 2 * nb.nmh + 4) : 1;
    }
    if (gauss || cgauss) {
        if (mask & BTF_SAMPLE_NU2) {
            // constrained Gaussian: the GASS steps leave no residual by-product, so the direct pass runs every sweep
            if (!e->resid_valid || c.resid_direct || cgauss) {
                int nb = 0;
                launch_residual(e->cnt, e->S, e->Ppad, e->W + (size_t)c.row_begin * e->K, e->V, e->nloc_pad, e->Ppad,
                                e->K, e->partials, &nb, st);
                launch_set_resid(e->scal, e->partials, nb, st);
                e->launches += 2;
                if (e->shard) {
                    // resid = ss_total + sum(partials) on every rank: combine the partial sums only
                    if (nccl_allreduce_resid(e->shard, e->scal, st)) return set_err(BTF_ENCCL, "all-reduce(resid) failed");
                }
            }
            ScalarStepArgs sa{e->scal, c.seed, c.nu2_a, c.nu2_b, inj(e, "g_nu2")};
            launch_nu2(sa, st); e->launches++;
        }
    } else if (e->omega && ((mask & BTF_SAMPLE_NU2) || inj(e, "omega"))) {
        const double* om = inj(e, "omega");
        if (om) {
            cudaMemcpy2DAsync(e->omega, (size_t)e->Ppad * 8, om, (size_t)e->P * 8, (size_t)e->P * 8, e->nloc,
                              cudaMemcpyDeviceToDevice, st);
        } else {
            PgArgs pa;
            pa.obs = e->cnt; pa.ntr = e->ntr; pa.omega = e->omega; pa.ld = e->Ppad;
            pa.W = e->W + (size_t)c.row_begin * e->K; pa.V = e->V;
            pa.nloc = e->nloc; pa.nrows_pad = e->nloc_pad; pa.P = e->P; pa.Ppad = e->Ppad; pa.K = e->K; pa.row_begin = c.row_begin;
            pa.scal = e->scal; pa.seed = c.seed;
            launch_pg_draw(pa, st); e->launches++;
        }
    }
    phase_mark(e, PH_SIGMA2);
    if (mask & BTF_SAMPLE_SIGMA2) {
        launch_w_sumsq(e->W, e->N, e->K, e->scal, e->lam_partials + e->M, st);
        ScalarStepArgs sa{e->scal, c.seed, c.sigma2_a, c.sigma2_b, inj(e, "g_sigma2")};
        const double nfree = e->N >= e->K ? (double)e->L + (double)(e->N - e->K) * e->K : 0.5 * e->N * (e->N + 1.0);
        launch_sigma2(sa, nfree, st);
        e->launches += 3;
    }
    phase_mark(e, PH_TAU2);
    HyperArgs ha;
    ha.scal = e->scal; ha.V = e->V; ha.M = e->M; ha.T = e->T; ha.K = e->K; ha.RD = e->RD;
    ha.d_start = e->d_start; ha.d_width = e->d_width; ha.d_coef = e->d_coef; ha.d_maxw = e->d_maxw;
    ha.Tau2 = e->Tau2; ha.Tau2_a = e->Tau2_a; ha.Tau2_b = e->Tau2_b; ha.Tau2_c = e->Tau2_c;
    ha.stability = c.stability; ha.g_inject = inj(e, "g_tau"); ha.seed = c.seed;
    ha.lam_partials = nullptr; ha.col_begin = 0; ha.col_end = e->M;   // Philox is keyed by (j, r): identical on every rank
    if (mask & BTF_SAMPLE_TAU2) {
        if (e->tau_sharded) {
            // own columns only (the band solve needs no others); the reference's lam2 step reads the LAST column
            // (factor.py:150), which every rank therefore updates too; the blocks are gathered at API boundaries
            HyperArgs hs = ha;
            hs.col_begin = c.col_begin; hs.col_end = c.col_end;
            launch_tau2(hs, st);
            if (c.col_end != e->M) { hs.col_begin = e->M - 1; hs.col_end = e->M; launch_tau2(hs, st); e->launches++; }
        } else {
            launch_tau2(ha, st);
        }
        e->launches++;
    }
    phase_mark(e, PH_LAM2);
    if (mask & BTF_SAMPLE_LAM2) {
        HyperArgs hl = ha;
        hl.Tau2_a = nullptr; hl.lam_partials = e->lam_partials;
        if (c.ref_compat_lam2) { hl.col_begin = e->M - 1; hl.col_end = e->M; }
        launch_tau2(hl, st);
        ScalarStepArgs sa{e->scal, c.seed, 0.0, 0.0, inj(e, "g_lam")};
        const double shape = 0.5 * ((double)e->RD * e->M * e->K + 1.0);
        launch_lam2(sa, e->lam_partials, e->M, c.ref_compat_lam2, shape, st);
        e->launches += 2;
    }
    // ---- W | rest
    phase_mark(e, PH_ROW_STATS);
    // GASS models: the statistics of the EP approximation (weights 1 / sigma^2, right-hand side mu / sigma^2), none without it
    const bool gass = gass_likelihood(c.likelihood);
    const bool no_stats = gass && !e->ep_on;
    const void* wt = (percell || gass) ? (const void*)e->wc : gauss ? (const void*)e->cnt : (const void*)e->omega;
    const double* sv = (percell || gass) ? e->sc : e->S;
    const bool wf64 = !homo;
    const StatsPlan& prow = stats_plan(e, false);
    const StatsPlan& pcol = stats_plan(e, true);
    if (doW) {
        if (e->i8_on) {
            if (!fork) { int rc = begin_row_stats_i8(e, false, 0, &pend_row); if (rc) return rc; }
            { int rc = finish_row_stats_i8(e, fork, pend_row); if (rc) return rc; }
        } else if (!no_stats) {
            launch_stats(prow, false, wf64, wt, sv, e->V, e->Ppad, e->Ppad, e->nloc, e->row_stats, e->zbuf, st);
            e->launches += prow.zpre ? 2 : 1;
        }
        phase_mark(e, PH_ROW_SOLVE);
        RowSolveArgs ra;
        ra.stats = e->row_stats; ra.nsplit = no_stats ? 0 : e->i8_on ? 1 : prow.nsplit; ra.split_stride = prow.out_elems_per_split;
        ra.nloc = e->nloc; ra.row_begin = c.row_begin; ra.K = e->K;
        ra.scale_from_nu2 = homo ? &e->scal->nu2 : nullptr; ra.scal = e->scal; ra.W = e->W;
        ra.z_inject = inj(e, "z_W"); ra.seed = c.seed;
        ra.diag_Q = diag_get(e, "W_Q", (size_t)e->N * e->K * e->K);
        ra.diag_L = diag_get(e, "W_L", (size_t)e->N * e->K * e->K);
        ra.diag_mean = diag_get(e, "W_mean", (size_t)e->N * e->K);
        ra.diag_b = diag_get(e, "W_b", (size_t)e->N * e->K);
        if (gass) {
            // GASS needs the old state and, with EP, the centre of the ellipse
            CK(cudaMemcpyAsync(e->Wold, e->W, (size_t)e->N * e->K * 8, cudaMemcpyDeviceToDevice, st));
            if (e->ep_on && !ra.diag_mean) ra.diag_mean = e->gmeanW;
        }
        launch_row_solve(ra, nullptr, st); e->launches++;
        if (gass) {
            GassArgs ga = gass_args(e, false);
            ga.Wmean = e->ep_on ? ra.diag_mean : nullptr;
            launch_gass(ga, st); e->launches++;
        }
        e->resid_valid = false;
    } else {
        phase_mark(e, PH_ROW_SOLVE);
    }
    phase_mark(e, PH_COL_STATS);
    if (e->shard && (mask & BTF_SAMPLE_W)) {
        if (nccl_allgather_rows(e->shard, e->W, e->K, st)) return set_err(BTF_ENCCL, "all-gather(W) failed");
    }
    // ---- V | rest
    if (mask & BTF_SAMPLE_V) {
        BandSolveArgs ba;
        ba.stats = e->col_stats; ba.nsplit = 1; ba.split_stride = pcol.out_elems_per_split;
        ba.col_begin = c.col_begin; ba.ncols_loc = e->Mloc; ba.T = e->T; ba.K = e->K; ba.order = e->order; ba.RD = e->RD;
        ba.homoskedastic = homo ? 1 : 0; ba.scal = e->scal; ba.Tau2 = e->Tau2;
        ba.prior_clip = c.clip_prior_precision ? c.stability : 0.0;
        ba.pm_ptr = e->pm_ptr; ba.pm_row = e->pm_row; ba.pm_coef = e->pm_coef;
        ba.V = e->V; ba.z_inject = inj(e, "z_V"); ba.seed = c.seed;
        ba.work_L = e->work_L; ba.work_y = e->work_y;
        ba.work_L_stride = e->wL_stride; ba.work_y_stride = e->wy_stride;
        ba.force_psd = c.force_psd; ba.attempts = c.force_psd_attempts; ba.eps = c.force_psd_eps;
        ba.force_scalar = e->env.band_scalar;
        const size_t bn = (size_t)e->Mloc * e->n * (e->kd + 1);
        ba.diag_band = diag_get(e, "V_band", bn);
        ba.diag_chol = diag_get(e, "V_chol", bn);
        ba.diag_mean = diag_get(e, "V_mean", (size_t)e->P * e->K);
        if (gass && e->ep_on && !ba.diag_mean) ba.diag_mean = e->gmeanV;
        ba.diag_retries = e->diag_retries;
        ba.resid_partials = homo ? e->resid_partials + c.col_begin : nullptr;
        auto band = [&]() {
            if (gass) CK(cudaMemcpyAsync(e->Vold, e->V, (size_t)e->P * e->K * 8, cudaMemcpyDeviceToDevice, st));
            launch_band_solve(ba, st); e->launches++;
            if (gass) {
                GassArgs ga = gass_args(e, true);
                ga.Vmean = e->ep_on ? ba.diag_mean : nullptr;
                launch_gass(ga, st); e->launches++;
            }
            return BTF_OK;
        };
        if (e->i8_on) {
            e->col_collapsed = false;
            int rc = col_step_i8(e, fork, 1, band);
            if (rc) return rc;
        } else {
            int nsplit = pcol.nsplit;
            if (no_stats) {
                ba.stats = nullptr;           // prior-only system
                nsplit = 0;
            } else {
                launch_stats(pcol, true, wf64, wt, sv, e->W + (size_t)c.row_begin * e->K, e->nloc_pad, e->Ppad, e->P,
                             e->col_stats, e->zbuf, st);
                e->launches += pcol.zpre ? 2 : 1;
            }
            if (e->shard) {
                // FP64 statistics path across GPUs: partial statistics over the local rows for all columns, collapsed
                // over the splits, then reduce-scattered by column block
                if (nccl_reduce_col_stats(e->shard, e->col_stats, nsplit, pcol.out_elems_per_split, e->T * e->nco, st))
                    return set_err(BTF_ENCCL, "reduce-scatter(col stats) failed");
                nsplit = 1;
                e->col_collapsed = true;
            } else if (nsplit > 2) {
                // deep split-K (few columns): one pass that sums the partials in split order, instead of
                // nsplit dependent loads per statistic inside the latency-bound band kernel
                launch_collapse_splits(e->col_stats, nsplit, pcol.out_elems_per_split, st);
                e->launches++;
                nsplit = 1;
                e->col_collapsed = true;
            } else {
                e->col_collapsed = false;
            }
            ba.nsplit = nsplit;
            phase_mark(e, PH_BAND_SOLVE);
            if (e->Mloc > 0) { int rc = band(); if (rc) return rc; }
        }
        phase_mark(e, PH_COMM);
        if (e->shard) {
            if (nccl_allgather_cols(e->shard, e->V, e->n, st)) return set_err(BTF_ENCCL, "all-gather(V) failed");
        }
        if (homo && !c.resid_direct) {
            // nu2 by-product: resid = ss_total + sum_j [v^T A v - 2 v.b]
            if (e->shard) {
                if (nccl_allgather_doubles(e->shard, e->resid_partials, st)) return set_err(BTF_ENCCL, "all-gather(resid) failed");
            }
            launch_set_resid(e->scal, e->resid_partials, e->M, st); e->launches++;
            e->resid_valid = true;
        }
    } else {
        phase_mark(e, PH_BAND_SOLVE);
        phase_mark(e, PH_COMM);
    }
    if (percell) e->resid_valid = false;   // no residual by-product: a later nu2 step takes the direct pass
    phase_mark(e, PH_COUNT);
    return BTF_OK;
}

// Sharded engines update the Tau2 chain for their own columns only: make the four arrays whole again
// (every rank calls the same API sequence, so the collectives match).
static int sync_tau(btf_engine* e) {
    if (!e->shard || !e->tau_stale) return BTF_OK;
    double* arrs[4] = {e->Tau2, e->Tau2_a, e->Tau2_b, e->Tau2_c};
    if (nccl_allgather_tau(e->shard, arrs, 4, e->RD, e->stream)) return set_err(BTF_ENCCL, "all-gather(Tau2) failed: %s", nccl_shard_error());
    e->tau_stale = false;
    return BTF_OK;
}

static int check_info(btf_engine* e) {
    CK(cudaMemcpyAsync(e->pinned_scal, e->scal, sizeof(Scalars), cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaGetLastError());
    Scalars h;
    memcpy(&h, e->pinned_scal, sizeof(h));
    if (h.info_w > 0) return set_err(BTF_ENOTPD, "W step: Cholesky failed for %d row(s) (factor.py:357 has no retry)", h.info_w);
    if (h.info_v > 0) return set_err(BTF_ENOTPD, "V step: Cholesky failed for %d column(s) after %d jitter attempts", h.info_v, e->cfg.force_psd_attempts);
    return BTF_OK;
}

static bool graph_ok(btf_engine* e) {
    // (sharded engines: the NCCL collectives are captured with the kernels; the first sweep runs eagerly
    //  so that NCCL has set up its channels before a capture)
    return e->cfg.use_graph && (!e->shard || e->eager_sweeps > 0) && e->inject.empty() && !e->diag && !e->time_phases &&
           (e->resid_valid || e->cfg.likelihood != BTF_GAUSSIAN || e->cfg.resid_direct || !(e->cfg.sample_mask & BTF_SAMPLE_NU2));
}

static int build_graph(btf_engine* e) {
    cudaGraph_t g = nullptr;
    int64_t before = e->launches;
    CK(cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
    int rc = enqueue_sweep(e);
    cudaError_t ce = cudaStreamEndCapture(e->stream, &g);
    e->graph_launches = (int)(e->launches - before);
    e->launches = before;
    if (rc) { if (g) cudaGraphDestroy(g); return rc; }
    if (ce != cudaSuccess) return set_err(BTF_ECUDA, "graph capture failed: %s", cudaGetErrorString(ce));
    ce = cudaGraphInstantiate(&e->graph_exec, g, 0);
    cudaGraphDestroy(g);
    if (ce != cudaSuccess) { e->graph_exec = nullptr; return set_err(BTF_ECUDA, "graph instantiate failed: %s", cudaGetErrorString(ce)); }
    return BTF_OK;
}

// one sweep, by graph replay when the sequence is static
static int one_sweep(btf_engine* e) {
    // (set here, not while enqueueing: a graph replay does not run the enqueue code)
    if (e->tau_sharded && (e->cfg.sample_mask & BTF_SAMPLE_TAU2)) e->tau_stale = true;
    if (graph_ok(e)) {
        if (!e->graph_exec) { int rc = build_graph(e); if (rc) return rc; }
        CK(cudaGraphLaunch(e->graph_exec, e->stream));
        e->launches += e->graph_launches;
        return BTF_OK;
    }
    int rc = enqueue_sweep(e);
    e->eager_sweeps++;
    if (!e->inject.empty()) {
        // injected noise is consumed by exactly one sweep
        CK(cudaStreamSynchronize(e->stream));
        clear_inject(e);
    }
    return rc;
}

static int pre_run(btf_engine* e) {
    if (!e) return set_err(BTF_EINVAL, "null engine");
    // the hyper-parameter steps (sigma2, Tau2, lam2) only read the factors: no data needed for them
    const int needs_data = BTF_SAMPLE_NU2 | BTF_SAMPLE_W | BTF_SAMPLE_V | BTF_SAMPLE_R;
    if (!e->has_data && ((e->cfg.sample_mask & needs_data) || e->cfg.likelihood != BTF_GAUSSIAN))
        return set_err(BTF_ESTATE, "no data: call btf_set_data_* first");
    CK(cudaSetDevice(e->cfg.device));
    if (e->nu2_cells) {
        if (e->cfg.sample_mask & BTF_SAMPLE_NU2)
            return set_err(BTF_ESTATE, "the nu2 step does not run with per-cell noise variances: clear BTF_SAMPLE_NU2 or "
                                       "return to a scalar nu2 with btf_set_nu2_cells(e, NULL)");
        if (e->nu2_dirty && e->has_data) {
            // the data changed since the weights were formed
            CK(cudaMemsetAsync(e->nu2_nbad, 0, sizeof(unsigned long long), e->stream));
            enqueue_nu2_weights(e, e->nu2c, e->Ppad, 0, e->nloc, false);
            int rc = read_nu2_bad(e);
            if (rc) return rc;
            e->nu2_dirty = false;
        }
        if (e->nu2_bad) return nu2_bad_error(e);
    }
    if (gass_likelihood(e->cfg.likelihood)) {
        if (!e->gass_set) return set_err(BTF_ESTATE, "no constraints: call btf_set_gass first");
        int rc = gass_check_start(e);
        if (rc) return rc;
    }
    int rc = ensure_data_reduced(e);
    if (rc) return rc;
    launch_clear_info(e->scal, e->stream); e->launches++;
    return BTF_OK;
}

int btf_sweep(btf_engine* e, int32_t nsweeps) {
    int rc = pre_run(e);
    if (rc) return rc;
    for (int s = 0; s < nsweeps; ++s) { rc = one_sweep(e); if (rc) return rc; }
    rc = sync_tau(e);
    if (rc) return rc;
    return check_info(e);
}

int btf_sweep_timed(btf_engine* e, int32_t nsweeps, double* ms_out) {
    int rc = pre_run(e);
    if (rc) return rc;
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaEventRecord(a, e->stream));
    for (int s = 0; s < nsweeps; ++s) { rc = one_sweep(e); if (rc) break; }
    CK(cudaEventRecord(b, e->stream));
    CK(cudaEventSynchronize(b));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, a, b));
    cudaEventDestroy(a); cudaEventDestroy(b);
    if (ms_out) *ms_out = ms;
    if (rc) return rc;
    rc = sync_tau(e);
    if (rc) return rc;
    return check_info(e);
}

int btf_time_phases(btf_engine* e, int32_t nsweeps, double* ms_out, int32_t nphases) {
    int rc = pre_run(e);
    if (rc) return rc;
    if (nphases < PH_COUNT) return set_err(BTF_EINVAL, "need room for %d phases", (int)PH_COUNT);
    for (int i = 0; i < nphases; ++i) ms_out[i] = 0.0;
    e->time_phases = true;
    for (int s = 0; s < nsweeps; ++s) {
        if (e->tau_sharded && (e->cfg.sample_mask & BTF_SAMPLE_TAU2)) e->tau_stale = true;
        rc = enqueue_sweep(e);
        if (rc) break;
        CK(cudaStreamSynchronize(e->stream));
        for (int i = 0; i < PH_COUNT; ++i) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, e->ph_ev[i], e->ph_ev[i + 1]) == cudaSuccess) ms_out[i] += ms;
            else cudaGetLastError();
        }
        // sub-phases of the integer statistics path: int8 GEMM and FP64 linear block, rows then columns
        if (e->i8_on && nphases >= PH_COUNT + 4) {
            const int msk = e->cfg.sample_mask;
            for (int rc2 = 0; rc2 < 2; ++rc2) {
                if (!(msk & (rc2 == 0 ? BTF_SAMPLE_W : BTF_SAMPLE_V))) continue;
                for (int q = 0; q < 2; ++q) {
                    float ms = 0.f;
                    if (cudaEventElapsedTime(&ms, e->i8_ev[rc2][q], e->i8_ev[rc2][q + 1]) == cudaSuccess) ms_out[PH_COUNT + 2 * rc2 + q] += ms;
                    else cudaGetLastError();
                }
            }
        }
    }
    e->time_phases = false;
    for (int i = 0; i < nphases; ++i) ms_out[i] /= std::max(1, nsweeps);
    if (rc) return rc;
    rc = sync_tau(e);
    if (rc) return rc;
    return check_info(e);
}

int btf_synchronize(btf_engine* e) {
    if (!e) return set_err(BTF_EINVAL, "null engine");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaStreamSynchronize(e->copy_stream));
    return BTF_OK;
}

static int eval_enqueue(btf_engine* e, int slot);

__global__ void pack_scalars_kernel(const Scalars* s, double* out) {
    out[0] = s->sigma2; out[1] = s->lam2; out[2] = s->nu2; out[3] = s->lam2_a;
}

// run_gibbs (genlasso.py:37-66), generalised to a segment of a chain: exactly `nsweeps`
// sweeps; the state after local sweep indices first_save, first_save + nthin, ... is
// written to sample slots sample_offset, sample_offset + 1, ...
int btf_run_segment(btf_engine* e, int32_t nsweeps, int32_t first_save, int32_t nthin, int64_t sample_offset,
                    double* W_out, double* V_out, double* Tau2_out, double* scalars_out, double* R_out,
                    double* omega_out) {
    int rc = pre_run(e);
    if (rc) return rc;
    if (nsweeps < 0 || nthin < 1 || first_save < 0 || sample_offset < 0) return set_err(BTF_EINVAL, "bad chain lengths");
    const size_t wn = (size_t)e->N * e->K, vn = (size_t)e->P * e->K, tn = (size_t)e->M * e->RD;
    const size_t rn = (size_t)e->Rn * e->Rm * e->Rt;
    bool pending = false;
    for (int step = 0; step < nsweeps; ++step) {
        rc = one_sweep(e);
        if (rc) return rc;
        if (step >= first_save && (step - first_save) % nthin == 0) {
            const size_t sidx = (size_t)sample_offset + (size_t)(step - first_save) / nthin;
            if (e->mu_track) {
                e->mu_count += 1;
                launch_mu_moments(e->W + (size_t)e->cfg.row_begin * e->K, e->V, e->K, e->nloc, e->P, e->mu_mean, e->mu_m2,
                                  (double)e->mu_count, e->stream);
                e->launches++;
            }
            for (int sl = 0; sl < EVAL_SLOTS; ++sl)
                if (e->eval[sl].active && e->eval[sl].auto_update) { rc = eval_enqueue(e, sl); if (rc) return rc; }
            // snapshot on the compute stream (device-to-device), drain on the copy stream
            if (Tau2_out) { rc = sync_tau(e); if (rc) return rc; }
            if (pending) CK(cudaStreamWaitEvent(e->stream, e->ev_copied, 0));
            if (W_out) CK(cudaMemcpyAsync(e->snapW, e->W, wn * 8, cudaMemcpyDeviceToDevice, e->stream));
            if (V_out) CK(cudaMemcpyAsync(e->snapV, e->V, vn * 8, cudaMemcpyDeviceToDevice, e->stream));
            if (Tau2_out) CK(cudaMemcpyAsync(e->snapTau2, e->Tau2, tn * 8, cudaMemcpyDeviceToDevice, e->stream));
            if (scalars_out) { pack_scalars_kernel<<<1, 1, 0, e->stream>>>(e->scal, e->snapScal); e->launches++; }
            if (R_out && e->Rdisp) CK(cudaMemcpyAsync(e->snapR, e->Rdisp, rn * 8, cudaMemcpyDeviceToDevice, e->stream));
            if (omega_out && e->omega) {
                // omega is large: copy straight from the live buffer on the compute stream
                CK(cudaMemcpy2DAsync(omega_out + sidx * (size_t)e->nloc * e->P, (size_t)e->P * 8, e->omega,
                                     (size_t)e->Ppad * 8, (size_t)e->P * 8, e->nloc, cudaMemcpyDeviceToHost, e->stream));
            }
            CK(cudaEventRecord(e->ev_snap, e->stream));
            CK(cudaStreamWaitEvent(e->copy_stream, e->ev_snap, 0));
            if (W_out) CK(cudaMemcpyAsync(W_out + sidx * wn, e->snapW, wn * 8, cudaMemcpyDeviceToHost, e->copy_stream));
            if (V_out) CK(cudaMemcpyAsync(V_out + sidx * vn, e->snapV, vn * 8, cudaMemcpyDeviceToHost, e->copy_stream));
            if (Tau2_out) CK(cudaMemcpyAsync(Tau2_out + sidx * tn, e->snapTau2, tn * 8, cudaMemcpyDeviceToHost, e->copy_stream));
            if (scalars_out) CK(cudaMemcpyAsync(scalars_out + sidx * 4, e->snapScal, 4 * 8, cudaMemcpyDeviceToHost, e->copy_stream));
            if (R_out && e->Rdisp) CK(cudaMemcpyAsync(R_out + sidx * rn, e->snapR, rn * 8, cudaMemcpyDeviceToHost, e->copy_stream));
            CK(cudaEventRecord(e->ev_copied, e->copy_stream));
            pending = true;
        }
    }
    CK(cudaStreamSynchronize(e->copy_stream));
    rc = sync_tau(e);
    if (rc) return rc;
    return check_info(e);
}

int btf_run(btf_engine* e, int32_t nburn, int32_t nthin, int32_t nsamples, double* W_out, double* V_out,
            double* Tau2_out, double* scalars_out, double* R_out, double* omega_out) {
    if (nburn < 0 || nthin < 1 || nsamples < 0) return set_err(BTF_EINVAL, "bad chain lengths");
    return btf_run_segment(e, nburn + nthin * nsamples, nburn, nthin, 0, W_out, V_out, Tau2_out, scalars_out, R_out,
                           omega_out);
}

// Running posterior moments of Mu = einsum('nk,mtk->nmt', W, V) (genlasso.py:51-65 keeps every
// sample on the host instead): track != 0 (re)starts the accumulation, every sample saved by
// btf_run / btf_run_segment then updates mean and M2 on the device.
int btf_mu_stats_track(btf_engine* e, int32_t track) {
    if (!e) return set_err(BTF_EINVAL, "null engine");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    const size_t n = (size_t)e->nloc * e->P;
    if (track) {
        if (!e->mu_mean) { CK(dev_alloc(&e->mu_mean, n)); CK(dev_alloc(&e->mu_m2, n)); }
        else { CK(cudaMemsetAsync(e->mu_mean, 0, n * 8, e->stream)); CK(cudaMemsetAsync(e->mu_m2, 0, n * 8, e->stream)); }
        e->mu_count = 0;
    }
    e->mu_track = track != 0;
    return BTF_OK;
}
// mean_out, var_out: [nloc, M, T] (either may be NULL); variance with the 1/(count-1) normalisation
int btf_mu_stats_get(btf_engine* e, double* mean_out, double* var_out, int64_t* count_out) {
    if (!e) return set_err(BTF_EINVAL, "null engine");
    if (!e->mu_mean) return set_err(BTF_ESTATE, "posterior moments are not being tracked");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    const size_t n = (size_t)e->nloc * e->P;
    if (count_out) *count_out = e->mu_count;
    if (mean_out) CK(cudaMemcpy(mean_out, e->mu_mean, n * 8, cudaMemcpyDeviceToHost));
    if (var_out) {
        CK(cudaMemcpy(var_out, e->mu_m2, n * 8, cudaMemcpyDeviceToHost));
        const double sc = e->mu_count > 1 ? 1.0 / (double)(e->mu_count - 1) : 0.0;
        for (size_t i = 0; i < n; ++i) var_out[i] *= sc;
    }
    return BTF_OK;
}

// ------------------------------------------------------------------ held-out evaluation
// (politics/benchmark.py:163-180, flutrends/benchmark.py:129-143,
//  examples/poisson_tensor_filtering.py:20-23; kernels in eval_kernels.cu)
static EvalArgs eval_args(btf_engine* e, EvalSlot& s) {
    EvalArgs a{};
    a.W = e->W + (size_t)e->cfg.row_begin * e->K; a.V = e->V;
    a.K = e->K; a.nloc = e->nloc; a.P = e->P; a.T = e->T; a.row_begin = e->cfg.row_begin;
    a.target = s.target; a.cls = s.cls; a.ncls = s.ncls; a.transform = s.transform; a.loglik = s.loglik;
    a.Rdisp = e->Rdisp; a.Rn = e->Rn; a.Rm = e->Rm; a.Rt = e->Rt;
    a.scal = e->scal; a.count = (double)s.count;
    a.mean = s.mean; a.below = s.below; a.above = s.above; a.cdf = s.cdf; a.c_lt = s.c_lt; a.c_le = s.c_le;
    a.partial = s.partial;
    a.nu2c = s.nu2;
    return a;
}
static int eval_enqueue(btf_engine* e, int slot) {
    EvalSlot& s = e->eval[slot];
    if (s.count >= s.max_samples) return set_err(BTF_ESTATE, "evaluator is full (max_samples reached)");
    s.count += 1;
    launch_eval_update(eval_args(e, s), s.samples + (size_t)(s.count - 1) * s.ncls * 4, e->stream);
    e->launches += 2;
    CK(cudaGetLastError());
    return BTF_OK;
}

int btf_eval_set(btf_engine* e, int32_t slot, const double* target, const uint8_t* cls, int32_t nclasses,
                 int32_t transform, int32_t loglik, int32_t cell_state, int32_t auto_update, int64_t max_samples) {
    if (!e) return set_err(BTF_EINVAL, "null engine");
    if (slot < 0 || slot >= EVAL_SLOTS) return set_err(BTF_EINVAL, "evaluator slot out of range");
    if (!target) return set_err(BTF_EINVAL, "null target");
    if (nclasses < 1 || nclasses > EVAL_MAX_CLASSES) return set_err(BTF_EINVAL, "1..4 classes");
    if (transform < EVAL_IDENTITY || transform > EVAL_NB_MEAN) return set_err(BTF_EINVAL, "unknown mean transform");
    if (transform == EVAL_NB_MEAN && !e->Rdisp) return set_err(BTF_EINVAL, "the NB mean needs a negative-binomial engine");
    if (loglik < EVAL_LL_NONE || loglik > EVAL_LL_POISSON) return set_err(BTF_EINVAL, "unknown log-likelihood");
    if (max_samples < 1) return set_err(BTF_EINVAL, "max_samples must be positive");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    EvalSlot& s = e->eval[slot];
    eval_free(s);
    const size_t n = (size_t)e->nloc * e->P;
    s.ncls = nclasses; s.transform = transform; s.loglik = loglik; s.max_samples = max_samples;
    s.auto_update = auto_update != 0;
    CK(dev_alloc(&s.target, n, false));
    CK(cudaMemcpy(s.target, target, n * 8, cudaMemcpyDefault));
    if (cls) { CK(dev_alloc(&s.cls, n, false)); CK(cudaMemcpy(s.cls, cls, n, cudaMemcpyDefault)); }
    CK(cudaStreamSynchronize(cudaStreamLegacy));
    if (cell_state) {
        CK(dev_alloc(&s.mean, n)); CK(dev_alloc(&s.below, n, false)); CK(dev_alloc(&s.above, n, false));
        CK(dev_alloc(&s.c_lt, n)); CK(dev_alloc(&s.c_le, n));
        if (cell_state > 1) CK(dev_alloc(&s.cdf, n));
        launch_eval_init(s.below, s.above, (long long)n, e->stream);
        e->launches++;
    }
    const long long pe = std::max<long long>(eval_partial_elems(e->nloc, e->P, nclasses),
                                             (long long)eval_summary_blocks(e->nloc, e->P) * nclasses * 6);
    CK(dev_alloc(&s.partial, (size_t)pe));
    CK(dev_alloc(&s.samples, (size_t)max_samples * nclasses * 4));
    CK(dev_alloc(&s.summary, (size_t)nclasses * 6));
    CK(cudaStreamSynchronize(e->stream));
    s.active = true;
    return BTF_OK;
}

// known per-cell variances of the slot's cells [Nloc, M, T] (host or device memory) for the Gaussian log-likelihood and
// the predictive band; NULL: the sample's scalar nu2 again
int btf_eval_set_nu2(btf_engine* e, int32_t slot, const double* nu2) {
    if (!e) return set_err(BTF_EINVAL, "null engine");
    if (slot < 0 || slot >= EVAL_SLOTS || !e->eval[slot].active)
        return set_err(BTF_ESTATE, "no evaluator in this slot (btf_eval_set first)");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    EvalSlot& s = e->eval[slot];
    if (s.nu2) { CK(cudaFree(s.nu2)); s.nu2 = nullptr; }
    if (!nu2) return BTF_OK;
    const size_t n = (size_t)e->nloc * e->P;
    CK(dev_alloc(&s.nu2, n, false));
    CK(cudaMemcpy(s.nu2, nu2, n * 8, cudaMemcpyDefault));
    CK(cudaStreamSynchronize(cudaStreamLegacy));
    return BTF_OK;
}

int btf_eval_clear(btf_engine* e, int32_t slot) {
    if (!e) return set_err(BTF_EINVAL, "null engine");
    if (slot < 0 || slot >= EVAL_SLOTS) return set_err(BTF_EINVAL, "evaluator slot out of range");
    CK(cudaSetDevice(e->cfg.device));
    CK(cudaStreamSynchronize(e->stream));
    eval_free(e->eval[slot]);
    return BTF_OK;
}

#define EVAL_SLOT_OR_FAIL(e, slot)                                                              \
    if (!e) return set_err(BTF_EINVAL, "null engine");                                          \
    if (slot < 0 || slot >= EVAL_SLOTS || !e->eval[slot].active)                                \
        return set_err(BTF_ESTATE, "no evaluator in this slot (btf_eval_set first)");          \
    CK(cudaSetDevice(e->cfg.device));

// score the current device state as one more sample
int btf_eval_update(btf_engine* e, int32_t slot) {
    EVAL_SLOT_OR_FAIL(e, slot)
    return eval_enqueue(e, slot);
}

// out: [count][nclasses][4] = {n, sum (y - mu)^2, sum |y - mu|, sum loglik} per scored sample
int btf_eval_samples(btf_engine* e, int32_t slot, double* out, int64_t* count_out) {
    EVAL_SLOT_OR_FAIL(e, slot)
    EvalSlot& s = e->eval[slot];
    CK(cudaStreamSynchronize(e->stream));
    if (count_out) *count_out = s.count;
    if (out && s.count) CK(cudaMemcpy(out, s.samples, (size_t)s.count * s.ncls * 4 * 8, cudaMemcpyDeviceToHost));
    return BTF_OK;
}

// out: [nclasses][6] = {n, sum (y - mean)^2, sum |y - mean|, sum loglik(y | mean), # cells whose target lies
// inside the [lo_pct, hi_pct] percentile band of the scored samples (np.percentile, linear interpolation),
// # cells with pred_lo <= mean_s Phi((y - mu_s) / sqrt(nu2_s)) <= pred_hi}; mean_out (optional): [Nloc, M, T]
int btf_eval_summary(btf_engine* e, int32_t slot, double lo_pct, double hi_pct, double pred_lo, double pred_hi,
                     double* out, double* mean_out) {
    EVAL_SLOT_OR_FAIL(e, slot)
    EvalSlot& s = e->eval[slot];
    if (!s.mean) return set_err(BTF_ESTATE, "the evaluator keeps no per-cell state (cell_state = 0)");
    if (s.count < 1) return set_err(BTF_ESTATE, "no sample has been scored yet");
    if (!(lo_pct >= 0.0 && lo_pct <= hi_pct && hi_pct <= 100.0)) return set_err(BTF_EINVAL, "0 <= lo_pct <= hi_pct <= 100");
    launch_eval_summary(eval_args(e, s), lo_pct, hi_pct, pred_lo, pred_hi, s.partial, s.summary, e->stream);
    e->launches += 2;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(e->stream));
    if (out) CK(cudaMemcpy(out, s.summary, (size_t)s.ncls * 6 * 8, cudaMemcpyDeviceToHost));
    if (mean_out) CK(cudaMemcpy(mean_out, s.mean, (size_t)e->nloc * e->P * 8, cudaMemcpyDeviceToHost));
    return BTF_OK;
}

// pinned host buffers for the result arrays (async device-to-host copies need them)
void* btf_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void btf_host_free(void* p) { if (p) cudaFreeHost(p); }
// page-lock an existing host allocation in place (fallback when a fresh pinned allocation fails)
int btf_host_register(void* p, size_t bytes) {
    if (!p || !bytes) return set_err(BTF_EINVAL, "bad arguments");
    cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterDefault);
    if (e != cudaSuccess) { cudaGetLastError(); return set_err(BTF_ECUDA, "cudaHostRegister: %s", cudaGetErrorString(e)); }
    return BTF_OK;
}
int btf_host_unregister(void* p) {
    if (p && cudaHostUnregister(p) != cudaSuccess) cudaGetLastError();
    return BTF_OK;
}

// Initial state drawn from the priors on the device (factor.py:230-253, 293-304, 560-563).
// init_mask bits: 1 sigma2, 2 lam2(+lam2_a), 4 nu2, 8 Tau2(+a,b,c), 16 W, 32 V, 64 R
int btf_init_state(btf_engine* e, int32_t init_mask) {
    if (!e) return set_err(BTF_EINVAL, "null engine");
    CK(cudaSetDevice(e->cfg.device));
    const btf_config& c = e->cfg;
    cudaStream_t st = e->stream;
    if (init_mask & 7) { launch_init_scalars(e->scal, c.seed, init_mask & 7, c.sigma2_a, c.sigma2_b, c.nu2_a, c.nu2_b, st); e->launches++; }
    if (init_mask & 8) { launch_init_tau2(e->Tau2, e->Tau2_a, e->Tau2_b, e->Tau2_c, (size_t)e->M * e->RD, c.seed, st); e->launches++; }
    if (init_mask & 16) { launch_init_W(e->W, e->N, e->K, e->scal, c.seed, st); e->launches++; }
    if (init_mask & 32) {
        // one prior MVN draw per column: the banded solver with zero statistics (factor.py:235-242)
        BandSolveArgs ba;
        memset(&ba, 0, sizeof(ba));
        ba.stats = nullptr; ba.nsplit = 0; ba.split_stride = 0;
        ba.col_begin = 0; ba.ncols_loc = e->M; ba.T = e->T; ba.K = e->K; ba.order = e->order; ba.RD = e->RD;
        ba.homoskedastic = 0; ba.scal = e->scal; ba.Tau2 = e->Tau2;
        ba.pm_ptr = e->pm_ptr; ba.pm_row = e->pm_row; ba.pm_coef = e->pm_coef;
        ba.V = e->V; ba.z_inject = nullptr; ba.seed = c.seed ^ 0x5bd1e995u;
        double *wl = nullptr, *wy = nullptr;
        const bool tmp = e->Mloc < e->M;   // sharded engines own a smaller workspace
        if (tmp) {
            CK(cudaMalloc((void**)&wl, (size_t)e->M * e->wL_stride * sizeof(double)));
            CK(cudaMalloc((void**)&wy, (size_t)e->M * e->wy_stride * sizeof(double)));
        }
        ba.work_L = tmp ? wl : e->work_L; ba.work_y = tmp ? wy : e->work_y;
        ba.work_L_stride = e->wL_stride; ba.work_y_stride = e->wy_stride;
        ba.force_psd = c.force_psd; ba.attempts = c.force_psd_attempts; ba.eps = c.force_psd_eps;
        ba.force_scalar = e->env.band_scalar;
        launch_band_solve(ba, st);
        launch_clip(e->V, (size_t)e->P * e->K, -10.0, 10.0, st);
        e->launches += 2;
        CK(cudaStreamSynchronize(st));
        if (wl) cudaFree(wl);
        if (wy) cudaFree(wy);
    }
    if ((init_mask & 64) && e->Rdisp) {
        // R = exp(N(0, rstdev)) + 1  (factor.py:560-563), drawn on the host side of the ABI
        const size_t rn = (size_t)e->Rn * e->Rm * e->Rt;
        std::vector<double> r(rn);
        uint64_t x = c.seed * 6364136223846793005ull + 1442695040888963407ull;
        auto u01 = [&]() { x = x * 6364136223846793005ull + 1442695040888963407ull; return ((x >> 11) + 0.5) / 9007199254740992.0; };
        for (size_t i = 0; i < rn; ++i) {
            double z = std::sqrt(-2.0 * std::log(u01())) * std::cos(6.283185307179586 * u01());
            r[i] = std::exp(c.rstdev * z) + 1.0;
        }
        CK(h2d(e->Rdisp, r.data(), rn * sizeof(double)));
    }
    CK(cudaStreamSynchronize(st));
    e->resid_valid = false;
    return check_info(e);
}

// ------------------------------------------------------------------ sampler test hooks
int btf_pg_sample(int32_t device, const double* b, const double* z, double* out, int64_t n, uint64_t seed) {
    if (!b || !z || !out || n < 1) return set_err(BTF_EINVAL, "bad arguments");
    CK(cudaSetDevice(device));
    double *db = nullptr, *dz = nullptr, *dout = nullptr;
    CK(cudaMalloc((void**)&db, n * 8)); CK(cudaMalloc((void**)&dz, n * 8)); CK(cudaMalloc((void**)&dout, n * 8));
    CK(h2d(db, b, n * 8));
    CK(h2d(dz, z, n * 8));
    launch_pg_sample(db, dz, dout, n, seed, 1ull, 0);
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(out, dout, n * 8, cudaMemcpyDeviceToHost));
    cudaFree(db); cudaFree(dz); cudaFree(dout);
    return BTF_OK;
}

int btf_rng_sample(int32_t device, int32_t kind, double param, double* out, int64_t n, uint64_t seed) {
    if (!out || n < 1) return set_err(BTF_EINVAL, "bad arguments");
    CK(cudaSetDevice(device));
    double* dout = nullptr;
    CK(cudaMalloc((void**)&dout, n * 8));
    launch_rng_sample(kind, param, dout, n, seed, 0);
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(out, dout, n * 8, cudaMemcpyDeviceToHost));
    cudaFree(dout);
    return BTF_OK;
}

// ------------------------------------------------------------------ NCCL plumbing
int btf_nccl_unique_id(char* id128) {
    if (!id128) return set_err(BTF_EINVAL, "null argument");
    if (nccl_shard_unique_id(id128)) return set_err(BTF_ENCCL, "ncclGetUniqueId failed: %s", nccl_shard_error());
    return BTF_OK;
}

int btf_nccl_init(btf_engine* e, const char* id128) {
    if (!e || !id128) return set_err(BTF_EINVAL, "null argument");
    if (e->cfg.world_size <= 1) return BTF_OK;
    CK(cudaSetDevice(e->cfg.device));
    e->shard = nccl_shard_create(id128, e->cfg.world_size, e->cfg.rank, e->N, e->M, e->cfg.row_begin, e->cfg.row_end,
                                 e->cfg.col_begin, e->cfg.col_end);
    if (!e->shard) return set_err(BTF_ENCCL, "NCCL init failed: %s", nccl_shard_error());
    // the lam2 step in its all-columns form needs every column's new Tau2: keep the chain replicated there
    e->tau_sharded = e->cfg.ref_compat_lam2 != 0;
    e->i8_decided = false;
    return BTF_OK;
}
