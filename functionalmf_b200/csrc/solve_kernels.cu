// K2: batched small dense FP64 Cholesky + MVN draw for the W rows
//     (replaces np.linalg.cholesky / cho_solve / solve_triangular, factor.py:356-362)
// K3: batched banded FP64 Cholesky + MVN draw for the V columns
//     (replaces sample_mvn_from_precision + CHOLMOD, fast_mvn.py:33-74, and the
//      kron/SpGEMM assembly of factor.py:396-408: the band is assembled on the fly
//      from the per-(j,t) statistics and the trend-filtering stencils).
#include "kernels.h"
#include <stdlib.h>

namespace btf {

// ============================================================================ K2
// One warp per row, lane = matrix row.  Left-looking Cholesky in shared memory,
// one forward and one (two right-hand sides: mean and draw) backward solve.
__global__ void __launch_bounds__(128) row_solve_kernel(RowSolveArgs a) {
    extern __shared__ double sm[];
    const int K = a.K, KS = K | 1, L = K * (K + 1) / 2, nco = L + K;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* Lm = sm + warp * (K * KS);
    const int il = blockIdx.x * 4 + warp;
    if (il >= a.nloc) return;
    const int i = a.row_begin + il;
    const int d = min(i + 1, K);
    const double scale = a.scale_from_nu2 ? 1.0 / a.scal->nu2 : 1.0;
    const double prior = 1.0 / a.scal->sigma2;
    const unsigned full = 0xffffffffu;

    double bl = 0.0;
    if (lane < d) {
        for (int c = 0; c <= lane; ++c) {
            double q = 0.0;
            for (int s = 0; s < a.nsplit; ++s) q += a.stats[s * a.split_stride + (size_t)il * nco + tri(lane, c)];
            q *= scale;
            if (c == lane) q += prior;
            Lm[lane * KS + c] = q;
        }
        for (int s = 0; s < a.nsplit; ++s) bl += a.stats[s * a.split_stride + (size_t)il * nco + L + lane];
        bl *= scale;
        if (a.diag_Q) {
            for (int c = 0; c <= lane; ++c) {
                double q = Lm[lane * KS + c];
                a.diag_Q[((size_t)i * K + lane) * K + c] = q;
                a.diag_Q[((size_t)i * K + c) * K + lane] = q;
            }
            a.diag_b[(size_t)i * K + lane] = bl;
        }
    }
    __syncwarp();

    bool ok = true;
    for (int j = 0; j < d; ++j) {
        double s = 0.0;
        if (lane >= j && lane < d) {
            s = Lm[lane * KS + j];
            for (int k = 0; k < j; ++k) s -= Lm[lane * KS + k] * Lm[j * KS + k];
        }
        double djj = __shfl_sync(full, s, j);
        if (!(djj > 0.0) || isinf(djj)) { ok = false; break; }
        double ljj = sqrt(djj);
        __syncwarp();
        if (lane == j) Lm[lane * KS + j] = ljj;
        else if (lane > j && lane < d) Lm[lane * KS + j] = s / ljj;
        __syncwarp();
    }
    if (!ok) {
        if (lane == 0) atomicAdd(&a.scal->info_w, 1);
        return;
    }

    // forward  y = L^-1 b
    double y = 0.0;
    for (int j = 0; j < d; ++j) {
        double yj = __shfl_sync(full, bl, j) / Lm[j * KS + j];
        if (lane == j) y = yj;
        if (lane > j && lane < d) bl -= Lm[lane * KS + j] * yj;
    }
    // noise
    double z = 0.0;
    if (lane < d) {
        if (a.z_inject) z = a.z_inject[(size_t)i * K + lane];
        else { Rng rng(a.seed, STREAM_W, a.scal->sweep, (uint64_t)i * K + lane); z = rng.normal(); }
    }
    // backward  x = L^-T w  for w = y (mean) and w = y + z (draw)
    double wm = y, wd = y + z, xm = 0.0, xd = 0.0;
    for (int j = d - 1; j >= 0; --j) {
        double ljj = Lm[j * KS + j];
        double xmj = __shfl_sync(full, wm, j) / ljj;
        double xdj = __shfl_sync(full, wd, j) / ljj;
        if (lane == j) { xm = xmj; xd = xdj; }
        if (lane < j) { double l = Lm[j * KS + lane]; wm -= l * xmj; wd -= l * xdj; }
    }
    if (lane < d) {
        a.W[(size_t)i * K + lane] = xd;
        if (a.diag_L)
            for (int c = 0; c <= lane; ++c) a.diag_L[((size_t)i * K + lane) * K + c] = Lm[lane * KS + c];
        if (a.diag_mean) a.diag_mean[(size_t)i * K + lane] = xm;
    }
}

void launch_row_solve(const RowSolveArgs& a, int* nblocks_out, cudaStream_t st) {
    int nb = (a.nloc + 3) / 4;
    size_t smem = (size_t)4 * a.K * (a.K | 1) * sizeof(double);
    row_solve_kernel<<<nb, 128, smem, st>>>(a);
    if (nblocks_out) *nblocks_out = nb;
}

// ============================================================================ K3
// One CTA per column.  Scalar left-looking banded Cholesky of the t-major system
// (n = T K unknowns, half-bandwidth kd = (p+1) K) with a circular shared-memory
// window of the last kd factor columns; the forward substitution is fused in as an
// extra row.  The factor is spilled to global memory in row-band form and streamed
// back in kd-row chunks for the column-oriented backward substitution (mean and
// draw together).  Cholesky failure -> jitter eps, 10 eps, ... (fast_mvn.py:62-68).
__global__ void band_solve_kernel(BandSolveArgs a) {
    extern __shared__ double sm[];
    const int K = a.K, T = a.T, q = a.order + 1, kd = q * K, n = T * K;
    const int L = K * (K + 1) / 2, nco = L + K, LS = kd + 1, NB = kd + 1;
    const int tid = threadIdx.x, NT = blockDim.x;
    const int jl = blockIdx.x, jg = a.col_begin + jl;

    double* Lw = sm;                           // [kd][kd+1]   (reused as chunk buffer in the backward pass)
    double* yw = Lw + (size_t)kd * LS;         // [kd] (+ chunk y/z: 2*kd)
    double* ychunk = yw + kd;                  // [kd]
    double* zchunk = ychunk + kd;              // [kd]
    double* dchunk = zchunk + kd;              // [kd]
    double* Ablk = dchunk + kd;                // [L+K]
    double* Pband = Ablk + nco;                // [T][q+1]
    double* linv = Pband + (size_t)T * (q + 1);   // [RD]
    double* misc = linv + a.RD;                // [8]
    __shared__ int fail_flag;

    const double scale = a.homoskedastic ? 1.0 / a.scal->nu2 : 1.0;
    const double lam2 = a.scal->lam2;
    for (int r = tid; r < a.RD; r += NT) {
        double pv = 1.0 / (lam2 * a.Tau2[(size_t)jg * a.RD + r]);
        if (a.prior_clip > 0.0) pv = fmin(fmax(pv, a.prior_clip), 1.0 / a.prior_clip);
        linv[r] = pv;
    }
    if (tid == 0) fail_flag = 0;
    __syncthreads();
    for (int e = tid; e < T * (q + 1); e += NT) {
        double s = 0.0;
        for (int x = a.pm_ptr[e]; x < a.pm_ptr[e + 1]; ++x) s += a.pm_coef[x] * linv[a.pm_row[x]];
        Pband[e] = s;
    }

    double* Lrow = a.work_L + (size_t)jl * a.work_L_stride;
    double* yg = a.work_y + (size_t)jl * a.work_y_stride;      // [y (n) | 1 / diag(L) (n)]
    const bool have_stats = a.stats != nullptr;     // nullptr: prior-only system (V initialisation)
    const double* stats0 = have_stats ? a.stats + (size_t)jg * T * nco : nullptr;
    const int mblk = tid / K;
    const bool on_kdiag = (tid % K) == 0;

    double jitter = 0.0, eps = a.eps;
    int attempt = 0;
    bool failed = false;

    while (true) {
        // ---- factorisation + forward substitution
        // statistics of block t+1 are fetched while block t is being factorised: the raw loads
        // (two split partials) stay in registers and are only combined at the next block boundary
        double preA[4], preB[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            int c = tid + u * NT;
            preA[u] = 0.0; preB[u] = 0.0;
            if (c < nco && have_stats) {
                preA[u] = stats0[c];
                if (a.nsplit > 1) preB[u] = stats0[a.split_stride + c];
                for (int s = 2; s < a.nsplit; ++s) preA[u] += stats0[s * a.split_stride + c];
            }
        }
        __syncthreads();
        int t = 0, k = 0;
        bool broke = false;
        for (int j = 0; j < n; ++j) {
            if (k == 0) {
#pragma unroll
                for (int u = 0; u < 4; ++u) { int c = tid + u * NT; if (c < nco) Ablk[c] = (preA[u] + preB[u]) * scale; }
                __syncthreads();
                if (t + 1 < T && have_stats) {
                    const double* nx = stats0 + (size_t)(t + 1) * nco;
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        int c = tid + u * NT;
                        if (c < nco) {
                            preA[u] = nx[c];
                            preB[u] = a.nsplit > 1 ? nx[a.split_stride + c] : 0.0;
                            for (int s = 2; s < a.nsplit; ++s) preA[u] += nx[s * a.split_stride + c];
                        }
                    }
                }
            }
            double s = 0.0, q0 = 0.0;
            bool valid = false;
            // Dot products over the window columns c in [cs, j): column c lives in slot c % kd
            // and consecutive columns are kd doubles apart (slot + 1, offset - 1), so the
            // range splits into at most two contiguous runs; four independent accumulators
            // keep the shared-memory loads and DFMAs pipelined.
            if (tid <= kd + 1) {
                const bool rhs = tid == kd + 1;
                const int off = rhs ? 0 : tid;
                const int i = j + off;
                if (rhs || i < n) {
                    valid = true;
                    if (rhs) {
                        q0 = Ablk[L + k];
                    } else {
                        if (k + tid < K) q0 = Ablk[tri(k + tid, k)];
                        if (on_kdiag && t + mblk < T) q0 += Pband[t * (q + 1) + mblk];
                        if (tid == 0) q0 += jitter;
                    }
                    // All threads walk the SAME window columns c = cbeg .. j-1 in lock step, so
                    // L[j][c] is a shared-memory broadcast and L[i][c] is a unit-stride read
                    // (thread-private start columns would put every lane on one bank).  Row
                    // i = j + off only couples to columns with (j - c) + off <= kd.
                    int cbeg = j - kd; if (cbeg < 0) cbeg = 0;
                    int len = j - cbeg;
                    int s0 = cbeg % kd;
                    int o = j - cbeg;                      // offset of L[j][c] inside its slot row
                    const int lim = kd - off;              // active while o <= lim
                    double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll 1
                    for (int seg = 0; seg < 2 && len > 0; ++seg) {
                        const int run = min(len, kd - s0);
                        const double* pl = Lw + s0 * LS + o;              // L[j][c] at pl[0], L[i][c] at pl[off]
                        const double* py = yw + s0;
                        int x = 0;
                        if (!rhs) {
                            for (; x + 4 <= run; x += 4) {
                                const double l0 = (o - x <= lim) ? pl[off] : 0.0;
                                const double l1 = (o - x - 1 <= lim) ? pl[kd + off] : 0.0;
                                const double l2 = (o - x - 2 <= lim) ? pl[2 * kd + off] : 0.0;
                                const double l3 = (o - x - 3 <= lim) ? pl[3 * kd + off] : 0.0;
                                a0 += l0 * pl[0];
                                a1 += l1 * pl[kd];
                                a2 += l2 * pl[2 * kd];
                                a3 += l3 * pl[3 * kd];
                                pl += 4 * kd;
                            }
                            for (; x < run; ++x) { if (o - x <= lim) a0 += pl[off] * pl[0]; pl += kd; }
                        } else {
                            for (; x + 4 <= run; x += 4) {
                                a0 += pl[0] * py[x];
                                a1 += pl[kd] * py[x + 1];
                                a2 += pl[2 * kd] * py[x + 2];
                                a3 += pl[3 * kd] * py[x + 3];
                                pl += 4 * kd;
                            }
                            for (; x < run; ++x) { a0 += pl[0] * py[x]; pl += kd; }
                        }
                        o -= run; len -= run; s0 = 0;
                    }
                    s = q0 - ((a0 + a1) + (a2 + a3));
                }
            }
            if (tid == 0) {
                if (!(s > 0.0) || isinf(s)) fail_flag = 1;
                else { const double lj = sqrt(s); misc[0] = lj; misc[1] = 1.0 / lj; }
            }
            __syncthreads();
            if (fail_flag) { broke = true; break; }
            const double ljj = misc[0], rinv = misc[1];
            const int slot_j = j % kd;
            if (tid <= kd) {
                double val = tid == 0 ? ljj : (valid ? s * rinv : 0.0);
                Lw[slot_j * LS + tid] = val;
                if (valid) {
                    Lrow[(size_t)(j + tid) * LS + kd - tid] = val;
                    if (a.diag_band) a.diag_band[((size_t)jl * n + j + tid) * LS + kd - tid] = q0;
                }
                if (tid == 0) yg[n + j] = rinv;
            } else if (tid == kd + 1) {
                double yj = s * rinv;
                yw[slot_j] = yj;
                yg[j] = yj;
            }
            __syncthreads();
            if (++k == K) { k = 0; ++t; }
        }
        if (!broke) break;
        // ---- jitter retry (all threads take the same branch: fail_flag is block-uniform)
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

    // ---- backward substitution  x = L^-T w, w = y (mean) and y + z (draw)
    double* Lc = Lw;                       // chunk of kd factor rows
    double* xs = misc + 2;                 // [2][2]
    const unsigned long long sweep = a.scal->sweep;
    auto noise = [&](int i) -> double {
        if (a.z_inject) return a.z_inject[(size_t)jg * n + i];
        Rng rng(a.seed, STREAM_V, sweep, (uint64_t)jg * n + i);
        return rng.normal();
    };
    int myrow = -1;
    double wm = 0.0, wd = 0.0;
    if (tid < NB && n - 1 >= tid) {
        myrow = tid + NB * ((n - 1 - tid) / NB);
        wm = yg[myrow];
        wd = wm + noise(myrow);
    }
    double* Vout = a.V + (size_t)jg * n;
    int par = 0;
    for (int jc = n - 1; jc >= 0; jc -= kd) {
        const int lo = jc - kd + 1 < 0 ? 0 : jc - kd + 1;
        const int cnt = jc - lo + 1;
        __syncthreads();
        {   // batched global -> shared copy of the chunk (8 independent loads in flight per thread)
            const double* src = Lrow + (size_t)lo * LS;
            const int total = cnt * LS;
            for (int base = tid; base < total; base += NT * 8) {
                double r8[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) { int e = base + u * NT; r8[u] = e < total ? src[e] : 0.0; }
#pragma unroll
                for (int u = 0; u < 8; ++u) { int e = base + u * NT; if (e < total) Lc[e] = r8[u]; }
            }
        }
        for (int e = tid; e < cnt; e += NT) {
            int i = lo - NB + e;
            if (i >= 0) { double yv = yg[i]; ychunk[e] = yv; zchunk[e] = noise(i); }
            dchunk[e] = yg[n + lo + e];
        }
        __syncthreads();
        for (int j = jc; j >= lo; --j) {
            const int jj = j - lo;
            if (tid < NB && myrow == j) {
                const double rj = dchunk[jj];
                const double xm = wm * rj, xd = wd * rj;
                xs[par * 2] = xm; xs[par * 2 + 1] = xd;
                Vout[j] = xd;
                if (a.diag_mean) a.diag_mean[(size_t)jg * n + j] = xm;
                myrow = j - NB;
                if (myrow >= 0) { wm = ychunk[jj]; wd = wm + zchunk[jj]; }
            }
            __syncthreads();
            if (tid < NB && myrow >= 0 && myrow < j && myrow >= j - kd) {
                const double l = Lc[jj * LS + kd - (j - myrow)];
                wm -= l * xs[par * 2];
                wd -= l * xs[par * 2 + 1];
            }
            par ^= 1;
        }
    }
    __syncthreads();
    if (a.diag_chol) {
        for (size_t e = tid; e < (size_t)n * LS; e += NT) a.diag_chol[(size_t)jl * n * LS + e] = Lrow[e];
    }

    // ---- nu2 by-product: sum_t v_t^T A_t v_t - 2 v_t . b_t with the UNSCALED statistics
    if (a.resid_partials && have_stats) {
        double accum = 0.0;
        for (int c = tid; c < nco; c += NT) {
            int k1 = 0, k2 = 0;
            double wgt = -2.0;
            if (c < L) {
                k1 = (int)((sqrt(8.0 * c + 1.0) - 1.0) * 0.5);
                while (k1 * (k1 + 1) / 2 > c) --k1;
                while ((k1 + 1) * (k1 + 2) / 2 <= c) ++k1;
                k2 = c - k1 * (k1 + 1) / 2;
                wgt = k1 == k2 ? 1.0 : 2.0;
            } else {
                k1 = c - L;
            }
            for (int t = 0; t < T; ++t) {
                const double* sb = stats0 + (size_t)t * nco + c;
                const double* v = Vout + (size_t)t * K;
                double sv = 0.0;
                for (int s = 0; s < a.nsplit; ++s) sv += sb[s * a.split_stride];
                accum += wgt * sv * v[k1] * (c < L ? v[k2] : 1.0);
            }
        }
        double tot = block_sum(accum, misc + 8);
        if (tid == 0) a.resid_partials[jl] = tot;
    }
}

void launch_band_solve(const BandSolveArgs& a, cudaStream_t st) {
    if (!a.force_scalar && launch_band_solve_lookahead(a, st)) return;    // blocked look-ahead kernel (band_lookahead.cu): K <= 32, order <= 3
    const int q = a.order + 1, kd = q * a.K, L = a.K * (a.K + 1) / 2, nco = L + a.K;
    int nt = ((kd + 2 + 31) / 32) * 32;
    int nt2 = (((nco + 3) / 4 + 31) / 32) * 32;
    if (nt2 > nt) nt = nt2;
    size_t smem = ((size_t)kd * (kd + 1) + 4 * (size_t)kd + nco + (size_t)a.T * (q + 1) + a.RD + 8 + 40) * sizeof(double);
    static PerDeviceMax max_set;
    if (smem > 48 * 1024 && max_set.raise(smem))
        cudaFuncSetAttribute(band_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    band_solve_kernel<<<a.ncols_loc, nt, smem, st>>>(a);
}

}  // namespace btf
