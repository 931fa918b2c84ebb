// K0 (replicate pre-reduction), K1 (NaN-masked sufficient-statistic contractions
// on the FP64 tensor pipe) and the nu2 residual pass.
//
// K1 replaces the per-row / per-column Python loops of the reference
// (factor.py:333-360 for W, factor.py:378-401 for V; the latter builds
// kron(W, I_T)[~missing] and two sparse products per column).  Both are the same
// GEMM-shaped contraction
//     out[m, c] = sum_k  A[m, k] * Z[k, c]
// with a *generated* right operand: Z[k, (k1,k2)] = F[k,k1] F[k,k2] for the packed
// lower triangle (L = K(K+1)/2 columns, weight operand A = counts or omega) and
// Z[k, L + k1] = F[k,k1] (K columns, A = replicate sums / kappa).
//   row statistics  (trans = false): m = row i, k = p = (j,t), F = V
//   col statistics  (trans = true ): m = p = (j,t), k = row i, F = W
// The data operand is read once from HBM with coalesced 16-byte cp.async into a
// two-stage shared-memory ring; Z tiles are generated on chip from the small
// factor tile; products run as mma.sync.m8n8k4.f64 (DMMA) -- tcgen05 has no FP64
// kind, so this is the B200 FP64 tensor path.
#include "stats_common.cuh"
#include <stdio.h>
#include <algorithm>
#include <stdlib.h>

namespace btf {

// ------------------------------------------------------------------ K0
__global__ void prereduce_gaussian_kernel(const double* __restrict__ Y, int rows, int P, int R,
                                          uint8_t* __restrict__ cnt, double* __restrict__ S, long long ld,
                                          double* __restrict__ partials) {
    __shared__ double sh[64];
    double ss = 0.0, no = 0.0;
    long long total = (long long)rows * P;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        int i = (int)(e / P), p = (int)(e - (long long)i * P);
        const double* y = Y + e * R;
        double s = 0.0;
        int c = 0;
        for (int r = 0; r < R; ++r) {
            double v = y[r];
            if (v == v) { s += v; ss += v * v; ++c; }
        }
        cnt[(long long)i * ld + p] = (uint8_t)c;
        S[(long long)i * ld + p] = s;
        no += (double)c;
    }
    double a = block_sum(ss, sh);
    double b = block_sum(no, sh + 32);
    if (threadIdx.x == 0) { partials[2 * blockIdx.x] = a; partials[2 * blockIdx.x + 1] = b; }
}

void launch_prereduce_gaussian(const double* Y, int rows, int P, int R, uint8_t* cnt, double* S,
                               long long ld, double* partials, int* nblocks_out, cudaStream_t st) {
    long long total = (long long)rows * P;
    int nb = (int)((total + 255) / 256);
    if (nb > 148 * 16) nb = 148 * 16;
    if (nb < 1) nb = 1;
    prereduce_gaussian_kernel<<<nb, 256, 0, st>>>(Y, rows, P, R, cnt, S, ld, partials);
    *nblocks_out = nb;
}

__global__ void prereduce_binomial_kernel(const double* __restrict__ Y, const double* __restrict__ Nt,
                                          int rows, int P, uint8_t* __restrict__ obs,
                                          double* __restrict__ kappa, double* __restrict__ ntr, long long ld) {
    long long total = (long long)rows * P;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        int i = (int)(e / P), p = (int)(e - (long long)i * P);
        double y = Y[e], n = Nt[e];
        bool ok = (y == y) && (n == n);
        long long o = (long long)i * ld + p;
        obs[o] = ok ? 1 : 0;
        kappa[o] = ok ? (y - 0.5 * n) : 0.0;
        ntr[o] = ok ? n : 0.0;
    }
}

void launch_prereduce_binomial(const double* Y, const double* Nt, int rows, int P, uint8_t* obs,
                               double* kappa, double* ntr, long long ld, cudaStream_t st) {
    long long total = (long long)rows * P;
    int nb = (int)((total + 255) / 256);
    if (nb > 148 * 16) nb = 148 * 16;
    if (nb < 1) nb = 1;
    prereduce_binomial_kernel<<<nb, 256, 0, st>>>(Y, Nt, rows, P, obs, kappa, ntr, ld);
}

// Known per-cell noise variances (the reference's heteroskedastic Gaussian branch, factor.py:345-346 and 390-391
// with an [N, M, T] nu2): weight w = cnt / nu2 and right-hand side S / nu2 of the statistics, both 0 where nothing is
// observed or nu2 = +inf (such a cell counts as missing); w = s = nullptr: no weights (the constrained Gaussian model,
// whose GASS steps read the variances).  Observed cells whose variance is NaN or <= 0 are counted.
__global__ void nu2_weights_kernel(const double* __restrict__ nu2, long long lds, int rows, int P,
                                   const uint8_t* __restrict__ cnt, const double* __restrict__ S, long long ld,
                                   double* __restrict__ keep, double* __restrict__ w, double* __restrict__ s,
                                   unsigned long long* __restrict__ nbad) {
    unsigned bad = 0;
    long long total = (long long)rows * P;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        int i = (int)(e / P), p = (int)(e - (long long)i * P);
        const double v = nu2[(long long)i * lds + p];
        const long long o = (long long)i * ld + p;
        const double c = (double)cnt[o];
        const bool on = c > 0.0 && v < INFINITY;
        bad += (c > 0.0 && !(v > 0.0)) ? 1u : 0u;
        if (w) {
            w[o] = on ? c / v : 0.0;
            s[o] = on ? S[o] / v : 0.0;
        }
        if (keep) keep[o] = v;
    }
    for (int d = 16; d > 0; d >>= 1) bad += __shfl_down_sync(0xffffffffu, bad, d);
    if ((threadIdx.x & 31) == 0 && bad) atomicAdd(nbad, (unsigned long long)bad);
}

void launch_nu2_weights(const double* nu2, long long lds, int rows, int P, const uint8_t* cnt, const double* S,
                        long long ld, double* keep, double* w, double* s, unsigned long long* nbad, cudaStream_t st) {
    long long total = (long long)rows * P;
    int nb = (int)((total + 255) / 256);
    if (nb > 148 * 16) nb = 148 * 16;
    if (nb < 1) nb = 1;
    nu2_weights_kernel<<<nb, 256, 0, st>>>(nu2, lds, rows, P, cnt, S, ld, keep, w, s, nbad);
}

__global__ void reduce_add_kernel(const double* __restrict__ src, int n, int stride, double* dst) {
    __shared__ double sh[32];
    double v = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) v += src[(long long)i * stride];
    v = block_sum(v, sh);
    if (threadIdx.x == 0) dst[0] += v;
}
void launch_reduce_add(const double* src, int n, int stride, double* dst, cudaStream_t st) {
    reduce_add_kernel<<<1, 256, 0, st>>>(src, n, stride, dst);
}

// ------------------------------------------------------------------ K1
// Column tiles (8 generated columns each): nct_z tiles of packed products, then nct_f
// tiles of plain factor columns.  Warp column-group wc owns product tiles
// [wc*ZPW, (wc+1)*ZPW) and factor tiles [wc*FPW, (wc+1)*FPW).  With KFIX > 0 all of this
// is compile-time: the inner loop has no branches and out-of-range tile slots compute
// into accumulators that are never stored.
template <int BM, int WR, int WC, int CTM, int KC, bool TRANS, typename WT, int KFIX>
__global__ void __launch_bounds__(32 * WR* WC, 1) stats_kernel(StatsKArgs a) {
    constexpr int NT = 32 * WR * WC;
    constexpr int RT = BM / 8 / WR;
    constexpr bool FIX = KFIX > 0;
    using G = TileGeom<TRANS, WT, BM, KC>;
    extern __shared__ __align__(16) unsigned char smem[];

    const int K = FIX ? KFIX : a.K;
    const int L = K * (K + 1) / 2;
    const int nct_z = cdiv(L, 8), nct_f = cdiv(K, 8);
    const int ZPW = cdiv(nct_z, WC), FPW = cdiv(nct_f, WC);     // ZPW + FPW <= CTM (checked on the host)
    const int zw = a.zw;
    const int ncw = (nct_z + nct_f) * 8;
    constexpr int CZ = FIX ? cdiv((cdiv(KFIX * (KFIX + 1) / 2, 8) + cdiv(KFIX, 8)) * 8, 32) : cdiv(CTM * WC * 8, 32);
    const int fbytes = ((KC * K * 8) + 15) & ~15;
    const int stage_bytes = G::WBYTES + G::SBYTES + fbytes;
    unsigned char* stage0 = smem;
    double* ztile = reinterpret_cast<double*>(smem + 2 * stage_bytes);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wr = warp / WC, wc = warp % WC;
    const int m0 = blockIdx.x * BM;
    const int split = blockIdx.y;
    const int c_begin = split * a.chunks_per_split;
    const int c_end = min(a.nchunks, c_begin + a.chunks_per_split);

    // which generated column(s) this lane fills during Z generation
    // code: bits 31..30 type (0 zero, 1 product, 2 copy), k1 = bits 8..15, k2 = bits 0..7
    int zcode[CZ];
#pragma unroll
    for (int q = 0; q < CZ; ++q) {
        int c = lane + 32 * q;
        int code = 0;
        if (c < ncw) {
            if (c < nct_z * 8) {
                if (c < L) {
                    int k1 = (int)((sqrt(8.0 * c + 1.0) - 1.0) * 0.5);
                    while (k1 * (k1 + 1) / 2 > c) --k1;
                    while ((k1 + 1) * (k1 + 2) / 2 <= c) ++k1;
                    int k2 = c - k1 * (k1 + 1) / 2;
                    code = (1 << 30) | (k1 << 8) | k2;
                }
            } else {
                int cf = c - nct_z * 8;
                if (cf < K) code = (2 << 30) | (cf << 8);
            }
        }
        zcode[q] = code;
    }

    double acc[RT][CTM][2];
#pragma unroll
    for (int r = 0; r < RT; ++r)
#pragma unroll
        for (int c = 0; c < CTM; ++c) acc[r][c][0] = acc[r][c][1] = 0.0;

    auto load_chunk = [&](int stage, int chunk) {
        unsigned char* base = stage0 + stage * stage_bytes;
        WT* wtile = reinterpret_cast<WT*>(base);
        double* stile = reinterpret_cast<double*>(base + G::WBYTES);
        double* ftile = reinterpret_cast<double*>(base + G::WBYTES + G::SBYTES);
        const int k0 = chunk * KC;
        const WT* wsrc = reinterpret_cast<const WT*>(a.wt);
        if (!TRANS) {
            // rows m0..m0+BM of the data, columns k0..k0+KC
            constexpr int WP = KC * (int)sizeof(WT) / 16;   // 16-byte pieces per row
            for (int e = tid; e < BM * WP; e += NT) {
                int r = e / WP, q = e % WP;
                cp_async16(reinterpret_cast<unsigned char*>(wtile + r * G::WSTR) + 16 * q,
                           reinterpret_cast<const unsigned char*>(wsrc + (long long)(m0 + r) * a.ld + k0) + 16 * q);
            }
            constexpr int SP = KC / 2;
            for (int e = tid; e < BM * SP; e += NT) {
                int r = e / SP, q = e % SP;
                cp_async16(stile + r * G::SSTR + 2 * q, a.sv + (long long)(m0 + r) * a.ld + k0 + 2 * q);
            }
        } else {
            // rows k0..k0+KC of the data, columns m0..m0+BM
            constexpr int WP = BM * (int)sizeof(WT) / 16;
            for (int e = tid; e < KC * WP; e += NT) {
                int r = e / WP, q = e % WP;
                cp_async16(reinterpret_cast<unsigned char*>(wtile + r * G::WSTR) + 16 * q,
                           reinterpret_cast<const unsigned char*>(wsrc + (long long)(k0 + r) * a.ld + m0) + 16 * q);
            }
            constexpr int SP = BM / 2;
            for (int e = tid; e < KC * SP; e += NT) {
                int r = e / SP, q = e % SP;
                cp_async16(stile + r * G::SSTR + 2 * q, a.sv + (long long)(k0 + r) * a.ld + m0 + 2 * q);
            }
        }
        // factor rows k0..k0+KC (contiguous KC*K doubles)
        const double* fsrc = a.F + (long long)k0 * K;
        for (int e = tid; e < (KC * K) / 2; e += NT) cp_async16(ftile + 2 * e, fsrc + 2 * e);
    };

    // per-warp column offsets of the tile slots inside a Z row
    const int zoff_z = wc * ZPW * 8 + (lane >> 2);
    const int zoff_f = (nct_z + wc * FPW) * 8 + (lane >> 2);

    if (c_begin < c_end) load_chunk(0, c_begin);
    cp_async_commit();

    for (int c = c_begin; c < c_end; ++c) {
        const int stg = (c - c_begin) & 1;
        if (c + 1 < c_end) load_chunk(stg ^ 1, c + 1);
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();

        unsigned char* base = stage0 + stg * stage_bytes;
        const WT* wtile = reinterpret_cast<const WT*>(base);
        const double* stile = reinterpret_cast<const double*>(base + G::WBYTES);
        const double* ftile = reinterpret_cast<const double*>(base + G::WBYTES + G::SBYTES);

        // ---- generate the Z tile [KC][zw] from the factor tile
        for (int k = warp; k < KC; k += NT / 32) {
            const double* fr = ftile + k * K;
#pragma unroll
            for (int q = 0; q < CZ; ++q) {
                int cc = lane + 32 * q;
                if (cc < ncw) {
                    int code = zcode[q];
                    int ty = (unsigned)code >> 30;
                    double v = 0.0;
                    if (ty == 1) v = fr[(code >> 8) & 0xff] * fr[code & 0xff];
                    else if (ty == 2) v = fr[(code >> 8) & 0xff];
                    ztile[k * zw + cc] = v;
                }
            }
        }
        __syncthreads();

        // ---- DMMA over the chunk
#pragma unroll 2
        for (int kk = 0; kk < KC / 4; ++kk) {
            const int kl = kk * 4 + (lane & 3);
            double aw[RT], as[RT];
#pragma unroll
            for (int r = 0; r < RT; ++r) {
                const int ml = (wr * RT + r) * 8 + (lane >> 2);
                if (!TRANS) {
                    aw[r] = (double)wtile[ml * G::WSTR + kl];
                    as[r] = stile[ml * G::SSTR + kl];
                } else {
                    aw[r] = (double)wtile[kl * G::WSTR + ml];
                    as[r] = stile[kl * G::SSTR + ml];
                }
            }
            const double* zrow = ztile + kl * zw;
            if (FIX) {
#pragma unroll
                for (int ci = 0; ci < CTM; ++ci) {
                    // compile-time operand choice: the first ZPW slots are product tiles
                    const bool isz = ci < ZPW;
                    const double b = isz ? zrow[zoff_z + ci * 8] : zrow[zoff_f + (ci - ZPW) * 8];
#pragma unroll
                    for (int r = 0; r < RT; ++r) dmma(acc[r][ci][0], acc[r][ci][1], isz ? aw[r] : as[r], b);
                }
            } else {
#pragma unroll
                for (int ci = 0; ci < CTM; ++ci) {
                    const bool isz = ci < ZPW;
                    const int tl = isz ? wc * ZPW + ci : wc * FPW + (ci - ZPW);
                    if (ci < ZPW + FPW && tl < (isz ? nct_z : nct_f)) {
                        const double b = isz ? zrow[zoff_z + ci * 8] : zrow[zoff_f + (ci - ZPW) * 8];
#pragma unroll
                        for (int r = 0; r < RT; ++r) dmma(acc[r][ci][0], acc[r][ci][1], isz ? aw[r] : as[r], b);
                    }
                }
            }
        }
        __syncthreads();
    }
    cp_async_wait<0>();

    // ---- epilogue: packed lower triangle then the K linear terms
    double* out = a.out + (long long)split * a.out_split_stride;
    const int nco = L + K;
#pragma unroll
    for (int r = 0; r < RT; ++r) {
        const int m = m0 + (wr * RT + r) * 8 + (lane >> 2);
        if (m < a.m_valid) {
#pragma unroll
            for (int ci = 0; ci < CTM; ++ci) {
                const bool isz = ci < ZPW;
                const int tl = isz ? wc * ZPW + ci : wc * FPW + (ci - ZPW);
                if (ci < ZPW + FPW && tl < (isz ? nct_z : nct_f)) {
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int cc = tl * 8 + (lane & 3) * 2 + h;
                        int oc = -1;
                        if (isz) { if (cc < L) oc = cc; }
                        else if (cc < K) oc = L + cc;
                        if (oc >= 0) out[(long long)m * nco + oc] = acc[r][ci][h];
                    }
                }
            }
        }
    }
}

// Overlapped variant (compile-time K only): the Z tile of chunk c+1 is generated INSIDE the
// DMMA loop of chunk c (four rows per k-step, spread over the 8 warps), from a factor tile
// that is prefetched two chunks ahead; Z is double buffered.  The tensor pipe no longer idles
// during Z generation and one barrier per chunk replaces three.
// UNI: the product and factor tiles form ONE list that is dealt to the column warps in runs of
// CTM tiles (K = 32: 70 tiles over 8 warps -> 9 per warp, 2 idle slots instead of 10).  Slots
// whose tile index can exceed the product range are "late" slots: they are product tiles for
// every warp but the last one, whose late slots are factor tiles (or idle).
// NH > 1 (implies UNI): the column tiles are split into NH parts handled by different CTAs
// (blockIdx.z) that share the data tile through L2; each CTA generates only its part of Z, so a
// twice as tall row tile fits and the generation / barrier cost per DMMA halves (K = 32).
template <int BM, int WR, int WC, int CTM, int KC, bool TRANS, typename WT, int KFIX, bool UNI, int NH>
__global__ void __launch_bounds__(32 * WR* WC, 1) stats_kernel_ovl(StatsKArgs a) {
    static_assert(WR * WC == 8, "Z generation inside the DMMA loop is laid out for 8 warps");
    static_assert(NH == 1 || UNI, "column parts use the unified tile list");
    constexpr int NT = 32 * WR * WC;
    constexpr int RT = BM / 8 / WR;
    using G = TileGeom<TRANS, WT, BM, KC>;
    extern __shared__ __align__(16) unsigned char smem[];

    constexpr int K = KFIX, L = K * (K + 1) / 2;
    constexpr int nct_z = cdiv(L, 8), nct_f = cdiv(K, 8);
    constexpr int ZPW = cdiv(nct_z, WC), FPW = cdiv(nct_f, WC);
    constexpr int nct = nct_z + nct_f;
    constexpr int TP = cdiv(nct, NH);                    // column tiles per part
    const int part = NH > 1 ? blockIdx.z : 0;
    const int gcol0 = part * TP * 8;                     // first global generated column of this part
    const int ncw = (min(nct, (part + 1) * TP) - part * TP) * 8;   // generated columns held by this CTA
    constexpr int CZ = cdiv(TP * 8, 32), CZH = (CZ + 1) / 2;
    constexpr int fbytes = ((KC * K * 8) + 15) & ~15;
    constexpr int dbytes = G::WBYTES + G::SBYTES;
    const int zw = a.zw;
    unsigned char* data0 = smem;                                   // [2][dbytes]
    unsigned char* f0 = smem + 2 * dbytes;                         // [3][fbytes]
    double* z0 = reinterpret_cast<double*>(smem + 2 * dbytes + 3 * fbytes);   // [2][KC][zw]
    const int zstride = KC * zw;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wr = warp / WC, wc = warp % WC;
    const int m0 = blockIdx.x * BM;
    const int split = blockIdx.y;
    const int c_begin = split * a.chunks_per_split;
    const int c_end = min(a.nchunks, c_begin + a.chunks_per_split);

    int zcode[CZ];
#pragma unroll
    for (int q = 0; q < CZ; ++q) {
        const int cl = lane + 32 * q;                    // local column of this CTA's Z tile
        const int c = gcol0 + cl;                        // global generated column
        int code = 0;
        if (cl < ncw) {
            if (c < nct_z * 8) {
                if (c < L) {
                    int k1 = (int)((sqrt(8.0 * c + 1.0) - 1.0) * 0.5);
                    while (k1 * (k1 + 1) / 2 > c) --k1;
                    while ((k1 + 1) * (k1 + 2) / 2 <= c) ++k1;
                    int k2 = c - k1 * (k1 + 1) / 2;
                    code = (1 << 30) | (k1 << 8) | k2;
                }
            } else {
                int cf = c - nct_z * 8;
                if (cf < K) code = (2 << 30) | (cf << 8);
            }
        }
        zcode[q] = code;
    }

    double acc[RT][CTM][2];
#pragma unroll
    for (int r = 0; r < RT; ++r)
#pragma unroll
        for (int c = 0; c < CTM; ++c) acc[r][c][0] = acc[r][c][1] = 0.0;

    auto load_data = [&](int stage, int chunk) {
        unsigned char* base = data0 + stage * dbytes;
        WT* wtile = reinterpret_cast<WT*>(base);
        double* stile = reinterpret_cast<double*>(base + G::WBYTES);
        const int k0 = chunk * KC;
        const WT* wsrc = reinterpret_cast<const WT*>(a.wt);
        if (!TRANS) {
            constexpr int WP = KC * (int)sizeof(WT) / 16;
            for (int e = tid; e < BM * WP; e += NT) {
                int r = e / WP, q = e % WP;
                cp_async16(reinterpret_cast<unsigned char*>(wtile + r * G::WSTR) + 16 * q,
                           reinterpret_cast<const unsigned char*>(wsrc + (long long)(m0 + r) * a.ld + k0) + 16 * q);
            }
            constexpr int SP = KC / 2;
            for (int e = tid; e < BM * SP; e += NT) {
                int r = e / SP, q = e % SP;
                cp_async16(stile + r * G::SSTR + 2 * q, a.sv + (long long)(m0 + r) * a.ld + k0 + 2 * q);
            }
        } else {
            constexpr int WP = BM * (int)sizeof(WT) / 16;
            for (int e = tid; e < KC * WP; e += NT) {
                int r = e / WP, q = e % WP;
                cp_async16(reinterpret_cast<unsigned char*>(wtile + r * G::WSTR) + 16 * q,
                           reinterpret_cast<const unsigned char*>(wsrc + (long long)(k0 + r) * a.ld + m0) + 16 * q);
            }
            constexpr int SP = BM / 2;
            for (int e = tid; e < KC * SP; e += NT) {
                int r = e / SP, q = e % SP;
                cp_async16(stile + r * G::SSTR + 2 * q, a.sv + (long long)(k0 + r) * a.ld + m0 + 2 * q);
            }
        }
    };
    auto load_f = [&](int fstage, int chunk) {
        double* ftile = reinterpret_cast<double*>(f0 + fstage * fbytes);
        const double* fsrc = a.F + (long long)chunk * KC * K;
        for (int e = tid; e < (KC * K) / 2; e += NT) cp_async16(ftile + 2 * e, fsrc + 2 * e);
    };
    // one row of Z for the columns zcode[qlo..qhi) of this lane
    auto gen_row = [&](double* zdst, const double* fr, int qlo, int qhi) {
#pragma unroll
        for (int q = 0; q < CZ; ++q) {
            if (q >= qlo && q < qhi) {
                const int cc = lane + 32 * q;
                if (cc < ncw) {
                    const int code = zcode[q];
                    const int ty = (unsigned)code >> 30;
                    double v = 0.0;
                    if (ty == 1) v = fr[(code >> 8) & 0xff] * fr[code & 0xff];
                    else if (ty == 2) v = fr[(code >> 8) & 0xff];
                    zdst[cc] = v;
                }
            }
        }
    };

    const int zoff_z = wc * ZPW * 8 + (lane >> 2);
    const int zoff_f = (nct_z + wc * FPW) * 8 + (lane >> 2);
    static_assert(!UNI || (NH - 1) * TP + (WC - 1) * CTM <= nct_z,
                  "only the last column warp of the last part may own factor tiles");
    const int zoff_u = wc * CTM * 8 + (lane >> 2);
    const bool last_wc = wc == WC - 1 && part == NH - 1;

    if (c_begin < c_end) {
        load_data(0, c_begin);
        load_f(0, c_begin);
        if (c_begin + 1 < c_end) load_f(1, c_begin + 1);
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    if (c_begin < c_end) {
        const double* ftile = reinterpret_cast<const double*>(f0);
        for (int k = warp; k < KC; k += NT / 32) gen_row(z0 + k * zw, ftile + k * K, 0, CZ);
    }
    __syncthreads();

    const int grow = warp & 3;                    // row (within a k-step) this warp generates
    const int gqlo = (warp >> 2) ? CZH : 0, gqhi = (warp >> 2) ? CZ : CZH;

    for (int c = c_begin; c < c_end; ++c) {
        const int it = c - c_begin;
        const bool more = c + 1 < c_end;
        if (more) load_data((it + 1) & 1, c + 1);
        if (c + 2 < c_end) load_f((it + 2) % 3, c + 2);
        cp_async_commit();

        unsigned char* base = data0 + (it & 1) * dbytes;
        const WT* wtile = reinterpret_cast<const WT*>(base);
        const double* stile = reinterpret_cast<const double*>(base + G::WBYTES);
        const double* zcur = z0 + (it & 1) * zstride;
        double* znext = z0 + ((it + 1) & 1) * zstride;
        const double* fnext = reinterpret_cast<const double*>(f0 + ((it + 1) % 3) * fbytes);

#pragma unroll 2
        for (int kk = 0; kk < KC / 4; ++kk) {
            const int kl = kk * 4 + (lane & 3);
            double aw[RT], as[RT];
#pragma unroll
            for (int r = 0; r < RT; ++r) {
                const int ml = (wr * RT + r) * 8 + (lane >> 2);
                if (!TRANS) {
                    aw[r] = (double)wtile[ml * G::WSTR + kl];
                    as[r] = stile[ml * G::SSTR + kl];
                } else {
                    aw[r] = (double)wtile[kl * G::WSTR + ml];
                    as[r] = stile[kl * G::SSTR + ml];
                }
            }
            const double* zrow = zcur + kl * zw;
            if (UNI) {
                double al[RT];                    // operand of the late slots: one select per k-step
#pragma unroll
                for (int r = 0; r < RT; ++r) al[r] = last_wc ? as[r] : aw[r];
#pragma unroll
                for (int ci = 0; ci < CTM; ++ci) {
                    const bool late = (NH - 1) * TP + (WC - 1) * CTM + ci >= nct_z;        // compile-time
                    const double b = zrow[zoff_u + ci * 8];
#pragma unroll
                    for (int r = 0; r < RT; ++r) dmma(acc[r][ci][0], acc[r][ci][1], late ? al[r] : aw[r], b);
                }
            } else {
#pragma unroll
                for (int ci = 0; ci < CTM; ++ci) {
                    const bool isz = ci < ZPW;
                    const double b = isz ? zrow[zoff_z + ci * 8] : zrow[zoff_f + (ci - ZPW) * 8];
#pragma unroll
                    for (int r = 0; r < RT; ++r) dmma(acc[r][ci][0], acc[r][ci][1], isz ? aw[r] : as[r], b);
                }
            }
            // four rows of the NEXT chunk's Z tile, issued in the shadow of the DMMAs above
            if (more) {
                const int gk = kk * 4 + grow;
                gen_row(znext + gk * zw, fnext + gk * K, gqlo, gqhi);
            }
        }
        cp_async_wait<0>();
        __syncthreads();
    }

    double* out = a.out + (long long)split * a.out_split_stride;
    constexpr int nco = L + K;
#pragma unroll
    for (int r = 0; r < RT; ++r) {
        const int m = m0 + (wr * RT + r) * 8 + (lane >> 2);
        if (m < a.m_valid) {
#pragma unroll
            for (int ci = 0; ci < CTM; ++ci) {
                bool isz, valid;
                int tl;
                if (UNI) {
                    const int tloc = wc * CTM + ci, tix = part * TP + tloc;
                    isz = tix < nct_z; tl = isz ? tix : tix - nct_z; valid = tloc < TP && tix < nct;
                } else {
                    isz = ci < ZPW; tl = isz ? wc * ZPW + ci : wc * FPW + (ci - ZPW);
                    valid = ci < ZPW + FPW && tl < (isz ? nct_z : nct_f);
                }
                if (valid) {
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int cc = tl * 8 + (lane & 3) * 2 + h;
                        int oc = -1;
                        if (isz) { if (cc < L) oc = cc; }
                        else if (cc < K) oc = L + cc;
                        if (oc >= 0) out[(long long)m * nco + oc] = acc[r][ci][h];
                    }
                }
            }
        }
    }
}

template <int BM, int WR, int WC, int CTM, int KC, bool TRANS, typename WT>
static size_t stats_smem_ovl(int K, int zw) {
    using G = TileGeom<TRANS, WT, BM, KC>;
    size_t fbytes = ((size_t)(KC * K * 8) + 15) & ~(size_t)15;
    return 2 * (size_t)(G::WBYTES + G::SBYTES) + 3 * fbytes + 2 * (size_t)KC * zw * 8;
}

template <int BM, int WR, int WC, int CTM, int KC, bool TRANS, typename WT>
static size_t stats_smem(int K, int zw) {
    using G = TileGeom<TRANS, WT, BM, KC>;
    size_t fbytes = ((size_t)(KC * K * 8) + 15) & ~(size_t)15;
    return 2 * (G::WBYTES + G::SBYTES + fbytes) + (size_t)KC * zw * 8;
}

template <int BM, int WR, int WC, int CTM, int KC, bool TRANS, typename WT, int KFIX>
static void launch_stats_t(const StatsPlan& p, const void* wt, const double* sv, const double* F,
                           long long ld, int m_valid, double* out, cudaStream_t st) {
    StatsKArgs a;
    a.wt = wt; a.sv = sv; a.F = F; a.out = out; a.ld = ld;
    a.K = p.K; a.L = p.L; a.nct_z = p.nct_z; a.nct_f = p.nct_f; a.zw = p.zw;
    a.nchunks = p.nchunks; a.chunks_per_split = p.chunks_per_split;
    a.m_valid = m_valid; a.out_split_stride = (long long)p.out_elems_per_split;
    auto kern = stats_kernel<BM, WR, WC, CTM, KC, TRANS, WT, KFIX>;
    static PerDeviceOnce attr_once;
    if (attr_once.first()) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
    dim3 grid(p.mtiles, p.nsplit);
    kern<<<grid, 32 * WR * WC, p.smem_bytes, st>>>(a);
}

template <int BM, int WR, int WC, int CTM, int KC, bool TRANS, typename WT, int KFIX, bool UNI, int NH>
static void launch_stats_ovl_t(const StatsPlan& p, const void* wt, const double* sv, const double* F,
                               long long ld, int m_valid, double* out, cudaStream_t st) {
    StatsKArgs a;
    a.wt = wt; a.sv = sv; a.F = F; a.out = out; a.ld = ld;
    a.K = p.K; a.L = p.L; a.nct_z = p.nct_z; a.nct_f = p.nct_f; a.zw = p.zw;
    a.nchunks = p.nchunks; a.chunks_per_split = p.chunks_per_split;
    a.m_valid = m_valid; a.out_split_stride = (long long)p.out_elems_per_split;
    auto kern = stats_kernel_ovl<BM, WR, WC, CTM, KC, TRANS, WT, KFIX, UNI, NH>;
    static PerDeviceOnce attr_once;
    if (attr_once.first()) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024);
    dim3 grid(p.mtiles, p.nsplit, NH);
    kern<<<grid, 32 * WR * WC, p.smem_bytes, st>>>(a);
}

// Tile configurations  (BM, WR, WC, CTM, KC):
//   cfg 0: generic K <= 16   128 rows, 8x1 warps, 19 column-tile slots, KC 32
//   cfg 1: generic K <= 32    32 rows, 1x8 warps, 10 slots per warp,    KC 16
//   cfg 2: generic K <=  8   128 rows, 8x1 warps,  6 slots,             KC 32
//   cfg 3: K == 16 (compile-time) 128 rows, 4x2 warps, 9+1 slots per warp, KC 32
//   cfg 4: K == 32 (compile-time)  32 rows, 1x8 warps, 9+1 slots per warp, KC 16
//   cfg 5: K ==  8 (compile-time) 128 rows, 8x1 warps, 5+1 slots,          KC 32
#define BTF_CFG0 128, 8, 1, 19, 32
#define BTF_CFG1 32, 1, 8, 10, 16
#define BTF_CFG2 128, 8, 1, 6, 32
#define BTF_CFG3 128, 4, 2, 10, 32
#define BTF_CFG4 32, 1, 8, 10, 16
#define BTF_CFG5 128, 8, 1, 6, 32
#define BTF_CFG4U 32, 1, 8, 9, 16      // K == 32 with the unified tile list (overlapped kernel)

static int cfg_wc(int cfg) { return (cfg == 1 || cfg == 4) ? 8 : (cfg == 3 ? 2 : 1); }

bool plan_stats(StatsPlan* p, int K, bool trans, bool weights_f64, int mdim_pad, int kdim_pad, int m_valid,
                int nsplit_request, int sm_count) {
    if (K < 1 || K > 32) return false;
    p->K = K;
    p->L = K * (K + 1) / 2;
    p->nct_z = (p->L + 7) / 8;
    p->nct_f = (K + 7) / 8;
    const int nct = p->nct_z + p->nct_f;
    if (K == 16) p->cfg = 3;
    else if (K == 32) p->cfg = 4;
    else if (K == 8) p->cfg = 5;
    else p->cfg = (nct <= 6) ? 2 : (nct <= 19 ? 0 : 1);
    const int WC = cfg_wc(p->cfg);
    // Z row width: every tile slot any warp may touch, rounded so that zw = 4 or 12 (mod 16)
    int need = std::max(nct, std::max(WC * cdiv(p->nct_z, WC), p->nct_z + WC * cdiv(p->nct_f, WC))) * 8;
    if (p->cfg == 4) need = std::max(need, 8 * 9 * 8);     // unified list: 8 warps x 9 tile slots
    int zw = need;
    while (!((zw % 16) == 4 || (zw % 16) == 12)) ++zw;
    p->zw = zw;
    p->BM = (p->cfg == 1 || p->cfg == 4) ? 32 : 128;
    p->KC = (p->cfg == 1 || p->cfg == 4) ? 16 : 32;
    if (mdim_pad % p->BM || kdim_pad % p->KC) return false;
    p->mtiles = mdim_pad / p->BM;
    p->nchunks = kdim_pad / p->KC;
    // split the contraction so the grid fills the machine in (nearly) whole waves
    int ns = nsplit_request;
    if (ns <= 0) {
        ns = 1;
        double best = -1.0;
        int maxs = p->nchunks < 64 ? p->nchunks : 64;
        for (int s = 1; s <= maxs; ++s) {
            long long ctas = (long long)p->mtiles * s;
            long long waves = (ctas + sm_count - 1) / sm_count;
            double eff = (double)ctas / (double)(waves * sm_count);
            // prefer few splits: demand a clear efficiency gain for more partial traffic
            if (eff > best + 0.03) { best = eff; ns = s; }
            if (best > 0.97) break;
        }
    }
    if (ns > p->nchunks) ns = p->nchunks;
    if (ns < 1) ns = 1;
    p->chunks_per_split = (p->nchunks + ns - 1) / ns;
    p->nsplit = (p->nchunks + p->chunks_per_split - 1) / p->chunks_per_split;
    p->out_elems_per_split = (size_t)m_valid * (size_t)(p->L + K);
#define SMEM_OF(...) (trans ? (weights_f64 ? stats_smem<__VA_ARGS__, true, double>(K, p->zw)   \
                                           : stats_smem<__VA_ARGS__, true, uint8_t>(K, p->zw)) \
                            : (weights_f64 ? stats_smem<__VA_ARGS__, false, double>(K, p->zw)  \
                                           : stats_smem<__VA_ARGS__, false, uint8_t>(K, p->zw)))
    switch (p->cfg) {
        case 0: p->smem_bytes = SMEM_OF(BTF_CFG0); break;
        case 1: p->smem_bytes = SMEM_OF(BTF_CFG1); break;
        case 2: p->smem_bytes = SMEM_OF(BTF_CFG2); break;
        case 3: p->smem_bytes = SMEM_OF(BTF_CFG3); break;
        case 4: p->smem_bytes = SMEM_OF(BTF_CFG4); break;
        default: p->smem_bytes = SMEM_OF(BTF_CFG5); break;
    }
#undef SMEM_OF
    // K = 32 with f64 weights: Z generation overlapped with the DMMAs (unified tile list, 185 KB).  K = 16 with f64
    // weights keeps the three-phase kernel (its overlapped form would need 234 KB).
    p->overlap = 0;
    if (p->cfg == 4 && weights_f64) {
        p->overlap = 1;
        p->smem_bytes = trans ? stats_smem_ovl<BTF_CFG4U, true, double>(K, p->zw) : stats_smem_ovl<BTF_CFG4U, false, double>(K, p->zw);
    }
    p->zpre = 0; p->zwg = 0;
    // count weights at K = 16 / 32: the right operand is pre-generated in global memory (stats_zpre.cu)
    if (!weights_f64 && (K == 16 || K == 32)) return plan_stats_zpre(p, trans, mdim_pad, kdim_pad, nsplit_request, sm_count);
    return p->smem_bytes <= 226 * 1024;
}

void launch_stats(const StatsPlan& p, bool trans, bool weights_f64, const void* wt, const double* sv,
                  const double* F, long long frows, long long ld, int m_valid, double* out, double* zscratch,
                  cudaStream_t st) {
    if (p.zpre) { launch_stats_zpre(p, trans, wt, sv, F, frows, ld, m_valid, out, zscratch, st); return; }
    if (p.overlap) {
        if (trans) launch_stats_ovl_t<BTF_CFG4U, true, double, 32, true, 1>(p, wt, sv, F, ld, m_valid, out, st);
        else launch_stats_ovl_t<BTF_CFG4U, false, double, 32, true, 1>(p, wt, sv, F, ld, m_valid, out, st);
        return;
    }
    if (p.cfg == 3) {   // K = 16 with count weights takes the zpre kernel
        if (trans) launch_stats_t<BTF_CFG3, true, double, 16>(p, wt, sv, F, ld, m_valid, out, st);
        else launch_stats_t<BTF_CFG3, false, double, 16>(p, wt, sv, F, ld, m_valid, out, st);
        return;
    }
#define DISPATCH(KF, ...)                                                                                        \
    do {                                                                                                         \
        if (trans) {                                                                                             \
            if (weights_f64) launch_stats_t<__VA_ARGS__, true, double, KF>(p, wt, sv, F, ld, m_valid, out, st);  \
            else launch_stats_t<__VA_ARGS__, true, uint8_t, KF>(p, wt, sv, F, ld, m_valid, out, st);             \
        } else {                                                                                                 \
            if (weights_f64) launch_stats_t<__VA_ARGS__, false, double, KF>(p, wt, sv, F, ld, m_valid, out, st); \
            else launch_stats_t<__VA_ARGS__, false, uint8_t, KF>(p, wt, sv, F, ld, m_valid, out, st);            \
        }                                                                                                        \
    } while (0)
    switch (p.cfg) {
        case 0: DISPATCH(0, BTF_CFG0); break;
        case 1: DISPATCH(0, BTF_CFG1); break;
        case 2: DISPATCH(0, BTF_CFG2); break;
        default: DISPATCH(8, BTF_CFG5); break;   // cfg 5 (cfg 4 is always overlapped or zpre)
    }
#undef DISPATCH
}

// ------------------------------------------------------------------ nu2 residual (direct pass)
// One block = 64 rows x 256 cells; partial = sum cnt*Mu^2 - 2*Mu*S over the block.
template <int KMAX>
__global__ void __launch_bounds__(256) residual_kernel(const uint8_t* __restrict__ cnt, const double* __restrict__ S,
                                                       long long ld, const double* __restrict__ W,
                                                       const double* __restrict__ V, int K,
                                                       double* __restrict__ partials) {
    __shared__ double ws[64 * KMAX];
    __shared__ double sh[32];
    const int p = blockIdx.x * 256 + threadIdx.x;
    const int i0 = blockIdx.y * 64;
    for (int e = threadIdx.x; e < 64 * K; e += 256) ws[e] = W[(long long)i0 * K + e];
    double v[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) v[k] = k < K ? V[(long long)p * K + k] : 0.0;
    __syncthreads();
    double accum = 0.0;
    for (int r = 0; r < 64; ++r) {
        long long o = (long long)(i0 + r) * ld + p;
        double c = (double)cnt[o];
        double s = S[o];
        double mu = 0.0;
#pragma unroll
        for (int k = 0; k < KMAX; ++k)
            if (k < K) mu += ws[r * K + k] * v[k];
        accum += mu * (c * mu - 2.0 * s);
    }
    double tot = block_sum(accum, sh);
    if (threadIdx.x == 0) partials[blockIdx.y * gridDim.x + blockIdx.x] = tot;
}

void launch_residual(const uint8_t* cnt, const double* S, long long ld, const double* W, const double* V,
                     int nrows_pad, int Ppad, int K, double* partials, int* nblocks_out, cudaStream_t st) {
    dim3 grid(Ppad / 256 > 0 ? Ppad / 256 : 1, nrows_pad / 64);
    if (K <= 8) residual_kernel<8><<<grid, 256, 0, st>>>(cnt, S, ld, W, V, K, partials);
    else if (K <= 16) residual_kernel<16><<<grid, 256, 0, st>>>(cnt, S, ld, W, V, K, partials);
    else residual_kernel<32><<<grid, 256, 0, st>>>(cnt, S, ld, W, V, K, partials);
    *nblocks_out = grid.x * grid.y;
}


// ------------------------------------------------------------------ running posterior moments of Mu
// Welford update of mean and M2 of Mu[i,p] = w_i . v_p for every local cell, one pass per saved
// sample (SURVEY.md 8f row 2: at C2 a thousand saved (W, V) samples are 10 GB, the two moment
// tensors 4.3 GB).  Same tiling as the residual pass: 64 rows x 256 cells per block.
template <int KMAX>
__global__ void __launch_bounds__(256) mu_moments_kernel(const double* __restrict__ W, const double* __restrict__ V,
                                                         int K, int nloc, int P, double* __restrict__ mean,
                                                         double* __restrict__ m2, double count) {
    __shared__ double ws[64 * KMAX];
    const int p = blockIdx.x * 256 + threadIdx.x;
    const int i0 = blockIdx.y * 64;
    for (int e = threadIdx.x; e < 64 * K; e += 256) ws[e] = W[(long long)i0 * K + e];
    double v[KMAX];
#pragma unroll
    for (int k = 0; k < KMAX; ++k) v[k] = (k < K && p < P) ? V[(long long)p * K + k] : 0.0;
    __syncthreads();
    if (p >= P) return;
    const double inv = 1.0 / count;
    const int nr = min(64, nloc - i0);
    // batches of 4 rows: all loads of a batch are in flight before the first update
    for (int r0 = 0; r0 < nr; r0 += 4) {
        double m[4], q[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const bool ok = r0 + u < nr;
            const long long o = (long long)(i0 + r0 + u) * P + p;
            m[u] = ok ? mean[o] : 0.0;
            q[u] = ok ? m2[o] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int r = r0 + u;
            if (r >= nr) break;
            double mu = 0.0;
#pragma unroll
            for (int k = 0; k < KMAX; ++k)
                if (k < K) mu += ws[r * K + k] * v[k];
            const long long o = (long long)(i0 + r) * P + p;
            const double d = mu - m[u];
            const double mn = m[u] + d * inv;
            mean[o] = mn;
            m2[o] = q[u] + d * (mu - mn);
        }
    }
}

void launch_mu_moments(const double* W, const double* V, int K, int nloc, int P, double* mean, double* m2,
                       double count, cudaStream_t st) {
    dim3 grid((P + 255) / 256, (nloc + 63) / 64);
    if (K <= 8) mu_moments_kernel<8><<<grid, 256, 0, st>>>(W, V, K, nloc, P, mean, m2, count);
    else if (K <= 16) mu_moments_kernel<16><<<grid, 256, 0, st>>>(W, V, K, nloc, P, mean, m2, count);
    else mu_moments_kernel<32><<<grid, 256, 0, st>>>(W, V, K, nloc, P, mean, m2, count);
}

}  // namespace btf
