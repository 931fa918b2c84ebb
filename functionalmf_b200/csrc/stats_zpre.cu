// K1 with a PRE-GENERATED right operand (compile-time K = 16 / 32).
//
// ncu on the generated-operand kernel (stats_kernels.cu) shows the Z products competing with
// the DMMAs: DMUL and DMMA share the FP64 pipe, every DMUL waits behind 16-cycle DMMAs
// ("math pipe throttle" on 10 % (K = 16) to 21 % (K = 32) of the samples) and stalls its
// in-order warp.  Here Z[k, :] = [F[k,k1] F[k,k2] (k2 <= k1) | F[k,:]] is written once per
// sweep by a tiny kernel (C2: 80 MB for V, 5 MB for W; it stays in the 126 MB L2 or is
// re-streamed from HBM, of which the statistics kernels use < 10 %), and the contraction
// kernel becomes a pure FP64 tensor GEMM: data tile and Z tile arrive through one cp.async
// pipeline, the loop contains nothing but LDS and DMMA.
#include "stats_common.cuh"
#include <stdlib.h>

namespace btf {

// Z[k][c], c < nct*8: packed products, then the factor columns, zero padded
__global__ void zgen_kernel(const double* __restrict__ F, long long rows, int K, int L, int nct_z, int zwg,
                            double* __restrict__ Z) {
    const long long total = rows * zwg;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long k = e / zwg;
        const int c = (int)(e - k * zwg);
        const double* fr = F + k * K;
        double v = 0.0;
        if (c < nct_z * 8) {
            if (c < L) {
                int k1 = (int)((sqrt(8.0 * c + 1.0) - 1.0) * 0.5);
                while (k1 * (k1 + 1) / 2 > c) --k1;
                while ((k1 + 1) * (k1 + 2) / 2 <= c) ++k1;
                v = fr[k1] * fr[c - k1 * (k1 + 1) / 2];
            }
        } else {
            const int cf = c - nct_z * 8;
            if (cf < K) v = fr[cf];
        }
        Z[e] = v;
    }
}

template <int BM, int WR, int WC, int CTM, int KC, bool TRANS, typename WT, int KFIX, int NH>
__global__ void __launch_bounds__(32 * WR* WC, 1) stats_kernel_zpre(StatsKArgs a, const double* __restrict__ Zg) {
    constexpr int NT = 32 * WR * WC;
    constexpr int RT = BM / 8 / WR;
    using G = TileGeom<TRANS, WT, BM, KC>;
    extern __shared__ __align__(16) unsigned char smem[];

    constexpr int K = KFIX, L = K * (K + 1) / 2;
    constexpr int nct_z = cdiv(L, 8), nct_f = cdiv(K, 8), nct = nct_z + nct_f;
    constexpr int zwg = nct * 8;                          // row pitch of the global Z
    constexpr int TP = cdiv(nct, NH);                     // column tiles per part
    static_assert((NH - 1) * TP + (WC - 1) * CTM <= nct_z, "only the last warp of the last part owns factor tiles");
    static_assert(WC * CTM >= TP, "tile slots must cover a part");
    const int part = NH > 1 ? blockIdx.z : 0;
    const int ntile = min(nct, (part + 1) * TP) - part * TP;      // tiles of this part
    const int zw = a.zw;                                  // shared-memory pitch (= 4 or 12 mod 16)
    constexpr int dbytes = G::WBYTES + G::SBYTES;
    const int zbytes = KC * zw * 8;
    const int stage_bytes = dbytes + zbytes;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wr = warp / WC, wc = warp % WC;
    const int m0 = blockIdx.x * BM;
    const int split = blockIdx.y;
    const int c_begin = split * a.chunks_per_split;
    const int c_end = min(a.nchunks, c_begin + a.chunks_per_split);

    double acc[RT][CTM][2];
#pragma unroll
    for (int r = 0; r < RT; ++r)
#pragma unroll
        for (int c = 0; c < CTM; ++c) acc[r][c][0] = acc[r][c][1] = 0.0;

    auto load_chunk = [&](int stage, int chunk) {
        unsigned char* base = smem + stage * stage_bytes;
        WT* wtile = reinterpret_cast<WT*>(base);
        double* stile = reinterpret_cast<double*>(base + G::WBYTES);
        double* ztile = reinterpret_cast<double*>(base + dbytes);
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
        // Z rows k0..k0+KC, columns of this part: ntile*4 16-byte pieces per row
        const int zp = ntile * 4;
        const double* zsrc = Zg + (long long)k0 * zwg + part * TP * 8;
        for (int e = tid; e < KC * zp; e += NT) {
            int r = e / zp, q = e - r * zp;
            cp_async16(ztile + r * zw + 2 * q, zsrc + (long long)r * zwg + 2 * q);
        }
    };

    const int zoff = wc * CTM * 8 + (lane >> 2);
    const bool last_wc = wc == WC - 1 && part == NH - 1;

    if (c_begin < c_end) load_chunk(0, c_begin);
    cp_async_commit();

    for (int c = c_begin; c < c_end; ++c) {
        const int stg = (c - c_begin) & 1;
        if (c + 1 < c_end) load_chunk(stg ^ 1, c + 1);
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();

        const unsigned char* base = smem + stg * stage_bytes;
        const WT* wtile = reinterpret_cast<const WT*>(base);
        const double* stile = reinterpret_cast<const double*>(base + G::WBYTES);
        const double* ztile = reinterpret_cast<const double*>(base + dbytes);

#pragma unroll 2
        for (int kk = 0; kk < KC / 4; ++kk) {
            const int kl = kk * 4 + (lane & 3);
            double aw[RT], al[RT];
#pragma unroll
            for (int r = 0; r < RT; ++r) {
                const int ml = (wr * RT + r) * 8 + (lane >> 2);
                double as;
                if (!TRANS) {
                    aw[r] = (double)wtile[ml * G::WSTR + kl];
                    as = stile[ml * G::SSTR + kl];
                } else {
                    aw[r] = (double)wtile[kl * G::WSTR + ml];
                    as = stile[kl * G::SSTR + ml];
                }
                al[r] = last_wc ? as : aw[r];             // operand of the late (factor) slots
            }
            const double* zrow = ztile + kl * zw + zoff;
#pragma unroll
            for (int ci = 0; ci < CTM; ++ci) {
                const bool late = (NH - 1) * TP + (WC - 1) * CTM + ci >= nct_z;      // compile-time
                const double b = zrow[ci * 8];
#pragma unroll
                for (int r = 0; r < RT; ++r) dmma(acc[r][ci][0], acc[r][ci][1], late ? al[r] : aw[r], b);
            }
        }
        __syncthreads();
    }
    cp_async_wait<0>();

    double* out = a.out + (long long)split * a.out_split_stride;
    constexpr int nco = L + K;
#pragma unroll
    for (int r = 0; r < RT; ++r) {
        const int m = m0 + (wr * RT + r) * 8 + (lane >> 2);
        if (m < a.m_valid) {
#pragma unroll
            for (int ci = 0; ci < CTM; ++ci) {
                const int tloc = wc * CTM + ci, tix = part * TP + tloc;
                const bool isz = tix < nct_z;
                const int tl = isz ? tix : tix - nct_z;
                if (tloc < TP && tix < nct) {
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
static size_t zpre_smem(int zw) {
    using G = TileGeom<TRANS, WT, BM, KC>;
    return 2 * ((size_t)(G::WBYTES + G::SBYTES) + (size_t)KC * zw * 8);
}

template <int BM, int WR, int WC, int CTM, int KC, bool TRANS, typename WT, int KFIX, int NH>
static void launch_zpre_t(const StatsPlan& p, const void* wt, const double* sv, long long ld, int m_valid, double* out,
                          const double* Zg, cudaStream_t st) {
    StatsKArgs a;
    a.wt = wt; a.sv = sv; a.F = nullptr; a.out = out; a.ld = ld;
    a.K = p.K; a.L = p.L; a.nct_z = p.nct_z; a.nct_f = p.nct_f; a.zw = p.zw;
    a.nchunks = p.nchunks; a.chunks_per_split = p.chunks_per_split;
    a.m_valid = m_valid; a.out_split_stride = (long long)p.out_elems_per_split;
    auto kern = stats_kernel_zpre<BM, WR, WC, CTM, KC, TRANS, WT, KFIX, NH>;
    static PerDeviceOnce attr_once;
    if (attr_once.first()) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024);
    dim3 grid(p.mtiles, p.nsplit, NH);
    kern<<<grid, 32 * WR * WC, p.smem_bytes, st>>>(a, Zg);
}

// tile configurations of the pre-generated-operand kernels (BM, WR, WC, CTM, KC)
#define ZP16R 128, 8, 1, 19, 32      // K = 16 rows:    every warp owns all 19 tiles
#define ZP16C 128, 4, 2, 10, 32      // K = 16 columns: 4 x 2 warps
#define ZP32  64, 2, 4, 9, 32        // K = 32: two column parts per 64-row tile

static int zpre_pitch(int ntiles) {
    int zw = ntiles * 8;
    while (!((zw % 16) == 4 || (zw % 16) == 12)) ++zw;
    return zw;
}

// Fill in the plan for the pre-generated-operand path (count weights, K = 16 or 32); false when the shape has no such kernel.
bool plan_stats_zpre(StatsPlan* p, bool trans, int mdim_pad, int kdim_pad, int nsplit_request, int sm_count) {
    if (p->K != 16 && p->K != 32) return false;
    const int nct = p->nct_z + p->nct_f;
    int parts = 1;
    size_t smem;
    if (p->K == 16) {
        p->BM = 128; p->KC = 32;
        p->zw = zpre_pitch(trans ? 2 * 10 : 19);
        smem = trans ? zpre_smem<ZP16C, true, uint8_t>(p->zw) : zpre_smem<ZP16R, false, uint8_t>(p->zw);
    } else {
        p->BM = 64; p->KC = 32; parts = 2;
        p->zw = zpre_pitch(4 * 9);
        smem = trans ? zpre_smem<ZP32, true, uint8_t>(p->zw) : zpre_smem<ZP32, false, uint8_t>(p->zw);
    }
    if (smem > 226 * 1024 || mdim_pad % p->BM || kdim_pad % p->KC) return false;
    p->smem_bytes = smem;
    p->zpre = 1;
    p->zwg = nct * 8;
    p->overlap = 0;
    p->mtiles = mdim_pad / p->BM;
    p->nchunks = kdim_pad / p->KC;
    int ns = nsplit_request;
    if (ns <= 0) {
        ns = 1;
        double best = -1.0;
        int maxs = p->nchunks < 64 ? p->nchunks : 64;
        for (int s = 1; s <= maxs; ++s) {
            long long ctas = (long long)p->mtiles * s * parts;
            long long waves = (ctas + sm_count - 1) / sm_count;
            double eff = (double)ctas / (double)(waves * sm_count);
            if (eff > best + 0.03) { best = eff; ns = s; }
            if (best > 0.97) break;
        }
    }
    if (ns > p->nchunks) ns = p->nchunks;
    if (ns < 1) ns = 1;
    p->chunks_per_split = (p->nchunks + ns - 1) / ns;
    p->nsplit = (p->nchunks + p->chunks_per_split - 1) / p->chunks_per_split;
    return true;
}

void launch_stats_zpre(const StatsPlan& p, bool trans, const void* wt, const double* sv, const double* F,
                       long long frows, long long ld, int m_valid, double* out, double* Zg, cudaStream_t st) {
    // 1. the right operand, once per launch
    const long long total = frows * p.zwg;
    int nb = (int)((total + 255) / 256);
    if (nb > 148 * 16) nb = 148 * 16;
    if (nb < 1) nb = 1;
    zgen_kernel<<<nb, 256, 0, st>>>(F, frows, p.K, p.L, p.nct_z, p.zwg, Zg);
    // 2. the contraction
    if (p.K == 16) {
        if (trans) launch_zpre_t<ZP16C, true, uint8_t, 16, 1>(p, wt, sv, ld, m_valid, out, Zg, st);
        else launch_zpre_t<ZP16R, false, uint8_t, 16, 1>(p, wt, sv, ld, m_valid, out, Zg, st);
    } else {
        if (trans) launch_zpre_t<ZP32, true, uint8_t, 32, 2>(p, wt, sv, ld, m_valid, out, Zg, st);
        else launch_zpre_t<ZP32, false, uint8_t, 32, 2>(p, wt, sv, ld, m_valid, out, Zg, st);
    }
}

}  // namespace btf
