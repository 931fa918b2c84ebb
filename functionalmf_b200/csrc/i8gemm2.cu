// The product block of the sufficient statistics as a Blackwell-native GEMM (tcgen05, 2-CTA pairs, TMA, persistent):
//
//   out[m][c] = 2^(e_c - 54) * sum_{s<7} 256^s * sum_k cnt[m][k] * d_s[k][c],      m < M,  c < L
//
// cnt: counts (int8, K-major, [M][ldc]); d_s: the 7 signed base-256 digit planes of the fixed-point column c of Z
// (int8, K-major, stored tile-major: plane row (c / 36) * 252 + s * 36 + (c % 36), see stats_i8.cu).  Exact integer
// contraction, recombined and rounded ONCE in the epilogue: no int32 intermediate in global memory.
//
// Shape of the kernel (what the earlier single-CTA 128 x 256 kernel lacked - it was bound by operand traffic from L2 at
// 87 MAC/B):
//   * one CTA PAIR (cluster of 2, tcgen05 cta_group::2) owns a 256 x 256 tile: each CTA stages 128 count rows and 128
//     digit rows per 128-byte K chunk (32 KB per stage, 6 stages) for 256 x 256 x 128 MACs of the pair
//     = 128 MAC per byte read from L2, 1.5x the single-CTA 128 x 256 tile;
//   * operands arrive by TMA (cp.async.bulk.tensor.2d, 128-byte swizzle, out-of-range rows zero-filled), one elected
//     thread per CTA; both CTAs' copies complete on the LEADER's mbarrier (.cta_group::2);
//   * one elected thread of the leader issues tcgen05.mma.cta_group::2.kind::i8 (M = 256, N = 256, K = 32) and releases
//     the stages of both CTAs with a multicast tcgen05.commit;
//   * persistent: pairs loop over tiles; TWO accumulator stages in tensor memory (2 x 256 columns), so the epilogue of
//     tile i (tcgen05.ld, integer Horner recombination of the 7 planes, one rounding, FP64 stores) runs under the main
//     loop of tile i + 1;
//   * a tile's 256 accumulator columns are 7 planes x 36 product columns, plane-major, so 7 aligned 4-column
//     tcgen05.ld give a thread (= one count row) all planes of 4 product columns.
#include <cuda.h>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "kernels.h"

namespace btf {

namespace {

constexpr int G2_ROWS = 128;                 // count rows / digit rows per CTA and stage
constexpr int G2_BK = 128;                   // bytes of K per stage
constexpr int G2_STAGES = 6;                              // operand stages (196 KB)
constexpr int G2_TILE_BYTES = G2_ROWS * G2_BK;            // 16 KB
constexpr int G2_STAGE_BYTES = 2 * G2_TILE_BYTES;         // counts + digits
constexpr int G2_SMEM = G2_STAGES * G2_STAGE_BYTES + 1024 /*alignment*/ + 256 /*barriers*/;
constexpr int G2_TMEM_COLS = 512;            // two accumulator stages of 256 columns
constexpr int G2_THREADS = 192;              // warp 0: TMA, warp 1: MMA + tensor-memory allocation, warps 2-5: epilogue
constexpr int G2_CPT = I8_COLS_PER_TILE;     // 36 product columns per tile
constexpr int G2_NP = I8_NPLANES;            // 7 planes
constexpr uint32_t G2_PEER_MASK = 0xFEFFFFFFu;   // clears the CTA-rank bit of a shared::cluster address: the leader's copy

__device__ __forceinline__ uint32_t s_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;\n" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;\n" ::: "memory");
}
__device__ __forceinline__ void g2_mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(s_u32(bar)), "r"(count));
}
__device__ __forceinline__ void g2_mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "G2_WAIT:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra G2_DONE;\n\t"
        "bra G2_WAIT;\n\t"
        "G2_DONE:\n\t}\n" ::"r"(s_u32(bar)), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void g2_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(s_u32(bar)), "r"(bytes) : "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ void g2_arrive_cluster(uint64_t* bar, uint32_t rank) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}\n" ::"r"(s_u32(bar)), "r"(rank)
        : "memory");
}
// TMA: 2-D tile (inner coordinate = byte offset along K, outer = row) into this CTA's shared memory; the bytes are
// credited to the LEADER's barrier (both CTAs of the pair feed one MMA)
__device__ __forceinline__ void g2_tma_load(const CUtensorMap* tm, uint64_t* bar, void* dst, int k0, int row0) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];\n" ::
            "r"(s_u32(dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(s_u32(bar) & G2_PEER_MASK), "r"(k0), "r"(row0)
        : "memory");
}
// shared-memory matrix descriptor, K-major, 128-byte swizzle: 8-row x 128-byte atoms, 1024 bytes apart
__device__ __forceinline__ uint64_t g2_desc(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// D = S32, A = B = signed 8-bit, both K-major, M = 256 (pair), N = 256
constexpr uint32_t G2_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(256 >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);

__device__ __forceinline__ void g2_mma(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}\n" ::"r"(tmem_d),
        "l"(da), "l"(db), "r"(G2_IDESC), "r"(accumulate), "r"(0u)
        : "memory");
}
// completion of all MMAs issued so far -> arrive on `bar` in BOTH CTAs of the pair
__device__ __forceinline__ void g2_commit_pair(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n" ::
                     "r"(s_u32(bar)), "h"((uint16_t)3)
                 : "memory");
}

struct G2Args {
    int M;            // count rows
    int L;            // product columns
    int k_chunks;     // K / 128
    int m_tiles, n_tiles;
    const int* expo;  // [L] column exponents
    double* out;      // out[m * ldo + c]
    long long ldo;
    // element-wise guard (stats_i8.cu): rows whose diagonal entries cannot be guaranteed to `tol` relative are flagged
    const unsigned* cntsum; unsigned char* flags; double tol;
    unsigned long long diag_mask[16];   // per column tile: bit q set when product column nt * 36 + q is a diagonal (k, k)
    // split-K mode (few tiles: narrow shards): nsplit > 1 jobs per tile, each over chunks_per_split K chunks; the exact int32
    // partial sums are added into D[i8_plane_row][m] with integer atomics (order independent) and recombined by i8_combine
    int nsplit, chunks_per_split;
    int32_t* D; long long ldd;
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(G2_THREADS, 1)
i8gemm2_kernel(const __grid_constant__ CUtensorMap tm_cnt, const __grid_constant__ CUtensorMap tm_dig, G2Args p) {
    const CUtensorMap* tm_cnt_p = &tm_cnt;     // counts
    const CUtensorMap* tm_dig_p = &tm_dig;     // digit planes
    extern __shared__ uint8_t smraw[];
    uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smraw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(sm + G2_STAGES * G2_STAGE_BYTES);   // [STAGES]  TMA -> MMA      (leader's copy is used)
    uint64_t* empty = full + G2_STAGES;                                              // [STAGES]  MMA -> TMA      (per CTA, multicast commit)
    uint64_t* tfull = empty + G2_STAGES;                                             // [2]       MMA -> epilogue (per CTA, multicast commit)
    uint64_t* tempty = tfull + 2;                                                    // [2]       epilogue -> MMA (leader's copy: 8 warp arrivals)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t rank = cluster_ctarank();
    const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
    const int ntiles = p.m_tiles * p.n_tiles * p.nsplit;       // jobs: (tile, K split), tile index fastest
    const int tiles_only = p.m_tiles * p.n_tiles;

    if (tid == 0) {
        for (int s = 0; s < G2_STAGES; ++s) { g2_mbar_init(full + s, 1); g2_mbar_init(empty + s, 1); }
        for (int a = 0; a < 2; ++a) { g2_mbar_init(tfull + a, 1); g2_mbar_init(tempty + a, 8); }
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(s_u32(tmem_slot)), "n"(G2_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;\n");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    cluster_sync_all();                       // barriers of both CTAs initialised, tensor memory allocated
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===== TMA producer (one lane): this CTA's half of the pair's operands
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];\n" ::"l"(reinterpret_cast<uint64_t>(tm_cnt_p)) : "memory");
            asm volatile("prefetch.tensormap [%0];\n" ::"l"(reinterpret_cast<uint64_t>(tm_dig_p)) : "memory");
            int stage = 0; uint32_t phase = 0;
            for (int t = pair; t < ntiles; t += npairs) {
                const int sp = t / tiles_only, tt = t - sp * tiles_only;
                const int mt = tt / p.n_tiles, nt = tt - mt * p.n_tiles;
                const int row_c = mt * 256 + (int)rank * G2_ROWS;                       // count rows of this CTA
                const int row_d = nt * (G2_CPT * G2_NP) + (int)rank * G2_ROWS;          // digit rows (N half) of this CTA
                const int c_lo = sp * p.chunks_per_split, c_hi = min(p.k_chunks, c_lo + p.chunks_per_split);
                for (int c = c_lo; c < c_hi; ++c) {
                    g2_mbar_wait(empty + stage, phase ^ 1u);                            // (a fresh barrier passes parity 1)
                    if (rank == 0) g2_expect_tx(full + stage, 2u * G2_STAGE_BYTES);     // both CTAs' bytes land on the leader's barrier
                    uint8_t* sa = sm + stage * G2_STAGE_BYTES;
                    g2_tma_load(tm_cnt_p, full + stage, sa, c * G2_BK, row_c);
                    g2_tma_load(tm_dig_p, full + stage, sa + G2_TILE_BYTES, c * G2_BK, row_d);
                    if (++stage == G2_STAGES) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: one lane of the leader CTA
        if (rank == 0 && lane == 0) {
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int t = pair; t < ntiles; t += npairs) {
                g2_mbar_wait(tempty + acc, acc_phase ^ 1u);                             // both CTAs' epilogues have drained this accumulator
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                const uint32_t tmem_d = tmem_base + (uint32_t)(acc * 256);
                const int sp = t / tiles_only;
                const int c_lo = sp * p.chunks_per_split, c_hi = min(p.k_chunks, c_lo + p.chunks_per_split);
                for (int c = c_lo; c < c_hi; ++c) {
                    g2_mbar_wait(full + stage, phase);
                    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                    const uint32_t a0 = s_u32(sm + stage * G2_STAGE_BYTES), b0 = a0 + G2_TILE_BYTES;
#pragma unroll
                    for (int k = 0; k < G2_BK / 32; ++k)
                        g2_mma(tmem_d, g2_desc(a0 + 32 * k), g2_desc(b0 + 32 * k), (c > c_lo || k > 0) ? 1u : 0u);
                    g2_commit_pair(empty + stage);                                      // frees the stage in both CTAs
                    if (++stage == G2_STAGES) { stage = 0; phase ^= 1u; }
                }
                g2_commit_pair(tfull + acc);                                            // accumulator complete: both epilogues
                if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
            }
        }
    } else {
        // ===== epilogue: warp w reads the 32 tensor-memory lanes of its quarter (w mod 4); lane = count row
        const int quarter = warp & 3;
        int acc = 0; uint32_t acc_phase = 0;
        for (int t = pair; t < ntiles; t += npairs) {
            const int tt = t % tiles_only;
            const int mt = tt / p.n_tiles, nt = tt - mt * p.n_tiles;
            g2_mbar_wait(tfull + acc, acc_phase);
            asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
            const int row = mt * 256 + (int)rank * G2_ROWS + quarter * 32 + lane;
            if (p.nsplit > 1) {
                // split-K: raw int32 partial sums, integer atomics (the 32 lanes of a warp are 32 consecutive count rows)
                const uint32_t tb = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * 256);
#pragma unroll 1
                for (int n = 0; n < G2_CPT * G2_NP; n += 4) {
                    uint32_t v0, v1, v2, v3;
                    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];\n"
                                 : "=r"(v0), "=r"(v1), "=r"(v2), "=r"(v3)
                                 : "r"(tb + (uint32_t)n));
                    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
                    if (row < p.M) {
                        int32_t* d = p.D + (long long)(nt * (G2_CPT * G2_NP) + n) * p.ldd + row;
                        if (v0) atomicAdd(d, (int)v0);
                        if (v1) atomicAdd(d + p.ldd, (int)v1);
                        if (v2) atomicAdd(d + 2 * p.ldd, (int)v2);
                        if (v3) atomicAdd(d + 3 * p.ldd, (int)v3);
                    }
                }
                asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
                __syncwarp();
                if (lane == 0) g2_arrive_cluster(tempty + acc, 0u);
                if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
                continue;
            }
            const unsigned long long dmask = p.cntsum ? p.diag_mask[nt] : 0ull;
            const double n_half = (dmask && row < p.M) ? 0.5 * (double)p.cntsum[row] : 0.0;     // error bound = n_m 2^(e_c - 55)
            bool bad = false;
            const uint32_t tbase = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * 256);
#pragma unroll 1
            for (int i = 0; i < G2_CPT / 4; ++i) {
                uint32_t v[G2_NP][4];
#pragma unroll
                for (int s = 0; s < G2_NP; ++s)
                    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];\n"
                                 : "=r"(v[s][0]), "=r"(v[s][1]), "=r"(v[s][2]), "=r"(v[s][3])
                                 : "r"(tbase + (uint32_t)(s * G2_CPT + 4 * i)));
                asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
                const int c0 = nt * G2_CPT + 4 * i;
                if (row < p.M && c0 < p.L) {
                    double r4[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        // sum_s 256^s D_s exactly: hi = D6..D4, lo = D3..D0 (int64), then H = hi 2^5 + (lo >> 27) and the low
                        // 27 bits are both exactly representable, so fma(H, 2^27, lo27) rounds the exact integer ONCE
                        long long hi = (int)v[6][j];
                        hi = hi * 256 + (int)v[5][j];
                        hi = hi * 256 + (int)v[4][j];
                        long long lo = (int)v[3][j];
                        lo = lo * 256 + (int)v[2][j];
                        lo = lo * 256 + (int)v[1][j];
                        lo = lo * 256 + (int)v[0][j];
                        const long long H = hi * 32 + (lo >> 27);
                        const long long l27 = lo & ((1ll << 27) - 1);
                        const int c = c0 + j;
                        const int ex = c < p.L ? p.expo[c] - I8_FIXBITS : 0;
                        const double sc = __longlong_as_double((long long)(1023 + ex) << 52);   // 2^(e_c - 54), exact
                        r4[j] = fma((double)H, 134217728.0, (double)l27) * sc;
                        if ((dmask >> (4 * i + j)) & 1ull) bad = bad || (n_half * sc > p.tol * r4[j]);
                    }
                    double* o = p.out + (long long)row * p.ldo + c0;
                    if (c0 + 4 <= p.L && (p.ldo & 1) == 0 && (c0 & 1) == 0) {
                        *reinterpret_cast<double2*>(o) = make_double2(r4[0], r4[1]);
                        *reinterpret_cast<double2*>(o + 2) = make_double2(r4[2], r4[3]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if (c0 + j < p.L) o[j] = r4[j];
                    }
                }
            }
            if (bad) p.flags[row] = 1;
            // this warp has read its lanes of the accumulator: tell the MMA issuer (leader CTA)
            asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
            __syncwarp();
            if (lane == 0) g2_arrive_cluster(tempty + acc, 0u);
            if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    cluster_sync_all();                       // no CTA frees tensor memory or exits while its partner still uses the pair's resources
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_base), "n"(G2_TMEM_COLS));
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* f = nullptr;
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(f);
        else
            cudaGetLastError();
    }
    return fn;
}

// int8 matrix [rows][ld] (K-major), K bytes valid per row: boxes of 128 rows x 128 bytes, 128-byte swizzle, zero fill
bool make_map(CUtensorMap* tm, const void* base, long long rows, long long ld, long long K) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return false;
    cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t gstr[1] = {(cuuint64_t)ld};
    cuuint32_t box[2] = {(cuuint32_t)G2_BK, (cuuint32_t)G2_ROWS};
    cuuint32_t estr[2] = {1, 1};
    return fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(base), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace

// The 2-CTA kernel runs on the current device: the driver exports the TMA descriptor encoder, and the kernel may use its
// shared memory (the attribute is set here, before the first launch or graph capture on this device).
bool i8gemm2_ready() {
    if (!encode_fn()) return false;
    if (cudaFuncSetAttribute(i8gemm2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, G2_SMEM) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return true;
}

// out[m][c] (c < L) for counts [M][ldc] and tile-major digit planes [n_tiles * 252][ldp], contraction length K.
// Fused route: the epilogue recombines the planes, writes `out` and applies the guard.  Split-K route, when the 256 x 256
// tiles are too few to fill the CTA pairs (< 48) and the contraction is long enough to split: the exact int32 partial sums
// go to the planes D [i8_plane_rows(L)][ldd], and stats_i8_combine recombines them (and applies the guard).
// Needs i8gemm2_ready() on this device, K a multiple of 128, ldc and ldp multiples of 16, 16-byte aligned operands and at
// most 16 column tiles (K <= 32): the engine's buffers always satisfy them.  Returns the I8Route taken, 0 when one of
// these conditions fails or the launch does.
int launch_i8gemm2(const int8_t* Cn, long long ldc, int M, const int8_t* Pl, long long ldp, int L, int K, const int* expo,
                   double* out, long long ldo, const I8Guard* guard, int32_t* D, long long ldd, cudaStream_t st) {
    const int mt = (M + 255) / 256, nt = (L + G2_CPT - 1) / G2_CPT;
    if (K % G2_BK != 0 || (ldc % 16) || (ldp % 16) || M < 1 || L < 1 || nt > 16) return 0;
    if ((reinterpret_cast<uintptr_t>(Cn) & 15) || (reinterpret_cast<uintptr_t>(Pl) & 15)) return 0;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // few tiles (narrow shards, small tensors): split the contraction so that one wave of jobs fills the CTA pairs, with
    // at least 8 chunks per job
    const int kc = K / G2_BK;
    const int nsplit = mt * nt < 48 ? std::max(1, std::min(kc / 8, (sms / 2) / (mt * nt))) : 1;
    // the descriptors travel as kernel parameters (a CUDA graph keeps its own copy of them)
    alignas(64) CUtensorMap tm_cnt, tm_dig;
    if (!make_map(&tm_cnt, Cn, M, ldc, K) || !make_map(&tm_dig, Pl, (long long)nt * G2_CPT * G2_NP, ldp, K)) return 0;
    G2Args p{};
    p.M = M; p.L = L; p.k_chunks = kc; p.m_tiles = mt; p.n_tiles = nt; p.expo = expo; p.out = out; p.ldo = ldo;
    p.chunks_per_split = (kc + nsplit - 1) / nsplit;
    p.nsplit = (kc + p.chunks_per_split - 1) / p.chunks_per_split;
    p.D = D; p.ldd = ldd;
    if (p.nsplit > 1 &&
        cudaMemset2DAsync(D, (size_t)ldd * sizeof(int32_t), 0, (size_t)M * sizeof(int32_t), (size_t)nt * G2_CPT * G2_NP, st) != cudaSuccess)
        return 0;
    if (guard && p.nsplit == 1) {
        p.cntsum = guard->cntsum; p.flags = guard->flags; p.tol = guard->tol;
        for (int k = 0; k * (k + 3) / 2 < L; ++k) { const int c = k * (k + 3) / 2; p.diag_mask[c / G2_CPT] |= 1ull << (c % G2_CPT); }
    }
    const int pairs = std::min(sms / 2, mt * nt * p.nsplit);
    i8gemm2_kernel<<<2 * pairs, G2_THREADS, G2_SMEM, st>>>(tm_cnt, tm_dig, p);
    if (cudaGetLastError() != cudaSuccess) return 0;
    return p.nsplit > 1 ? I8_ROUTE_SPLITK : I8_ROUTE_FUSED;
}

}  // namespace btf
