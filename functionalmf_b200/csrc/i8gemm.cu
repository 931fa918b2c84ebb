// Exact integer GEMM on the 5th-generation tensor cores:  D[M x N] (int32) = A[M x K] (int8) . B[N x K]^T (int8),
// both operands K-major in global memory.  tcgen05.mma.kind::i8 with the accumulator in tensor memory,
// operands staged in shared memory in the canonical 128-byte-swizzled K-major layout.
//
// Why it exists: the sufficient-statistic contractions out[m, l] = sum_k cnt[m, k] Z[k, l] have an
// INTEGER left operand (cnt = number of observed replicates, 0..R).  Writing every column of Z as a
// fixed-point number  Z[k, l] = scale_l 2^-54 sum_s 256^s d_s[k, l]  with signed 8-bit digits d_s turns
// the FP64 contraction into 7 int8 x int8 -> int32 contractions whose results are EXACT; the digits
// are recombined in integer arithmetic and rounded once (stats_i8.cu).  This file is the single-CTA 128 x 256 kernel
// with split-K (shapes with few tiles, the raw GEMM test hook); the large contractions run in i8gemm2.cu.  The FP64 pipe of the
// B200 peaks at 37 TFLOP/s; the int8 tensor pipe is two orders of magnitude faster, so even with
// eight digit planes the exact contraction is several times cheaper than the DMMA kernel.
//
// One CTA = one 128 x 256 tile of D, K streamed in 128-byte chunks through a 4-stage pipeline:
//   warps 1-4 (128 threads): cp.async producers (16-byte copies into the swizzled layout), later the epilogue
//   warp 0, one lane:        tcgen05.mma issuer; tcgen05.commit releases a stage / publishes the accumulator
// mbarriers: full[stage] (producers -> MMA), empty[stage] (MMA -> producers), accum (MMA -> epilogue).
#include <cstdio>
#include <cstdlib>
#include "kernels.h"

namespace btf {

namespace {

constexpr int I8_BM = 128, I8_BN = 256, I8_BK = 128, I8_STAGES = 4, I8_LAG = 2;
constexpr int I8_A_BYTES = I8_BM * I8_BK, I8_B_BYTES = I8_BN * I8_BK, I8_STAGE_BYTES = I8_A_BYTES + I8_B_BYTES;
constexpr int I8_SMEM = I8_STAGES * I8_STAGE_BYTES + 1024 /*alignment*/ + 256 /*barriers*/;
constexpr int I8_SMEM2 = 2 * I8_STAGE_BYTES + 1024 + 256;     // two-stage variant: two CTAs per SM
constexpr int I8_TMEM_COLS = 256;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t}\n" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}

// shared-memory matrix descriptor, K-major, 128-byte swizzle: 8-row x 128-byte atoms, 1024 bytes apart
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);        // start address, 16-byte units
    d |= (uint64_t)1 << 16;                         // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;               // stride byte offset between 8-row groups
    d |= (uint64_t)1 << 46;                         // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                         // SWIZZLE_128B
    return d;
}
// instruction descriptor: D = S32, A = B = signed 8-bit, both K-major, M = 128, N = 256
constexpr uint32_t I8_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(I8_BN >> 3) << 17) | ((uint32_t)(I8_BM >> 4) << 24);

__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(da), "l"(db), "r"(I8_IDESC), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}

struct I8Args {
    const int8_t* A; long long lda; int M;       // digits   [M][lda]
    const int8_t* B; long long ldb; int N;       // counts   [N][ldb]
    int K;                                       // multiple of 128 (both operands readable up to K)
    int32_t* D; long long ldd;                   // [M][ldd]
    int chunks_per_split;                        // gridDim.z > 1: split-K, partial tiles are added with integer atomics (exact, order independent)
};

}  // namespace

// STAGES = 4: one CTA per SM, deep pipeline (long contractions).  STAGES = 2: two CTAs per SM, so that one CTA's
// prologue (tensor-memory allocation, pipeline fill) and epilogue overlap the other's main loop (short contractions).
template <int STAGES>
__global__ void __launch_bounds__(160, STAGES > 2 ? 1 : 2) i8gemm_kernel(I8Args p) {
    constexpr int LAG = STAGES > 2 ? 2 : 1;
    extern __shared__ uint8_t smraw[];
    uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smraw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full = reinterpret_cast<uint64_t*>(sm + STAGES * I8_STAGE_BYTES);
    uint64_t* empty = full + STAGES;
    uint64_t* accum = empty + STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int m0 = blockIdx.x * I8_BM, n0 = blockIdx.y * I8_BN;
    const int c_first = blockIdx.z * p.chunks_per_split;
    const int nchunks = min(p.K / I8_BK - c_first, p.chunks_per_split);     // this CTA's share of the contraction
    const bool split = gridDim.z > 1;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full + s, 128); mbar_init(empty + s, 1); }
        mbar_init(accum, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "n"(I8_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem_d = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            // ===== MMA issuer
            for (int c = 0; c < nchunks; ++c) {
                const int s = c % STAGES;
                mbar_wait(full + s, (uint32_t)((c / STAGES) & 1));
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                const uint32_t a0 = smem_u32(sm + s * I8_STAGE_BYTES), b0 = a0 + I8_A_BYTES;
#pragma unroll
                for (int k = 0; k < I8_BK / 32; ++k)
                    umma_i8(tmem_d, umma_desc_sw128(a0 + 32 * k), umma_desc_sw128(b0 + 32 * k), (c > 0 || k > 0) ? 1u : 0u);
                umma_commit(empty + s);          // the stage is free once these MMAs have read it
            }
            umma_commit(accum);
        }
    } else {
        // ===== producers: 3072 16-byte copies per stage, 24 per thread; 8 consecutive threads cover one 128-byte row
        const int pt = tid - 32;
        auto issue = [&](int c) {
            const int s = c % STAGES;
            uint8_t* sa = sm + s * I8_STAGE_BYTES;
            uint8_t* sb = sa + I8_A_BYTES;
            const long long k0 = (long long)(c_first + c) * I8_BK;
#pragma unroll
            for (int j = 0; j < (I8_BM + I8_BN) * 8 / 128; ++j) {
                const int q = pt + 128 * j;
                const bool isA = q < I8_BM * 8;
                const int qq = isA ? q : q - I8_BM * 8;
                const int row = qq >> 3, c16 = qq & 7;
                const int grow = (isA ? m0 : n0) + row;
                const bool ok = grow < (isA ? p.M : p.N);
                const int8_t* src = (isA ? p.A + (long long)(ok ? grow : 0) * p.lda : p.B + (long long)(ok ? grow : 0) * p.ldb) + k0 + 16 * c16;
                uint8_t* dst = (isA ? sa : sb) + (row >> 3) * 1024 + (row & 7) * 128 + ((c16 ^ (row & 7)) << 4);
                const int nbytes = ok ? 16 : 0;      // rows past the end are zero-filled
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(smem_u32(dst)), "l"(src), "r"(nbytes));
            }
            asm volatile("cp.async.commit_group;\n" ::);
        };
        auto publish = [&](int c) {
            // the copies of chunk c have landed (generic proxy) -> make them visible to the tensor core (async proxy)
            asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
            mbar_arrive(full + (c % STAGES));
        };
        for (int c = 0; c < nchunks; ++c) {
            if (c >= STAGES) mbar_wait(empty + (c % STAGES), (uint32_t)(((c / STAGES) - 1) & 1));
            issue(c);
            if (c >= LAG) {
                asm volatile("cp.async.wait_group %0;\n" ::"n"(LAG));
                publish(c - LAG);
            }
        }
        // drain
        if (LAG >= 2 && nchunks >= 2) { asm volatile("cp.async.wait_group 1;\n" ::); publish(nchunks - 2); }
        asm volatile("cp.async.wait_group 0;\n" ::);
        if (nchunks >= 1) publish(nchunks - 1);

        // ===== epilogue: tensor memory -> registers -> global (a warp reads the 32 lanes of its quarter)
        mbar_wait(accum, 0);
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
        const int quarter = warp & 3;
        const int row = m0 + quarter * 32 + lane;
#pragma unroll 1
        for (int j = 0; j < I8_BN / 32; ++j) {
            uint32_t v[32];
            const uint32_t taddr = tmem_d + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(j * 32);
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
                : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
                  "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
                  "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
                  "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                : "r"(taddr));
            asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
            if (row < p.M) {
                int32_t* drow = p.D + (long long)row * p.ldd + n0 + j * 32;
                if (split) {
#pragma unroll
                    for (int q = 0; q < 32; ++q)
                        if (n0 + j * 32 + q < p.N && v[q] != 0u) atomicAdd(drow + q, (int)v[q]);
                } else if (n0 + j * 32 + 32 <= p.N) {
#pragma unroll
                    for (int q = 0; q < 8; ++q)
                        *reinterpret_cast<int4*>(drow + 4 * q) = make_int4((int)v[4 * q], (int)v[4 * q + 1], (int)v[4 * q + 2], (int)v[4 * q + 3]);
                } else {
#pragma unroll
                    for (int q = 0; q < 32; ++q)
                        if (n0 + j * 32 + q < p.N) drow[q] = (int)v[q];
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (warp == 0) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_d), "n"(I8_TMEM_COLS));
    }
}

// D[M][ldd] = A[M][lda] . B[N][ldb]^T over k < K (K a multiple of 128); device pointers
int launch_i8gemm(const int8_t* A, long long lda, int M, const int8_t* B, long long ldb, int N, int K, int32_t* D,
                  long long ldd, cudaStream_t st) {
    if (K % I8_BK != 0 || (lda % 16) || (ldb % 16) || (ldd % 4)) return 1;
    static PerDeviceOnce attr_once;
    if (attr_once.first()) {
        if (cudaFuncSetAttribute(i8gemm_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, I8_SMEM) != cudaSuccess) return 2;
        if (cudaFuncSetAttribute(i8gemm_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, I8_SMEM2) != cudaSuccess) return 2;
    }
    const int mt = (M + I8_BM - 1) / I8_BM, nt = (N + I8_BN - 1) / I8_BN, nchunks = K / I8_BK;
    // split-K when the tiles alone cannot fill the GPU (few rows: multi-GPU shards, small tensors)
    int nsplit = 1;
    if (mt * nt < 148) {
        nsplit = 148 / (mt * nt);
        const int cap = nchunks / 8 > 0 ? nchunks / 8 : 1;      // keep at least 8 chunks per CTA
        if (nsplit > cap) nsplit = cap;
        if (nsplit < 1) nsplit = 1;
    }
    const int cps = (nchunks + nsplit - 1) / nsplit;
    nsplit = (nchunks + cps - 1) / cps;
    if (nsplit > 1) {
        if (cudaMemsetAsync(D, 0, (size_t)M * ldd * sizeof(int32_t), st) != cudaSuccess) return 4;
    }
    I8Args p{A, lda, M, B, ldb, N, K, D, ldd, cps};
    dim3 grid(mt, nt, nsplit);
    // short contractions with many tiles: two CTAs per SM hide the per-CTA prologue and epilogue
    if (cps <= 64 && mt * nt * nsplit >= 2 * 148) i8gemm_kernel<2><<<grid, 160, I8_SMEM2, st>>>(p);
    else i8gemm_kernel<4><<<grid, 160, I8_SMEM, st>>>(p);
    return cudaGetLastError() == cudaSuccess ? 0 : 3;
}

}  // namespace btf

// test / benchmark entry: host operands in, int32 result out; returns the kernel time of `reps` launches (ms) or < 0
extern "C" double btf_i8gemm_test(int device, const int8_t* A, const int8_t* B, int32_t* D, int M, int N, int K, int reps) {
    using namespace btf;
    if (cudaSetDevice(device) != cudaSuccess) return -1.0;
    int8_t *dA = nullptr, *dB = nullptr;
    int32_t* dD = nullptr;
    const long long ldd = (N + 3) & ~3;                      // rows of D start on 16-byte boundaries
    const size_t na = (size_t)M * K, nb = (size_t)N * K, nd = (size_t)M * ldd;
    if (cudaMalloc(&dA, na) || cudaMalloc(&dB, nb) || cudaMalloc(&dD, nd * 4)) return -2.0;
    cudaMemcpy(dA, A, na, cudaMemcpyHostToDevice);
    cudaMemcpy(dB, B, nb, cudaMemcpyHostToDevice);
    cudaMemset(dD, 0xff, nd * 4);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    int rc = launch_i8gemm(dA, K, M, dB, K, N, K, dD, ldd, 0);
    if (rc || cudaDeviceSynchronize() != cudaSuccess) {
        fprintf(stderr, "i8gemm: rc %d, %s\n", rc, cudaGetErrorString(cudaGetLastError()));
        return -3.0;
    }
    cudaEventRecord(e0);
    for (int r = 0; r < reps; ++r) launch_i8gemm(dA, K, M, dB, K, N, K, dD, ldd, 0);
    cudaEventRecord(e1);
    if (cudaDeviceSynchronize() != cudaSuccess) return -4.0;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaMemcpy2D(D, (size_t)N * 4, dD, (size_t)ldd * 4, (size_t)N * 4, M, cudaMemcpyDeviceToHost);
    cudaFree(dA); cudaFree(dB); cudaFree(dD);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return (double)ms;
}

// ---------------------------------------------------------------------------------------------------------
// Roofline denominator of the int8 tensor pipe: every SM issues tcgen05.mma.kind::i8 (M = 128, N = 256, K = 32) on
// operands that stay in shared memory - no loads, no epilogue - so the rate is the pipe's, not the memory system's.
namespace btf {
namespace {
__global__ void __launch_bounds__(128, 1) i8_peak_kernel(int iters, int* sink) {
    extern __shared__ uint8_t smraw[];
    uint8_t* sm = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smraw) + 1023) & ~(uintptr_t)1023);
    uint64_t* done = reinterpret_cast<uint64_t*>(sm + I8_STAGE_BYTES);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int e = tid; e < I8_STAGE_BYTES / 4; e += 128) reinterpret_cast<uint32_t*>(sm)[e] = 0x01ff0201u * (uint32_t)(e % 7);
    if (tid == 0) { mbar_init(done, 1); asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(tmem_slot)), "n"(I8_TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
    }
    asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem_d = *tmem_slot;
    if (tid == 0) {
        const uint32_t a0 = smem_u32(sm), b0 = a0 + I8_A_BYTES;
        for (int it = 0; it < iters; ++it) {
#pragma unroll
            for (int k = 0; k < I8_BK / 32; ++k)
                umma_i8(tmem_d, umma_desc_sw128(a0 + 32 * k), umma_desc_sw128(b0 + 32 * k), (it > 0 || k > 0) ? 1u : 0u);
        }
        umma_commit(done);
        mbar_wait(done, 0);
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    }
    __syncthreads();
    if (warp == 0) {
        uint32_t v;
        asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];\n" : "=r"(v) : "r"(tmem_d));
        asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
        if (v == 0x7fffffffu) sink[0] = (int)v;
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem_d), "n"(I8_TMEM_COLS));
}
}  // namespace
}  // namespace btf

// int8 tensor throughput with resident operands, in Top/s (2 * MACs); best of 3 timed launches after a warm-up
extern "C" double btf_i8_peak(int32_t device, int32_t iters) {
    using namespace btf;
    if (cudaSetDevice(device) != cudaSuccess) return -1.0;
    int sms = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    const int smem = I8_STAGE_BYTES + 1024 + 64;
    if (cudaFuncSetAttribute(i8_peak_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) return -2.0;
    int* sink = nullptr;
    if (cudaMalloc(&sink, 4) != cudaSuccess) return -2.0;
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {
        cudaEventRecord(e0);
        i8_peak_kernel<<<sms, 128, smem>>>(iters, sink);
        cudaEventRecord(e1);
        if (cudaEventSynchronize(e1) != cudaSuccess) { best = -3.0; break; }
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        const double ops = 2.0 * I8_BM * I8_BN * I8_BK * (double)iters * sms;
        const double tops = ops / (ms * 1e-3) / 1e12;
        if (rep > 0 && tops > best) best = tops;
    }
    if (cudaGetLastError() != cudaSuccess && best > 0) best = -4.0;
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(sink);
    return best;
}
