// FP64, HBM and int8 tensor-core micro-benchmarks: the roofline denominators of the statistics kernels.
// MEASURED_PEAKS.json (driver-written) has HBM copy bandwidth and bf16 GEMM only; the
// FP64 pipes are measured here: independent DFMA chains and mma.sync.m8n8k4.f64 chains,
// and the int8 tensor pipe with resident operands (btf_i8_peak).
#include "../../include/btf_b200.h"
#include <cuda_runtime.h>
#include <stdio.h>

namespace {

template <int CH>
__global__ void __launch_bounds__(256) dfma_kernel(double* out, int iters, double a, double b) {
    double x[CH];
#pragma unroll
    for (int c = 0; c < CH; ++c) x[c] = threadIdx.x * 1e-3 + c;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int c = 0; c < CH; ++c) x[c] = fma(x[c], a, b);
    }
    double s = 0.0;
#pragma unroll
    for (int c = 0; c < CH; ++c) s += x[c];
    if (s == 123.456) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

template <int CH>
__global__ void __launch_bounds__(256) dmma_kernel(double* out, int iters, double a, double b) {
    double c0[CH], c1[CH];
#pragma unroll
    for (int c = 0; c < CH; ++c) { c0[c] = threadIdx.x * 1e-3; c1[c] = c; }
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int c = 0; c < CH; ++c)
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                         : "+d"(c0[c]), "+d"(c1[c]) : "d"(a), "d"(b));
    }
    double s = 0.0;
#pragma unroll
    for (int c = 0; c < CH; ++c) s += c0[c] + c1[c];
    if (s == 123.456) out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

__global__ void copy_kernel(const double4* __restrict__ src, double4* __restrict__ dst, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = src[i];
}

}  // namespace

extern "C" double btf_fp64_peak(int32_t device, int32_t mode, int32_t iters) {
    if (cudaSetDevice(device) != cudaSuccess) return -1.0;
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    const int blocks = prop.multiProcessorCount * 4;
    double* out = nullptr;
    cudaMalloc(&out, (size_t)blocks * 256 * sizeof(double));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    if (iters < 1) iters = 20000;
    constexpr int CH = 16;
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {
        cudaEventRecord(e0);
        if (mode == 0) dfma_kernel<CH><<<blocks, 256>>>(out, iters, 0.999999, 1e-9);
        else dmma_kernel<CH><<<blocks, 256>>>(out, iters, 0.999999, 1e-9);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        double flops;
        if (mode == 0) flops = 2.0 * CH * (double)iters * blocks * 256;
        else flops = 2.0 * 256.0 * CH * (double)iters * blocks * 8;   // 8 warps/block, 8x8x4 FMAs per DMMA
        double tf = flops / (ms * 1e-3) / 1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaError_t err = cudaGetLastError();
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(out);
    return err == cudaSuccess ? best : -1.0;
}

extern "C" double btf_hbm_copy_gbs(int32_t device, size_t bytes, int32_t iters) {
    if (cudaSetDevice(device) != cudaSuccess) return -1.0;
    double4 *a = nullptr, *b = nullptr;
    bytes = bytes / 32 * 32;
    if (cudaMalloc(&a, bytes) != cudaSuccess || cudaMalloc(&b, bytes) != cudaSuccess) { cudaFree(a); return -1.0; }
    cudaMemset(a, 1, bytes);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    double best = 0.0;
    for (int it = 0; it < iters + 1; ++it) {
        cudaEventRecord(e0);
        copy_kernel<<<148 * 16, 512>>>(a, b, bytes / 32);
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, e0, e1);
        double gbs = 2.0 * bytes / (ms * 1e-3) / 1e9;
        if (it > 0 && gbs > best) best = gbs;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(a); cudaFree(b);
    return best;
}

// ---- int8 tensor pipe (tcgen05.mma.kind::i8): every SM issues M = 128, N = 256, K = 32 MMAs on operands that stay in
// shared memory - no loads, no epilogue - so the rate is the pipe's, not the memory system's.
namespace btf {
namespace {

constexpr int I8_BM = 128, I8_BN = 256, I8_BK = 128;
constexpr int I8_A_BYTES = I8_BM * I8_BK, I8_B_BYTES = I8_BN * I8_BK, I8_STAGE_BYTES = I8_A_BYTES + I8_B_BYTES;
constexpr int I8_TMEM_COLS = 256;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(bar)), "r"(count));
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
