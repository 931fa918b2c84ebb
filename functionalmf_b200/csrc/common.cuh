// Shared device utilities of the BTF engine: device scalar block, Philox4x32-10
// counter-based RNG, FP64 normal / gamma variates, reductions.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

namespace btf {

// All scalar state lives on the device so a sweep needs no host round trip
// (and can be replayed as a CUDA graph).
struct Scalars {
    double nu2;        // Gaussian observation variance (factor.py:411-416)
    double sigma2;     // row-embedding variance (factor.py:130-132)
    double lam2;       // global shrinkage (factor.py:143-153)
    double lam2_a;
    double ss_total;   // sum of squares of all observed entries (constant)
    double n_obs;      // number of observed entries (constant)
    double resid;      // sum (Mu - Y)^2 over observed entries for the current (W, V)
    double w_sumsq;    // sum of squares of the free entries of W
    double nu2_a_post, nu2_b_post;       // diagnostics
    double lam2_rate, lam2_shape;        // diagnostics
    unsigned long long sweep;            // sweep counter (Philox counter word)
    int info_w;        // # rows whose Cholesky failed in the last sweep
    int info_v;        // # columns whose Cholesky failed after all retries
    int retries_v;     // total jitter retries in the last sweep
    int pad;
};

// RNG stream identifiers (mixed into the Philox key)
enum Stream : uint32_t {
    STREAM_W = 1, STREAM_V = 2, STREAM_TAU = 3, STREAM_LAM = 4, STREAM_SIGMA = 5,
    STREAM_NU = 6, STREAM_PG = 7, STREAM_R = 8, STREAM_GASS_W = 9, STREAM_GASS_V = 10
};

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
        uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += W0; k.y += W1;
    }
    return c;
}

// A per-element generator: counter = (index lo, index hi, draw #, sweep),
// key = (seed lo ^ stream * golden, seed hi ^ sweep hi).
struct Rng {
    uint4 ctr;
    uint2 key;
    __device__ __forceinline__ Rng(uint64_t seed, uint32_t stream, unsigned long long sweep, uint64_t index) {
        key = make_uint2((uint32_t)seed ^ (stream * 0x9E3779B9u), (uint32_t)(seed >> 32) ^ (uint32_t)(sweep >> 32));
        ctr = make_uint4((uint32_t)index, (uint32_t)(index >> 32), 0u, (uint32_t)sweep);
    }
    __device__ __forceinline__ uint4 next4() { uint4 r = philox4x32_10(ctr, key); ctr.z += 1u; return r; }
    static __device__ __forceinline__ double to_unit(uint32_t hi, uint32_t lo) {
        // 53-bit uniform in the open interval (0, 1)
        unsigned long long b = (((unsigned long long)hi << 32) | lo) >> 11;
        return ((double)b + 0.5) * (1.0 / 9007199254740992.0);
    }
    __device__ __forceinline__ double2 uniform2() { uint4 r = next4(); return make_double2(to_unit(r.x, r.y), to_unit(r.z, r.w)); }
    __device__ __forceinline__ double uniform() { return uniform2().x; }
    __device__ __forceinline__ double2 normal2() {
        double2 u = uniform2();
        double r = sqrt(-2.0 * log(u.x));
        double s, c;
        sincospi(2.0 * u.y, &s, &c);
        return make_double2(r * c, r * s);
    }
    __device__ __forceinline__ double normal() { return normal2().x; }
    __device__ __forceinline__ double exponential() { return -log(uniform()); }
    // Marsaglia & Tsang (2000) Gamma(a, 1); a < 1 by the boost G(a+1) U^(1/a)
    __device__ double gamma(double a) {
        if (a == 1.0) return exponential();
        double boost = 1.0;
        if (a < 1.0) { boost = pow(uniform(), 1.0 / a); a += 1.0; }
        const double d = a - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
        for (int it = 0; it < 1000; ++it) {
            double2 nu = normal2();            // .x normal; reuse .y? keep independent draws simple
            double x = nu.x, v = 1.0 + c * x;
            if (v <= 0.0) continue;
            v = v * v * v;
            double u = uniform();
            double x2 = x * x;
            if (u < 1.0 - 0.0331 * x2 * x2) return d * v * boost;
            if (log(u) < 0.5 * x2 + d * (1.0 - v + log(v))) return d * v * boost;
        }
        return d * boost;
    }
};

__device__ __forceinline__ double clampd(double x, double lo, double hi) { return fmin(fmax(x, lo), hi); }

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Deterministic block sum (fixed tree); result valid in thread 0. `sh` >= 32 doubles.
__device__ __forceinline__ double block_sum(double v, double* sh) {
    v = warp_sum(v);
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (lane == 0) sh[w] = v;
    __syncthreads();
    double r = 0.0;
    if (w == 0) {
        r = lane < nw ? sh[lane] : 0.0;
        r = warp_sum(r);
    }
    return r;
}

__host__ __device__ __forceinline__ int tri(int k1, int k2) { return k1 * (k1 + 1) / 2 + k2; }   // k2 <= k1

}  // namespace btf
