// K1 on the integer tensor cores: the Gaussian sufficient statistics with count weights,
//   out[m, c] = sum_k cnt[m, k] Z[k, c]   (c < L: packed products F[k,k1] F[k,k2]),   out[m, L + j] = sum_k S[m, k] F[k, j],
// computed EXACTLY for the product block and in FP64 for the (small) linear block.
//
// The left operand of the product block is an integer (cnt = number of observed replicates), so every
// column of Z is written as a fixed-point number against a power-of-two column scale,
//   Z[k, c] ~ 2^(e_c - 54) q[k, c],   q = round(Z 2^(54 - e_c)),  |q| <= 2^54,   q = sum_{s<7} 256^s d_s,  d_s in [-128, 127],
// and the seven digit planes are contracted with the counts by ONE exact int8 x int8 -> int32 GEMM on the
// tcgen05 tensor cores (i8gemm2.cu: 2-CTA pairs, TMA, recombination in the epilogue, or split-K through int32 planes
// for shapes with few tiles):  D[(s, c), m] = sum_k d_s[k, c] cnt[m, k].  The planes are recombined in integer arithmetic
// (two int64 Horner sums re-split into parts that are exactly representable in a double) and rounded once.  The only error is the 2^-55 (relative to the column maximum) rounding of Z
// itself - below the rounding noise of an FP64 accumulation over the same number of terms - and the result
// does not depend on the order of summation at all.
// Replaces the DMMA kernel for the product block (L of the L + K columns: 89 % of the flops at K = 16);
// the linear block stays on the FP64 pipe (sf_kernel, HBM bound: it has to read S once).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include "kernels.h"
#include "stats_common.cuh"

namespace btf {

bool i8gemm2_ready();
int launch_i8gemm2(const int8_t* Cn, long long ldc, int M, const int8_t* Pl, long long ldp, int L, int K, const int* expo,
                   double* out, long long ldo, const I8Guard* guard, int32_t* D, long long ldd, cudaStream_t st);

namespace {

constexpr int NPLANES = I8_NPLANES;
constexpr int FIXBITS = I8_FIXBITS;

__device__ __forceinline__ void pair_of(int c, int& k1, int& k2) {
    k1 = (int)((sqrt(8.0 * c + 1.0) - 1.0) * 0.5);
    while (k1 * (k1 + 1) / 2 > c) --k1;
    while ((k1 + 1) * (k1 + 2) / 2 <= c) ++k1;
    k2 = c - k1 * (k1 + 1) / 2;
}

// colmax[c] = max_r |F[r,k1] F[r,k2]| (bit pattern of a non-negative double, so an integer max is exact).
// A block stages 128 rows of F in shared memory; thread c (and c + 256, ...) scans them.
__global__ void __launch_bounds__(256) zmax_kernel(const double* __restrict__ F, int rows, int K, int L,
                                                   unsigned long long* __restrict__ colmax) {
    extern __shared__ __align__(16) double zms[];
    const int rb = blockIdx.x * 128;
    const int nr = min(128, rows - rb);
    for (int e = threadIdx.x; e < nr * K; e += 256) zms[e] = F[(long long)rb * K + e];
    __syncthreads();
    for (int c = threadIdx.x + 256 * blockIdx.y; c < L; c += 256 * gridDim.y) {
        int k1, k2;
        pair_of(c, k1, k2);
        double m0 = 0.0, m1 = 0.0;
        int r = 0;
        for (; r + 2 <= nr; r += 2) {
            m0 = fmax(m0, fabs(zms[r * K + k1] * zms[r * K + k2]));
            m1 = fmax(m1, fabs(zms[(r + 1) * K + k1] * zms[(r + 1) * K + k2]));
        }
        if (r < nr) m0 = fmax(m0, fabs(zms[r * K + k1] * zms[r * K + k2]));
        const double m = fmax(m0, m1);
        if (m > 0.0) atomicMax(colmax + c, (unsigned long long)__double_as_longlong(m));
    }
}

// digit planes, tile-major: planes[i8_plane_row(c, s) ldk + r] = d_s of q[r, c] (zero for the padding columns
// L <= c < n_tiles 36).  A block stages 256 rows of F in shared memory;
// thread (tx, ty): rows 4 tx .. 4 tx + 3 (one 4-byte store per plane), columns c = ty, ty + 4, ...
__global__ void __launch_bounds__(256) zdigits_kernel(const double* __restrict__ F, int rows, int rows_pad, int K, int L,
                                                      const unsigned long long* __restrict__ colmax,
                                                      int* __restrict__ expo, int8_t* __restrict__ planes, long long ldk) {
    extern __shared__ __align__(16) double zsm[];
    const int KS = K + 1;
    double* Fs = zsm;                                              // [256][K + 1]
    unsigned short* pairs = reinterpret_cast<unsigned short*>(Fs + 256 * KS);   // [L]  (k1 << 8 | k2)
    const int rb = blockIdx.x * 256;
    for (int e = threadIdx.x; e < 256 * K; e += 256) {
        const int r = e / K, k = e - r * K;
        Fs[r * KS + k] = (rb + r < rows) ? F[(long long)(rb + r) * K + k] : 0.0;
    }
    for (int c = threadIdx.x; c < L; c += 256) {
        int k1, k2;
        pair_of(c, k1, k2);
        pairs[c] = (unsigned short)((k1 << 8) | k2);
    }
    __syncthreads();
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
    const int r0 = rb + 4 * tx;
    if (r0 >= rows_pad) return;
    const int Lslots = (L + I8_COLS_PER_TILE - 1) / I8_COLS_PER_TILE * I8_COLS_PER_TILE;
    for (int c = ty + 4 * blockIdx.y; c < Lslots; c += 4 * gridDim.y) {       // gridDim.y: column groups (few factor rows)
        unsigned dig[NPLANES];
#pragma unroll
        for (int s = 0; s < NPLANES; ++s) dig[s] = 0u;
        if (c < L) {
            const int k1 = pairs[c] >> 8, k2 = pairs[c] & 0xff;
            const double mx = __longlong_as_double((long long)colmax[c]);
            const int e = mx > 0.0 ? ilogb(mx) + 1 : 0;                // max < 2^e
            if (r0 == 0) expo[c] = e;
            // 2^(54 - e) as a double: the scaling is then ONE exact multiplication per entry (scalbn is a library call of ~25
            // instructions); exponents outside the normal range (column maxima below 2^-968 or above 2^1000) keep scalbn
            const int se = FIXBITS - e;
            const bool fast = se > -1000 && se < 1000;
            const double sc = fast ? __longlong_as_double((long long)(1023 + se) << 52) : 1.0;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const double* fr = Fs + (4 * tx + u) * KS;
                const double z = fr[k1] * fr[k2];
                // signed base-256 digits without a carry chain: add 128 at every digit position (C = sum_{s<7} 128 256^s
                // < 2^55.1, so q + C is in (0, 2^56)), read the unsigned 8-bit fields, subtract 128 from each
                const unsigned long long qq =
                    (unsigned long long)(__double2ll_rn(fast ? z * sc : scalbn(z, se)) + 0x0080808080808080ll);
#pragma unroll
                for (int s = 0; s < NPLANES; ++s) {
                    const int d = (int)((qq >> (8 * s)) & 255ull) - 128;   // in [-128, 127]
                    dig[s] |= ((unsigned)(d & 0xff)) << (8 * u);
                }
            }
        }
#pragma unroll
        for (int s = 0; s < NPLANES; ++s)
            *reinterpret_cast<unsigned*>(planes + (long long)i8_plane_row(c, s) * ldk + r0) = dig[s];
    }
}

// out[split][m][j] = sum_k S[m,k] F[k,j] over the split's k range: FP64 tensor pipe, HBM bound.
// 128 rows x KC contraction elements per stage, NST stages; a warp owns 16 rows x all columns = 2 CT independent
// accumulator chains (the FP64 mma has a long latency: two chains left the pipe 40 % idle).
// Work items (row tile, split) are dealt round-robin to the CTAs of the grid; launch_sf_t gives every item its own
// CTA (KC = 32, two stages, two CTAs per SM).
template <int KB, bool TRANS, int KC, int NST, int MINB>
__global__ void __launch_bounds__(256, MINB) sf_kernel(const double* __restrict__ S, long long lds, const double* __restrict__ F,
                                                       int K, int m_valid, int nchunks, int chunks_per_split, int m_tiles,
                                                       int nitems, double* __restrict__ out) {
    constexpr int BM = 128, FS = KB + 4, CT = KB / 8;
    constexpr int SROWS = TRANS ? KC : BM, SCOLS = TRANS ? BM : KC, SS = SCOLS + 4;   // strides = 4 (mod 16) doubles
    extern __shared__ __align__(16) double smf[];
    double* Ssm = smf;                         // [NST][SROWS][SS]   (!TRANS: [m][k], TRANS: [k][m])
    double* Fsm = smf + NST * SROWS * SS;      // [NST][KC][FS]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // zero the padding columns of the F tiles once (K < KB)
    for (int e = tid; e < NST * KC * FS; e += 256) Fsm[e] = 0.0;
    __syncthreads();
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
        const int mt = item % m_tiles, sp = item / m_tiles;
        const int m0 = mt * BM;
        const int c_begin = sp * chunks_per_split, c_end = min(nchunks, c_begin + chunks_per_split);
        auto load = [&](int stage, int chunk) {
            const long long k0 = (long long)chunk * KC;
            double* sd = Ssm + stage * SROWS * SS;
            constexpr int CPR = SCOLS / 2;       // 16-byte copies per row
            for (int e = tid; e < SROWS * CPR; e += 256) {
                const int r = e / CPR, q = e - r * CPR;
                const double* src = TRANS ? S + (k0 + r) * lds + m0 + 2 * q : S + (long long)(m0 + r) * lds + k0 + 2 * q;
                cp_async16(sd + r * SS + 2 * q, src);
            }
            double* fd = Fsm + stage * KC * FS;
            for (int e = tid; e < KC * K / 2; e += 256) {
                const int r = (2 * e) / K, cidx = (2 * e) - r * K;
                cp_async16(fd + r * FS + cidx, F + (k0 + r) * K + cidx);
            }
        };
        double acc[2][CT][2];
#pragma unroll
        for (int r = 0; r < 2; ++r)
#pragma unroll
            for (int c = 0; c < CT; ++c) acc[r][c][0] = acc[r][c][1] = 0.0;
#pragma unroll
        for (int s0 = 0; s0 < NST - 1; ++s0) {
            if (c_begin + s0 < c_end) load(s0, c_begin + s0);
            cp_async_commit();
        }
        for (int c = c_begin; c < c_end; ++c) {
            const int stg = (c - c_begin) % NST;
            if (c + NST - 1 < c_end) load((c - c_begin + NST - 1) % NST, c + NST - 1);
            cp_async_commit();
            cp_async_wait<NST - 1>();
            __syncthreads();
            const double* sd = Ssm + stg * SROWS * SS;
            const double* fd = Fsm + stg * KC * FS;
            const int ml = warp * 16 + (lane >> 2);
#pragma unroll
            for (int kk = 0; kk < KC / 4; ++kk) {
                const int kl = kk * 4 + (lane & 3);
                const double a0 = TRANS ? sd[kl * SS + ml] : sd[ml * SS + kl];
                const double a1 = TRANS ? sd[kl * SS + ml + 8] : sd[(ml + 8) * SS + kl];
#pragma unroll
                for (int ct = 0; ct < CT; ++ct) {
                    const double bv = fd[kl * FS + ct * 8 + (lane >> 2)];
                    dmma(acc[0][ct][0], acc[0][ct][1], a0, bv);
                    dmma(acc[1][ct][0], acc[1][ct][1], a1, bv);
                }
            }
            __syncthreads();
        }
        cp_async_wait<0>();
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int m = m0 + warp * 16 + r * 8 + (lane >> 2);
            if (m < m_valid) {
                double* o = out + ((long long)sp * m_valid + m) * K;
#pragma unroll
                for (int ct = 0; ct < CT; ++ct)
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int j = ct * 8 + (lane & 3) * 2 + h;
                        if (j < K) o[j] = acc[r][ct][h];
                    }
            }
        }
    }
}

// out[m][c] = 2^(e_c - 54) sum_s 256^s D[i8_plane_row(c, s) ldn + m]  (32 x 32 tiles through shared memory),
// out[m][L + j] = sum_split bpart[split][m][j]
__global__ void __launch_bounds__(256) i8_combine_kernel(const int32_t* __restrict__ D, long long ldn, const int* __restrict__ expo,
                                                         const double* __restrict__ bpart, int nsplit_b, int m_valid, int L,
                                                         int K, double* __restrict__ out, int first_cy,
                                                         long long bpart_m0, long long bpart_rows, I8Guard g, int use_guard) {
    __shared__ double tile[32][33];
    const int nco = L + K;
    const int m0 = blockIdx.x * 32, c0 = (blockIdx.y + first_cy) * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;     // 32 x 8
    if (c0 < L) {
        for (int cy = ty; cy < 32; cy += 8) {
            const int c = c0 + cy, m = m0 + tx;
            double v = 0.0;
            if (c < L && m < m_valid) {
                const int32_t* d = D + m;
                long long hi = d[(long long)i8_plane_row(c, 6) * ldn];
                hi = hi * 256 + d[(long long)i8_plane_row(c, 5) * ldn];
                hi = hi * 256 + d[(long long)i8_plane_row(c, 4) * ldn];
                long long lo = d[(long long)i8_plane_row(c, 3) * ldn];
                lo = lo * 256 + d[(long long)i8_plane_row(c, 2) * ldn];
                lo = lo * 256 + d[(long long)i8_plane_row(c, 1) * ldn];
                lo = lo * 256 + d[(long long)i8_plane_row(c, 0) * ldn];
                // H = hi 2^5 + (lo >> 27) and the low 27 bits are exactly representable: one rounding of the exact integer
                const long long H = hi * 32 + (lo >> 27);
                const long long l27 = lo & ((1ll << 27) - 1);
                v = scalbn(fma((double)H, 134217728.0, (double)l27), expo[c] - FIXBITS);
                if (use_guard) {
                    int kk = (int)((sqrtf(8.0f * c + 9.0f) - 3.0f) * 0.5f);             // is c a diagonal column k (k + 3) / 2 ?
                    while (kk * (kk + 3) / 2 > c) --kk;
                    while ((kk + 1) * (kk + 4) / 2 <= c) ++kk;
                    if (kk * (kk + 3) / 2 == c && scalbn((double)g.cntsum[m], expo[c] - (FIXBITS + 1)) > g.tol * v) g.flags[m] = 1;
                }
            }
            tile[cy][tx] = v;
        }
        __syncthreads();
        for (int my = ty; my < 32; my += 8) {
            const int m = m0 + my, c = c0 + tx;
            if (m < m_valid && c < L) out[(long long)m * nco + c] = tile[tx][my];
        }
    } else {
        if (use_guard && blockIdx.x == 0 && threadIdx.x == 0) *g.nflag = 0;     // (the fallback kernel counts what it recomputes)
        // the linear block: columns L .. L+K-1 (this block row handles all of them for its 32 rows)
        for (int e = threadIdx.x; e < 32 * K; e += 256) {
            const int m = m0 + e / K, j = e % K;
            if (m < m_valid) {
                double s = 0.0;
                for (int sp = 0; sp < nsplit_b; ++sp) s += bpart[((long long)sp * bpart_rows + bpart_m0 + m) * K + j];
                out[(long long)m * nco + L + j] = s;
            }
        }
    }
}

// ---- element-wise guard of the fixed-point product block.
// Every entry of Z is rounded to a multiple of 2^(e_c - 54), so |out[m][c] - exact| <= 2^(e_c - 55) n_m with
// n_m = sum_k cnt[m][k].  That is 2^-55 relative to the COLUMN maximum: fine normwise, but a row whose observed cells
// all sit where |Z| is far below the column maximum (structured missingness + badly scaled factors) gets a large
// RELATIVE error.  The diagonal columns c = (k, k) are sums of non-negative terms, so bound / out[m][(k,k)] is the true
// relative accuracy of the row's precision matrix; the kernels that produce the block (the GEMM epilogue / the
// recombination kernel) flag the rows where it exceeds `tol`, and this kernel recomputes those rows in plain FP64:
// out[m][c] (c < L) = sum_k B[m][k] F[k,k1] F[k,k2].  A CTA scans a contiguous range of flags, then works through the
// rows it found: 128-row slabs of F in shared memory, thread t owns the packed columns t, t + 256, ...
template <int MAXC>
__global__ void __launch_bounds__(256) i8_fallback_kernel(const uint8_t* __restrict__ B, long long ldb, const double* __restrict__ F,
                                                          int f_rows, int K, int L, int m_valid, unsigned char* __restrict__ flags,
                                                          int* __restrict__ nflag, double* __restrict__ out, int nco) {
    extern __shared__ __align__(16) double fsm[];               // [128][K] + 128 counts
    __shared__ int list[64];
    __shared__ int nlist;
    double* Fs = fsm;
    double* Cs = fsm + 128 * K;
    const int per = (m_valid + gridDim.x - 1) / gridDim.x;
    const int lo = blockIdx.x * per, hi = min(m_valid, lo + per);
    int k1[MAXC], k2[MAXC];
#pragma unroll
    for (int q = 0; q < MAXC; ++q) { k1[q] = k2[q] = 0; const int c = threadIdx.x + 256 * q; if (c < L) pair_of(c, k1[q], k2[q]); }
    for (int base = lo; base < hi; base += 64) {                // (at most 64 rows per round keeps the list in shared memory)
        if (threadIdx.x == 0) nlist = 0;
        __syncthreads();
        if (threadIdx.x < 64 && base + (int)threadIdx.x < hi && flags[base + threadIdx.x]) {
            list[atomicAdd(&nlist, 1)] = base + threadIdx.x;
            flags[base + threadIdx.x] = 0;
        }
        __syncthreads();
        const int n = nlist;
        if (n && threadIdx.x == 0) atomicAdd(nflag, n);
        for (int it = 0; it < n; ++it) {
            const int m = list[it];
            double acc[MAXC][2];
#pragma unroll
            for (int q = 0; q < MAXC; ++q) acc[q][0] = acc[q][1] = 0.0;
            for (int r0 = 0; r0 < f_rows; r0 += 128) {
                const int nr = min(128, f_rows - r0);
                __syncthreads();
                for (int e = threadIdx.x; e < nr * K; e += 256) Fs[e] = F[(long long)r0 * K + e];
                for (int e = threadIdx.x; e < 128; e += 256) Cs[e] = e < nr ? (double)B[(long long)m * ldb + r0 + e] : 0.0;
                __syncthreads();
#pragma unroll
                for (int q = 0; q < MAXC; ++q) {
                    if (threadIdx.x + 256 * q < L) {
                        for (int r = 0; r < nr; r += 2) {
                            const double c0 = Cs[r], c1 = (r + 1 < nr) ? Cs[r + 1] : 0.0;
                            if (c0 != 0.0) acc[q][0] = fma(c0, Fs[r * K + k1[q]] * Fs[r * K + k2[q]], acc[q][0]);
                            if (c1 != 0.0) acc[q][1] = fma(c1, Fs[(r + 1) * K + k1[q]] * Fs[(r + 1) * K + k2[q]], acc[q][1]);
                        }
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < MAXC; ++q) {
                const int c = threadIdx.x + 256 * q;
                if (c < L) out[(long long)m * nco + c] = acc[q][0] + acc[q][1];
            }
        }
        __syncthreads();
    }
}

// cntsum[m] = sum_k B[m][k] (uint8 rows of length kdim, 16-byte aligned): one warp per row
__global__ void __launch_bounds__(256) count_rows_kernel(const uint8_t* __restrict__ B, long long ldb, int m_valid, int kdim,
                                                         unsigned* __restrict__ cntsum) {
    const int m = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (m >= m_valid) return;
    const uint4* row = reinterpret_cast<const uint4*>(B + (long long)m * ldb);
    unsigned s = 0;
    for (int q = lane; q < kdim / 16; q += 32) {
        const uint4 v = row[q];
        s += __vsadu4(v.x, 0u) + __vsadu4(v.y, 0u) + __vsadu4(v.z, 0u) + __vsadu4(v.w, 0u);     // sum of the 4 bytes of each word
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) cntsum[m] = s;
}

// dst[p][i] = src[i][p]  (uint8), 32 x 32 tiles
__global__ void __launch_bounds__(256) transpose_u8_kernel(const uint8_t* __restrict__ src, long long lds, int rows, int cols,
                                                           uint8_t* __restrict__ dst, long long ldd) {
    __shared__ uint8_t tile[32][33];
    const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int y = ty; y < 32; y += 8) {
        const int r = r0 + y, c = c0 + tx;
        tile[y][tx] = (r < rows && c < cols) ? src[(long long)r * lds + c] : (uint8_t)0;
    }
    __syncthreads();
    for (int y = ty; y < 32; y += 8) {
        const int c = c0 + y, r = r0 + tx;
        if (c < cols && r < rows) dst[(long long)c * ldd + r] = tile[tx][y];
    }
}

// contraction chunks of 32 through a 2-stage ring, two CTAs per SM, one CTA per (tile, split) item
template <int KB, bool TRANS>
void launch_sf_t(const double* S, long long lds, const double* F, int K, int m_valid, int m_tiles, int nchunks, int nsplit,
                 double* out, cudaStream_t st) {
    constexpr int KC = 32, NST = 2;
    const size_t smem = (size_t)(NST * (TRANS ? KC * 132 : 128 * (KC + 4)) + NST * KC * (KB + 4)) * sizeof(double);
    auto kern = sf_kernel<KB, TRANS, KC, NST, 2>;
    static PerDeviceOnce once;
    if (once.first()) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    const int cps = (nchunks + nsplit - 1) / nsplit;
    const int nitems = m_tiles * nsplit;
    kern<<<nitems, 256, smem, st>>>(S, lds, F, K, m_valid, nchunks, cps, m_tiles, nitems, out);
}

}  // namespace

bool stats_i8_supported(int K, int nreps, long long kdim_row, long long kdim_col) {
    if (!(K == 8 || K == 16 || K == 32)) return false;
    if (nreps < 1 || nreps > 127) return false;
    const long long kd = kdim_row > kdim_col ? kdim_row : kdim_col;
    if (kd * nreps * 128 >= (1ll << 31)) return false;      // the int32 accumulators cannot overflow
    return i8gemm2_ready();
}

void stats_i8_sizes(int K, int nloc_pad, int Ppad, int nloc, int P, int nall_pad, int ploc, StatsI8Sizes* s) {
    const long long L = (long long)K * (K + 1) / 2;
    const long long kd = std::max(nall_pad, Ppad);                          // contraction lengths: rows over p, columns over ALL rows
    const long long nd = std::max<long long>(nloc_pad, (ploc + 255) / 256 * 256);   // output rows: local rows / local columns
    s->planes_bytes = (size_t)i8_plane_rows((int)L) * kd;
    s->d_elems = (size_t)i8_plane_rows((int)L) * nd;
    s->cntT_bytes = (size_t)std::max(ploc, 1) * nall_pad;
    s->nsplit_b_row = 64;            // upper bound of the split count of the row-variant linear block (buffer size)
    s->bpart_elems = std::max((size_t)s->nsplit_b_row * nloc * K, (size_t)2 * P * K);   // columns: the split counts fit in 2 P K
    s->L = (int)L;
}

void launch_transpose_u8(const uint8_t* src, long long lds, int rows, int cols, uint8_t* dst, long long ldd, cudaStream_t st) {
    transpose_u8_kernel<<<dim3((cols + 31) / 32, (rows + 31) / 32), 256, 0, st>>>(src, lds, rows, cols, dst, ldd);
}

// ---- the integer path in stages, so that the engine can put the tensor-core contraction and the HBM-bound
// linear block on different streams (they use disjoint resources) and shard the column side by columns.
//
// 1. column scales and digit planes of Z = [F (x) F packed]: planes [8 L][kdim_pad]
void stats_i8_digits(const StatsI8Buffers& w, int K, const double* F, int f_rows, int kdim_pad, cudaStream_t st) {
    const int L = K * (K + 1) / 2;
    cudaMemsetAsync(w.colmax, 0, (size_t)L * 8, st);
    zmax_kernel<<<dim3((f_rows + 127) / 128, (L + 255) / 256), 256, (size_t)128 * K * 8, st>>>(F, f_rows, K, L, w.colmax);
    const size_t zs = (size_t)256 * (K + 1) * 8 + (size_t)((L + 3) / 4) * 8;
    static PerDeviceMax zs_set;
    if (zs > 48 * 1024 && zs_set.raise(zs)) cudaFuncSetAttribute(zdigits_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)zs);
    // few factor rows (the column side: W has N rows): split the product columns over gridDim.y so the launch fills the GPU
    const int nbx = (kdim_pad + 255) / 256;
    const int nby = std::max(1, std::min((L + 3) / 4, 592 / nbx));
    zdigits_kernel<<<dim3(nbx, nby), 256, zs, st>>>(F, f_rows, kdim_pad, K, L, w.colmax, w.expo, w.planes, (long long)kdim_pad);
}

// 2. exact product block on the tensor cores, D[(s, c)][m] = sum_k d_s[k, c] B[m][k], m < m_valid (B = counts, K-major):
//    recombined into `out` by the GEMM's epilogue (fused route), or left as int32 planes in w.D (split-K route)
int stats_i8_product(const StatsI8Buffers& w, int K, const uint8_t* B, long long ldb, int kdim_pad, int m_valid, int m_pad,
                     double* out, const I8Guard* guard, cudaStream_t st) {
    const int L = K * (K + 1) / 2;
    return launch_i8gemm2(reinterpret_cast<const int8_t*>(B), ldb, m_valid, w.planes, kdim_pad, L, kdim_pad, w.expo, out, L + K,
                          guard, w.D, m_pad, st);
}

// 3. linear block in FP64: bpart[split][m][j] = sum_k S[m, k] F[k, j] over the split's k range; returns the split count
int stats_i8_linear(const StatsI8Buffers& w, bool trans, int K, const double* S, long long lds, const double* F,
                    int kdim_pad, int m_valid, int max_split, double* out, cudaStream_t st) {
    const int nchunks = kdim_pad / 32;
    const int m_tiles = (m_valid + 127) / 128;
    int sms = 148;
    { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); if (sms < 1) sms = 148; }
    // split-K partials are summed in split order by the recombination kernel
    int nsplit = 1;
    const int target = 2 * sms;      // one wave of two CTAs per SM
    if (m_tiles < target) {
        nsplit = target / m_tiles;       // never a partial last wave
        if (nsplit > nchunks / 8) nsplit = nchunks / 8 > 0 ? nchunks / 8 : 1;
        if (nsplit > max_split) nsplit = max_split;
    } else if (max_split > 1) {
        // more tiles than CTA slots: the items run in ceil(items / slots) rounds, and a partial last round idles part of the
        // GPU (C2 columns: 512 tiles on 296 slots = 2 rounds for 1.73 rounds of work).  Splitting the contraction s ways
        // makes the rounds s times shorter: pick the s with the least rounds / s, 2 % per extra split for the partial sums.
        double best = 1e30;
        for (int s = 1; s <= max_split && s <= std::max(1, nchunks / 8); ++s) {
            const int cps = (nchunks + s - 1) / s, se = (nchunks + cps - 1) / cps;
            const long long rounds = ((long long)m_tiles * se + target - 1) / target;
            const double cost = (double)rounds / se * (1.0 + 0.02 * (se - 1));
            if (cost < best - 1e-12) { best = cost; nsplit = se; }
        }
    }
    { const int cps = (nchunks + nsplit - 1) / nsplit; nsplit = (nchunks + cps - 1) / cps; }
    if (K <= 8) { if (trans) launch_sf_t<8, true>(S, lds, F, K, m_valid, m_tiles, nchunks, nsplit, out, st); else launch_sf_t<8, false>(S, lds, F, K, m_valid, m_tiles, nchunks, nsplit, out, st); }
    else if (K <= 16) { if (trans) launch_sf_t<16, true>(S, lds, F, K, m_valid, m_tiles, nchunks, nsplit, out, st); else launch_sf_t<16, false>(S, lds, F, K, m_valid, m_tiles, nchunks, nsplit, out, st); }
    else { if (trans) launch_sf_t<32, true>(S, lds, F, K, m_valid, m_tiles, nchunks, nsplit, out, st); else launch_sf_t<32, false>(S, lds, F, K, m_valid, m_tiles, nchunks, nsplit, out, st); }
    return nsplit;
}

// 4. recombination of the int32 planes (skipped when the fused epilogue already wrote them) and the sum of the
//    linear-block partials: out[m][0..L) from D, out[m][L..L+K) from bpart[split][bpart_m0 + m][.] (row pitch of a
//    split = bpart_rows)
void stats_i8_combine(const StatsI8Buffers& w, int K, int m_valid, int m_pad, bool product_done,
                      const double* bpart, int nsplit_b, long long bpart_m0, long long bpart_rows, double* out,
                      const I8Guard* guard, cudaStream_t st) {
    const int L = K * (K + 1) / 2;
    const int ncy = (L + 31) / 32;
    const I8Guard g = guard ? *guard : I8Guard{nullptr, nullptr, nullptr, 0.0};
    if (product_done)
        i8_combine_kernel<<<dim3((m_valid + 31) / 32, 1), 256, 0, st>>>(w.D, m_pad, w.expo, bpart, nsplit_b, m_valid, L, K, out, ncy,
                                                                       bpart_m0, bpart_rows, g, guard != nullptr);
    else
        i8_combine_kernel<<<dim3((m_valid + 31) / 32, ncy + 1), 256, 0, st>>>(w.D, m_pad, w.expo, bpart, nsplit_b, m_valid, L, K, out, 0,
                                                                             bpart_m0, bpart_rows, g, guard != nullptr);
}

// 5. FP64 recomputation of the rows flagged by the element-wise guard (see i8_fallback_kernel)
void stats_i8_count_rows(const uint8_t* B, long long ldb, int m_valid, int kdim_pad, unsigned* cntsum, cudaStream_t st) {
    if (m_valid > 0) count_rows_kernel<<<(m_valid + 7) / 8, 256, 0, st>>>(B, ldb, m_valid, kdim_pad, cntsum);
}
void stats_i8_fallback(int K, const uint8_t* B, long long ldb, const double* F, int f_rows, int m_valid, double* out,
                       const I8Guard& g, cudaStream_t st) {
    if (m_valid <= 0) return;
    const int L = K * (K + 1) / 2, nco = L + K;
    const size_t smem = (size_t)(128 * K + 128) * sizeof(double);
    const int grid = std::min((m_valid + 63) / 64, 592);
    if (L <= 256) i8_fallback_kernel<1><<<grid, 256, smem, st>>>(B, ldb, F, f_rows, K, L, m_valid, g.flags, g.nflag, out, nco);
    else i8_fallback_kernel<3><<<grid, 256, smem, st>>>(B, ldb, F, f_rows, K, L, m_valid, g.flags, g.nflag, out, nco);
}

}  // namespace btf
