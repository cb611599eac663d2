// iq_correction.cuh -- per-block DC and IQ-imbalance correction of the FIR front ends (rt_ddc.cu, rt_fbank.cu; the definition
// is in include/rt_ddc.h and include/rt_fbank.h).  For every input and wideband block of block_samples normalised samples x:
//
//     m = mean(x)      p = mean(|x - m|^2)      c = mean((x - m)^2)
//     w = -c / (p + sqrt(p^2 - |c|^2))  (0 when p = 0)      y = (x - m) + w conj(x - m)
//
// and the filter runs on y.  Kernels (on the front end's stream, ahead of its filter kernel, no host synchronisation):
//   iq_moments_kernel   one CTA = one tile of IQ_TILE samples of one block of one input: the five sums S_I, S_Q, S_II, S_QQ,
//                       S_IQ of the tile's elements (ci8, ci16: the element; cu8: the byte - 128; exact int64) or of its values
//                       (cf32: float64, each thread in sample order, then a fixed shuffle tree and the warps in order)
//   iq_coef_kernel      one warp = one (input, block): the sums of its tiles in a fixed order (lane l takes the tiles l, l + 32,
//                       ..., then a fixed shuffle tree); lane 0 forms m and w in float64 and stores them as fp32
// Tiles start at the block's first sample, so the sums of a block never depend on how many blocks a call carries, on the batch
// or on the grid.
//
// The filter kernels read the coefficients through fir_sample<FMT, true> (fir_history.cuh).  A CTA's span may straddle block
// boundaries (a block can be as short as D samples): each thread divides its first in-call sample index by block_samples once
// (int64) and every later index by a multiply-high with a per-handle magic number (IqCorrArgs).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>

#include "sample_format.cuh"

namespace rt {

constexpr int IQ_THREADS = 256;
constexpr int IQ_TILE = 16384;                  // samples per moments CTA (64 per thread)
constexpr long long IQ_MAX_BLOCK = 1LL << 30;   // block_samples with the correction on: exact int64 sums, 32-bit in-span division

// What the filter kernels need: the member `corr` of the argument struct of the corrected kernels, which derives from the front
// end's own struct (the uncorrected kernels keep the parameter block, and with it the code, they had before the correction).
struct IqCorrArgs {
    const float4* coef;         // [n_inputs][n_blocks] (m.re, m.im, w.re, w.im) of this call
    long long block;            // block_samples
    int n_blocks;               // blocks in this call
    uint32_t magic;             // q = umulhi(v, magic) >> shift equals v / block for every v < 2^31
    int shift;
};

// magic and shift of the division by d (2 <= d <= 2^30) for dividends below 2^31 (Granlund and Montgomery, "Division by
// invariant integers using multiplication", 1994, Theorem 4.2 with N = 31: l = ceil(log2 d), magic = ceil(2^(31 + l) / d) < 2^32)
inline void iq_division_magic(long long d, uint32_t* magic, int* shift) {
    int l = 0;
    while ((1LL << l) < d) ++l;
    const unsigned __int128 num = (unsigned __int128)1 << (31 + l);
    *magic = (uint32_t)((num + (unsigned __int128)d - 1) / (unsigned __int128)d);
    *shift = l - 1;
}

// per-thread state of the corrected loader: the block of the in-call sample `base` and its offset in that block
template <bool IQ>
struct IqSpan {};
template <>
struct IqSpan<true> {
    const float4* coef;         // this input's row
    long long base, b_base;
    uint32_t r0;
};

template <bool IQ, class A>
__device__ __forceinline__ IqSpan<IQ> iq_span(const A& a, int input, long long base) {
    if constexpr (IQ) {
        IqSpan<true> s;
        s.coef = a.corr.coef + (size_t)input * a.corr.n_blocks;
        s.base = base < 0 ? 0 : base;
        s.b_base = s.base / a.corr.block;
        s.r0 = (uint32_t)(s.base - s.b_base * a.corr.block);
        return s;
    } else {
        return {};
    }
}

// y of the normalised sample x of in-call index rel >= s.base (rel - s.base < 2^31 - block_samples)
__device__ __forceinline__ float2 iq_apply(const IqCorrArgs& c, const IqSpan<true>& s, long long rel, float2 x) {
    const uint32_t v = (uint32_t)(rel - s.base) + s.r0;
    const float4 k = __ldg(s.coef + s.b_base + (__umulhi(v, c.magic) >> c.shift));
    const float dr = __fsub_rn(x.x, k.x), di = __fsub_rn(x.y, k.y);
    // (x - m) + w conj(x - m) = (dr (1 + w.re) + w.im di, di (1 - w.re) + w.im dr), each rounded as written
    return make_float2(__fmaf_rn(k.w, di, __fmaf_rn(k.z, dr, dr)), __fmaf_rn(k.w, dr, __fmaf_rn(-k.z, di, di)));
}

namespace {   // every source that includes this file gets its own kernels

// element sums of one tile; part[((input * n_blocks + b) * tiles + tile) * 5 + j], S = long long (integer formats) or double
template <int FMT, class S>
__global__ void __launch_bounds__(IQ_THREADS) iq_moments_kernel(const unsigned char* iq, size_t in_stride, long long block, int n_blocks,
                                                                int tiles, S* part) {
    const int input = blockIdx.y, tile = (int)(blockIdx.x % (unsigned)tiles), b = (int)(blockIdx.x / (unsigned)tiles);
    const long long t0 = (long long)tile * IQ_TILE;
    const int len = (int)min((long long)IQ_TILE, block - t0);
    constexpr int BYTES = FMT == RT_SAMPLE_CU8 || FMT == RT_SAMPLE_CI8 ? 2 : FMT == RT_SAMPLE_CI16 ? 4 : 8;
    const unsigned char* row = iq + (size_t)input * in_stride + (size_t)((long long)b * block + t0) * BYTES;
    S s[5] = {0, 0, 0, 0, 0};
    for (int t = threadIdx.x; t < len; t += IQ_THREADS) {
        S re, im;
        if (FMT == RT_SAMPLE_CU8) {
            const uchar2 v = reinterpret_cast<const uchar2*>(row)[t];
            re = (int)v.x - 128; im = (int)v.y - 128;
        } else if (FMT == RT_SAMPLE_CI8) {
            const char2 v = reinterpret_cast<const char2*>(row)[t];
            re = v.x; im = v.y;
        } else if (FMT == RT_SAMPLE_CI16) {
            const short2 v = reinterpret_cast<const short2*>(row)[t];
            re = v.x; im = v.y;
        } else {
            const float2 v = reinterpret_cast<const float2*>(row)[t];
            re = v.x; im = v.y;
        }
        s[0] += re;
        s[1] += im;
        s[2] += re * re;
        s[3] += im * im;
        s[4] += re * im;
    }
    __shared__ S ws[IQ_THREADS / 32][5];
#pragma unroll
    for (int j = 0; j < 5; ++j) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s[j] += __shfl_xor_sync(0xffffffffu, s[j], o);
        if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5][j] = s[j];
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        S acc = 0;
#pragma unroll
        for (int w = 0; w < IQ_THREADS / 32; ++w) acc += ws[w][threadIdx.x];
        part[(((size_t)input * n_blocks + b) * tiles + tile) * 5 + threadIdx.x] = acc;
    }
}

// m and w of every (input, block) from the tile sums; elements map to normalised samples as e * scale + offset
template <class S>
__global__ void iq_coef_kernel(const S* part, int n_inputs, int n_blocks, int tiles, long long block, double scale, double offset,
                               float4* coef) {
    const int pair = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (pair >= n_inputs * n_blocks) return;                  // whole warps leave together (blockDim.x is a multiple of 32)
    const S* src = part + (size_t)pair * tiles * 5;
    S s[5] = {0, 0, 0, 0, 0};
    for (int t = lane; t < tiles; t += 32)
#pragma unroll
        for (int j = 0; j < 5; ++j) s[j] += src[(size_t)t * 5 + j];
#pragma unroll
    for (int j = 0; j < 5; ++j)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s[j] += __shfl_xor_sync(0xffffffffu, s[j], o);
    if (lane != 0) return;
    const double n = (double)block;
    const double mI = (double)s[0] / n, mQ = (double)s[1] / n;
    // central moments of the elements; p and c do not depend on the scale of x, only w and m are needed
    const double sII = (double)s[2] / n - mI * mI, sQQ = (double)s[3] / n - mQ * mQ, sIQ = (double)s[4] / n - mI * mQ;
    const double p = sII + sQQ, cr = sII - sQQ, ci = 2.0 * sIQ;
    double wr = 0.0, wi = 0.0;
    if (p > 0.0) {
        const double den = p + sqrt(fmax(p * p - (cr * cr + ci * ci), 0.0));
        wr = -cr / den;
        wi = -ci / den;
    }
    coef[pair] = make_float4((float)(mI * scale + offset), (float)(mQ * scale + offset), (float)wr, (float)wi);
}

}  // namespace

inline size_t iq_tiles(long long block) { return (size_t)((block + IQ_TILE - 1) / IQ_TILE); }

// Host side of one handle: the setting, the coefficient and tile-sum buffers (grown when a call carries more blocks, after the
// previous run has finished with them) and what the last run did.
struct IqState {
    bool on = false;                    // set_iq_correction: applied from the next run
    bool applied = false;               // the last run corrected
    int blocks = 0;                     // blocks of that run
    float4* coef = nullptr;             // [n_inputs][blocks]
    size_t coef_bytes = 0;
    void* part = nullptr;               // [n_inputs][blocks][tiles][5] int64 or float64 tile sums
    size_t part_bytes = 0;
    void release() {
        cudaFree(coef);
        cudaFree(part);
        coef = nullptr;
        part = nullptr;
    }
};

inline cudaError_t iq_grow(void** buf, size_t* have, size_t need, cudaEvent_t done, bool ran) {
    if (need <= *have) return cudaSuccess;
    cudaError_t e;
    if (ran && (e = cudaEventSynchronize(done)) != cudaSuccess) return e;
    if ((e = cudaFree(*buf)) != cudaSuccess) return e;
    *buf = nullptr;
    *have = 0;
    if ((e = cudaMalloc(buf, need)) != cudaSuccess) return e;
    *have = need;
    return cudaSuccess;
}

// One run: with the correction on, enqueue the tile sums and the coefficients of `blocks` blocks of every input (rows at
// src + i * stride) on `st` and describe them in *args; off, *args is zero and nothing is enqueued.  `done` / `ran`: the
// handle's last run, which may still read the buffers.
inline cudaError_t iq_prepare(IqState& s, cudaStream_t st, cudaEvent_t done, bool ran, int fmt, const SampleFormatInfo& info,
                              const unsigned char* src, size_t stride, int n_in, long long block, int blocks, IqCorrArgs* args) {
    *args = IqCorrArgs{};
    s.applied = false;
    if (!s.on) return cudaSuccess;
    const int tiles = (int)iq_tiles(block);
    cudaError_t e;
    if ((e = iq_grow((void**)&s.coef, &s.coef_bytes, (size_t)n_in * blocks * sizeof(float4), done, ran)) != cudaSuccess) return e;
    if ((e = iq_grow(&s.part, &s.part_bytes, (size_t)n_in * blocks * tiles * 5 * 8, done, ran)) != cudaSuccess) return e;
    // elements e map to x = e * scale + offset (scale = (float)(1 / full_scale), as rt::load_normalised); the cu8 sums are of b - 128
    const double scale = (double)(float)(1.0 / info.full_scale);
    const double offset = fmt == RT_SAMPLE_CU8 ? info.offset + 128.0 * scale : info.offset;
    const dim3 grid((unsigned)((size_t)tiles * blocks), (unsigned)n_in);
    const unsigned cgrid = (unsigned)(((size_t)n_in * blocks * 32 + 255) / 256);
    long long* pi = (long long*)s.part;
    switch (fmt) {
        case RT_SAMPLE_CU8: iq_moments_kernel<RT_SAMPLE_CU8><<<grid, IQ_THREADS, 0, st>>>(src, stride, block, blocks, tiles, pi); break;
        case RT_SAMPLE_CI8: iq_moments_kernel<RT_SAMPLE_CI8><<<grid, IQ_THREADS, 0, st>>>(src, stride, block, blocks, tiles, pi); break;
        case RT_SAMPLE_CI16: iq_moments_kernel<RT_SAMPLE_CI16><<<grid, IQ_THREADS, 0, st>>>(src, stride, block, blocks, tiles, pi); break;
        default: break;
    }
    if (fmt == RT_SAMPLE_CF32) {
        double* pd = (double*)s.part;
        iq_moments_kernel<RT_SAMPLE_CF32><<<grid, IQ_THREADS, 0, st>>>(src, stride, block, blocks, tiles, pd);
        iq_coef_kernel<<<cgrid, 256, 0, st>>>((const double*)pd, n_in, blocks, tiles, block, scale, offset, s.coef);
    } else {
        iq_coef_kernel<<<cgrid, 256, 0, st>>>((const long long*)pi, n_in, blocks, tiles, block, scale, offset, s.coef);
    }
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    args->coef = s.coef;
    args->block = block;
    args->n_blocks = blocks;
    iq_division_magic(block, &args->magic, &args->shift);
    s.applied = true;
    s.blocks = blocks;
    return cudaSuccess;
}

// m and w of (input, block) of the last run, after it has finished: out = {m.re, m.im, w.re, w.im}
inline cudaError_t iq_read(const IqState& s, cudaEvent_t done, int input, int block, float out[4]) {
    cudaError_t e;
    if ((e = cudaEventSynchronize(done)) != cudaSuccess) return e;
    float4 v;
    if ((e = cudaMemcpy(&v, s.coef + (size_t)input * s.blocks + block, sizeof(v), cudaMemcpyDeviceToHost)) != cudaSuccess) return e;
    out[0] = v.x;
    out[1] = v.y;
    out[2] = v.z;
    out[3] = v.w;
    return cudaSuccess;
}

}  // namespace rt
