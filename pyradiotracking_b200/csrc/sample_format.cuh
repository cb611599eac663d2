// sample_format.cuh -- the input sample formats of the engine (rt_config.sample_format, RT_SAMPLE_*): the host-side table and
// the device-side front end of the generic spectrogram kernel.
//
// Every format is centred on its segment mean (scipy detrend='constant') and the remaining scale is folded into the window, so
// the kernels see (element - mean) and the host divides by the format's full scale (sample_format_info).  The byte kernels
// (register, tensor-core, radix-16) take ci8 as cu8 with the top bit of every byte flipped: v ^ 0x80 is v + 128 as an unsigned
// byte, and the constant 128 vanishes in the exact integer detrend.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rt_engine.h"

namespace rt {

// host-side table: bytes per complex sample, and the divisor and offset that map an element to the normalised sample
// element / full_scale + offset (cu8: b / 127.5 - 1; the spectrogram kernels drop the offset, the detrend removes it)
struct SampleFormatInfo {
    int bytes;
    double full_scale;
    double offset;
};
inline bool sample_format_info(int fmt, SampleFormatInfo* out) {
    switch (fmt) {
        case RT_SAMPLE_CU8: *out = {2, 127.5, -1.0}; return true;
        case RT_SAMPLE_CI8: *out = {2, 128.0, 0.0}; return true;
        case RT_SAMPLE_CI16: *out = {4, 32768.0, 0.0}; return true;
        case RT_SAMPLE_CF32: *out = {8, 1.0, 0.0}; return true;
        default: return false;
    }
}
// the formats the byte kernels (register, tensor-core, radix-16) read
constexpr bool sample_format_is_byte(int fmt) { return fmt == RT_SAMPLE_CU8 || fmt == RT_SAMPLE_CI8; }

// Device side of the generic kernel: centre one segment of n complex samples (`seg` in global memory) on its mean, multiply by
// the window and write it to `out` (shared memory).  NT threads (`tid`) take part; the function ends after a CTA barrier that follows
// the reduction, and the caller synchronises before reading `out`.  `sums` (2 ints) and `scratch` (NT / 32 float2, not `out`)
// are shared-memory scratch.
template <int FMT>
struct SegmentIn;

// cu8 / ci8: byte sums are exact integers, the mean (sum / n, n a power of two) is exact in fp32
template <int FMT>
struct SegmentInBytes {
    static constexpr int BYTES = 2;
    template <int NT>
    __device__ __forceinline__ static void centre(const unsigned char* seg, int n, int tid, const float* win, float2* out, int* sums, float2*) {
        const uchar2* src = reinterpret_cast<const uchar2*>(seg);
        if (tid == 0) sums[0] = sums[1] = 0;
        __syncthreads();
        int sI = 0, sQ = 0;
        for (int i = tid; i < n; i += NT) {
            uchar2 v = src[i];
            if (FMT == RT_SAMPLE_CI8) { v.x ^= 0x80; v.y ^= 0x80; }
            sI += v.x;
            sQ += v.y;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            sI += __shfl_xor_sync(0xffffffffu, sI, o);
            sQ += __shfl_xor_sync(0xffffffffu, sQ, o);
        }
        if ((tid & 31) == 0) {
            atomicAdd(&sums[0], sI);
            atomicAdd(&sums[1], sQ);
        }
        __syncthreads();
        const float mI = (float)sums[0] / (float)n;   // exact: sum < 2^24, n a power of two
        const float mQ = (float)sums[1] / (float)n;
        for (int i = tid; i < n; i += NT) {
            uchar2 v = src[i];
            if (FMT == RT_SAMPLE_CI8) { v.x ^= 0x80; v.y ^= 0x80; }
            float w = win[i];
            out[i] = make_float2(((float)v.x - mI) * w, ((float)v.y - mQ) * w);
        }
    }
};
template <> struct SegmentIn<RT_SAMPLE_CU8> : SegmentInBytes<RT_SAMPLE_CU8> {};
template <> struct SegmentIn<RT_SAMPLE_CI8> : SegmentInBytes<RT_SAMPLE_CI8> {};

// ci16: int32 sums are exact (|sum| <= 2^27).  n v no longer fits fp32 exactly, so the mean is split exactly: sum = q n + r with
// q = floor(sum / n), 0 <= r < n, and v - sum / n = (v - q) - r / n: an exact integer minus an exact fraction, rounded once
template <>
struct SegmentIn<RT_SAMPLE_CI16> {
    static constexpr int BYTES = 4;
    template <int NT>
    __device__ __forceinline__ static void centre(const unsigned char* seg, int n, int tid, const float* win, float2* out, int* sums, float2*) {
        const short2* src = reinterpret_cast<const short2*>(seg);
        if (tid == 0) sums[0] = sums[1] = 0;
        __syncthreads();
        int sI = 0, sQ = 0;
        for (int i = tid; i < n; i += NT) {
            const short2 v = src[i];
            sI += v.x;
            sQ += v.y;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            sI += __shfl_xor_sync(0xffffffffu, sI, o);
            sQ += __shfl_xor_sync(0xffffffffu, sQ, o);
        }
        if ((tid & 31) == 0) {
            atomicAdd(&sums[0], sI);
            atomicAdd(&sums[1], sQ);
        }
        __syncthreads();
        const int lg = __ffs(n) - 1;
        const int qI = sums[0] >> lg, qQ = sums[1] >> lg;                      // arithmetic shift: floor
        const float inv_n = 1.f / (float)n;                                    // exact: n a power of two
        const float rI = (float)(sums[0] - (qI << lg)) * inv_n, rQ = (float)(sums[1] - (qQ << lg)) * inv_n;
        for (int i = tid; i < n; i += NT) {
            const short2 v = src[i];
            const float w = win[i];
            out[i] = make_float2(((float)(v.x - qI) - rI) * w, ((float)(v.y - qQ) - rQ) * w);
        }
    }
};

// cf32: fp32 sums in a fixed order (per thread, a shuffle tree, then the warps in order), so every run gives the same bits.
// Error bound: include/rt_engine.h (RT_SAMPLE_CF32)
template <>
struct SegmentIn<RT_SAMPLE_CF32> {
    static constexpr int BYTES = 8;
    template <int NT>
    __device__ __forceinline__ static void centre(const unsigned char* seg, int n, int tid, const float* win, float2* out, int*, float2* scratch) {
        const float2* src = reinterpret_cast<const float2*>(seg);
        float sI = 0.f, sQ = 0.f;
        for (int i = tid; i < n; i += NT) {
            const float2 v = src[i];
            sI += v.x;
            sQ += v.y;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {     // a + b == b + a: every lane ends with the same bits
            sI += __shfl_xor_sync(0xffffffffu, sI, o);
            sQ += __shfl_xor_sync(0xffffffffu, sQ, o);
        }
        if ((tid & 31) == 0) scratch[tid >> 5] = make_float2(sI, sQ);
        __syncthreads();
        float tI = 0.f, tQ = 0.f;
#pragma unroll
        for (int w = 0; w < NT / 32; ++w) {
            const float2 p = scratch[w];
            tI += p.x;
            tQ += p.y;
        }
        const float inv_n = 1.f / (float)n;
        const float mI = tI * inv_n, mQ = tQ * inv_n;
        for (int i = tid; i < n; i += NT) {
            const float2 v = src[i];
            const float w = win[i];
            out[i] = make_float2((v.x - mI) * w, (v.y - mQ) * w);
        }
    }
};

// The normalised complex sample i of an interleaved I,Q row: fma(element, scale, offset) with scale = (float)(1 / full_scale) and
// offset from sample_format_info (cf32: scale 1, offset 0, the value as stored).
template <int FMT>
__device__ __forceinline__ float2 load_normalised(const unsigned char* row, long long i, float scale, float offset) {
    float re, im;
    if (FMT == RT_SAMPLE_CU8) {
        const uchar2 v = reinterpret_cast<const uchar2*>(row)[i];
        re = v.x; im = v.y;
    } else if (FMT == RT_SAMPLE_CI8) {
        const char2 v = reinterpret_cast<const char2*>(row)[i];
        re = v.x; im = v.y;
    } else if (FMT == RT_SAMPLE_CI16) {
        const short2 v = reinterpret_cast<const short2*>(row)[i];
        re = v.x; im = v.y;
    } else {
        return reinterpret_cast<const float2*>(row)[i];
    }
    return make_float2(__fmaf_rn(re, scale, offset), __fmaf_rn(im, scale, offset));
}

}  // namespace rt
