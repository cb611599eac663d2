// fir_history.cuh -- what the FIR front ends of librtb200.so (rt_ddc.cu, rt_fbank.cu) share: the per-input history of the last
// L - 1 normalised samples, its reset in stream order, and the staging copy of a host input.
//
// The kernels take the front end's own argument struct A, which has these fields:
//   const unsigned char* iq; size_t in_stride;   input i at iq + i * in_stride
//   const float2* hist; float2* hist_out;         [n_inputs][hist_len] samples before the call, and the same after it
//   int hist_len;                                 L - 1
//   long long n_samples;                          input samples per input in this call
//   float scale, offset;                          rt::load_normalised
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "sample_format.cuh"

namespace rt {
namespace {   // every source that includes this file gets its own kernels

// sample `rel` of the call (negative: the history before it; past the end: zero, read only by outputs that are not stored)
template <int FMT, class A>
__device__ __forceinline__ float2 fir_sample(const A& a, const unsigned char* row, const float2* hist, long long rel) {
    if (rel < 0) return hist[a.hist_len + rel];
    if (rel >= a.n_samples) return make_float2(0.f, 0.f);
    return load_normalised<FMT>(row, rel, a.scale, a.offset);
}

// the last L - 1 normalised samples of every input, for the next call; grid (ceil(hist_len / blockDim.x), n_inputs)
template <int FMT, class A>
__global__ void fir_history_kernel(const A a) {
    const int input = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.hist_len) return;
    const unsigned char* row = a.iq + (size_t)input * a.in_stride;
    const float2* hist = a.hist + (size_t)input * a.hist_len;
    a.hist_out[(size_t)input * a.hist_len + j] = fir_sample<FMT>(a, row, hist, a.n_samples - a.hist_len + j);
}

// reset_input, applied in stream order at the next run: zero history, and the phase offset of the input
__global__ void fir_reset_kernel(float2* hist, uint32_t* off, int input, int hist_len, uint32_t off_value) {
    for (int j = threadIdx.x; j < hist_len; j += blockDim.x) hist[(size_t)input * hist_len + j] = make_float2(0.f, 0.f);
    if (threadIdx.x == 0) off[input] = off_value;
}

}  // namespace

// Copy n_in host rows of row_bytes (stride `stride`) into the device staging buffer (*stage, grown when too small, rows 256-byte
// aligned) on `st`; *src and *stride then describe the staged copy.
inline cudaError_t fir_stage_host_input(cudaStream_t st, const unsigned char** src, size_t* stride, size_t row_bytes, int n_in,
                                        unsigned char** stage, size_t* stage_bytes) {
    const size_t sstride = (row_bytes + 255) & ~(size_t)255;
    cudaError_t e;
    if (sstride * n_in > *stage_bytes) {
        if ((e = cudaStreamSynchronize(st)) != cudaSuccess) return e;
        if ((e = cudaFree(*stage)) != cudaSuccess) return e;
        *stage = nullptr;
        *stage_bytes = 0;
        if ((e = cudaMalloc(stage, sstride * n_in)) != cudaSuccess) return e;
        *stage_bytes = sstride * n_in;
    }
    if ((e = cudaMemcpy2DAsync(*stage, sstride, *src, *stride, row_bytes, n_in, cudaMemcpyHostToDevice, st)) != cudaSuccess) return e;
    *src = *stage;
    *stride = sstride;
    return cudaSuccess;
}

}  // namespace rt
