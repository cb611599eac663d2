// fir_history.cuh -- the device side that the FIR front ends of librtb200.so (rt_ddc.cu, rt_fbank.cu) share: the loader of one
// normalised sample of a call, which reads the per-input history of the last L - 1 samples for indices before the call, and the
// kernel that saves that history for the next call.  The history's reset and the rest of the host side are in fir_frontend.cu.
//
// The kernels take the front end's own argument struct A, which has these fields:
//   const unsigned char* iq; size_t in_stride;   input i at iq + i * in_stride
//   const float2* hist; float2* hist_out;         [n_inputs][hist_len] samples before the call, and the same after it
//   int hist_len;                                 L - 1
//   long long n_samples;                          input samples per input in this call
//   float scale, offset;                          rt::load_normalised
//   IqCorrArgs corr;                              only with IQ = true: the DC / IQ-imbalance coefficients (iq_correction.cuh)
// IQ = false is the uncorrected front end; its kernels compile to the code they had before the correction existed.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "iq_correction.cuh"
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

// the same with the per-block correction when IQ (`sp` from iq_span with a base <= every in-call rel this thread reads): history
// samples are corrected already, and past the end there is nothing to correct
template <int FMT, bool IQ, class A>
__device__ __forceinline__ float2 fir_sample(const A& a, const unsigned char* row, const float2* hist, long long rel, const IqSpan<IQ>& sp) {
    if constexpr (IQ) {
        if (rel < 0) return hist[a.hist_len + rel];
        if (rel >= a.n_samples) return make_float2(0.f, 0.f);
        return iq_apply(a.corr, sp, rel, load_normalised<FMT>(row, rel, a.scale, a.offset));
    } else {
        return fir_sample<FMT>(a, row, hist, rel);
    }
}

// the last L - 1 normalised samples of every input, for the next call; grid (ceil(hist_len / blockDim.x), n_inputs)
template <int FMT, bool IQ, class A>
__global__ void fir_history_kernel(const A a) {
    const int input = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= a.hist_len) return;
    const unsigned char* row = a.iq + (size_t)input * a.in_stride;
    const float2* hist = a.hist + (size_t)input * a.hist_len;
    const long long rel = a.n_samples - a.hist_len + j;
    a.hist_out[(size_t)input * a.hist_len + j] = fir_sample<FMT, IQ>(a, row, hist, rel, iq_span<IQ>(a, input, rel));
}

}  // namespace

}  // namespace rt
