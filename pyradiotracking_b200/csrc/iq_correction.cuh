// iq_correction.cuh -- per-block DC and IQ-imbalance correction of the FIR front ends (rt_ddc.cu, rt_fbank.cu; the definition
// is in include/rt_ddc.h and include/rt_fbank.h).  For every input and wideband block of block_samples normalised samples x:
//
//     m = mean(x)      p = mean(|x - m|^2)      c = mean((x - m)^2)
//     w = -c / (p + sqrt(p^2 - |c|^2))  (0 when p = 0)      y = (x - m) + w conj(x - m)
//
// and the filter runs on y.  The kernels that form m and w of every block are in fir_frontend.cu; this file is what the filter
// kernels need to apply them.  They read the coefficients through fir_sample<FMT, true> (fir_history.cuh).  A CTA's span may
// straddle block boundaries (a block can be as short as D samples): each thread divides its first in-call sample index by
// block_samples once (int64) and every later index by a multiply-high with a per-handle magic number (IqCorrArgs).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rt {

// What the filter kernels need: the member `corr` of the argument struct of the corrected kernels, which derives from the front
// end's own struct (the uncorrected kernels keep the parameter block, and with it the code, they had before the correction).
struct IqCorrArgs {
    const float4* coef;         // [n_inputs][n_blocks] (m.re, m.im, w.re, w.im) of this call
    long long block;            // block_samples
    int n_blocks;               // blocks in this call
    uint32_t magic;             // q = umulhi(v, magic) >> shift equals v / block for every v < 2^31
    int shift;
};

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

}  // namespace rt
