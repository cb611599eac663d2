// rt_fbank.cu -- polyphase FFT filter bank (include/rt_fbank.h): all 2 D - 1 in-band channels of the uniform grid k fs / (2 D)
// of many wideband inputs, in fp32 on the CUDA cores.
//
// Kernels (all on the caller's stream):
//   fbank_kernel        one CTA = one input and a tile of MT output frames.  It decodes the input span those frames read
//                       ((MT - 1) D + L samples, the history for indices before the call) into shared memory once, forms the
//                       C = 2 D polyphase partial sums u_r of every frame (a thread owns one (frame, tap phase) pair and sums
//                       its <= 9 taps), writes them in bit-reversed order, runs an in-place radix-2 FFT per frame in shared
//                       memory and stores each channel row's MT outputs contiguously (the frames are padded to C + 1 points,
//                       so reading one bin across frames is free of bank conflicts)
//   fir_history_kernel  the last L - 1 normalised samples of every input, for the next call (double-buffered; fir_history.cuh)
// With rt_fbank_set_iq_correction on, the IQ = true instantiations of both apply each block's DC and IQ-imbalance coefficients
// as they decode (iq_correction.cuh).  The handle, the checks and steps a run shares with the down-converter, the reset kernel
// and the kernels that form the coefficients are in fir_frontend.cu.
#include <cuda_runtime.h>

#include <cmath>
#include <memory>
#include <type_traits>
#include <vector>

#include "../../include/rt_fbank.h"
#include "fir_frontend.cuh"

namespace {

constexpr int FB_THREADS = 256;
constexpr int FB_MAX_MT = 64;                       // output frames per CTA: 512-byte row segments at most
constexpr size_t FB_SMEM_TARGET = 112 * 1024;       // two CTAs per SM

using rt::fail;

struct FbankArgs {
    const unsigned char* iq;        // input i at iq + i * in_stride
    size_t in_stride;
    const float2* hist;             // [n_inputs][hist_len] normalised samples before the call
    float2* hist_out;               // the same after the call
    int hist_len;                   // L - 1
    const float* taps;              // h[0 .. L-1]
    const float2* twiddle;          // exp(-2 pi i t / C), t < C / 2
    const uint32_t* off;            // [n_inputs]: index of the call's first sample = advance + off[i]  (mod 2^32)
    uint32_t advance;
    float2* out;
    size_t out_stride;
    long long n_samples;            // input samples per input in this call
    long long m_total;              // output frames per input
    int D, L, lg_c, mt;
    float scale, offset;
};
// the arguments of the corrected kernels (rt_fbank_set_iq_correction)
struct FbankArgsIq : FbankArgs {
    rt::IqCorrArgs corr;
};
template <bool IQ>
using FbankArgsOf = typename std::conditional<IQ, FbankArgsIq, FbankArgs>::type;

inline size_t fbank_smem(int mt, int D, int L) {
    const int C = 2 * D;
    return ((size_t)(mt - 1) * D + L + (size_t)mt * (C + 1) + C / 2) * sizeof(float2);
}

template <int FMT, bool IQ>
__global__ void __launch_bounds__(FB_THREADS) fbank_kernel(const FbankArgsOf<IQ> a) {
    extern __shared__ float2 sm[];
    const int C = 1 << a.lg_c, CP = C + 1, D = a.D, L = a.L, tid = threadIdx.x;
    const int span = (a.mt - 1) * D + L;
    float2* xs = sm;                                    // [span] local sample t = the call's sample m0 D - (L - 1) + t
    float2* fr = sm + span;                             // [mt][C + 1] frames
    float2* tw = fr + (size_t)a.mt * CP;                // [C / 2]
    const int input = blockIdx.y;
    const long long m0 = (long long)blockIdx.x * a.mt;
    const unsigned char* row = a.iq + (size_t)input * a.in_stride;
    const float2* hist = a.hist + (size_t)input * a.hist_len;
    const long long rel0 = m0 * D - (L - 1);
    const rt::IqSpan<IQ> sp = rt::iq_span<IQ>(a, input, rel0);
    for (int t = tid; t < span; t += FB_THREADS) xs[t] = rt::fir_sample<FMT, IQ>(a, row, hist, rel0 + t, sp);
    for (int t = tid; t < C / 2; t += FB_THREADS) tw[t] = a.twiddle[t];
    __syncthreads();

    // u_r of frame mm: tap k = s + q C of output n = n0 + (m0 + mm) D reads the local sample mm D + L - 1 - k, whose global
    // index is = n0 + (m0 + mm) D - s (mod C).  Sum order: q ascending.  Stored at the bit-reversed position of r.
    const uint32_t n0 = a.advance + a.off[input];
    const int n_s = min(C, L);
    for (int i = tid; i < a.mt * C; i += FB_THREADS) {
        const int mm = i >> a.lg_c, s = i & (C - 1);
        float2 acc = make_float2(0.f, 0.f);
        if (s < n_s) {
            const float2* x = xs + mm * D + L - 1 - s;
            for (int k = s; k < L; k += C) {
                const float h = a.taps[k];
                const float2 v = x[s - k];
                acc.x = __fmaf_rn(h, v.x, acc.x);
                acc.y = __fmaf_rn(h, v.y, acc.y);
            }
        }
        const uint32_t r = (n0 + (uint32_t)(m0 + mm) * (uint32_t)D - (uint32_t)s) & (uint32_t)(C - 1);
        fr[mm * CP + (__brev(r) >> (32 - a.lg_c))] = acc;
    }
    __syncthreads();

    // in-place radix-2 decimation-in-time FFT of every frame: bit-reversed in, natural order out, y_k = sum_r e^{-2 pi i k r / C} u_r
    for (int lh = 0; lh < a.lg_c; ++lh) {
        const int h = 1 << lh;
        for (int b = tid; b < a.mt * (C / 2); b += FB_THREADS) {
            const int mm = b >> (a.lg_c - 1), bb = b & (C / 2 - 1);
            const int j = bb & (h - 1);
            float2* f = fr + mm * CP + ((bb - j) << 1) + j;
            const float2 w = tw[j << (a.lg_c - 1 - lh)];
            const float2 p = f[0], q = f[h];
            const float2 t = make_float2(__fmaf_rn(q.x, w.x, -__fmul_rn(q.y, w.y)), __fmaf_rn(q.x, w.y, __fmul_rn(q.y, w.x)));
            f[0] = make_float2(__fadd_rn(p.x, t.x), __fadd_rn(p.y, t.y));
            f[h] = make_float2(__fsub_rn(p.x, t.x), __fsub_rn(p.y, t.y));
        }
        __syncthreads();
    }

    // channel k = rho - (D - 1) is FFT bin k mod C; each row's frames are contiguous in the output
    const int n_rows = C - 1;
    const int mt_here = (int)min((long long)a.mt, a.m_total - m0);
    for (int i = tid; i < n_rows * a.mt; i += FB_THREADS) {
        const int rho = i / a.mt, mm = i - rho * a.mt;
        if (mm < mt_here) {
            const int bin = (rho - (D - 1)) & (C - 1);
            float2* orow = reinterpret_cast<float2*>(reinterpret_cast<unsigned char*>(a.out) +
                                                     (size_t)((long long)input * n_rows + rho) * a.out_stride);
            orow[m0 + mm] = fr[mm * CP + bin];
        }
    }
}

// fbank_kernel of a format and IQ, given as std::integral_constant values (rt::fir_kernels, rt::fir_launch)
constexpr auto fbank_main = [](auto fmt, auto iq) { return fbank_kernel<decltype(fmt)::value, decltype(iq)::value>; };

}  // namespace

struct rt_fbank : rt::FirFrontEnd {
    int lg_c = 0;                                       // log2 of the FFT length C = 2 D
};

extern "C" {

int rt_fbank_create(const rt_fbank_config* cfg, rt_fbank** out) {
    if (!cfg || !out) return fail(RT_ERR_INVALID, "null argument");
    *out = nullptr;
    if (cfg->abi_version != RT_FBANK_ABI_VERSION) return fail(RT_ERR_INVALID, "rt_fbank_config.abi_version mismatch");
    if (cfg->reserved != 0) return fail(RT_ERR_INVALID, "rt_fbank_config.reserved must be zero");
    const int D = cfg->decimation;
    if (D < RT_FBANK_MIN_DECIMATION || D > RT_FBANK_MAX_DECIMATION || (D & (D - 1)) != 0)
        return fail(RT_ERR_INVALID, "decimation must be a power of two in [RT_FBANK_MIN_DECIMATION, RT_FBANK_MAX_DECIMATION]");
    if ((long long)cfg->n_inputs * (2 * D - 1) > (1 << 30)) return fail(RT_ERR_INVALID, "n_inputs * (2 decimation - 1) must be <= 2^30");
    const rt::FirPlan p{cfg->cuda_device, cfg->sample_format, cfg->n_inputs, 2 * D - 1, D, cfg->n_taps, cfg->block_samples, cfg->taps};
    int rc = rt::fir_check(p, RT_FBANK_MAX_TAPS(D), "16 decimation + 1");
    if (rc != RT_OK) return rc;

    // geometry: the largest power-of-two tile of frames whose span and frames fit two CTAs per SM (one frame always fits)
    const int L = p.L;
    int mt = FB_MAX_MT;
    while (mt > 1 && fbank_smem(mt, D, L) > FB_SMEM_TARGET) mt >>= 1;

    // taps rounded to fp32 once; twiddles exp(-2 pi i t / C) in float64, rounded once
    const int C = 2 * D;
    std::vector<float> h(L);
    for (int k = 0; k < L; ++k) h[k] = (float)cfg->taps[k];
    std::vector<float2> w(C / 2);
    for (int t = 0; t < C / 2; ++t) {
        const double ang = -2.0 * M_PI * (double)t / (double)C;
        w[t] = make_float2((float)std::cos(ang), (float)std::sin(ang));
    }
    std::unique_ptr<rt_fbank> f(new rt_fbank());
    while ((1 << f->lg_c) < C) ++f->lg_c;
    rc = rt::fir_open(f.get(), p, mt, fbank_smem(mt, D, L), rt::fir_kernels(fbank_main, p.fmt),
                      {{h.data(), h.size() * sizeof(float)}, {w.data(), w.size() * sizeof(float2)}});
    if (rc == RT_OK) *out = f.release();
    return rc;
}

void rt_fbank_destroy(rt_fbank* f) { delete f; }

int rt_fbank_reset_input(rt_fbank* f, int32_t input, int64_t first_sample) { return rt::fir_reset_input(f, input, first_sample); }

int rt_fbank_run(rt_fbank* f, void* cuda_stream, const void* iq, int32_t iq_on_device, size_t in_stride_bytes, int32_t blocks,
                 void* out, size_t out_stride_bytes) {
    rt::FirRun r;
    const int rc = rt::fir_run_begin(f, cuda_stream, iq, iq_on_device, in_stride_bytes, blocks, out, out_stride_bytes, &r);
    if (rc != RT_OK) return rc;
    FbankArgs a;
    rt::fir_args(a, *f, r);
    a.taps = static_cast<const float*>(f->tables[0]);
    a.twiddle = static_cast<const float2*>(f->tables[1]);
    a.lg_c = f->lg_c;
    const dim3 grid((unsigned)((r.m_total + f->mt - 1) / f->mt), (unsigned)f->n_in);
    rt::fir_launch<FbankArgsIq>(*f, r, a, fbank_main, grid, FB_THREADS);
    return rt::fir_run_end(f, r);
}

int rt_fbank_set_iq_correction(rt_fbank* f, int32_t enable) { return rt::fir_set_iq_correction(f, enable); }

int rt_fbank_read_iq_correction(rt_fbank* f, int32_t input, int32_t block, float out[4]) {
    return rt::fir_read_iq_correction(f, input, block, out);
}

}  // extern "C"
