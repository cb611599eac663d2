// rt_ddc.cu -- wideband down-converter (include/rt_ddc.h): mix every channel to baseband, filter with real taps, keep every
// D-th sample, for many channels of many wideband inputs at once, in fp32 on the CUDA cores.
//
// Kernels (all on the caller's stream):
//   ddc_kernel          one CTA = one tile of MT outputs of CW channels of one input.  It decodes the input span those outputs
//                       read ((MT - 1) D + L samples, the history for indices before the call) into shared memory once, in
//                       polyphase order (row b holds the samples whose local index is b mod D), and holds the complex taps
//                       g_c of its CW channels.  A thread owns one channel and DDC_MR consecutive outputs: for a tap phase r
//                       the outputs read consecutive samples of one polyphase row, so eight taps of a phase need 15 samples
//                       and 8 taps (shared loads) for 64 complex products (128 packed fp32x2 FMAs, fft_cpk.cuh)
//   fir_history_kernel  the last L - 1 normalised samples of every input, for the next call (double-buffered; fir_history.cuh)
// With rt_ddc_set_iq_correction on, the IQ = true instantiations of both apply each block's DC and IQ-imbalance coefficients as
// they decode (iq_correction.cuh).  The handle, the checks and steps a run shares with the filter bank, the reset kernel and
// the kernels that form the coefficients are in fir_frontend.cu.
#include <cuda_runtime.h>

#include <cmath>
#include <memory>
#include <type_traits>
#include <vector>

#include "../../include/rt_ddc.h"
#include "fft_cpk.cuh"
#include "fir_frontend.cuh"

namespace {

constexpr int DDC_THREADS = 128;
constexpr int DDC_MR = 8;                           // consecutive outputs per thread
constexpr int DDC_PAD = 8;                          // zero samples in front of every polyphase row (masked tap tails read them)
constexpr size_t DDC_TAP_BUDGET = 66 * 1024;        // shared memory for the taps of one channel group
constexpr size_t DDC_SMEM_TARGET = 112 * 1024;      // two CTAs per SM

using rt::fail;

struct DdcArgs {
    const unsigned char* iq;        // input i at iq + i * in_stride
    size_t in_stride;
    const float2* hist;             // [n_inputs][hist_len] normalised samples before the call
    float2* hist_out;               // the same after the call
    int hist_len;                   // L - 1
    const float2* taps;             // [n_channels][L] g_c
    const uint32_t* inc;            // [n_channels]
    const uint32_t* off;            // [n_inputs]: index of the call's first sample = advance + off[i]  (mod 2^32)
    uint32_t advance;
    float2* out;
    size_t out_stride;
    long long n_samples;            // input samples per input in this call
    long long m_total;              // outputs per channel
    int D, L, n_channels, cw, lg_cw, mt, rows;
    float scale, offset;
};
// the arguments of the corrected kernels (rt_ddc_set_iq_correction)
struct DdcArgsIq : DdcArgs {
    rt::IqCorrArgs corr;
};
template <bool IQ>
using DdcArgsOf = typename std::conditional<IQ, DdcArgsIq, DdcArgs>::type;

// polyphase row length: a zero pad, the MT outputs' own samples and the (L - 1) / D earlier ones, odd (conflict-free fills)
inline int ddc_rows(int mt, int D, int L) { return (DDC_PAD + mt + (L - 1) / D) | 1; }
inline size_t ddc_smem(int cw, int mt, int D, int L) {
    return (size_t)cw * L * sizeof(float2) + (size_t)D * ddc_rows(mt, D, L) * sizeof(float2);
}

template <int FMT, bool IQ>
__global__ void __launch_bounds__(DDC_THREADS) ddc_kernel(const DdcArgsOf<IQ> a) {
    extern __shared__ float2 sm[];
    float2* gs = sm;                                    // [cw][L]
    float2* xs = sm + (size_t)a.cw * a.L;               // [D][rows]
    const int input = blockIdx.z, c0 = blockIdx.y * a.cw, tid = threadIdx.x;
    const long long m0 = (long long)blockIdx.x * a.mt;
    for (int i = tid; i < a.cw * a.L; i += DDC_THREADS) {
        const int cl = i / a.L, c = c0 + cl;
        gs[i] = c < a.n_channels ? a.taps[(size_t)c * a.L + (i - cl * a.L)] : make_float2(0.f, 0.f);
    }
    // local sample t is the call's sample m0 D - (L - 1) + t; it lives at xs[(t % D) * rows + DDC_PAD + t / D]
    const unsigned char* row = a.iq + (size_t)input * a.in_stride;
    const float2* hist = a.hist + (size_t)input * a.hist_len;
    const long long rel0 = m0 * a.D - (a.L - 1);
    const long long span = (long long)(a.mt - 1) * a.D + a.L;
    const int n_fill = (a.rows - DDC_PAD) * a.D;
    const rt::IqSpan<IQ> sp = rt::iq_span<IQ>(a, input, rel0);
    for (int t = tid; t < n_fill; t += DDC_THREADS) {
        const int q = t / a.D, b = t - q * a.D;
        xs[b * a.rows + DDC_PAD + q] = t < span ? rt::fir_sample<FMT, IQ>(a, row, hist, rel0 + t, sp) : make_float2(0.f, 0.f);
    }
    for (int p = tid; p < DDC_PAD * a.D; p += DDC_THREADS) {
        const int q = p / a.D;
        xs[(p - q * a.D) * a.rows + q] = make_float2(0.f, 0.f);
    }
    __syncthreads();

    const int lane = tid & 31, cl = lane & (a.cw - 1), c = c0 + cl;
    const int groups = DDC_THREADS >> a.lg_cw;
    const float2* gch = gs + cl * a.L;
    const int n_r = min(a.D, a.L);
    for (int og = (tid >> 5) * (32 >> a.lg_cw) + (lane >> a.lg_cw); og < a.mt / DDC_MR; og += groups) {
        rt::cpk acc[DDC_MR];
#pragma unroll
        for (int j = 0; j < DDC_MR; ++j) acc[j] = rt::c_make(0.f, 0.f);
        // term k = q D + r of output mm = og MR + j reads the local sample (mm - q) D + L - 1 - r: polyphase row b = e % D,
        // position mm - q + e / D with e = L - 1 - r.  Order of the sum: r ascending, then q ascending.
        for (int r = 0; r < n_r; ++r) {
            const int e = a.L - 1 - r, a0 = e / a.D, b = e - a0 * a.D, Q = a0 + 1;
            const float2* xrow = xs + b * a.rows + DDC_PAD + og * DDC_MR + a0;     // sample (j, q) at xrow[j - q]
            for (int q0 = 0; q0 < Q; q0 += 8) {
                float2 v[DDC_MR + 7];
#pragma unroll
                for (int t = 0; t < DDC_MR + 7; ++t) v[t] = xrow[t - 7 - q0];      // t = j - u + 7 for q = q0 + u
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    // taps past the phase's last one are zero (they meet the zero pad or real samples: 0 * x adds nothing)
                    const float2 g = q0 + u < Q ? gch[(q0 + u) * a.D + r] : make_float2(0.f, 0.f);
                    const rt::cpk gp = rt::c_make(g.x, g.y), gq = rt::c_make(-g.y, g.x);
#pragma unroll
                    for (int j = 0; j < DDC_MR; ++j) {
                        const float2 x = v[j - u + 7];
                        acc[j] = rt::c_fma_s(gq, x.y, rt::c_fma_s(gp, x.x, acc[j]));   // += g * x
                    }
                }
            }
        }
        if (c < a.n_channels) {
            const uint32_t inc = a.inc[c];
            const uint32_t n0 = a.advance + a.off[input];
            float2* orow = reinterpret_cast<float2*>(reinterpret_cast<unsigned char*>(a.out) + (size_t)(input * a.n_channels + c) * a.out_stride);
#pragma unroll
            for (int j = 0; j < DDC_MR; ++j) {
                const long long m = m0 + og * DDC_MR + j;
                if (m < a.m_total) {
                    // exp(-2 pi i ph / 2^32) with ph = inc (n0 + m D) mod 2^32, as a signed fraction of pi
                    const uint32_t ph = inc * (n0 + (uint32_t)m * (uint32_t)a.D);
                    float s, co;
                    sincospif((float)(int32_t)ph * 0x1p-31f, &s, &co);
                    const float ar = rt::c_re(acc[j]), ai = rt::c_im(acc[j]);
                    orow[m] = make_float2(__fmaf_rn(ar, co, __fmul_rn(ai, s)), __fmaf_rn(ai, co, -__fmul_rn(ar, s)));
                }
            }
        }
    }
}

// ddc_kernel of a format and IQ, given as std::integral_constant values (rt::fir_kernels, rt::fir_launch)
constexpr auto ddc_main = [](auto fmt, auto iq) { return ddc_kernel<decltype(fmt)::value, decltype(iq)::value>; };

}  // namespace

struct rt_ddc : rt::FirFrontEnd {
    int cw = 1, lg_cw = 0;                              // channels per CTA, its log2
};

extern "C" {

int rt_ddc_create(const rt_ddc_config* cfg, rt_ddc** out) {
    if (!cfg || !out) return fail(RT_ERR_INVALID, "null argument");
    *out = nullptr;
    if (cfg->abi_version != RT_DDC_ABI_VERSION) return fail(RT_ERR_INVALID, "rt_ddc_config.abi_version mismatch");
    if (cfg->reserved != 0) return fail(RT_ERR_INVALID, "rt_ddc_config.reserved must be zero");
    if (cfg->n_channels < 1 || (long long)cfg->n_inputs * cfg->n_channels > (1 << 30)) return fail(RT_ERR_INVALID, "n_channels must be >= 1");
    if (cfg->decimation < 2 || cfg->decimation > RT_DDC_MAX_DECIMATION) return fail(RT_ERR_INVALID, "decimation must be in [2, RT_DDC_MAX_DECIMATION]");
    if (!cfg->taps || !cfg->phase_inc) return fail(RT_ERR_INVALID, "taps / phase_inc missing");
    const rt::FirPlan p{cfg->cuda_device, cfg->sample_format, cfg->n_inputs, cfg->n_channels, cfg->decimation, cfg->n_taps,
                        cfg->block_samples, cfg->taps};
    int rc = rt::fir_check(p, RT_DDC_MAX_TAPS, "RT_DDC_MAX_TAPS");
    if (rc != RT_OK) return rc;

    // geometry: CW channels per CTA (a power of two <= 16 whose taps fit DDC_TAP_BUDGET), MT outputs per CTA (every thread group
    // busy unless the span would not fit two CTAs per SM)
    const int D = p.D, L = p.L;
    int cw = 1, lg = 0;
    while (cw < 16 && cw < p.nch && (size_t)(2 * cw) * L * sizeof(float2) <= DDC_TAP_BUDGET) { cw <<= 1; ++lg; }
    int mt = (DDC_THREADS / cw) * DDC_MR;
    while (mt > DDC_MR && ddc_smem(cw, mt, D, L) > DDC_SMEM_TARGET) mt -= DDC_MR;

    // g_c[k] = h[k] exp(+2 pi i ((inc_c k) mod 2^32) / 2^32), in float64, rounded once
    std::vector<float2> g((size_t)p.nch * L);
    for (int c = 0; c < p.nch; ++c)
        for (int k = 0; k < L; ++k) {
            const uint32_t ph = cfg->phase_inc[c] * (uint32_t)k;
            const double ang = 2.0 * M_PI * (double)ph / 4294967296.0;
            g[(size_t)c * L + k] = make_float2((float)(cfg->taps[k] * std::cos(ang)), (float)(cfg->taps[k] * std::sin(ang)));
        }
    std::unique_ptr<rt_ddc> d(new rt_ddc());
    d->cw = cw;
    d->lg_cw = lg;
    rc = rt::fir_open(d.get(), p, mt, ddc_smem(cw, mt, D, L), rt::fir_kernels(ddc_main, p.fmt),
                      {{g.data(), g.size() * sizeof(float2)}, {cfg->phase_inc, (size_t)p.nch * sizeof(uint32_t)}});
    if (rc == RT_OK) *out = d.release();
    return rc;
}

void rt_ddc_destroy(rt_ddc* d) { delete d; }

int rt_ddc_reset_input(rt_ddc* d, int32_t input, int64_t first_sample) { return rt::fir_reset_input(d, input, first_sample); }

int rt_ddc_run(rt_ddc* d, void* cuda_stream, const void* iq, int32_t iq_on_device, size_t in_stride_bytes, int32_t blocks,
               void* out, size_t out_stride_bytes) {
    rt::FirRun r;
    const int rc = rt::fir_run_begin(d, cuda_stream, iq, iq_on_device, in_stride_bytes, blocks, out, out_stride_bytes, &r);
    if (rc != RT_OK) return rc;
    DdcArgs a;
    rt::fir_args(a, *d, r);
    a.taps = static_cast<const float2*>(d->tables[0]);
    a.inc = static_cast<const uint32_t*>(d->tables[1]);
    a.n_channels = d->nch;
    a.cw = d->cw;
    a.lg_cw = d->lg_cw;
    a.rows = ddc_rows(d->mt, d->D, d->L);
    const dim3 grid((unsigned)((r.m_total + d->mt - 1) / d->mt), (unsigned)((d->nch + d->cw - 1) / d->cw), (unsigned)d->n_in);
    rt::fir_launch<DdcArgsIq>(*d, r, a, ddc_main, grid, DDC_THREADS);
    return rt::fir_run_end(d, r);
}

int rt_ddc_set_iq_correction(rt_ddc* d, int32_t enable) { return rt::fir_set_iq_correction(d, enable); }

int rt_ddc_read_iq_correction(rt_ddc* d, int32_t input, int32_t block, float out[4]) {
    return rt::fir_read_iq_correction(d, input, block, out);
}

}  // extern "C"
