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
//   fir_reset_kernel    rt_ddc_reset_input, applied in stream order at the next run (fir_history.cuh)
//   iq_moments_kernel, iq_coef_kernel   with rt_ddc_set_iq_correction on: each block's DC and IQ-imbalance coefficients,
//                       which the IQ = true instantiations of the two kernels above apply as they decode (iq_correction.cuh)
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <mutex>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "../../include/rt_ddc.h"
#include "fft_cpk.cuh"
#include "fir_history.cuh"
#include "sample_format.cuh"

int rt_internal_fail(int code, const char* msg);   // rt_engine.cu: sets the thread-local rt_last_error() text

namespace {

constexpr int DDC_THREADS = 128;
constexpr int DDC_MR = 8;                           // consecutive outputs per thread
constexpr int DDC_PAD = 8;                          // zero samples in front of every polyphase row (masked tap tails read them)
constexpr size_t DDC_TAP_BUDGET = 66 * 1024;        // shared memory for the taps of one channel group
constexpr size_t DDC_SMEM_TARGET = 112 * 1024;      // two CTAs per SM
constexpr size_t DDC_SMEM_MAX = 227 * 1024;

int fail(int code, const std::string& msg) { return rt_internal_fail(code, msg.c_str()); }

#define DCU(call)                                                                                  \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess)                                                                     \
            return fail(RT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e));          \
    } while (0)

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

template <bool IQ>
using DdcKernel = void (*)(const DdcArgsOf<IQ>);
template <bool IQ>
DdcKernel<IQ> ddc_main(int fmt) {
    switch (fmt) {
        case RT_SAMPLE_CU8: return ddc_kernel<RT_SAMPLE_CU8, IQ>;
        case RT_SAMPLE_CI8: return ddc_kernel<RT_SAMPLE_CI8, IQ>;
        case RT_SAMPLE_CI16: return ddc_kernel<RT_SAMPLE_CI16, IQ>;
        default: return ddc_kernel<RT_SAMPLE_CF32, IQ>;
    }
}
template <bool IQ>
DdcKernel<IQ> ddc_history(int fmt) {
    switch (fmt) {
        case RT_SAMPLE_CU8: return rt::fir_history_kernel<RT_SAMPLE_CU8, IQ, DdcArgsOf<IQ>>;
        case RT_SAMPLE_CI8: return rt::fir_history_kernel<RT_SAMPLE_CI8, IQ, DdcArgsOf<IQ>>;
        case RT_SAMPLE_CI16: return rt::fir_history_kernel<RT_SAMPLE_CI16, IQ, DdcArgsOf<IQ>>;
        default: return rt::fir_history_kernel<RT_SAMPLE_CF32, IQ, DdcArgsOf<IQ>>;
    }
}

// the filter kernel and the history kernel of one run
template <bool IQ>
void ddc_launch(const DdcArgsOf<IQ>& a, int fmt, dim3 grid, size_t smem, int n_in, cudaStream_t st) {
    ddc_main<IQ>(fmt)<<<grid, DDC_THREADS, smem, st>>>(a);
    if (a.L > 1) ddc_history<IQ>(fmt)<<<dim3((unsigned)((a.L - 1 + 127) / 128), (unsigned)n_in), 128, 0, st>>>(a);
}

// the limit belongs to the kernel: only ever raise it (handles with other geometries may exist in this process)
template <class Kernel>
int raise_smem_limit(Kernel k, size_t smem) {
    cudaFuncAttributes fa;
    cudaError_t ferr = cudaFuncGetAttributes(&fa, k);
    if (ferr != cudaSuccess)
        return fail(RT_ERR_CUDA, std::string("kernels not loadable on this device (built for sm_100a only): ") + cudaGetErrorString(ferr));
    if ((size_t)fa.maxDynamicSharedSizeBytes < smem) DCU(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return RT_OK;
}

}  // namespace

struct rt_ddc {
    int dev = 0, fmt = 0, n_in = 0, nch = 0, D = 0, L = 0;
    long long block = 0;
    rt::SampleFormatInfo info{};
    int cw = 1, lg_cw = 0, mt = DDC_MR;
    size_t smem = 0;
    float2* d_taps = nullptr;
    uint32_t* d_inc = nullptr;
    uint32_t* d_off = nullptr;
    float2* d_hist[2] = {nullptr, nullptr};
    int cur = 0;                                        // d_hist[cur] holds the history before the next run
    uint32_t advance = 0;                               // input samples per input since create, mod 2^32
    std::vector<std::pair<int, uint32_t>> resets;       // (input, first sample mod 2^32), applied at the next run
    unsigned char* d_stage = nullptr;
    size_t stage_bytes = 0;
    cudaEvent_t done = nullptr;
    bool ran = false;
    rt::IqState iq;                                     // rt_ddc_set_iq_correction
};

static void free_ddc(rt_ddc* d) {
    if (!d) return;
    cudaSetDevice(d->dev);
    if (d->done) {
        cudaEventSynchronize(d->done);
        cudaEventDestroy(d->done);
    }
    cudaFree(d->d_taps);
    cudaFree(d->d_inc);
    cudaFree(d->d_off);
    cudaFree(d->d_hist[0]);
    cudaFree(d->d_hist[1]);
    cudaFree(d->d_stage);
    d->iq.release();
    delete d;
}

extern "C" {

int rt_ddc_create(const rt_ddc_config* cfg, rt_ddc** out) {
    if (!cfg || !out) return fail(RT_ERR_INVALID, "null argument");
    *out = nullptr;
    if (cfg->abi_version != RT_DDC_ABI_VERSION) return fail(RT_ERR_INVALID, "rt_ddc_config.abi_version mismatch");
    if (cfg->n_inputs < 1 || cfg->n_inputs > 65535) return fail(RT_ERR_INVALID, "n_inputs must be in [1, 65535]");
    if (cfg->n_channels < 1 || (long long)cfg->n_inputs * cfg->n_channels > (1 << 30)) return fail(RT_ERR_INVALID, "n_channels must be >= 1");
    if (cfg->decimation < 2 || cfg->decimation > RT_DDC_MAX_DECIMATION) return fail(RT_ERR_INVALID, "decimation must be in [2, RT_DDC_MAX_DECIMATION]");
    if (cfg->n_taps < 1 || cfg->n_taps > RT_DDC_MAX_TAPS || cfg->n_taps % 2 == 0) return fail(RT_ERR_INVALID, "n_taps must be odd and in [1, RT_DDC_MAX_TAPS]");
    if (cfg->block_samples < cfg->decimation || cfg->block_samples % cfg->decimation != 0)
        return fail(RT_ERR_INVALID, "block_samples must be a positive multiple of decimation");
    rt::SampleFormatInfo info;
    if (!rt::sample_format_info(cfg->sample_format, &info)) return fail(RT_ERR_INVALID, "unknown sample_format");
    if (!cfg->taps || !cfg->phase_inc) return fail(RT_ERR_INVALID, "taps / phase_inc missing");
    if (cfg->reserved != 0) return fail(RT_ERR_INVALID, "rt_ddc_config.reserved must be zero");
    for (int k = 0; k < cfg->n_taps; ++k)
        if (!std::isfinite(cfg->taps[k])) return fail(RT_ERR_INVALID, "taps must be finite");

    // geometry: CW channels per CTA (a power of two <= 16 whose taps fit DDC_TAP_BUDGET), MT outputs per CTA (every thread group
    // busy unless the span would not fit two CTAs per SM)
    const int D = cfg->decimation, L = cfg->n_taps;
    int cw = 1, lg = 0;
    while (cw < 16 && cw < cfg->n_channels && (size_t)(2 * cw) * L * sizeof(float2) <= DDC_TAP_BUDGET) { cw <<= 1; ++lg; }
    int mt = (DDC_THREADS / cw) * DDC_MR;
    while (mt > DDC_MR && ddc_smem(cw, mt, D, L) > DDC_SMEM_TARGET) mt -= DDC_MR;
    const size_t smem = ddc_smem(cw, mt, D, L);
    if (smem > DDC_SMEM_MAX) return fail(RT_ERR_INVALID, "decimation and n_taps need more shared memory than a CTA has");

    int ndev = 0;
    DCU(cudaGetDeviceCount(&ndev));
    if (cfg->cuda_device < 0 || cfg->cuda_device >= ndev) return fail(RT_ERR_CUDA, "no such CUDA device (this engine has no CPU fallback)");
    DCU(cudaSetDevice(cfg->cuda_device));
    {
        static std::mutex mu;
        std::lock_guard<std::mutex> lock(mu);
        int rc = raise_smem_limit(ddc_main<false>(cfg->sample_format), smem);
        if (rc == RT_OK) rc = raise_smem_limit(ddc_main<true>(cfg->sample_format), smem);
        if (rc != RT_OK) return rc;
    }

    rt_ddc* d = new rt_ddc();
    d->dev = cfg->cuda_device;
    d->fmt = cfg->sample_format;
    d->n_in = cfg->n_inputs;
    d->nch = cfg->n_channels;
    d->D = D;
    d->L = L;
    d->block = cfg->block_samples;
    d->info = info;
    d->cw = cw;
    d->lg_cw = lg;
    d->mt = mt;
    d->smem = smem;

    // g_c[k] = h[k] exp(+2 pi i ((inc_c k) mod 2^32) / 2^32), in float64, rounded once
    std::vector<float2> g((size_t)d->nch * L);
    for (int c = 0; c < d->nch; ++c)
        for (int k = 0; k < L; ++k) {
            const uint32_t ph = cfg->phase_inc[c] * (uint32_t)k;
            const double ang = 2.0 * M_PI * (double)ph / 4294967296.0;
            g[(size_t)c * L + k] = make_float2((float)(cfg->taps[k] * std::cos(ang)), (float)(cfg->taps[k] * std::sin(ang)));
        }
    const size_t hist_bytes = (size_t)d->n_in * std::max(1, L - 1) * sizeof(float2);
#define DCUE(call)                                                                                 \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            free_ddc(d);                                                                           \
            return fail(RT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e));          \
        }                                                                                          \
    } while (0)
    DCUE(cudaMalloc(&d->d_taps, g.size() * sizeof(float2)));
    DCUE(cudaMalloc(&d->d_inc, d->nch * sizeof(uint32_t)));
    DCUE(cudaMalloc(&d->d_off, d->n_in * sizeof(uint32_t)));
    DCUE(cudaMalloc(&d->d_hist[0], hist_bytes));
    DCUE(cudaMalloc(&d->d_hist[1], hist_bytes));
    DCUE(cudaMemcpy(d->d_taps, g.data(), g.size() * sizeof(float2), cudaMemcpyHostToDevice));
    DCUE(cudaMemcpy(d->d_inc, cfg->phase_inc, d->nch * sizeof(uint32_t), cudaMemcpyHostToDevice));
    DCUE(cudaMemset(d->d_off, 0, d->n_in * sizeof(uint32_t)));
    DCUE(cudaMemset(d->d_hist[0], 0, hist_bytes));
    DCUE(cudaEventCreateWithFlags(&d->done, cudaEventDisableTiming));
#undef DCUE
    *out = d;
    return RT_OK;
}

void rt_ddc_destroy(rt_ddc* d) { free_ddc(d); }

int rt_ddc_reset_input(rt_ddc* d, int32_t input, int64_t first_sample) {
    if (!d || input < 0 || input >= d->n_in) return fail(RT_ERR_INVALID, "bad input index");
    d->resets.emplace_back(input, (uint32_t)(uint64_t)first_sample);
    return RT_OK;
}

int rt_ddc_run(rt_ddc* d, void* cuda_stream, const void* iq, int32_t iq_on_device, size_t in_stride_bytes, int32_t blocks,
               void* out, size_t out_stride_bytes) {
    if (!d || !iq || !out) return fail(RT_ERR_INVALID, "null argument");
    if (blocks < 1) return fail(RT_ERR_INVALID, "blocks must be >= 1");
    const long long n = d->block * blocks;
    const long long m_total = n / d->D;
    const size_t row_bytes = (size_t)d->info.bytes * (size_t)n;
    if (d->n_in > 1 && in_stride_bytes < row_bytes) return fail(RT_ERR_INVALID, "in_stride_bytes smaller than one input's blocks");
    if (out_stride_bytes < (size_t)m_total * sizeof(float2) && (long long)d->n_in * d->nch > 1)
        return fail(RT_ERR_INVALID, "out_stride_bytes smaller than one channel's outputs");
    if (((uintptr_t)out | out_stride_bytes) % sizeof(float2) != 0) return fail(RT_ERR_INVALID, "output pointer / stride not aligned to 8 bytes");
    if ((m_total + d->mt - 1) / d->mt > 0x7fffffffLL) return fail(RT_ERR_INVALID, "call too long");
    DCU(cudaSetDevice(d->dev));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    if (d->ran) DCU(cudaStreamWaitEvent(st, d->done, 0));      // history, offsets and the staging buffer of the previous run

    const unsigned char* src = static_cast<const unsigned char*>(iq);
    size_t stride = d->n_in > 1 ? in_stride_bytes : row_bytes;
    if (!iq_on_device) {
        DCU(rt::fir_stage_host_input(st, &src, &stride, row_bytes, d->n_in, &d->d_stage, &d->stage_bytes));
    } else if (((uintptr_t)src | (d->n_in > 1 ? stride : 0)) % (uintptr_t)d->info.bytes != 0) {
        return fail(RT_ERR_INVALID, "IQ pointer / input stride not aligned to one complex sample");
    }

    rt::IqCorrArgs corr;
    DCU(rt::iq_prepare(d->iq, st, d->done, d->ran, d->fmt, d->info, src, stride, d->n_in, d->block, blocks, &corr));
    for (const auto& r : d->resets)
        rt::fir_reset_kernel<<<1, 256, 0, st>>>(d->d_hist[d->cur], d->d_off, r.first, d->L - 1, r.second - d->advance);

    DdcArgs a;
    a.iq = src;
    a.in_stride = stride;
    a.hist = d->d_hist[d->cur];
    a.hist_out = d->d_hist[d->cur ^ 1];
    a.hist_len = d->L - 1;
    a.taps = d->d_taps;
    a.inc = d->d_inc;
    a.off = d->d_off;
    a.advance = d->advance;
    a.out = static_cast<float2*>(out);
    a.out_stride = out_stride_bytes;
    a.n_samples = n;
    a.m_total = m_total;
    a.D = d->D;
    a.L = d->L;
    a.n_channels = d->nch;
    a.cw = d->cw;
    a.lg_cw = d->lg_cw;
    a.mt = d->mt;
    a.rows = ddc_rows(d->mt, d->D, d->L);
    a.scale = (float)(1.0 / d->info.full_scale);
    a.offset = (float)d->info.offset;
    const dim3 grid((unsigned)((m_total + d->mt - 1) / d->mt), (unsigned)((d->nch + d->cw - 1) / d->cw), (unsigned)d->n_in);
    if (d->iq.applied) {
        DdcArgsIq ai;
        static_cast<DdcArgs&>(ai) = a;
        ai.corr = corr;
        ddc_launch<true>(ai, d->fmt, grid, d->smem, d->n_in, st);
    } else {
        ddc_launch<false>(a, d->fmt, grid, d->smem, d->n_in, st);
    }
    DCU(cudaGetLastError());
    DCU(cudaEventRecord(d->done, st));
    d->ran = true;
    d->resets.clear();
    d->cur ^= d->L > 1 ? 1 : 0;
    d->advance += (uint32_t)(uint64_t)n;
    return RT_OK;
}

int rt_ddc_set_iq_correction(rt_ddc* d, int32_t enable) {
    if (!d) return fail(RT_ERR_INVALID, "null handle");
    if (enable && d->block > rt::IQ_MAX_BLOCK) return fail(RT_ERR_INVALID, "block_samples must be <= 2^30 for the IQ correction");
    d->iq.on = enable != 0;
    return RT_OK;
}

int rt_ddc_read_iq_correction(rt_ddc* d, int32_t input, int32_t block, float out[4]) {
    if (!d || !out) return fail(RT_ERR_INVALID, "null argument");
    if (!d->iq.applied) return fail(RT_ERR_INVALID, "the last run did not apply the IQ correction");
    if (input < 0 || input >= d->n_in || block < 0 || block >= d->iq.blocks) return fail(RT_ERR_INVALID, "bad input / block index");
    DCU(cudaSetDevice(d->dev));
    DCU(rt::iq_read(d->iq, d->done, input, block, out));
    return RT_OK;
}

}  // extern "C"
