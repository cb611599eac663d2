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
//   fir_reset_kernel    rt_fbank_reset_input, applied in stream order at the next run (fir_history.cuh)
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "../../include/rt_fbank.h"
#include "fir_history.cuh"
#include "sample_format.cuh"

int rt_internal_fail(int code, const char* msg);   // rt_engine.cu: sets the thread-local rt_last_error() text

namespace {

constexpr int FB_THREADS = 256;
constexpr int FB_MAX_MT = 64;                       // output frames per CTA: 512-byte row segments at most
constexpr size_t FB_SMEM_TARGET = 112 * 1024;       // two CTAs per SM
constexpr size_t FB_SMEM_MAX = 227 * 1024;

int fail(int code, const std::string& msg) { return rt_internal_fail(code, msg.c_str()); }

#define FCU(call)                                                                                  \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess)                                                                     \
            return fail(RT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e));          \
    } while (0)

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

inline size_t fbank_smem(int mt, int D, int L) {
    const int C = 2 * D;
    return ((size_t)(mt - 1) * D + L + (size_t)mt * (C + 1) + C / 2) * sizeof(float2);
}

template <int FMT>
__global__ void __launch_bounds__(FB_THREADS) fbank_kernel(const FbankArgs a) {
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
    for (int t = tid; t < span; t += FB_THREADS) xs[t] = rt::fir_sample<FMT>(a, row, hist, rel0 + t);
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

typedef void (*FbankKernel)(const FbankArgs);
FbankKernel fbank_main(int fmt) {
    switch (fmt) {
        case RT_SAMPLE_CU8: return fbank_kernel<RT_SAMPLE_CU8>;
        case RT_SAMPLE_CI8: return fbank_kernel<RT_SAMPLE_CI8>;
        case RT_SAMPLE_CI16: return fbank_kernel<RT_SAMPLE_CI16>;
        default: return fbank_kernel<RT_SAMPLE_CF32>;
    }
}
FbankKernel fbank_history(int fmt) {
    switch (fmt) {
        case RT_SAMPLE_CU8: return rt::fir_history_kernel<RT_SAMPLE_CU8, FbankArgs>;
        case RT_SAMPLE_CI8: return rt::fir_history_kernel<RT_SAMPLE_CI8, FbankArgs>;
        case RT_SAMPLE_CI16: return rt::fir_history_kernel<RT_SAMPLE_CI16, FbankArgs>;
        default: return rt::fir_history_kernel<RT_SAMPLE_CF32, FbankArgs>;
    }
}

}  // namespace

struct rt_fbank {
    int dev = 0, fmt = 0, n_in = 0, D = 0, L = 0, lg_c = 0;
    long long block = 0;
    rt::SampleFormatInfo info{};
    int mt = 1;
    size_t smem = 0;
    float* d_taps = nullptr;
    float2* d_twiddle = nullptr;
    uint32_t* d_off = nullptr;
    float2* d_hist[2] = {nullptr, nullptr};
    int cur = 0;                                        // d_hist[cur] holds the history before the next run
    uint32_t advance = 0;                               // input samples per input since create, mod 2^32
    std::vector<std::pair<int, uint32_t>> resets;       // (input, first sample mod 2^32), applied at the next run
    unsigned char* d_stage = nullptr;
    size_t stage_bytes = 0;
    cudaEvent_t done = nullptr;
    bool ran = false;
};

static void free_fbank(rt_fbank* f) {
    if (!f) return;
    cudaSetDevice(f->dev);
    if (f->done) {
        cudaEventSynchronize(f->done);
        cudaEventDestroy(f->done);
    }
    cudaFree(f->d_taps);
    cudaFree(f->d_twiddle);
    cudaFree(f->d_off);
    cudaFree(f->d_hist[0]);
    cudaFree(f->d_hist[1]);
    cudaFree(f->d_stage);
    delete f;
}

extern "C" {

int rt_fbank_create(const rt_fbank_config* cfg, rt_fbank** out) {
    if (!cfg || !out) return fail(RT_ERR_INVALID, "null argument");
    *out = nullptr;
    if (cfg->abi_version != RT_FBANK_ABI_VERSION) return fail(RT_ERR_INVALID, "rt_fbank_config.abi_version mismatch");
    if (cfg->reserved != 0) return fail(RT_ERR_INVALID, "rt_fbank_config.reserved must be zero");
    if (cfg->n_inputs < 1 || cfg->n_inputs > 65535) return fail(RT_ERR_INVALID, "n_inputs must be in [1, 65535]");
    const int D = cfg->decimation;
    if (D < RT_FBANK_MIN_DECIMATION || D > RT_FBANK_MAX_DECIMATION || (D & (D - 1)) != 0)
        return fail(RT_ERR_INVALID, "decimation must be a power of two in [RT_FBANK_MIN_DECIMATION, RT_FBANK_MAX_DECIMATION]");
    if ((long long)cfg->n_inputs * (2 * D - 1) > (1 << 30)) return fail(RT_ERR_INVALID, "n_inputs * (2 decimation - 1) must be <= 2^30");
    if (cfg->n_taps < 1 || cfg->n_taps > RT_FBANK_MAX_TAPS(D) || cfg->n_taps % 2 == 0)
        return fail(RT_ERR_INVALID, "n_taps must be odd and in [1, 16 decimation + 1]");
    if (cfg->block_samples < D || cfg->block_samples % D != 0)
        return fail(RT_ERR_INVALID, "block_samples must be a positive multiple of decimation");
    rt::SampleFormatInfo info;
    if (!rt::sample_format_info(cfg->sample_format, &info)) return fail(RT_ERR_INVALID, "unknown sample_format");
    if (!cfg->taps) return fail(RT_ERR_INVALID, "taps missing");
    for (int k = 0; k < cfg->n_taps; ++k)
        if (!std::isfinite(cfg->taps[k])) return fail(RT_ERR_INVALID, "taps must be finite");

    // geometry: the largest power-of-two tile of frames whose span and frames fit two CTAs per SM (one frame always fits)
    const int L = cfg->n_taps;
    int mt = FB_MAX_MT;
    while (mt > 1 && fbank_smem(mt, D, L) > FB_SMEM_TARGET) mt >>= 1;
    const size_t smem = fbank_smem(mt, D, L);
    if (smem > FB_SMEM_MAX) return fail(RT_ERR_INVALID, "decimation and n_taps need more shared memory than a CTA has");

    int ndev = 0;
    FCU(cudaGetDeviceCount(&ndev));
    if (cfg->cuda_device < 0 || cfg->cuda_device >= ndev) return fail(RT_ERR_CUDA, "no such CUDA device (this engine has no CPU fallback)");
    FCU(cudaSetDevice(cfg->cuda_device));
    {
        // the limit belongs to the kernel: only ever raise it (handles with other geometries may exist in this process)
        static std::mutex mu;
        std::lock_guard<std::mutex> lock(mu);
        cudaFuncAttributes fa;
        cudaError_t ferr = cudaFuncGetAttributes(&fa, fbank_main(cfg->sample_format));
        if (ferr != cudaSuccess)
            return fail(RT_ERR_CUDA, std::string("kernels not loadable on this device (built for sm_100a only): ") + cudaGetErrorString(ferr));
        if ((size_t)fa.maxDynamicSharedSizeBytes < smem)
            FCU(cudaFuncSetAttribute(fbank_main(cfg->sample_format), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }

    rt_fbank* f = new rt_fbank();
    f->dev = cfg->cuda_device;
    f->fmt = cfg->sample_format;
    f->n_in = cfg->n_inputs;
    f->D = D;
    f->L = L;
    while ((1 << f->lg_c) < 2 * D) ++f->lg_c;
    f->block = cfg->block_samples;
    f->info = info;
    f->mt = mt;
    f->smem = smem;

    // taps rounded to fp32 once; twiddles exp(-2 pi i t / C) in float64, rounded once
    const int C = 2 * D;
    std::vector<float> h(L);
    for (int k = 0; k < L; ++k) h[k] = (float)cfg->taps[k];
    std::vector<float2> w(C / 2);
    for (int t = 0; t < C / 2; ++t) {
        const double ang = -2.0 * M_PI * (double)t / (double)C;
        w[t] = make_float2((float)std::cos(ang), (float)std::sin(ang));
    }
    const size_t hist_bytes = (size_t)f->n_in * std::max(1, L - 1) * sizeof(float2);
#define FCUE(call)                                                                                 \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            free_fbank(f);                                                                         \
            return fail(RT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e));          \
        }                                                                                          \
    } while (0)
    FCUE(cudaMalloc(&f->d_taps, h.size() * sizeof(float)));
    FCUE(cudaMalloc(&f->d_twiddle, w.size() * sizeof(float2)));
    FCUE(cudaMalloc(&f->d_off, f->n_in * sizeof(uint32_t)));
    FCUE(cudaMalloc(&f->d_hist[0], hist_bytes));
    FCUE(cudaMalloc(&f->d_hist[1], hist_bytes));
    FCUE(cudaMemcpy(f->d_taps, h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
    FCUE(cudaMemcpy(f->d_twiddle, w.data(), w.size() * sizeof(float2), cudaMemcpyHostToDevice));
    FCUE(cudaMemset(f->d_off, 0, f->n_in * sizeof(uint32_t)));
    FCUE(cudaMemset(f->d_hist[0], 0, hist_bytes));
    FCUE(cudaEventCreateWithFlags(&f->done, cudaEventDisableTiming));
#undef FCUE
    *out = f;
    return RT_OK;
}

void rt_fbank_destroy(rt_fbank* f) { free_fbank(f); }

int rt_fbank_reset_input(rt_fbank* f, int32_t input, int64_t first_sample) {
    if (!f || input < 0 || input >= f->n_in) return fail(RT_ERR_INVALID, "bad input index");
    f->resets.emplace_back(input, (uint32_t)(uint64_t)first_sample);
    return RT_OK;
}

int rt_fbank_run(rt_fbank* f, void* cuda_stream, const void* iq, int32_t iq_on_device, size_t in_stride_bytes, int32_t blocks,
                 void* out, size_t out_stride_bytes) {
    if (!f || !iq || !out) return fail(RT_ERR_INVALID, "null argument");
    if (blocks < 1) return fail(RT_ERR_INVALID, "blocks must be >= 1");
    const long long n = f->block * blocks;
    const long long m_total = n / f->D;
    const size_t row_bytes = (size_t)f->info.bytes * (size_t)n;
    if (f->n_in > 1 && in_stride_bytes < row_bytes) return fail(RT_ERR_INVALID, "in_stride_bytes smaller than one input's blocks");
    if (out_stride_bytes < (size_t)m_total * sizeof(float2)) return fail(RT_ERR_INVALID, "out_stride_bytes smaller than one channel's outputs");
    if (((uintptr_t)out | out_stride_bytes) % sizeof(float2) != 0) return fail(RT_ERR_INVALID, "output pointer / stride not aligned to 8 bytes");
    if ((m_total + f->mt - 1) / f->mt > 0x7fffffffLL) return fail(RT_ERR_INVALID, "call too long");
    FCU(cudaSetDevice(f->dev));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    if (f->ran) FCU(cudaStreamWaitEvent(st, f->done, 0));      // history, offsets and the staging buffer of the previous run

    const unsigned char* src = static_cast<const unsigned char*>(iq);
    size_t stride = f->n_in > 1 ? in_stride_bytes : row_bytes;
    if (!iq_on_device) {
        FCU(rt::fir_stage_host_input(st, &src, &stride, row_bytes, f->n_in, &f->d_stage, &f->stage_bytes));
    } else if (((uintptr_t)src | (f->n_in > 1 ? stride : 0)) % (uintptr_t)f->info.bytes != 0) {
        return fail(RT_ERR_INVALID, "IQ pointer / input stride not aligned to one complex sample");
    }

    const int hist_len = std::max(1, f->L - 1);
    for (const auto& r : f->resets)
        rt::fir_reset_kernel<<<1, 256, 0, st>>>(f->d_hist[f->cur], f->d_off, r.first, f->L - 1, r.second - f->advance);

    FbankArgs a;
    a.iq = src;
    a.in_stride = stride;
    a.hist = f->d_hist[f->cur];
    a.hist_out = f->d_hist[f->cur ^ 1];
    a.hist_len = f->L - 1;
    a.taps = f->d_taps;
    a.twiddle = f->d_twiddle;
    a.off = f->d_off;
    a.advance = f->advance;
    a.out = static_cast<float2*>(out);
    a.out_stride = out_stride_bytes;
    a.n_samples = n;
    a.m_total = m_total;
    a.D = f->D;
    a.L = f->L;
    a.lg_c = f->lg_c;
    a.mt = f->mt;
    a.scale = (float)(1.0 / f->info.full_scale);
    a.offset = (float)f->info.offset;
    const dim3 grid((unsigned)((m_total + f->mt - 1) / f->mt), (unsigned)f->n_in);
    fbank_main(f->fmt)<<<grid, FB_THREADS, f->smem, st>>>(a);
    if (f->L > 1) fbank_history(f->fmt)<<<dim3((unsigned)((hist_len + 127) / 128), (unsigned)f->n_in), 128, 0, st>>>(a);
    FCU(cudaGetLastError());
    FCU(cudaEventRecord(f->done, st));
    f->ran = true;
    f->resets.clear();
    f->cur ^= f->L > 1 ? 1 : 0;
    f->advance += (uint32_t)(uint64_t)n;
    return RT_OK;
}

}  // extern "C"
