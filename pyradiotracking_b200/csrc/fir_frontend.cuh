// fir_frontend.cuh -- the host side that the FIR front ends of librtb200.so (the down-converter rt_ddc.cu and the filter bank
// rt_fbank.cu) share: the state of a handle, create's common checks and set-up, and the steps of a run around the front end's
// own filter kernel.  The functions are compiled once, in fir_frontend.cu.
//
// A front end keeps what is its own: its plan checks, its geometry, its constant tables, its argument struct, its grid and its
// filter kernel.  Its argument struct A has the fields fir_history.cuh lists and
//   const uint32_t* off; uint32_t advance;        index of the call's first sample = advance + off[i]  (mod 2^32)
//   float2* out; size_t out_stride;               output row r at out + r * out_stride bytes
//   long long m_total;                            outputs per row in this call
//   int D, L, mt;
// and its corrected kernels take a struct derived from A that adds `IqCorrArgs corr`.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <initializer_list>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "fir_history.cuh"
#include "iq_correction.cuh"
#include "sample_format.cuh"

namespace rt {

int fail(int code, const std::string& msg);         // sets the thread-local rt_last_error() text; returns code

// f(std::integral_constant<int, RT_SAMPLE_*>) for the run-time sample format `fmt` (one sample_format_info accepts)
template <class F>
auto with_format(int fmt, F&& f) {
    switch (fmt) {
        case RT_SAMPLE_CU8: return f(std::integral_constant<int, RT_SAMPLE_CU8>{});
        case RT_SAMPLE_CI8: return f(std::integral_constant<int, RT_SAMPLE_CI8>{});
        case RT_SAMPLE_CI16: return f(std::integral_constant<int, RT_SAMPLE_CI16>{});
        default: return f(std::integral_constant<int, RT_SAMPLE_CF32>{});
    }
}

// The host half of the IQ correction of one handle: the setting, the coefficient and tile-sum buffers (grown when a call carries
// more blocks, after the previous run has finished with them) and what the last run did.
struct IqState {
    bool on = false;                    // set_iq_correction: applied from the next run
    bool applied = false;               // the last run corrected
    int blocks = 0;                     // blocks of that run
    float4* coef = nullptr;             // [n_inputs][blocks]
    size_t coef_bytes = 0;
    void* part = nullptr;               // [n_inputs][blocks][tiles][5] int64 or float64 tile sums
    size_t part_bytes = 0;
};

// The state of a front-end handle; struct rt_ddc and struct rt_fbank derive from it.  The destructor waits for the last run and
// frees everything.
struct FirFrontEnd {
    int dev = -1;                                       // -1 until fir_open has selected the device
    int fmt = 0, n_in = 0, nch = 0, D = 0, L = 0;       // nch: output rows per input
    long long block = 0;
    SampleFormatInfo info{};
    int mt = 1;                                         // outputs (DDC) or output frames (filter bank) per CTA
    size_t smem = 0;                                    // dynamic shared memory of the filter kernel
    std::vector<void*> tables;                          // the front end's constant tables, in the order fir_open got them
    uint32_t* d_off = nullptr;
    float2* d_hist[2] = {nullptr, nullptr};
    int cur = 0;                                        // d_hist[cur] holds the history before the next run
    uint32_t advance = 0;                               // input samples per input since create, mod 2^32
    std::vector<std::pair<int, uint32_t>> resets;       // (input, first sample mod 2^32), applied at the next run
    unsigned char* d_stage = nullptr;
    size_t stage_bytes = 0;
    cudaEvent_t done = nullptr;
    bool ran = false;
    IqState iq;                                         // set_iq_correction
    ~FirFrontEnd();
};

// the configuration fields both front ends have
struct FirPlan {
    int dev, fmt, n_in, nch, D, L;
    long long block;
    const double* taps;
};

// create's checks of the fields in FirPlan, after the front end's own (which validate D): n_inputs, n_taps (odd, at most
// max_taps, which `max_taps_text` names), block_samples, sample_format and the taps
int fir_check(const FirPlan& p, int max_taps, const char* max_taps_text);

// The filter kernel's two instantiations (IQ = false, true) for the sample format `fmt`: kernel(fmt, iq) takes
// std::integral_constant values of the format and of IQ and returns the kernel.
template <class Kernel>
std::pair<const void*, const void*> fir_kernels(Kernel kernel, int fmt) {
    return with_format(fmt, [&](auto f) {
        return std::make_pair((const void*)kernel(f, std::false_type{}), (const void*)kernel(f, std::true_type{}));
    });
}

// a constant table of the front end, on the host
struct HostTable {
    const void* data;
    size_t bytes;
};

// The rest of create, on the checked plan `p` with the front end's geometry (mt, smem): select the device, raise the shared-memory
// limit of both filter kernels to smem, then set f's fields, and allocate and fill the offsets, the history, the event and the
// front end's constant tables.  On failure f holds what was allocated; the caller deletes it.
int fir_open(FirFrontEnd* f, const FirPlan& p, int mt, size_t smem, std::pair<const void*, const void*> kernels,
             std::initializer_list<HostTable> tables);

int fir_reset_input(FirFrontEnd* f, int input, int64_t first_sample);
int fir_set_iq_correction(FirFrontEnd* f, int enable);
int fir_read_iq_correction(FirFrontEnd* f, int input, int block, float out[4]);

// One run, as the steps before the front end's kernels leave it.
struct FirRun {
    cudaStream_t st;
    const unsigned char* src;           // input i at src + i * stride, on the device (the staged copy of a host input)
    size_t stride;
    long long n, m_total;               // input samples per input, outputs per row
    void* out;
    size_t out_stride;
    IqCorrArgs corr;                    // when f.iq.applied
};

// The steps of a run before the front end's kernels: the argument checks, the wait for the previous run, the staging copy of a
// host input, the alignment check of a device input, the IQ coefficients of this run and the pending resets.
int fir_run_begin(FirFrontEnd* f, void* cuda_stream, const void* iq, int iq_on_device, size_t in_stride_bytes, int blocks,
                  void* out, size_t out_stride_bytes, FirRun* r);
// ... and after them: the launch check, the event, the history flip and the advance.
int fir_run_end(FirFrontEnd* f, const FirRun& r);

// the fields of the argument struct A that fir_history.cuh and this file define
template <class A>
void fir_args(A& a, const FirFrontEnd& f, const FirRun& r) {
    a.iq = r.src;
    a.in_stride = r.stride;
    a.hist = f.d_hist[f.cur];
    a.hist_out = f.d_hist[f.cur ^ 1];
    a.hist_len = f.L - 1;
    a.off = f.d_off;
    a.advance = f.advance;
    a.out = static_cast<float2*>(r.out);
    a.out_stride = r.out_stride;
    a.n_samples = r.n;
    a.m_total = r.m_total;
    a.D = f.D;
    a.L = f.L;
    a.mt = f.mt;
    a.scale = (float)(1.0 / f.info.full_scale);
    a.offset = (float)f.info.offset;
}

// The kernels of a run: the filter kernel kernel(fmt, iq) (as for fir_kernels) on `grid` x `threads` and the history kernel,
// with the arguments `a`, or, when the run corrects, with AIq (derived from A) holding a and the run's coefficients.
template <class AIq, class A, class Kernel>
void fir_launch(const FirFrontEnd& f, const FirRun& r, const A& a, Kernel kernel, dim3 grid, int threads) {
    const auto launch = [&](auto iq, const auto& args) {
        with_format(f.fmt, [&](auto fmt) {
            kernel(fmt, iq)<<<grid, threads, f.smem, r.st>>>(args);
            if (f.L > 1)
                fir_history_kernel<decltype(fmt)::value, decltype(iq)::value>
                    <<<dim3((unsigned)((f.L - 1 + 127) / 128), (unsigned)f.n_in), 128, 0, r.st>>>(args);
        });
    };
    if (f.iq.applied) {
        AIq ai;
        static_cast<A&>(ai) = a;
        ai.corr = r.corr;
        launch(std::true_type{}, ai);
    } else {
        launch(std::false_type{}, a);
    }
}

}  // namespace rt
