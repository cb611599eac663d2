// fir_frontend.cu -- the host side of the FIR front ends of librtb200.so (fir_frontend.cuh), written once for the down-converter
// (rt_ddc.cu) and the filter bank (rt_fbank.cu), and their kernels that do not depend on the front end.
//
// Kernels (all on the front end's stream, ahead of its filter kernel, with no host synchronisation):
//   fir_reset_kernel    reset_input, applied in stream order at the next run
//   iq_moments_kernel   with set_iq_correction on: one CTA = one tile of IQ_TILE samples of one block of one input: the five sums
//                       S_I, S_Q, S_II, S_QQ, S_IQ of the tile's elements (ci8, ci16: the element; cu8: the byte - 128; exact
//                       int64) or of its values (cf32: float64, each thread in sample order, then a fixed shuffle tree and the
//                       warps in order)
//   iq_coef_kernel      one warp = one (input, block): the sums of its tiles in a fixed order (lane l takes the tiles l, l + 32,
//                       ..., then a fixed shuffle tree); lane 0 forms m and w (iq_correction.cuh) in float64 and stores them as
//                       fp32
// Tiles start at the block's first sample, so the sums of a block never depend on how many blocks a call carries, on the batch
// or on the grid.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <mutex>
#include <string>
#include <type_traits>

#include "fir_frontend.cuh"

int rt_internal_fail(int code, const char* msg);   // rt_engine.cu: sets the thread-local rt_last_error() text

namespace rt {

int fail(int code, const std::string& msg) { return rt_internal_fail(code, msg.c_str()); }

namespace {

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess)                                                                     \
            return fail(RT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e));          \
    } while (0)

constexpr size_t FIR_SMEM_MAX = 227 * 1024;     // dynamic shared memory of one CTA
constexpr int IQ_THREADS = 256;
constexpr int IQ_TILE = 16384;                  // samples per moments CTA (64 per thread)
constexpr long long IQ_MAX_BLOCK = 1LL << 30;   // block_samples with the correction on: exact int64 sums, 32-bit in-span division

// reset_input, applied in stream order at the next run: zero history, and the phase offset of the input
__global__ void fir_reset_kernel(float2* hist, uint32_t* off, int input, int hist_len, uint32_t off_value) {
    for (int j = threadIdx.x; j < hist_len; j += blockDim.x) hist[(size_t)input * hist_len + j] = make_float2(0.f, 0.f);
    if (threadIdx.x == 0) off[input] = off_value;
}

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

// the limit belongs to the kernel: only ever raise it (handles with other geometries may exist in this process)
int raise_smem_limit(const void* k, size_t smem) {
    cudaFuncAttributes fa;
    cudaError_t ferr = cudaFuncGetAttributes(&fa, k);
    if (ferr != cudaSuccess)
        return fail(RT_ERR_CUDA, std::string("kernels not loadable on this device (built for sm_100a only): ") + cudaGetErrorString(ferr));
    if ((size_t)fa.maxDynamicSharedSizeBytes < smem) CU(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return RT_OK;
}

// Copy n_in host rows of row_bytes (stride `stride`) into the device staging buffer (*stage, grown when too small, rows 256-byte
// aligned) on `st`; *src and *stride then describe the staged copy.
cudaError_t stage_host_input(cudaStream_t st, const unsigned char** src, size_t* stride, size_t row_bytes, int n_in,
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

// magic and shift of the division by d (2 <= d <= 2^30) for dividends below 2^31 (Granlund and Montgomery, "Division by
// invariant integers using multiplication", 1994, Theorem 4.2 with N = 31: l = ceil(log2 d), magic = ceil(2^(31 + l) / d) < 2^32)
void iq_division_magic(long long d, uint32_t* magic, int* shift) {
    int l = 0;
    while ((1LL << l) < d) ++l;
    const unsigned __int128 num = (unsigned __int128)1 << (31 + l);
    *magic = (uint32_t)((num + (unsigned __int128)d - 1) / (unsigned __int128)d);
    *shift = l - 1;
}

cudaError_t iq_grow(void** buf, size_t* have, size_t need, cudaEvent_t done, bool ran) {
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

// One run of f: with the correction on, enqueue the tile sums and the coefficients of `blocks` blocks of every input (rows at
// src + i * stride) on `st` and describe them in *args; off, *args is zero and nothing is enqueued.  The buffers are grown only
// after f's last run, which may still read them, has finished.
cudaError_t iq_prepare(FirFrontEnd& f, cudaStream_t st, const unsigned char* src, size_t stride, int blocks, IqCorrArgs* args) {
    IqState& s = f.iq;
    *args = IqCorrArgs{};
    s.applied = false;
    if (!s.on) return cudaSuccess;
    const long long block = f.block;
    const int n_in = f.n_in, tiles = (int)((block + IQ_TILE - 1) / IQ_TILE);
    cudaError_t e;
    if ((e = iq_grow((void**)&s.coef, &s.coef_bytes, (size_t)n_in * blocks * sizeof(float4), f.done, f.ran)) != cudaSuccess) return e;
    if ((e = iq_grow(&s.part, &s.part_bytes, (size_t)n_in * blocks * tiles * 5 * 8, f.done, f.ran)) != cudaSuccess) return e;
    // elements e map to x = e * scale + offset (scale = (float)(1 / full_scale), as rt::load_normalised); the cu8 sums are of b - 128
    const double scale = (double)(float)(1.0 / f.info.full_scale);
    const double offset = f.fmt == RT_SAMPLE_CU8 ? f.info.offset + 128.0 * scale : f.info.offset;
    const dim3 grid((unsigned)((size_t)tiles * blocks), (unsigned)n_in);
    const unsigned cgrid = (unsigned)(((size_t)n_in * blocks * 32 + 255) / 256);
    with_format(f.fmt, [&](auto fmt) {
        // exact int64 sums of the integer elements, float64 sums of cf32 values
        using S = typename std::conditional<decltype(fmt)::value == RT_SAMPLE_CF32, double, long long>::type;
        S* part = static_cast<S*>(s.part);
        iq_moments_kernel<decltype(fmt)::value><<<grid, IQ_THREADS, 0, st>>>(src, stride, block, blocks, tiles, part);
        iq_coef_kernel<<<cgrid, 256, 0, st>>>((const S*)part, n_in, blocks, tiles, block, scale, offset, s.coef);
    });
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    args->coef = s.coef;
    args->block = block;
    args->n_blocks = blocks;
    iq_division_magic(block, &args->magic, &args->shift);
    s.applied = true;
    s.blocks = blocks;
    return cudaSuccess;
}

}  // namespace

FirFrontEnd::~FirFrontEnd() {
    if (dev < 0) return;
    cudaSetDevice(dev);
    if (done) {
        cudaEventSynchronize(done);
        cudaEventDestroy(done);
    }
    for (void* t : tables) cudaFree(t);
    cudaFree(d_off);
    cudaFree(d_hist[0]);
    cudaFree(d_hist[1]);
    cudaFree(d_stage);
    cudaFree(iq.coef);
    cudaFree(iq.part);
}

int fir_check(const FirPlan& p, int max_taps, const char* max_taps_text) {
    if (p.n_in < 1 || p.n_in > 65535) return fail(RT_ERR_INVALID, "n_inputs must be in [1, 65535]");
    if (p.L < 1 || p.L > max_taps || p.L % 2 == 0)
        return fail(RT_ERR_INVALID, std::string("n_taps must be odd and in [1, ") + max_taps_text + "]");
    if (p.block < p.D || p.block % p.D != 0) return fail(RT_ERR_INVALID, "block_samples must be a positive multiple of decimation");
    SampleFormatInfo info;
    if (!sample_format_info(p.fmt, &info)) return fail(RT_ERR_INVALID, "unknown sample_format");
    if (!p.taps) return fail(RT_ERR_INVALID, "taps missing");
    for (int k = 0; k < p.L; ++k)
        if (!std::isfinite(p.taps[k])) return fail(RT_ERR_INVALID, "taps must be finite");
    return RT_OK;
}

int fir_open(FirFrontEnd* f, const FirPlan& p, int mt, size_t smem, std::pair<const void*, const void*> kernels,
             std::initializer_list<HostTable> tables) {
    if (smem > FIR_SMEM_MAX) return fail(RT_ERR_INVALID, "decimation and n_taps need more shared memory than a CTA has");
    int ndev = 0;
    CU(cudaGetDeviceCount(&ndev));
    if (p.dev < 0 || p.dev >= ndev) return fail(RT_ERR_CUDA, "no such CUDA device (this engine has no CPU fallback)");
    CU(cudaSetDevice(p.dev));
    {
        static std::mutex mu;
        std::lock_guard<std::mutex> lock(mu);
        int rc = raise_smem_limit(kernels.first, smem);
        if (rc == RT_OK) rc = raise_smem_limit(kernels.second, smem);
        if (rc != RT_OK) return rc;
    }

    f->dev = p.dev;
    f->fmt = p.fmt;
    f->n_in = p.n_in;
    f->nch = p.nch;
    f->D = p.D;
    f->L = p.L;
    f->block = p.block;
    sample_format_info(p.fmt, &f->info);
    f->mt = mt;
    f->smem = smem;
    const size_t hist_bytes = (size_t)f->n_in * std::max(1, f->L - 1) * sizeof(float2);
    for (const HostTable& t : tables) {
        void* d = nullptr;
        CU(cudaMalloc(&d, t.bytes));
        f->tables.push_back(d);
    }
    CU(cudaMalloc(&f->d_off, f->n_in * sizeof(uint32_t)));
    CU(cudaMalloc(&f->d_hist[0], hist_bytes));
    CU(cudaMalloc(&f->d_hist[1], hist_bytes));
    size_t i = 0;
    for (const HostTable& t : tables) CU(cudaMemcpy(f->tables[i++], t.data, t.bytes, cudaMemcpyHostToDevice));
    CU(cudaMemset(f->d_off, 0, f->n_in * sizeof(uint32_t)));
    CU(cudaMemset(f->d_hist[0], 0, hist_bytes));
    CU(cudaEventCreateWithFlags(&f->done, cudaEventDisableTiming));
    return RT_OK;
}

int fir_reset_input(FirFrontEnd* f, int input, int64_t first_sample) {
    if (!f || input < 0 || input >= f->n_in) return fail(RT_ERR_INVALID, "bad input index");
    f->resets.emplace_back(input, (uint32_t)(uint64_t)first_sample);
    return RT_OK;
}

int fir_set_iq_correction(FirFrontEnd* f, int enable) {
    if (!f) return fail(RT_ERR_INVALID, "null handle");
    if (enable && f->block > IQ_MAX_BLOCK) return fail(RT_ERR_INVALID, "block_samples must be <= 2^30 for the IQ correction");
    f->iq.on = enable != 0;
    return RT_OK;
}

// m and w of (input, block) of the last run, after it has finished: out = {m.re, m.im, w.re, w.im}
int fir_read_iq_correction(FirFrontEnd* f, int input, int block, float out[4]) {
    if (!f || !out) return fail(RT_ERR_INVALID, "null argument");
    if (!f->iq.applied) return fail(RT_ERR_INVALID, "the last run did not apply the IQ correction");
    if (input < 0 || input >= f->n_in || block < 0 || block >= f->iq.blocks) return fail(RT_ERR_INVALID, "bad input / block index");
    CU(cudaSetDevice(f->dev));
    CU(cudaEventSynchronize(f->done));
    float4 v;
    CU(cudaMemcpy(&v, f->iq.coef + (size_t)input * f->iq.blocks + block, sizeof(v), cudaMemcpyDeviceToHost));
    out[0] = v.x;
    out[1] = v.y;
    out[2] = v.z;
    out[3] = v.w;
    return RT_OK;
}

int fir_run_begin(FirFrontEnd* f, void* cuda_stream, const void* iq, int iq_on_device, size_t in_stride_bytes, int blocks,
                  void* out, size_t out_stride_bytes, FirRun* r) {
    if (!f || !iq || !out) return fail(RT_ERR_INVALID, "null argument");
    if (blocks < 1) return fail(RT_ERR_INVALID, "blocks must be >= 1");
    const long long n = f->block * blocks;
    const long long m_total = n / f->D;
    const size_t row_bytes = (size_t)f->info.bytes * (size_t)n;
    if (f->n_in > 1 && in_stride_bytes < row_bytes) return fail(RT_ERR_INVALID, "in_stride_bytes smaller than one input's blocks");
    if (out_stride_bytes < (size_t)m_total * sizeof(float2) && (long long)f->n_in * f->nch > 1)
        return fail(RT_ERR_INVALID, "out_stride_bytes smaller than one channel's outputs");
    if (((uintptr_t)out | out_stride_bytes) % sizeof(float2) != 0) return fail(RT_ERR_INVALID, "output pointer / stride not aligned to 8 bytes");
    if ((m_total + f->mt - 1) / f->mt > 0x7fffffffLL) return fail(RT_ERR_INVALID, "call too long");
    CU(cudaSetDevice(f->dev));
    cudaStream_t st = (cudaStream_t)cuda_stream;
    if (f->ran) CU(cudaStreamWaitEvent(st, f->done, 0));      // history, offsets and the staging buffer of the previous run

    const unsigned char* src = static_cast<const unsigned char*>(iq);
    size_t stride = f->n_in > 1 ? in_stride_bytes : row_bytes;
    if (!iq_on_device) {
        CU(stage_host_input(st, &src, &stride, row_bytes, f->n_in, &f->d_stage, &f->stage_bytes));
    } else if (((uintptr_t)src | (f->n_in > 1 ? stride : 0)) % (uintptr_t)f->info.bytes != 0) {
        return fail(RT_ERR_INVALID, "IQ pointer / input stride not aligned to one complex sample");
    }

    CU(iq_prepare(*f, st, src, stride, blocks, &r->corr));
    for (const auto& rs : f->resets)
        fir_reset_kernel<<<1, 256, 0, st>>>(f->d_hist[f->cur], f->d_off, rs.first, f->L - 1, rs.second - f->advance);
    r->st = st;
    r->src = src;
    r->stride = stride;
    r->n = n;
    r->m_total = m_total;
    r->out = out;
    r->out_stride = out_stride_bytes;
    return RT_OK;
}

int fir_run_end(FirFrontEnd* f, const FirRun& r) {
    CU(cudaGetLastError());
    CU(cudaEventRecord(f->done, r.st));
    f->ran = true;
    f->resets.clear();
    f->cur ^= f->L > 1 ? 1 : 0;
    f->advance += (uint32_t)(uint64_t)r.n;
    return RT_OK;
}

}  // namespace rt
