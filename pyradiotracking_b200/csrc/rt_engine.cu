// rt_engine.cu -- B200 (sm_100a) detection engine behind include/rt_engine.h.
//
// Path replaced: the inside of SignalAnalyzer.process_samples
// (/root/reference/radiotracking/analyze.py:234-245): scipy.signal.spectrogram
// (noverlap=0, two-sided, detrend='constant', density scaling) followed by
// extract_signals' probe / backward / forward scans and per-signal statistics.
//
// Kernels (one launch each per engine call, all streams of the batch at once):
//   spectro_*      IQ samples (rt_config.sample_format) -> power cells S (fp32, layout per kernel) + row sums / row means
//   probe          prologue: deterministic reduction of the chunk sums -> freq_avg[stream][bin] (the tensor-core
//                  kernel does this itself in the last warp-group run of each stream); then one thread per
//                  (stream, bin, 8 probe columns k*stride): predicate test, cheap pruning of short noise runs,
//                  survivors -> work list
//   extract        one warp per work item: run limits by ballot, carry into the
//                  previous block, coarse duration gate, statistics, record emission
//
// No CPU fallback and no library FFT: if this file is not built for the device present,
// rt_engine_create fails.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/rt_engine.h"
#include "predicate.h"
#include "sample_format.cuh"
#include "spectro256.cuh"
#include "spectro_tc256.cuh"
#include "spectro_r16.cuh"

namespace {

thread_local std::string g_err;
constexpr int RT_SLOTS = 2;     // launches that may be in flight before rt_engine_fetch
constexpr int RT_SBUFS = 3;     // spectrogram buffers (block being written, block being scanned, its carry)

int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess)                                                                     \
            return fail(RT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e));          \
    } while (0)

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------

// analyze.py:370-379: a cell is part of a run unless it undershoots either threshold (predicate.h)
using rt::Pred;
__device__ __forceinline__ bool above(float p, float thr, float avg, float snr) { return rt::above_exact(p, thr, avg, snr); }

// Spectrogram layouts.
//   LINEAR (generic kernel)        S[stream][t][bin]
//   PERM   (register kernel v7)    S[stream][t / TG][pos(bin) / 4][t % TG][pos % 4], pos = 64 (k2 >> 2) + 4 k1 + (k2 & 3) for bin = k1 + 16 k2:
//                                  thread k1 of a half-warp stores its bins as four float4; with TG = 2 the half-warps of a warp (time
//                                  steps t, t + 1) fill 512 contiguous bytes per store instruction and a walk along time finds two
//                                  cells per 32-byte sector
//   TILE   (tensor-core kernel)    S[stream][t / 32][quad][t % 32][4], quad = 4 k1 + (k2 >> 2) (rt::tile_cell_off): a thread owns a
//                                  segment, a warp stores 512 contiguous bytes, 32 time steps of a bin lie within 512 bytes
// (time-blocked variants of PERM were measured and rejected: DESIGN.md 5.7)
enum { LAYOUT_LINEAR = 0, LAYOUT_PERM = 1, LAYOUT_TILE = 2 };
// PERM time group (spectro256.cuh, TG): S[stream][t / TG][pos / 4][t % TG][pos % 4]; pairs of time steps (DESIGN.md 11.6)
constexpr int PERM_TG = 2;
// with time pairs the register kernel maps a segment's 16 threads onto the lanes {0-3, 8-11, ...} (spectro256.cuh, LMAP): every quarter-warp
// phase of its 128-bit stores then covers one whole 128-byte line; back to back 173.9 -> 169.7 us (one time step per row: 170.8 us)
using R256Prod = rt::R256v7T<4, 4, true>;
__host__ __device__ __forceinline__ constexpr int perm256(int k) { return ((k >> 6) << 6) | ((k & 15) << 2) | ((k >> 4) & 3); }                // bin -> position
__host__ __device__ constexpr int unperm256(int p) { return ((p >> 2) & 15) + 16 * (4 * (p >> 6) + (p & 3)); }                 // position -> bin
// row position -> FFT bin for the layouts whose rows are not in bin order
template <int L>
__device__ __forceinline__ int pos_to_bin(int idx) {
    return L == LAYOUT_PERM ? unperm256(idx) : idx;
}

struct CellRef {
    const float* base;     // stream base + the bin's constant part
    int step;              // LINEAR: floats per time step
    template <int L>
    __device__ __forceinline__ static CellRef make(const float* S, size_t stream_stride, int s, int fi, int n) {
        CellRef c;
        if (L == LAYOUT_TILE) { c.base = S + (size_t)s * stream_stride + (size_t)((fi & 15) * 4 + (fi >> 6)) * 128 + ((fi >> 4) & 3); c.step = 0; }
        else if (L == LAYOUT_PERM) {
            const int pos = perm256(fi);
            c.base = S + (size_t)s * stream_stride + (pos >> 2) * (4 * PERM_TG) + (pos & 3);
            c.step = 256;
        }
        else { c.base = S + (size_t)s * stream_stride + fi; c.step = n; }
        return c;
    }
    template <int L>
    __device__ __forceinline__ const float* ptr(int t) const {
        return L == LAYOUT_TILE ? base + ((size_t)(t >> 5) * 8192 + (size_t)(t & 31) * 4)
             : L == LAYOUT_PERM ? base + ((size_t)(t / PERM_TG) * (256 * PERM_TG) + (size_t)(t % PERM_TG) * 4)
                                : base + (size_t)t * step;
    }
    template <int L>
    __device__ __forceinline__ float at(int t) const { return *ptr<L>(t); }
};

// ---------------------------------------------------------------------------------------------
// spectrogram, generic: any power-of-two nperseg in [8, 4096]; Stockham radix-4 in shared memory
// ---------------------------------------------------------------------------------------------
using rt::SpectroArgs;

template <int NT, int FMT>
__global__ void __launch_bounds__(NT) spectro_generic(SpectroArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int n = a.n;
    float2* buf0 = reinterpret_cast<float2*>(smem_raw);
    float2* buf1 = buf0 + n;
    float* rowacc = reinterpret_cast<float*>(buf1 + n);
    int* sums = reinterpret_cast<int*>(rowacc + n);

    const int tid = threadIdx.x;
    const int s = blockIdx.y;
    const int seg0 = blockIdx.x * a.chunk_segs;
    const int seg1 = min(a.T, seg0 + a.chunk_segs);
    for (int i = tid; i < n; i += NT) rowacc[i] = 0.f;

    for (int seg = seg0; seg < seg1; ++seg) {
        // scipy detrend='constant' (the segment's complex mean) and the window, per sample format (sample_format.cuh); buf1 is
        // free until the first FFT pass
        using In = rt::SegmentIn<FMT>;
        In::template centre<NT>(a.unit_base(s) + (size_t)seg * In::BYTES * n, n, tid, a.win, buf0, sums, buf1);
        __syncthreads();
        float2* X = buf0;
        float2* Y = buf1;
        int st = 1, lst = 0, ncur = n;
        // radix-4 Stockham passes (decimation in frequency, self-sorting)
        for (; ncur >= 4; ncur >>= 2, st <<= 2, lst += 2) {
            const int m = ncur >> 2;
            for (int b = tid; b < (n >> 2); b += NT) {
                const int p = b >> lst, q = b & (st - 1);
                const float2 w1 = a.tw[p << lst], w2 = a.tw[(2 * p) << lst], w3 = a.tw[(3 * p) << lst];
                const float2 x0 = X[q + st * p], x1 = X[q + st * (p + m)];
                const float2 x2 = X[q + st * (p + 2 * m)], x3 = X[q + st * (p + 3 * m)];
                const float apr = x0.x + x2.x, api = x0.y + x2.y, amr = x0.x - x2.x, ami = x0.y - x2.y;
                const float bpr = x1.x + x3.x, bpi = x1.y + x3.y;
                const float jr = -(x1.y - x3.y), ji = x1.x - x3.x;          // j * (x1 - x3)
                float2* y = Y + q + st * 4 * p;
                y[0] = make_float2(apr + bpr, api + bpi);
                float tr = amr - jr, ti = ami - ji;
                y[st] = make_float2(tr * w1.x - ti * w1.y, tr * w1.y + ti * w1.x);
                tr = apr - bpr; ti = api - bpi;
                y[2 * st] = make_float2(tr * w2.x - ti * w2.y, tr * w2.y + ti * w2.x);
                tr = amr + jr; ti = ami + ji;
                y[3 * st] = make_float2(tr * w3.x - ti * w3.y, tr * w3.y + ti * w3.x);
            }
            __syncthreads();
            float2* t = X;
            X = Y;
            Y = t;
        }
        if (ncur == 2) {    // odd log2(n): one final radix-2 pass (twiddle-free)
            for (int q = tid; q < st; q += NT) {
                const float2 u = X[q], v = X[q + st];
                Y[q] = make_float2(u.x + v.x, u.y + v.y);
                Y[q + st] = make_float2(u.x - v.x, u.y - v.y);
            }
            __syncthreads();
            float2* t = X;
            X = Y;
            Y = t;
        }
        float* dst = a.S + ((size_t)s * a.T + seg) * n;
        for (int i = tid; i < n; i += NT) {
            const float2 x = X[i];
            const float p = x.x * x.x + x.y * x.y;
            dst[i] = p;
            rowacc[i] += p;
        }
        __syncthreads();
    }
    float* pd = a.part + ((size_t)s * a.n_chunks + blockIdx.x) * n;
    for (int i = tid; i < n; i += NT) pd[i] = rowacc[i];
}

// the generic kernel's instantiation for a sample format (RT_SAMPLE_*, validated by rt_engine_create)
using SpectroKernel = void (*)(SpectroArgs);
SpectroKernel generic_kernel(int fmt) {
    switch (fmt) {
        case RT_SAMPLE_CI8: return spectro_generic<256, RT_SAMPLE_CI8>;
        case RT_SAMPLE_CI16: return spectro_generic<256, RT_SAMPLE_CI16>;
        case RT_SAMPLE_CF32: return spectro_generic<256, RT_SAMPLE_CF32>;
        default: return spectro_generic<256, RT_SAMPLE_CU8>;
    }
}

// ---------------------------------------------------------------------------------------------
// row means (analyze.py:374-375), deterministic
// ---------------------------------------------------------------------------------------------
// fixed summation order (4 interleaved partial sums over the chunks), float64: run-to-run identical and
// identical in every CTA that evaluates it
__device__ __forceinline__ float row_mean_of(const float* part, int s, int fi, int n, int n_chunks, int T) {
    const float* p = part + (size_t)s * n_chunks * n + fi;
    double t[4] = {0.0, 0.0, 0.0, 0.0};
    if (n_chunks <= 48) {                                // the usual case: every chunk sum in flight at once (one round trip)
        float v[48];
#pragma unroll
        for (int i = 0; i < 48; ++i) v[i] = (i < n_chunks) ? p[(size_t)i * n] : 0.f;
#pragma unroll
        for (int i = 0; i < 48; ++i) t[i & 3] += (double)v[i];     // + 0.0 beyond n_chunks: same value as the loop below
    } else {
        for (int c0 = 0; c0 < n_chunks; c0 += 16) {      // 16 chunk sums per memory round trip
            float v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = (c0 + i < n_chunks) ? p[(size_t)(c0 + i) * n] : 0.f;
#pragma unroll
            for (int i = 0; i < 16; ++i) t[i & 3] += (double)v[i];
        }
    }
    return (float)(((t[0] + t[1]) + (t[2] + t[3])) / (double)T);
}

// stand-alone row means for kernels that leave many partial rows per stream (spectro_r16: one per CTA) and for the lean scan
// schedule.  Four threads per bin: thread k owns the partial sum t[k] of row_mean_of (chunks k, k + 4, ...: the same values in
// the same order), so the result is bit-identical to the one-thread version while the dependent round trips drop fourfold.
__global__ void __launch_bounds__(128, 16) row_mean_kernel(const float* part, float* avg, int n, int n_chunks, int T, int part_perm) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int fi = g >> 2, k = g & 3;
    const bool active = fi < n;
    // part_perm: the register kernel writes its chunk sums in PERM position order (n == 256)
    const int src = part_perm ? perm256(fi) : fi;
    const float* p = part + (size_t)blockIdx.y * n_chunks * n + (active ? src : 0);
    double t = 0.0;
    for (int c0 = k; c0 < n_chunks; c0 += 32) {          // 8 of this thread's chunk sums per memory round trip
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = (c0 + 4 * i < n_chunks) ? p[(size_t)(c0 + 4 * i) * n] : 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) t += (double)v[i];
    }
    const double t1 = __shfl_xor_sync(0xffffffffu, t, 1);            // k even: t[k] + t[k + 1]
    const double pair = (k & 1) ? t1 + t : t + t1;                   // always (t[even] + t[odd])
    const double other = __shfl_xor_sync(0xffffffffu, pair, 2);
    const double tot = (k & 2) ? other + pair : pair + other;        // (t0 + t1) + (t2 + t3)
    if (active && k == 0) avg[blockIdx.y * n + fi] = (float)(tot / (double)T);
}

// ---------------------------------------------------------------------------------------------
// probe + extraction (analyze.py:354-447)
// ---------------------------------------------------------------------------------------------
struct ScanArgs {
    const float* S;        // current block (LINEAR or TILE layout)
    const float* Sprev;    // previous block
    size_t stream_stride;  // floats per stream
    float* avg;            // [stream][n] row means: written by the probe kernel (from `part`) or by the tensor-core kernel
    const float* part;     // [stream][n_chunks][n] chunk row sums (nullptr: avg is already there)
    int part_perm;         // the chunk sums are stored in PERM position order (register kernel)
    int n_chunks;
    const float* thr;      // [stream]
    const int* has_prev;   // [stream]
    int bpl;               // blocks per launch: the carry of unit s is unit s - 1 of the same buffer unless s % bpl == 0
    float snr;
    int n, T, stride, n_probes, min_cols, max_cols;
    int n_streams_scan;    // streams of the batch (lean probe kernel: tiles are walked with a grid stride)
    uint4* work;           // (stream << 16 | fi, ti | (chain members - 1) << 24, row mean, threshold): consecutive probe columns ti, ti + stride, ...;
                           // the two floats save the extraction warp two dependent round trips in front of its first cells
    int max_work;          // capacity of the work list (worst case: every probe column of every bin)
    int widen;             // extraction: widen the forward walk after three round trips (small launches)
    int* counters;         // [0] work items, [1] records
    rt_record* rec;
    int max_records;
};

constexpr int PROBE_QUICK = 3;   // cells examined on each side before handing a probe hit to a warp
constexpr int PROBE_CHAIN = 8;   // consecutive surviving probe hits of a bin handed to ONE extraction warp (bounds its serial work)
constexpr int PROBE_PPT = 32;    // probe columns per thread: their loads are in flight together, and the row-mean prologue
                                 // is repeated once per PROBE_PPT columns (8 -> 32: 5x fewer instructions, 29 -> see DESIGN 5.4)

constexpr int PROBE_LIST = 2048; // probe hits a CTA resolves in parallel (more than that: resolved by the finding thread itself)

// One thread per (stream, bin, group of PPT probe columns); blockDim.x bins of one stream per CTA.
// Prologue: the bin's row mean from the chunk sums (analyze.py:374-375) -- every CTA of the stream computes the
// same value, the CTAs of probe group 0 publish it for the extraction kernel and the parity hook.
// Three phases, each ONE memory round trip: (1) chunk sums + probe cells of every thread, (2) the CTA's hits are pooled in
// shared memory and resolved one per thread (the neighbours of a hit), (3) every thread chains its surviving hits.
template <int TILE, int PPT>
__global__ void probe_kernel(ScanArgs a) {
    static_assert(PPT >= 1 && PPT <= 32, "hit mask is one word");
    __shared__ float s_avg[1024];
    __shared__ unsigned s_live[1024];
    __shared__ unsigned s_list[PROBE_LIST];
    __shared__ int s_n;
    const int tid = threadIdx.x;
    const int nbb = (a.n + blockDim.x - 1) / blockDim.x;           // bin blocks
    const int bb = blockIdx.x % nbb, g = blockIdx.x / nbb;
    const int idx = bb * blockDim.x + tid;
    const int s = blockIdx.y;
    const bool active = idx < a.n;
    // PERM layout: the thread index is the position inside the S row (and inside the chunk-sum rows, which the register
    // kernel writes in the same order), so a warp reads 128 contiguous bytes per load instead of 2 floats out of each of
    // 8 sectors; position 64 a + 4 k1 + b holds bin k1 + 16 (4 a + b)
    const int fi = pos_to_bin<TILE>(idx);
    const float thr = a.thr[s], snr = a.snr;
    if (tid == 0) s_n = 0;
    s_live[tid] = 0;
    float avg = 1.f;
    unsigned hits = 0;
    if (active) {
        // ~96 % of the probe cells fail the predicate: only a hit pays for its neighbours
        float c0[PPT];
        {
            const CellRef col = CellRef::make<TILE>(a.S, a.stream_stride, s, fi, a.n);
#pragma unroll
            for (int i = 0; i < PPT; ++i) {
                const int k = g * PPT + i;
                c0[i] = (k < a.n_probes) ? col.at<TILE>(k * a.stride) : -1.f;      // -1: no such probe column (never above)
            }
        }
        if (a.part != nullptr) {
            avg = row_mean_of(a.part, s, a.part_perm ? idx : fi, a.n, a.n_chunks, a.T);
            if (g == 0) a.avg[s * a.n + fi] = avg;
        } else {
            avg = a.avg[s * a.n + fi];
        }
#pragma unroll
        for (int i = 0; i < PPT; ++i) hits |= (c0[i] >= 0.f && above(c0[i], thr, avg, snr)) ? (1u << i) : 0u;
    }
    s_avg[tid] = avg;
    __syncthreads();

    // Most hits are 1-2 cell noise runs that the duration gate rejects anyway: resolve those here.  true = hand it to a warp
    auto resolve = [&](int fi_, float avg_, int i) -> bool {
        const CellRef col = CellRef::make<TILE>(a.S, a.stream_stride, s, fi_, a.n);
        const int ti = (g * PPT + i) * a.stride;
        float lo_c[PROBE_QUICK], hi_c[PROBE_QUICK];
#pragma unroll
        for (int d = 1; d <= PROBE_QUICK; ++d) {
            lo_c[d - 1] = (ti - d >= 0) ? col.at<TILE>(ti - d) : 0.f;
            hi_c[d - 1] = (ti + d < a.T) ? col.at<TILE>(ti + d) : 0.f;
        }
        int lo = -1, hi = -1;             // nearest not-above cells, if found within PROBE_QUICK
#pragma unroll
        for (int d = 1; d <= PROBE_QUICK; ++d) {
            const int t = ti - d;
            if (t < 0) break;             // run reaches column 0: carry logic, leave it to the warp
            if (!above(lo_c[d - 1], thr, avg_, snr)) { lo = t; break; }
        }
#pragma unroll
        for (int d = 1; d <= PROBE_QUICK; ++d) {
            const int t = ti + d;
            if (t >= a.T) return false;   // run touches the block end: dropped (analyze.py:415-417)
            if (!above(hi_c[d - 1], thr, avg_, snr)) { hi = t; break; }
        }
        return !(lo >= 0 && hi >= 0 && hi - lo < a.min_cols);      // window = [lo, hi): too short
    };

    unsigned live = 0;
    while (hits) {
        const int i = __ffs(hits) - 1;
        hits &= hits - 1;
        const int slot = atomicAdd(&s_n, 1);
        if (slot < PROBE_LIST) s_list[slot] = ((unsigned)tid << 5) | (unsigned)i;
        else if (resolve(fi, avg, i)) live |= 1u << i;
    }
    __syncthreads();
    const int n_list = min(s_n, PROBE_LIST);
    for (int e = tid; e < n_list; e += blockDim.x) {
        const unsigned ent = s_list[e];
        const int o = (int)(ent >> 5), i = (int)(ent & 31u);
        if (resolve(pos_to_bin<TILE>(bb * blockDim.x + o), s_avg[o], i)) atomicOr(&s_live[o], 1u << i);
    }
    __syncthreads();
    live |= s_live[tid];
    // Surviving hits at consecutive probe columns almost always lie in the same run (a pulse of 75-375 columns spans
    // 1-5 probes at config 2): they form one work item (head column + length, at most PROBE_CHAIN members), and the
    // extraction warp walks the members the way the reference's probe loop does (ti_skip, analyze.py:366).
    while (live) {
        const int head = __ffs(live) - 1;
        int len = 1;
        while (head + len < 32 && ((head + len) % PROBE_CHAIN) != 0 && ((live >> (head + len)) & 1u)) ++len;
        live &= ~(((1u << len) - 1u) << head);
        const int slot = atomicAdd(&a.counters[0], 1);
        a.work[slot] = make_uint4(((unsigned)s << 16) | (unsigned)fi, (unsigned)((g * PPT + head) * a.stride) | ((unsigned)(len - 1) << 24), __float_as_uint(avg), __float_as_uint(thr));
    }
}

// Lean variant for the two-stream schedule.  The register kernel keeps 4 CTAs x 128 threads x 120 registers resident per SM,
// which leaves exactly 4096 registers: a 128-thread CTA capped at 32 registers runs BESIDE them instead of waiting for (and
// then displacing) a spectrogram CTA.  One such CTA per SM walks the (stream, probe group, position block) tiles with a grid
// stride; 8 probe columns per thread and tile, hits resolved by the finding thread; row means come from row_mean_kernel.
constexpr int LEAN_PPT = 8;
static_assert(LEAN_PPT == PROBE_CHAIN, "a chain must not leave its tile");
template <int TILE>
__global__ void __launch_bounds__(128, 16) probe_lean_kernel(ScanArgs a) {
    const int lane = threadIdx.x & 31;
    const int warp = blockIdx.x * 4 + (threadIdx.x >> 5), n_warps = gridDim.x * 4;
    const int npb = (a.n + 31) / 32, ngr = (a.n_probes + LEAN_PPT - 1) / LEAN_PPT;
    const int n_tiles = npb * ngr * a.n_streams_scan;
    const float snr = a.snr;
    // a tile = 32 row positions x 8 probe columns of one stream; the warps walk the tiles independently (no CTA barrier)
    for (int tile = warp; tile < n_tiles; tile += n_warps) {
        const int pb = tile % npb, g = (tile / npb) % ngr, s = tile / (npb * ngr);
        const int idx = pb * 32 + lane;
        if (idx >= a.n) continue;
        const int fi = pos_to_bin<TILE>(idx);
        const CellRef col = CellRef::make<TILE>(a.S, a.stream_stride, s, fi, a.n);
        float c0[LEAN_PPT];
#pragma unroll
        for (int i = 0; i < LEAN_PPT; ++i) {
            const int k = g * LEAN_PPT + i;
            c0[i] = (k < a.n_probes) ? col.at<TILE>(k * a.stride) : -1.f;
        }
        const float thr = a.thr[s], avg = a.avg[s * a.n + fi];
        const Pred pred(thr, avg, snr);
        unsigned hits = 0;
#pragma unroll
        for (int i = 0; i < LEAN_PPT; ++i) hits |= (c0[i] >= 0.f && pred(c0[i])) ? (1u << i) : 0u;
        int head = -1, len = 0;              // open chain (LEAN_PPT == PROBE_CHAIN: a chain never leaves the tile)
        auto flush = [&]() {
            if (len > 0) {
                const int slot = atomicAdd(&a.counters[0], 1);
                a.work[slot] = make_uint4(((unsigned)s << 16) | (unsigned)fi, (unsigned)((g * LEAN_PPT + head) * a.stride) | ((unsigned)(len - 1) << 24), __float_as_uint(avg), __float_as_uint(thr));
            }
            len = 0;
        };
        while (hits) {
            const int i = __ffs(hits) - 1;
            hits &= hits - 1;
            const int ti = (g * LEAN_PPT + i) * a.stride;
            // neighbours by increasing distance, one round trip per distance and only on a side that is still open: ~92 % of the
            // hits are single noise cells and are settled by the first pair (2 sectors instead of 6; this kernel runs beside
            // the spectrogram, where DRAM sectors cost more than latency)
            bool keep = true;
            int lo = -1, hi = -1;
            bool lo_open = true, hi_open = true;
#pragma unroll 1
            for (int d = 1; d <= PROBE_QUICK && (lo_open || hi_open); ++d) {
                const int tl = ti - d, th = ti + d;
                if (lo_open && tl < 0) lo_open = false;                    // run reaches column 0: carry logic, leave it to the warp
                if (hi_open && th >= a.T) { keep = false; break; }         // run touches the block end: dropped (analyze.py:415-417)
                const float pl = lo_open ? col.at<TILE>(tl) : 0.f;
                const float ph = hi_open ? col.at<TILE>(th) : 0.f;
                if (lo_open && !pred(pl)) { lo = tl; lo_open = false; }
                if (hi_open && !pred(ph)) { hi = th; hi_open = false; }
            }
            if (keep && lo >= 0 && hi >= 0 && hi - lo < a.min_cols) keep = false;
            if (keep && len > 0 && i == head + len) { ++len; continue; }
            flush();
            if (keep) { head = i; len = 1; }
        }
        flush();
    }
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// extract2_kernel: one warp per work item (the round-1 extract_kernel at about half its memory sectors and round trips).  Measured
// (DESIGN.md 11.6, configs[1]): beside the spectrogram of the next launch the extraction alone costs the step 23 of its 30 us
// of scan overhead, and that cost follows the number of scattered 32-byte sectors it reads (a first version with wide
// speculative fetches -- 4 round trips per run instead of 11, the same ~340 sectors -- was 4 us SLOWER).
//   * cells travel in ALIGNED blocks of 32 columns (lane = column & 31), the probe's own block first, then one block down
//     and one block up per round trip for as long as that side of the run is still open: nothing is fetched speculatively;
//   * max / sum / sum dB / sum dB^2 are accumulated while the blocks pass through the registers -- no second pass over the
//     run, which was 150 of the ~340 sectors of a typical 150-column pulse;
//   * one fixed per-lane order of the float64 sums, so every schedule returns the same bits.
template <int TILE, int MINB, int WF = 1>
__global__ void __launch_bounds__(128, MINB) extract2_kernel(ScanArgs a) {
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int n_warps = (gridDim.x * blockDim.x) >> 5;
    // the first work item is fetched together with the item count (the list is allocated for the worst case, a stale entry is
    // harmless): one round trip in front of the first cells instead of three (count -> item -> row mean / threshold)
    uint4 wk = a.work[min(warp, a.max_work - 1)];
    const int n_work = a.counters[0];
    const int T = a.T, n = a.n;

    for (int item = warp; item < n_work; item += n_warps) {
        if (item != warp) wk = a.work[item];
        const int s = wk.x >> 16, fi = wk.x & 0xffff, ti0 = (int)(wk.y & 0xffffffu), members = (int)(wk.y >> 24) + 1;
        const CellRef col = CellRef::make<TILE>(a.S, a.stream_stride, s, fi, n);
        const float thr = __uint_as_float(wk.w), avg = __uint_as_float(wk.z), snr = a.snr;
        const Pred pred(thr, avg, snr);
        const int span_cap = a.max_cols + 2;             // a run longer than this fails the duration test anyway
        int skip_to = 0;                                 // every cell in [previous member's probe, skip_to) is known to be above
      for (int mem = 0; mem < members; ++mem) {
        const int ti = ti0 + mem * a.stride;
        if (ti < skip_to) continue;                      // inside the run the previous member evaluated (ti_skip, analyze.py:366)
        const int lo_lim = max(ti - a.stride, 0);        // the backward scan stops at the previous probe column (analyze.py:366)
        const int bh = ti >> 5, tl = ti & 31;

        // statistics over data = [start, end) (analyze.py:436-447), accumulated as the cells arrive
        float mx = 0.f;
        double sum = 0.0, sdb = 0.0, sdb2 = 0.0;
        auto acc = [&](float p) {
            mx = fmaxf(mx, p);
            sum += (double)p;
            // dB of one cell in float (MUFU.LG2: ~1e-6 dB absolute error, the record tolerance is 5e-4 dB); the sums stay float64
            const double db = (double)(3.0102999566398120f * __log2f(p));
            sdb += db;
            sdb2 += db * db;
        };

        int nb = -1, end = -1;                           // nearest not-above cell below / above the probe column
        {                                                // the probe's own block serves both directions
            const int t = 32 * bh + lane;
            const bool valid = t >= lo_lim && t < T;
            const float p = valid ? col.at<TILE>(t) : 0.f;
            const unsigned m = __ballot_sync(0xffffffffu, valid && !pred(p));
            const unsigned mb = m & ((1u << tl) - 1u), mf = m & ~((2u << tl) - 1u);      // tl == 31: no lane above
            if (mb) nb = 32 * bh + 31 - __clz(mb);
            if (mf) end = 32 * bh + __ffs(mf) - 1;
            if (valid && t >= nb && (end < 0 || t < end)) acc(p);
        }
        int kb = bh - 1, kf = bh + 1;                    // next block down / up
        bool bopen = nb < 0 && 32 * bh > lo_lim;
        bool fopen = end < 0 && 32 * kf < T;
        bool too_long = false;
        // forward blocks per round trip: 1, 1, 1, then (WF = 4 and a.widen: small launches, where the chain of round trips IS the kernel
        // time and the sectors cost nothing) 2, 2, 4, 4, ... -- a 25-block pulse of a 20 MS/s stream takes 9 round trips instead of 25.
        // The lean instantiation (WF = 1) keeps one block per direction: beside the spectrogram every sector counts and 32 registers
        // have no room for more loads in flight.
        int rounds = 0;
        while (bopen || fopen) {
            if (fopen && 32 * kf - (nb >= 0 ? nb : 32 * (kb + 1)) > span_cap) { too_long = true; skip_to = 32 * kf; break; }
            const int wf = WF == 1 || !a.widen || rounds < 3 ? 1 : (rounds < 5 ? 2 : 4);
            ++rounds;
            const int tb = 32 * kb + lane;
            const bool vb = bopen && tb >= lo_lim;
            const float pb = vb ? col.at<TILE>(tb) : 0.f;                    // every load of a round is in flight together
            float pf[WF];
#pragma unroll
            for (int w = 0; w < WF; ++w) {
                const int tf = 32 * (kf + w) + lane;
                pf[w] = (fopen && w < wf && tf < T) ? col.at<TILE>(tf) : -1.f;
            }
            if (bopen) {
                const unsigned m = __ballot_sync(0xffffffffu, vb && !pred(pb));
                if (m) nb = 32 * kb + 31 - __clz(m);
                if (vb && tb >= nb) acc(pb);
                bopen = nb < 0 && 32 * kb > lo_lim;
                --kb;
            }
            if (fopen) {
#pragma unroll
                for (int w = 0; w < WF; ++w) {
                    if (w < wf && end < 0) {
                        const int tf = 32 * (kf + w) + lane;
                        const unsigned m = __ballot_sync(0xffffffffu, pf[w] >= 0.f && !pred(pf[w]));
                        if (m) end = 32 * (kf + w) + __ffs(m) - 1;
                        if (pf[w] >= 0.f && (end < 0 || tf < end)) acc(pf[w]);
                    }
                }
                kf += wf;
                fopen = end < 0 && 32 * kf < T;
            }
        }
        int start;
        if (nb >= 0) {
            start = nb;                                  // the not-above cell is part of the window
        } else if (ti - a.stride >= 0) {
            continue;                                    // an earlier probe lies in the same run
        } else if (!a.has_prev[s]) {
            start = 0;                                   // analyze.py:382: start_min = 0
        } else if (too_long) {
            continue;
        } else {
            // analyze.py:383-398: walk into the previous block (the previous unit of the same launch, or the last unit of the
            // stream in the previous launch's buffer), tested against the CURRENT row mean; start_min = -T + 1 is never tested
            const CellRef pcol = (a.bpl == 1 || (s % a.bpl) == 0) ? CellRef::make<TILE>(a.Sprev, a.stream_stride, s + a.bpl - 1, fi, n)
                                                                   : CellRef::make<TILE>(a.S, a.stream_stride, s - 1, fi, n);
            const int jmax = T - 2;                      // cells last[T-1] ... last[2]
            const int jcap = min(jmax, a.max_cols + 2);
            int jf = 0;
            for (int base = 1; base <= jcap && jf == 0; base += 32) {
                const int jj = base + lane;
                const bool valid = jj <= jcap;
                const float p = valid ? pcol.at<TILE>(T - jj) : 0.f;
                const unsigned m = __ballot_sync(0xffffffffu, valid && !pred(p));
                if (m) jf = base + (__ffs(m) - 1);
                if (valid && (jf == 0 || jj <= jf)) acc(p);
            }
            if (jf > 0) start = -jf;
            else if (jcap == jmax) { start = -(T - 1); if (lane == 0) acc(pcol.at<TILE>(1)); }     // ran into start_min: last[1] is in the window, untested
            else continue;                               // longer than max_cols: fails the duration test
        }
        if (too_long || end < 0) {                       // end == T: dropped, re-found from the next block
            if (!too_long) skip_to = T;
            continue;
        }
        skip_to = end;
        const int cols = end - start + (start < 0 ? 1 : 0);
        if (cols < a.min_cols || cols > a.max_cols) continue;

        const int cnt = end - start;
        mx = warp_max(mx);
        sum = warp_sum(sum);
        sdb = warp_sum(sdb);
        sdb2 = warp_sum(sdb2);
        const double mdb = sdb / cnt;
        const double ss = fmax(sdb2 / cnt - mdb * mdb, 0.0) * cnt;
        if (lane == 0) {
            const int slot = atomicAdd(&a.counters[1], 1);
            if (slot < a.max_records) {
                rt_record r;
                r.stream = s; r.fi = fi; r.start = start; r.end = end;
                r.max_lin = mx; r.row_mean = avg;
                r.mean_lin = sum / cnt;
                r.std_db = sqrt(ss / cnt);
                a.rec[slot] = r;
            }
        }
      }
    }
}

// ---------------------------------------------------------------------------------------------
// band survey (rt_engine_set_survey): per unit and bin, the row mean, the peak and the columns that pass the scan's predicate
// ---------------------------------------------------------------------------------------------
// Its own argument struct: the scan kernels' ScanArgs stays as it is, so they compile to the same code with the survey off.
struct SurveyArgs {
    const float* S;        // current block, in the engine's layout
    size_t stream_stride;  // floats per unit
    const float* avg;      // [unit][n] row means of this launch (complete once the probe kernel has run)
    const float* thr;      // [unit]
    float snr;
    int n, T;
    float* noise;          // [unit][n] <- avg (the CTAs of column chunk 0)
    unsigned* peak;        // [unit][n] <- max_t S as a bit pattern (zeroed before): powers are >= 0, so atomicMax on the bits
                           //              is the float maximum, whatever order the chunks arrive in
    int* above;            // [unit][n] <- columns that pass the predicate (zeroed before; integer sums: order-free)
};

constexpr int SURVEY_COLS = 128;     // columns per thread: 74 chunks x 64 units x 256 bins = 1.2 M threads at configs[1]
constexpr int SURVEY_BATCH = 8;      // cells of a thread in flight together

// row position -> bin for the survey: as pos_to_bin, except that on TILE consecutive threads take consecutive floats of a time
// step (16-byte quads of 4 bins, 512 bytes apart), as the PERM positions do
template <int L>
__device__ __forceinline__ int survey_bin(int idx) {
    return L == LAYOUT_TILE ? (idx >> 4) + 16 * (idx & 3) + 64 * ((idx >> 2) & 3) : pos_to_bin<L>(idx);
}

// One thread per (unit, bin, chunk of SURVEY_COLS columns); min(n, 256) row positions of one unit per CTA.
template <int L>
__global__ void __launch_bounds__(256) survey_kernel(SurveyArgs a) {
    const int nbb = (a.n + blockDim.x - 1) / blockDim.x;           // bin blocks
    const int bb = blockIdx.x % nbb, chunk = blockIdx.x / nbb;
    const int idx = bb * blockDim.x + threadIdx.x;
    const int s = blockIdx.y;
    if (idx >= a.n) return;
    const int fi = survey_bin<L>(idx);
    const size_t cell = (size_t)s * a.n + fi;
    const float avg = a.avg[cell];
    if (chunk == 0) a.noise[cell] = avg;
    const Pred pred(a.thr[s], avg, a.snr);           // bit for bit the probe's above() (predicate.h)
    const CellRef col = CellRef::make<L>(a.S, a.stream_stride, s, fi, a.n);
    const int t0 = chunk * SURVEY_COLS, t1 = min(a.T, t0 + SURVEY_COLS);
    float mx = 0.f;
    int cnt = 0;
    for (int tb = t0; tb < t1; tb += SURVEY_BATCH) {
        float c[SURVEY_BATCH];
#pragma unroll
        for (int i = 0; i < SURVEY_BATCH; ++i) c[i] = (tb + i < t1) ? col.at<L>(tb + i) : -1.f;      // -1: no such column
#pragma unroll
        for (int i = 0; i < SURVEY_BATCH; ++i) {
            mx = fmaxf(mx, c[i]);
            cnt += (c[i] >= 0.f && pred(c[i])) ? 1 : 0;
        }
    }
    atomicMax(&a.peak[cell], __float_as_uint(mx));
    if (cnt) atomicAdd(&a.above[cell], cnt);
}

// ---------------------------------------------------------------------------------------------
// neighbour bins (rt_engine_set_neighbours): per record, the mean of bins fi - 1 and fi + 1 over the record's own cells
// ---------------------------------------------------------------------------------------------
// Its own argument struct, like SurveyArgs: ScanArgs stays as it is.
struct NeighbourArgs {
    const float* S;          // current block, in the engine's layout
    const float* Sprev;      // previous block (the carry of the first unit of every stream)
    size_t stream_stride;    // floats per unit
    const float* avg;        // [unit][n] row means of this launch
    const rt_record* rec;    // this launch's records, in the order the extraction kernel wrote them
    const int* counters;     // [1]: records emitted (may exceed max_records)
    int max_records;
    int bpl, n, T;
    rt_neighbours* out;      // [max_records], entry i for rec[i]
};

constexpr int NEIGHBOUR_CTAS = 296;       // 2 per SM of a B200; the warps grid-stride over the device-side record count

// One warp per record.  Lane l accumulates in double the carried columns T + start + l, + 32, ... and then the current columns
// max(start, 0) + l, + 32, ...; warp_sum's xor-butterfly adds the lanes.  That order depends only on the record, so every launch,
// batch and schedule returns the same bits.  The cells are exactly those extract2_kernel averaged into mean_lin, with its carry
// rule (the previous unit of the same launch, or the last unit of the stream in the previous launch's buffer).
template <int L>
__global__ void __launch_bounds__(256) neighbour_kernel(NeighbourArgs a) {
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int n_warps = (gridDim.x * blockDim.x) >> 5;
    const int n_rec = min(a.counters[1], a.max_records);
    const int n = a.n, T = a.T;
    for (int i = warp; i < n_rec; i += n_warps) {
        const rt_record r = a.rec[i];
        const int s = r.stream, lo = (r.fi + n - 1) % n, hi = (r.fi + 1) % n;
        double slo = 0.0, shi = 0.0;
        if (r.start < 0) {
            const bool own = a.bpl == 1 || (s % a.bpl) == 0;
            const float* P = own ? a.Sprev : a.S;
            const int ps = own ? s + a.bpl - 1 : s - 1;
            const CellRef plo = CellRef::make<L>(P, a.stream_stride, ps, lo, n), phi = CellRef::make<L>(P, a.stream_stride, ps, hi, n);
            for (int t = T + r.start + lane; t < T; t += 32) {
                slo += (double)plo.at<L>(t);
                shi += (double)phi.at<L>(t);
            }
        }
        const CellRef clo = CellRef::make<L>(a.S, a.stream_stride, s, lo, n), chi = CellRef::make<L>(a.S, a.stream_stride, s, hi, n);
        for (int t = max(r.start, 0) + lane; t < r.end; t += 32) {
            slo += (double)clo.at<L>(t);
            shi += (double)chi.at<L>(t);
        }
        slo = warp_sum(slo);
        shi = warp_sum(shi);
        if (lane == 0) {
            const int cnt = r.end - r.start;
            rt_neighbours o;
            o.mean_lo = slo / cnt; o.mean_hi = shi / cnt;
            o.row_mean_lo = a.avg[(size_t)s * n + lo]; o.row_mean_hi = a.avg[(size_t)s * n + hi];
            a.out[i] = o;
        }
    }
}

// PERM / TILE -> [T][n] for the parity hook, with the power scale of the tensor-core path undone (a power of two: exact)
template <int L>
__global__ void untile_kernel(const float* S, float* out, int total, int n, float inv_scale) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int t = idx / n, fi = idx % n;
    out[idx] = CellRef::make<L>(S, 0, 0, fi, n).template at<L>(t) * inv_scale;
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// The spectrogram kernels of the engine (choose_kernels decides one per engine)
enum class Spectro {
    GENERIC,     // spectro_generic: every nperseg and sample format, LINEAR layout
    REG256,      // nperseg 256, byte formats: register kernel spectro_reg256_v8 (spectro256.cuh), PERM layout
    TC256,       // nperseg 256, byte formats, RT_FFT_TC256: tensor-core stage 1 (spectro_tc256.cuh), TILE layout
    R16,         // nperseg 1024 / 4096, byte formats: radix-16 Stockham kernel (spectro_r16.cuh), LINEAR layout
};

}  // namespace

// error text for the other translation units of the library (rt_matcher.cpp)
int rt_internal_fail(int code, const char* msg) { return fail(code, msg); }

struct rt_engine {
    rt_config cfg{};
    int dev = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int n = 0, T = 0, n_streams = 0, bpl = 1, n_units = 0, n_chunks = 0, chunk_segs = 0, n_probes = 0;
    size_t block_bytes = 0;                  // bytes per block of one stream: bytes per complex sample * block_samples
    int sample_bytes = 2;                    // bytes per complex sample (rt_config.sample_format)
    bool ci8 = false;                        // RT_SAMPLE_CI8: the byte kernels' int8 instantiations
    int max_work = 0;                        // capacity of d_work
    int max_records = 0;                     // effective capacity of one launch's record list
    // ---- decided by choose_kernels
    Spectro kind = Spectro::GENERIC;
    int layout = LAYOUT_LINEAR;              // S layout
    size_t s_stride = 0;                     // floats per unit in a spectrogram buffer
    int part_rows = 0;                       // partial row sums per unit (d_part)
    bool part_perm = false;                  // the partial sums are in PERM position order (register kernel)
    bool sep_mean = false;                   // the scan runs row_mean_kernel (else the probe kernel or the tensor-core kernel does)
    int (*scan)(const rt_engine*, const ScanArgs&, cudaStream_t, cudaEvent_t) = nullptr;   // launch_scan<layout>, set by select_scan
    float pscale = 1.f;                      // power factor carried by S / row means / thresholds (tensor-core path), a power of two
    uint4* d_bmat = nullptr;                 // tensor-core operand image
    rt::TcTables tc_tab;
    int tc_grid = 0, tc_slots = 1, tc_bps = 0;
    int probe_ppt = PROBE_PPT;               // probe columns per thread: 8, 16 or 32 (chosen by launch size)
    bool scan_lean = false;                  // RT_SCAN_LEAN: 32-register scan CTAs that fit beside the resident spectrogram CTAs
    int lean_ctas = 148;
    float* d_win = nullptr;
    float2* d_tw = nullptr;
    float2* d_tw1 = nullptr;                 // spectro_r16: pass-1 twiddle table [15][n / 16]
    // three spectrogram buffers: launch i writes S[i % 3] while the scan of launch i-1 still reads
    // S[(i-1) % 3] (its block) and S[(i-2) % 3] (its carry) on the scan stream
    float* d_S[RT_SBUFS] = {nullptr, nullptr, nullptr};
    int cur = 0;
    float* d_part[RT_SLOTS] = {nullptr, nullptr};   // chunk row sums, by launch parity
    float* d_avg[RT_SLOTS] = {nullptr, nullptr};    // row means, by launch parity
    unsigned* d_ctr[RT_SLOTS] = {nullptr, nullptr}; // tensor-core kernel: finished-run tickets per unit, by launch parity (two launches
                                                    // may overlap on the two launch streams: they must not share tickets)
    cudaStream_t scan_stream = nullptr;      // row mean / probe / extract: overlaps the next launch's spectrogram
    // Consecutive spectrogram kernels alternate between two internal streams (forked from the launch stream by an event), so
    // that launch i+1 fills the SMs while the last CTAs of launch i drain: step 227.7 -> 213.9 us at config 2
    cudaStream_t lstream[2] = {nullptr, nullptr};
    cudaEvent_t fork_ev = nullptr;
    cudaEvent_t wait_ev = nullptr;           // rt_engine_wait_stream: the caller's stream, recorded (created on first use)
    int n_lstreams = 1;
    cudaEvent_t spec_done[RT_SLOTS] = {nullptr, nullptr};
    float* d_thr = nullptr;                  // [unit]
    int* d_hasprev = nullptr;                // [unit]
    std::vector<int> h_hasprev;              // [stream]: a previous launch exists (the carry of the first block of a launch)
    std::vector<int> h_hasprev_units;
    bool hasprev_dirty = true;
    // host input: two staging buffers filled on an upload stream, so the copy of launch i+1 overlaps the kernels of launch i
    uint8_t* d_stage[2] = {nullptr, nullptr};
    size_t stage_stride = 0;
    cudaStream_t h2d_stream = nullptr;
    cudaEvent_t h2d_done[2] = {nullptr, nullptr}, stage_free[2] = {nullptr, nullptr};
    unsigned long long h2d_seq = 0;
    uint4* d_work = nullptr;
    // results ring: up to RT_SLOTS launches may be in flight before their records are fetched
    int* d_counters = nullptr;              // [slot][2]
    rt_record* d_rec[RT_SLOTS] = {nullptr, nullptr};
    cudaEvent_t done[RT_SLOTS] = {nullptr, nullptr};
    cudaStream_t copy_stream = nullptr;
    unsigned long long launch_seq = 0, fetch_seq = 0;
    rt_record* h_rec = nullptr;     // pinned, grown on demand
    size_t h_rec_cap = 0;
    int* h_counters = nullptr;      // pinned
    bool peeked = false;            // h_counters holds the counters of the oldest unfetched launch
    float* d_tmp = nullptr;         // parity hook scratch
    bool launched = false;
    int last_work_items = 0, last_records = 0;   // counters of the last fetched launch
    // band survey (rt_engine_set_survey): [noise | peak bits | above columns], each [unit][n], per result slot
    bool survey = false;                         // survey the launches from the next one on
    bool surveyed[RT_SLOTS] = {false, false};    // the launch in this slot surveyed
    bool last_surveyed = false;                  // the last fetched launch surveyed: h_survey holds it
    uint32_t* d_survey[RT_SLOTS] = {nullptr, nullptr};
    uint32_t* h_survey = nullptr;                // pinned, allocated by the first fetch of a survey
    // neighbour bins (rt_engine_set_neighbours): one rt_neighbours per record, per result slot
    bool neighbours = false;                     // compute them for the launches from the next one on
    bool refined[RT_SLOTS] = {false, false};     // the launch in this slot computed them
    bool last_refined = false;                   // the last fetched launch computed them: h_nb_sorted holds them
    rt_neighbours* d_nb[RT_SLOTS] = {nullptr, nullptr};
    rt_neighbours* h_nb = nullptr;               // pinned, grown on demand like h_rec
    size_t h_nb_cap = 0;
    std::vector<rt_neighbours> h_nb_sorted;      // entry i for record i of the last fetch, power scale undone
    // timing
    struct EvSet { cudaEvent_t ev[6]; };   // launch stream: before / after spectrogram; scan stream: start, row mean, probe, extract
    std::vector<EvSet> ev_pool;
    size_t ev_used = 0;
    rt_timing acc{};
    // Per-kernel events are recorded on every timing_period-th launch only: two event records between consecutive spectrogram
    // kernels cost ~5 us of launch gap per step (232 -> 227 us at config 2).  The per-kernel sums reported by
    // rt_engine_get_timing are scaled to all launches (sum over the timed ones x launches / timed launches).
    int timing_period = 0;                 // 0: off
    int64_t timed_launches = 0, timing_launches = 0;      // launches with events / launches while timing was on
};

namespace {

int harvest_timing(rt_engine* e) {
    if (e->ev_used == 0) return RT_OK;
    CU(cudaStreamSynchronize(e->stream));
    for (auto& ls : e->lstream) if (ls) CU(cudaStreamSynchronize(ls));
    if (e->scan_stream) CU(cudaStreamSynchronize(e->scan_stream));
    for (size_t i = 0; i < e->ev_used; ++i) {
        float ms[4];
        CU(cudaEventElapsedTime(&ms[0], e->ev_pool[i].ev[0], e->ev_pool[i].ev[1]));
        for (int k = 1; k < 4; ++k) CU(cudaEventElapsedTime(&ms[k], e->ev_pool[i].ev[k + 1], e->ev_pool[i].ev[k + 2]));
        e->acc.spectrogram_ms += ms[0];
        e->acc.rowmean_ms += ms[1];
        e->acc.probe_ms += ms[2];
        e->acc.extract_ms += ms[3];
    }
    e->ev_used = 0;
    return RT_OK;
}

void free_engine(rt_engine* e) {
    if (!e) return;
    cudaSetDevice(e->dev);
    if (e->stream) cudaStreamSynchronize(e->stream);
    for (auto& ls : e->lstream) if (ls) cudaStreamSynchronize(ls);
    if (e->scan_stream) cudaStreamSynchronize(e->scan_stream);
    if (e->h2d_stream) cudaStreamSynchronize(e->h2d_stream);
    if (e->copy_stream) cudaStreamSynchronize(e->copy_stream);
    for (auto& s : e->ev_pool)
        for (auto& ev : s.ev) cudaEventDestroy(ev);
    cudaFree(e->d_win); cudaFree(e->d_tw); cudaFree(e->d_tw1);
    for (auto& p : e->d_S) cudaFree(p);
    for (int k = 0; k < RT_SLOTS; ++k) { cudaFree(e->d_part[k]); cudaFree(e->d_avg[k]); cudaFree(e->d_ctr[k]); cudaFree(e->d_rec[k]); cudaFree(e->d_survey[k]); cudaFree(e->d_nb[k]); }
    if (e->h_survey) cudaFreeHost(e->h_survey);
    if (e->h_nb) cudaFreeHost(e->h_nb);
    cudaFree(e->d_bmat); cudaFree(e->d_thr); cudaFree(e->d_hasprev);
    cudaFree(e->d_stage[0]); cudaFree(e->d_stage[1]); cudaFree(e->d_work); cudaFree(e->d_counters); cudaFree(e->d_tmp);
    for (int k = 0; k < 2; ++k) { if (e->h2d_done[k]) cudaEventDestroy(e->h2d_done[k]); if (e->stage_free[k]) cudaEventDestroy(e->stage_free[k]); }
    if (e->h2d_stream) cudaStreamDestroy(e->h2d_stream);
    for (auto& ev : e->done) if (ev) cudaEventDestroy(ev);
    for (auto& ev : e->spec_done) if (ev) cudaEventDestroy(ev);
    if (e->copy_stream) cudaStreamDestroy(e->copy_stream);
    if (e->scan_stream) cudaStreamDestroy(e->scan_stream);
    for (auto& ls : e->lstream) if (ls) cudaStreamDestroy(ls);
    if (e->fork_ev) cudaEventDestroy(e->fork_ev);
    if (e->wait_ev) cudaEventDestroy(e->wait_ev);
    if (e->h_rec) cudaFreeHost(e->h_rec);
    if (e->h_counters) cudaFreeHost(e->h_counters);
    if (e->own_stream && e->stream) cudaStreamDestroy(e->stream);
    delete e;
}

// wait for the oldest unfetched launch and read its two counters (work items, records)
int peek_oldest(rt_engine* e) {
    if (e->peeked) return RT_OK;
    const int slot = (int)(e->fetch_seq % RT_SLOTS);
    // copy on a side stream that only waits for THIS launch, so a later launch already queued does not delay it
    CU(cudaStreamWaitEvent(e->copy_stream, e->done[slot], 0));
    CU(cudaMemcpyAsync(e->h_counters, e->d_counters + 2 * slot, 2 * sizeof(int), cudaMemcpyDeviceToHost, e->copy_stream));
    CU(cudaStreamSynchronize(e->copy_stream));
    e->peeked = true;
    return RT_OK;
}

// The engine's spectrogram kernel and everything that follows from it: the S layout, the chunking, the partial row sums, who takes
// the row means, and the scan schedule that RT_SCAN_AUTO stands for (returned).  Called once, by rt_engine_create, on a validated
// configuration; it reads n, T, bpl, n_units and block_bytes.
int choose_kernels(rt_engine* e, const rt_config& cfg, bool byte_fmt, int sms) {
    const int n = e->n, T = e->T;
    // the register and tensor-core kernels read every unit's segments with 16-byte bulk copies: with blocks_per_launch > 1 the units
    // of a stream lie block_bytes apart (RT_FFT_AUTO runs the generic kernel then, RT_FFT_REG256 was refused)
    const bool units_aligned = e->bpl == 1 || e->block_bytes % 16 == 0;
    if (cfg.fft_impl == RT_FFT_TC256) e->kind = Spectro::TC256;
    else if (n == 256 && cfg.fft_impl != RT_FFT_GENERIC && byte_fmt && units_aligned) e->kind = Spectro::REG256;
    else if ((n == 1024 || n == 4096) && cfg.fft_impl == RT_FFT_AUTO && byte_fmt) e->kind = Spectro::R16;
    else e->kind = Spectro::GENERIC;

    // chunking: it depends on T only, so a stream gives bit-identical row means whether it runs alone or inside a batch
    e->chunk_segs = 32;
    if (e->kind == Spectro::REG256 || e->kind == Spectro::TC256) {
        // short blocks (300 kS/s SDRs, replay): shorter chunks = more CTAs per unit
        e->chunk_segs = T >= 8192 ? 192 : (T >= 2048 ? 128 : 64);   // 192 at T = 9375 (49 chunks per stream): step 205.0 -> 202.8 us vs 128, 209.8 at 256
        if (cfg.chunk_segs > 0) e->chunk_segs = cfg.chunk_segs;
    }
    e->n_chunks = (T + e->chunk_segs - 1) / e->chunk_segs;
    if (e->kind == Spectro::R16) {
        // segments are dealt round-robin over n_chunks CTAs (x teams) per unit: 148 SMs x the resident CTAs (3 at 1024, 2 at 4096)
        const int teams = n == 4096 ? 1 : 4;
        const int resident = 148 * (n == 4096 ? rt::R16Cfg<4096>::CTAS_PER_SM : rt::R16Cfg<1024>::CTAS_PER_SM);
        e->n_chunks = std::min(resident, (T + teams - 1) / teams);
        e->chunk_segs = (T + e->n_chunks - 1) / e->n_chunks;      // informational
    }
    e->part_rows = e->n_chunks;              // one partial row per CTA
    e->part_perm = e->kind == Spectro::REG256;

    switch (e->kind) {
        case Spectro::TC256: {
            e->layout = LAYOUT_TILE;
            e->s_stride = (size_t)((T + 31) / 32) * 8192;
            constexpr int NG = 2;
            e->tc_bps = (T + rt::Tc256<NG>::BATCH - 1) / rt::Tc256<NG>::BATCH;
            const long long Btot = (long long)e->n_units * e->tc_bps;
            e->tc_grid = (int)std::max<long long>(1, std::min<long long>(sms, Btot / NG));
            const long long G = (long long)e->tc_grid * NG;
            for (int s = 0; s < e->n_units; ++s)
                e->tc_slots = std::max(e->tc_slots, rt::tc_last_run(s, e->tc_bps, G, Btot) - rt::tc_first_run(s, e->tc_bps, G, Btot) + 1);
            e->part_rows = e->tc_slots;      // one partial row per warp-group run
            break;
        }
        case Spectro::REG256:
            e->layout = LAYOUT_PERM;
            e->s_stride = (size_t)((T + PERM_TG - 1) / PERM_TG) * PERM_TG * n;      // whole time groups
            break;
        default:
            e->layout = LAYOUT_LINEAR;
            e->s_stride = (size_t)T * n;
    }

    int sched = cfg.scan_schedule;
    if (sched == RT_SCAN_AUTO)
        // lean only where it was measured to win: the register kernel (the tensor-core kernel owns its SMs) with at least
        // ~100 us of spectrogram per launch (short launches: the slower lean kernels become the critical path)
        // (round-2 kernels, 2.4 MS/s streams: 32 streams 112.5 overlap / 113.9 lean, 48: 151.3 / 153.3, 64: 197.4 / 189.0 us;
        //  lean probe + full-size extraction: 188.0, full-size probe + lean extraction: 196.5)
        sched = (e->kind == Spectro::REG256 && (long long)e->n_units * T >= 500000) ? RT_SCAN_LEAN : RT_SCAN_OVERLAP;
    e->scan_lean = sched == RT_SCAN_LEAN;
    // the tensor-core kernel writes the row means itself; otherwise the probe kernel sums up to 48 partial rows (row_mean_of)
    // and row_mean_kernel runs for more, and always under the lean schedule (the lean probe reads finished row means)
    e->sep_mean = e->kind != Spectro::TC256 && (e->scan_lean || e->n_chunks > 48);
    return sched;
}

size_t generic_smem(int n) { return (size_t)n * (2 * sizeof(float2) + sizeof(float)) + 16; }

// The generic kernel's dynamic shared-memory limit.  The limit belongs to the kernel, not to this engine: only ever raise it, or an
// engine created later with a smaller nperseg would make every launch of a larger one in the same process fail
int raise_generic_smem(int sample_format, int n) {
    static std::mutex attr_mu;                  // engines may be created from several threads
    std::lock_guard<std::mutex> lock(attr_mu);
    const SpectroKernel gk = generic_kernel(sample_format);
    cudaFuncAttributes ga;
    CU(cudaFuncGetAttributes(&ga, gk));
    if (ga.maxDynamicSharedSizeBytes < (int)generic_smem(n))
        CU(cudaFuncSetAttribute(gk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)generic_smem(n)));
    return RT_OK;
}

// Kernel attributes of the engine's spectrogram kernel; CI8: the int8 instantiations of the byte kernels
template <bool CI8>
int set_spectro_attributes(const rt_engine* e) {
    constexpr cudaFuncAttribute SMEM = cudaFuncAttributeMaxDynamicSharedMemorySize;
    switch (e->kind) {
        case Spectro::TC256:
            CU((cudaFuncSetAttribute(rt::spectro_tc256_k<2, CI8>, SMEM, rt::Tc256<2>::SMEM)));
            return RT_OK;
        case Spectro::REG256:
            CU((cudaFuncSetAttribute(rt::spectro_reg256_v8<true, 2, CI8>, SMEM, R256Prod::SMEM)));
            CU((cudaFuncSetAttribute(rt::spectro_reg256_v8<true, 2, CI8>, cudaFuncAttributePreferredSharedMemoryCarveout, 100)));
            return RT_OK;
        case Spectro::R16:
            if (e->n == 4096) CU((cudaFuncSetAttribute(rt::spectro_r16_k<4096, CI8>, SMEM, rt::R16Cfg<4096>::SMEM)));
            else CU((cudaFuncSetAttribute(rt::spectro_r16_k<1024, CI8>, SMEM, rt::R16Cfg<1024>::SMEM)));
            return raise_generic_smem(e->cfg.sample_format, e->n);      // for unaligned input (launch_spectrogram)
        case Spectro::GENERIC:
            return raise_generic_smem(e->cfg.sample_format, e->n);
    }
    return RT_OK;
}

// The engine's spectrogram kernel for one launch; CI8 as above
template <bool CI8>
void launch_spectrogram(const rt_engine* e, const SpectroArgs& sa, int slot, bool aligned, cudaStream_t st) {
    const dim3 grid(e->n_chunks, e->n_units);
    switch (e->kind) {
        case Spectro::TC256: {
            rt::TcArgs ta;
            ta.iq = sa.iq; ta.stream_stride = sa.stream_stride; ta.T = e->T; ta.n_streams = e->n_units;
            ta.bps = e->tc_bps; ta.total_batches = e->n_units * e->tc_bps;
            ta.bmat = e->d_bmat; ta.wc0 = e->tc_tab.wc0; ta.wc1 = e->tc_tab.wc1; ta.wc255 = e->tc_tab.wc255;
            ta.S = sa.S; ta.S_stream_stride = e->s_stride;
            ta.part = sa.part; ta.part_slots = e->tc_slots; ta.avg = e->d_avg[slot]; ta.ctr = e->d_ctr[slot];
            ta.store = 1; ta.dbg = 0; ta.prof = nullptr;
            rt::spectro_tc256_k<2, CI8><<<e->tc_grid, 512, rt::Tc256<2>::SMEM, st>>>(ta);
            return;
        }
        case Spectro::REG256:
            rt::spectro_reg256_v8<true, 2, CI8><<<grid, R256Prod::THREADS, R256Prod::SMEM, st>>>(sa);
            return;
        case Spectro::R16:
            // the one choice made per launch: the radix-16 kernel reads 16-byte aligned input only.  Given anything else, the
            // generic kernel runs with the same chunking (one partial row per CTA) and writes the same LINEAR layout
            if (!aligned) break;
            if (e->n == 4096) rt::spectro_r16_k<4096, CI8><<<grid, 256, rt::R16Cfg<4096>::SMEM, st>>>(sa);
            else rt::spectro_r16_k<1024, CI8><<<grid, 256, rt::R16Cfg<1024>::SMEM, st>>>(sa);
            return;
        case Spectro::GENERIC:
            break;
    }
    generic_kernel(e->cfg.sample_format)<<<grid, 256, generic_smem(e->n), st>>>(sa);
}

// The probe and extraction kernels of one launch for S layout L (rt_engine::scan); probe_done is recorded between them (timing)
template <int L>
int launch_scan(const rt_engine* e, const ScanArgs& sc, cudaStream_t st, cudaEvent_t probe_done) {
    if (e->scan_lean) {
        probe_lean_kernel<L><<<e->lean_ctas, 128, 0, st>>>(sc);
    } else {
        const int pbins = std::min(e->n, 256), ppt = e->probe_ppt;
        const dim3 pgrid(((e->n + pbins - 1) / pbins) * ((e->n_probes + ppt - 1) / ppt), e->n_units);
        if (ppt == 8) probe_kernel<L, 8><<<pgrid, pbins, 0, st>>>(sc);
        else if (ppt == 16) probe_kernel<L, 16><<<pgrid, pbins, 0, st>>>(sc);
        else probe_kernel<L, 32><<<pgrid, pbins, 0, st>>>(sc);
    }
    CU(cudaGetLastError());
    if (probe_done) CU(cudaEventRecord(probe_done, st));
    // full size: one wave of 128-thread CTAs, four 32-cell windows per round trip; lean: one 32-cell window, no speculative
    // forward fetch (fewest sectors: the kernel runs beside the spectrogram of the next launch)
    if (e->scan_lean) extract2_kernel<L, 16><<<e->lean_ctas, 128, 0, st>>>(sc);
    else if (sc.widen) extract2_kernel<L, 8, 4><<<148 * 24, 128, 0, st>>>(sc);
    else extract2_kernel<L, 8><<<148 * 24, 128, 0, st>>>(sc);
    CU(cudaGetLastError());
    return RT_OK;
}

// The scan kernels of the engine's layout: rt_engine::scan, and the lean schedule's carve-out (the same as the resident spectrogram
// CTAs': an SM does not change its L1 / shared split while CTAs are resident, so a kernel asking for another split could not join them)
template <int L>
int use_scan_layout(rt_engine* e) {
    e->scan = launch_scan<L>;
    if (e->scan_lean) {
        CU(cudaFuncSetAttribute(row_mean_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        CU(cudaFuncSetAttribute(probe_lean_kernel<L>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
        CU((cudaFuncSetAttribute(extract2_kernel<L, 16>, cudaFuncAttributePreferredSharedMemoryCarveout, 100)));
    }
    return RT_OK;
}

int select_scan(rt_engine* e) {
    switch (e->layout) {
        case LAYOUT_PERM: return use_scan_layout<LAYOUT_PERM>(e);
        case LAYOUT_TILE: return use_scan_layout<LAYOUT_TILE>(e);
        default: return use_scan_layout<LAYOUT_LINEAR>(e);
    }
}

size_t survey_words(const rt_engine* e) { return (size_t)3 * e->n_units * e->n; }

// The band survey of one launch into d_survey[slot], on the scan stream behind the probe and extraction kernels (the row means are
// complete there under every schedule) and in front of done[slot], which orders the next writer of this S buffer and of
// d_survey[slot] after it.  So the fetch of a surveyed launch, which waits for done[slot], also waits for its survey, and the next
// launch's scan kernels queue behind it on the scan stream.
int launch_survey(const rt_engine* e, const float* S, int slot, cudaStream_t st) {
    const size_t cells = (size_t)e->n_units * e->n;
    uint32_t* buf = e->d_survey[slot];
    CU(cudaMemsetAsync(buf + cells, 0, 2 * cells * sizeof(uint32_t), st));
    SurveyArgs a;
    a.S = S; a.stream_stride = e->s_stride; a.avg = e->d_avg[slot]; a.thr = e->d_thr; a.snr = (float)e->cfg.snr_threshold;
    a.n = e->n; a.T = e->T;
    a.noise = reinterpret_cast<float*>(buf); a.peak = buf + cells; a.above = reinterpret_cast<int*>(buf + 2 * cells);
    const int bins = std::min(e->n, 256);
    const dim3 grid(((e->n + bins - 1) / bins) * ((e->T + SURVEY_COLS - 1) / SURVEY_COLS), e->n_units);
    switch (e->layout) {
        case LAYOUT_PERM: survey_kernel<LAYOUT_PERM><<<grid, bins, 0, st>>>(a); break;
        case LAYOUT_TILE: survey_kernel<LAYOUT_TILE><<<grid, bins, 0, st>>>(a); break;
        default: survey_kernel<LAYOUT_LINEAR><<<grid, bins, 0, st>>>(a);
    }
    CU(cudaGetLastError());
    return RT_OK;
}

// The neighbour bins of one launch's records into d_nb[slot], on the scan stream behind the extraction kernel (and the survey) and in
// front of done[slot], which orders the next writer of S[next], of the carry buffer, of d_rec[slot] and of d_nb[slot] after it.
// The record count stays on the device: the grid is fixed and the warps stride over it.
int launch_neighbours(const rt_engine* e, const float* S, const float* Sprev, int slot, const int* d_cnt, cudaStream_t st) {
    NeighbourArgs a;
    a.S = S; a.Sprev = Sprev; a.stream_stride = e->s_stride; a.avg = e->d_avg[slot];
    a.rec = e->d_rec[slot]; a.counters = d_cnt; a.max_records = e->max_records;
    a.bpl = e->bpl; a.n = e->n; a.T = e->T;
    a.out = e->d_nb[slot];
    switch (e->layout) {
        case LAYOUT_PERM: neighbour_kernel<LAYOUT_PERM><<<NEIGHBOUR_CTAS, 256, 0, st>>>(a); break;
        case LAYOUT_TILE: neighbour_kernel<LAYOUT_TILE><<<NEIGHBOUR_CTAS, 256, 0, st>>>(a); break;
        default: neighbour_kernel<LAYOUT_LINEAR><<<NEIGHBOUR_CTAS, 256, 0, st>>>(a);
    }
    CU(cudaGetLastError());
    return RT_OK;
}

}  // namespace

extern "C" {

const char* rt_last_error(void) { return g_err.c_str(); }
int rt_abi_version(void) { return RT_ABI_VERSION; }

int rt_device_count(void) {
    int n = 0;
    cudaError_t err = cudaGetDeviceCount(&n);
    if (err != cudaSuccess) return fail(RT_ERR_CUDA, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(err));
    return n;
}

int rt_engine_create(const rt_config* cfg, rt_engine** out) {
    if (!cfg || !out) return fail(RT_ERR_INVALID, "null argument");
    *out = nullptr;
    if (cfg->abi_version != RT_ABI_VERSION) return fail(RT_ERR_INVALID, "rt_config.abi_version mismatch");
    const int n = cfg->nperseg;
    if (n < 8 || n > 4096 || (n & (n - 1))) return fail(RT_ERR_INVALID, "nperseg must be a power of two in [8, 4096]");
    if (cfg->n_streams < 1 || cfg->n_streams > 65535) return fail(RT_ERR_INVALID, "n_streams must be in [1, 65535]");
    const int bpl = cfg->blocks_per_launch == 0 ? 1 : cfg->blocks_per_launch;
    if (bpl < 1 || (long long)cfg->n_streams * bpl > 65535) return fail(RT_ERR_INVALID, "blocks_per_launch must be >= 1 and n_streams * blocks_per_launch <= 65535");
    if (!cfg->window || !cfg->signal_threshold) return fail(RT_ERR_INVALID, "window / signal_threshold missing");
    if (cfg->block_samples / n < 2) return fail(RT_ERR_INVALID, "block_samples must hold at least two segments (analyze.py:354 indexes times[1])");
    if (cfg->block_samples / n > (1 << 24)) return fail(RT_ERR_INVALID, "block too long");
    if (cfg->probe_stride < 1 || cfg->min_cols < 0 || cfg->max_cols < cfg->min_cols || cfg->max_records < 0)
        return fail(RT_ERR_INVALID, "probe_stride / min_cols / max_cols / max_records out of range");
    if (!(cfg->sample_rate > 0) || !(cfg->snr_threshold >= 0)) return fail(RT_ERR_INVALID, "sample_rate / snr_threshold out of range");
    if (cfg->fft_impl < RT_FFT_AUTO || cfg->fft_impl > RT_FFT_TC256) return fail(RT_ERR_INVALID, "unknown fft_impl");
    if ((cfg->fft_impl == RT_FFT_REG256 || cfg->fft_impl == RT_FFT_TC256) && n != 256) return fail(RT_ERR_INVALID, "RT_FFT_REG256 / RT_FFT_TC256 need nperseg == 256");
    if (cfg->scan_schedule < RT_SCAN_AUTO || cfg->scan_schedule > RT_SCAN_LEAN) return fail(RT_ERR_INVALID, "unknown scan_schedule");
    if (cfg->launch_streams < 0 || cfg->launch_streams > 2) return fail(RT_ERR_INVALID, "launch_streams must be 0 (auto), 1 or 2");
    if (cfg->launch_streams == 2 && cfg->scan_schedule == RT_SCAN_SERIAL) return fail(RT_ERR_INVALID, "two launch streams need an overlapped scan schedule");
    if (cfg->chunk_segs < 0 || cfg->chunk_segs % 8 != 0) return fail(RT_ERR_INVALID, "chunk_segs must be 0 (auto) or a multiple of 8");
    if (cfg->fft_impl == RT_FFT_TC256 && bpl != 1) return fail(RT_ERR_INVALID, "RT_FFT_TC256 does not take blocks_per_launch > 1");
    rt::SampleFormatInfo fmt;
    if (!rt::sample_format_info(cfg->sample_format, &fmt)) return fail(RT_ERR_INVALID, "unknown sample_format");
    const bool byte_fmt = rt::sample_format_is_byte(cfg->sample_format);
    if (!byte_fmt && (cfg->fft_impl == RT_FFT_REG256 || cfg->fft_impl == RT_FFT_TC256))
        return fail(RT_ERR_INVALID, "RT_FFT_REG256 / RT_FFT_TC256 read bytes: RT_SAMPLE_CI16 / RT_SAMPLE_CF32 run on RT_FFT_GENERIC");
    // the register kernel reads every unit's segments with 16-byte bulk copies: with blocks_per_launch > 1 the units of a stream
    // lie block_bytes apart, so the block must be a multiple of 16 bytes (choose_kernels)
    if (cfg->fft_impl == RT_FFT_REG256 && bpl > 1 && (fmt.bytes * cfg->block_samples) % 16 != 0)
        return fail(RT_ERR_INVALID, "RT_FFT_REG256 with blocks_per_launch > 1 needs block_samples to be a multiple of 8");
    for (int r : cfg->reserved) if (r != 0) return fail(RT_ERR_INVALID, "rt_config.reserved must be zero");

    int ndev = 0;
    CU(cudaGetDeviceCount(&ndev));
    if (cfg->cuda_device < 0 || cfg->cuda_device >= ndev) return fail(RT_ERR_CUDA, "no such CUDA device (this engine has no CPU fallback)");
    CU(cudaSetDevice(cfg->cuda_device));
    cudaFuncAttributes fa;
    cudaError_t ferr = cudaFuncGetAttributes(&fa, probe_kernel<LAYOUT_PERM, PROBE_PPT>);
    if (ferr != cudaSuccess)
        return fail(RT_ERR_CUDA, std::string("kernels not loadable on this device (built for sm_100a only): ") + cudaGetErrorString(ferr));

    rt_engine* e = new rt_engine();
    e->cfg = *cfg;
    e->dev = cfg->cuda_device;
    e->n = n;
    e->T = (int)(cfg->block_samples / n);
    e->n_streams = cfg->n_streams;
    e->bpl = bpl;
    e->n_units = cfg->n_streams * bpl;
    e->sample_bytes = fmt.bytes;
    e->ci8 = cfg->sample_format == RT_SAMPLE_CI8;
    e->block_bytes = (size_t)fmt.bytes * (size_t)cfg->block_samples;
    e->n_probes = (e->T + cfg->probe_stride - 1) / cfg->probe_stride;
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, e->dev) != cudaSuccess || sms < 1) sms = 148;
    const int sched = choose_kernels(e, *cfg, byte_fmt, sms);
    {
        // full-size probe kernel: as many CTAs as fit in ONE wave beside the resident spectrogram CTAs of the next launch (about one
        // 256-thread CTA per SM).  Fewer probe columns per thread = more CTAs and shorter chains of round trips, but a second wave
        // doubles the kernel: a 20 MS/s nperseg-4096 block took 46 us at 8 columns per thread (256 CTAs), 18 us at 16 (128 CTAs) and
        // 57 us at 32 (64 CTAs); step 85.5 -> 67.2 us
        const long long bin_blocks = (n + 255) / 256;
        for (int ppt = 8; ppt <= 32; ppt <<= 1) {
            e->probe_ppt = ppt;
            if (bin_blocks * ((e->n_probes + ppt - 1) / ppt) * e->n_units <= 148) break;
        }
    }
    const size_t max_work = (size_t)e->n_units * n * e->n_probes;    // every probe cell a hit: the work list cannot overflow
    // every record belongs to a different probe hit, so max_work records is the worst case; capped at 4 Mi (160 MB per slot)
    e->max_records = cfg->max_records > 0 ? cfg->max_records : (int)std::min<size_t>(max_work, (size_t)4 << 20);

#define CUE(call)                                                                                  \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            free_engine(e);                                                                        \
            return fail(RT_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e));          \
        }                                                                                          \
    } while (0)

    CUE(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    e->own_stream = true;

    // window with the density scaling and the full scale of the sample format folded in (sample_format.cuh):
    // S = |FFT(w (x - mean))|^2 / (fs sum w^2),  x = b / scale (- 1 for cu8)  =>  S = |FFT(w' (b - mean_b))|^2
    double sw2 = 0.0;
    for (int i = 0; i < n; ++i) sw2 += cfg->window[i] * cfg->window[i];
    if (!(sw2 > 0)) { free_engine(e); return fail(RT_ERR_INVALID, "window has no energy"); }
    const double amp = std::sqrt(1.0 / (cfg->sample_rate * sw2)) / fmt.full_scale;
    std::vector<float> hwin(n);
    for (int i = 0; i < n; ++i) hwin[i] = (float)(cfg->window[i] * amp);
    if (e->kind == Spectro::TC256) {
        e->tc_tab = rt::tc_make_tables(cfg->window, amp);
        if (!e->tc_tab.eligible) { free_engine(e); return fail(RT_ERR_INVALID, "RT_FFT_TC256 needs a window whose DFT is confined to the bins 0 and +-1 (boxcar, hann, hamming)"); }
        e->pscale = e->tc_tab.pscale;
    }
    std::vector<float2> htw(n);
    for (int k = 0; k < n; ++k) {
        const double ang = -2.0 * M_PI * (double)k / (double)n;
        htw[k] = make_float2((float)std::cos(ang), (float)std::sin(ang));
    }
    std::vector<float> hthr(e->n_units);
    for (int u = 0; u < e->n_units; ++u) hthr[u] = (float)cfg->signal_threshold[u / bpl] * e->pscale;   // pscale is a power of two: exact

    const size_t cells = (size_t)e->n_units * e->s_stride;
    const size_t part_cells = (size_t)e->n_units * e->part_rows * n;
    CUE(cudaMalloc(&e->d_win, n * sizeof(float)));
    CUE(cudaMalloc(&e->d_tw, n * sizeof(float2)));
    for (int k = 0; k < RT_SBUFS; ++k) CUE(cudaMalloc(&e->d_S[k], cells * sizeof(float)));
    for (int k = 0; k < RT_SLOTS; ++k) {
        CUE(cudaMalloc(&e->d_part[k], part_cells * sizeof(float)));
        CUE(cudaMemset(e->d_part[k], 0, part_cells * sizeof(float)));
        CUE(cudaMalloc(&e->d_avg[k], (size_t)e->n_units * n * sizeof(float)));
        CUE(cudaMalloc(&e->d_ctr[k], e->n_units * sizeof(unsigned)));
        CUE(cudaMemset(e->d_ctr[k], 0, e->n_units * sizeof(unsigned)));
        CUE(cudaMalloc(&e->d_rec[k], (size_t)e->max_records * sizeof(rt_record)));
        CUE(cudaEventCreateWithFlags(&e->done[k], cudaEventDisableTiming));
        CUE(cudaEventCreateWithFlags(&e->spec_done[k], cudaEventDisableTiming));
    }
    if (e->kind == Spectro::TC256) {
        CUE(cudaMalloc(&e->d_bmat, e->tc_tab.bmat.size() * sizeof(uint16_t)));
        CUE(cudaMemcpy(e->d_bmat, e->tc_tab.bmat.data(), e->tc_tab.bmat.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
    }
    CUE(cudaMalloc(&e->d_thr, e->n_units * sizeof(float)));
    CUE(cudaMalloc(&e->d_hasprev, e->n_units * sizeof(int)));
    CUE(cudaMalloc(&e->d_work, max_work * sizeof(uint4)));
    e->max_work = (int)std::min<size_t>(max_work, 0x7fffffff);
    CUE(cudaMalloc(&e->d_counters, 2 * RT_SLOTS * sizeof(int)));
    CUE(cudaStreamCreateWithFlags(&e->copy_stream, cudaStreamNonBlocking));

    // ---- schedule (rt_config.scan_schedule / launch_streams, resolved by choose_kernels; DESIGN.md 5.7)
    if (sched != RT_SCAN_SERIAL) {
        // the scan kernels are small and latency bound: give them priority over the next launch's spectrogram CTAs
        int prio_lo = 0, prio_hi = 0;
        CUE(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        CUE(cudaStreamCreateWithPriority(&e->scan_stream, cudaStreamNonBlocking, prio_hi));
        if (cfg->launch_streams != 1) {
            for (auto& q : e->lstream) CUE(cudaStreamCreateWithFlags(&q, cudaStreamNonBlocking));
            CUE(cudaEventCreateWithFlags(&e->fork_ev, cudaEventDisableTiming));
            e->n_lstreams = 2;
        }
    }
    // lean scan kernels: 128-thread CTAs capped at 32 registers (4096 per CTA -- what four resident spectrogram CTAs leave free
    // on an SM), 12 per SM (8 ... 16 time the same within 1 %)
    e->lean_ctas = sms * 12;
    CUE(cudaMallocHost(&e->h_counters, 2 * sizeof(int)));
    CUE(cudaMemcpy(e->d_win, hwin.data(), n * sizeof(float), cudaMemcpyHostToDevice));
    CUE(cudaMemcpy(e->d_tw, htw.data(), n * sizeof(float2), cudaMemcpyHostToDevice));
    CUE(cudaMemcpy(e->d_thr, hthr.data(), e->n_units * sizeof(float), cudaMemcpyHostToDevice));
    e->h_hasprev.assign(e->n_streams, 0);
    e->h_hasprev_units.assign(e->n_units, 0);
    e->hasprev_dirty = true;
    if (e->kind == Spectro::R16) {
        const int bt = n / 16;
        std::vector<float2> htw1((size_t)15 * bt);
        for (int i = 1; i < 16; ++i)
            for (int b = 0; b < bt; ++b) htw1[(size_t)(i - 1) * bt + b] = htw[(b * i) & (n - 1)];
        CUE(cudaMalloc(&e->d_tw1, htw1.size() * sizeof(float2)));
        CUE(cudaMemcpy(e->d_tw1, htw1.data(), htw1.size() * sizeof(float2), cudaMemcpyHostToDevice));
    }
#undef CUE
    int rc = e->ci8 ? set_spectro_attributes<true>(e) : set_spectro_attributes<false>(e);
    if (rc == RT_OK) rc = select_scan(e);
    if (rc != RT_OK) { free_engine(e); return rc; }
    *out = e;
    return RT_OK;
}

void rt_engine_destroy(rt_engine* e) { free_engine(e); }

int rt_engine_set_stream(rt_engine* e, void* cuda_stream) {
    if (!e) return fail(RT_ERR_INVALID, "null engine");
    CU(cudaSetDevice(e->dev));
    CU(cudaStreamSynchronize(e->stream));
    for (auto& ls : e->lstream) if (ls) CU(cudaStreamSynchronize(ls));
    if (e->scan_stream) CU(cudaStreamSynchronize(e->scan_stream));
    if (e->own_stream) {
        CU(cudaStreamDestroy(e->stream));
        e->own_stream = false;
    }
    e->stream = (cudaStream_t)cuda_stream;
    return RT_OK;
}

int rt_engine_wait_stream(rt_engine* e, void* cuda_stream) {
    if (!e) return fail(RT_ERR_INVALID, "null engine");
    CU(cudaSetDevice(e->dev));
    if (!e->wait_ev) CU(cudaEventCreateWithFlags(&e->wait_ev, cudaEventDisableTiming));
    // the internal launch streams fork from e->stream at the next launch, so they inherit this wait
    CU(cudaEventRecord(e->wait_ev, (cudaStream_t)cuda_stream));
    CU(cudaStreamWaitEvent(e->stream, e->wait_ev, 0));
    return RT_OK;
}

int rt_engine_reset_stream(rt_engine* e, int32_t stream) {
    if (!e || stream < 0 || stream >= e->n_streams) return fail(RT_ERR_INVALID, "bad stream index");
    e->h_hasprev[stream] = 0;
    e->hasprev_dirty = true;
    return RT_OK;
}

int rt_engine_shape(const rt_engine* e, int32_t* n_streams, int32_t* nperseg, int32_t* T) {
    if (!e) return fail(RT_ERR_INVALID, "null engine");
    if (n_streams) *n_streams = e->n_units;
    if (nperseg) *nperseg = e->n;
    if (T) *T = e->T;
    return RT_OK;
}


int rt_engine_launch(rt_engine* e, const uint8_t* iq, int32_t iq_on_device, size_t stream_stride_bytes) {
    if (!e || !iq) return fail(RT_ERR_INVALID, "null argument");
    const size_t stream_bytes = e->block_bytes * (size_t)e->bpl;     // the consecutive blocks of one stream
    if (stream_stride_bytes < stream_bytes && e->n_streams > 1) return fail(RT_ERR_INVALID, "stream_stride_bytes smaller than one stream's blocks");
    CU(cudaSetDevice(e->dev));
    cudaStream_t st = e->stream;
    if (e->n_lstreams == 2) {
        CU(cudaEventRecord(e->fork_ev, e->stream));
        st = e->lstream[e->launch_seq & 1];
        CU(cudaStreamWaitEvent(st, e->fork_ev, 0));
    }

    const uint8_t* d_iq = iq;
    size_t stride = stream_stride_bytes;
    if (!iq_on_device) {
        if (!e->d_stage[0]) {
            e->stage_stride = (stream_bytes + 255) & ~(size_t)255;
            for (int k = 0; k < 2; ++k) {
                CU(cudaMalloc(&e->d_stage[k], e->stage_stride * e->n_streams));
                CU(cudaEventCreateWithFlags(&e->h2d_done[k], cudaEventDisableTiming));
                CU(cudaEventCreateWithFlags(&e->stage_free[k], cudaEventDisableTiming));
            }
            CU(cudaStreamCreateWithFlags(&e->h2d_stream, cudaStreamNonBlocking));
        }
        const int sb = (int)(e->h2d_seq & 1);
        if (e->h2d_seq >= 2) CU(cudaStreamWaitEvent(e->h2d_stream, e->stage_free[sb], 0));   // the spectrogram kernel that read this buffer is done
        if (e->stage_stride == stream_stride_bytes || e->n_streams == 1)    // packed batch: one linear DMA instead of n_streams row copies
            CU(cudaMemcpyAsync(e->d_stage[sb], iq, e->n_streams == 1 ? stream_bytes : e->stage_stride * e->n_streams, cudaMemcpyHostToDevice, e->h2d_stream));
        else
            CU(cudaMemcpy2DAsync(e->d_stage[sb], e->stage_stride, iq, stream_stride_bytes, stream_bytes, e->n_streams,
                                 cudaMemcpyHostToDevice, e->h2d_stream));
        CU(cudaEventRecord(e->h2d_done[sb], e->h2d_stream));
        CU(cudaStreamWaitEvent(st, e->h2d_done[sb], 0));
        d_iq = e->d_stage[sb];
        stride = e->stage_stride;
    }
    if (((uintptr_t)d_iq | (e->n_streams > 1 ? stride : 0)) % (uintptr_t)e->sample_bytes != 0)
        return fail(RT_ERR_INVALID, "IQ pointer / stream stride not aligned to one complex sample");
    const bool aligned = (((uintptr_t)d_iq | stride | (e->bpl > 1 ? e->block_bytes : 0)) & 15) == 0;
    if ((e->kind == Spectro::REG256 || e->kind == Spectro::TC256) && !aligned) return fail(RT_ERR_INVALID, "register FFT path needs 16-byte aligned IQ, stream stride and (blocks_per_launch > 1) block size");
    const int slot = (int)(e->launch_seq % RT_SLOTS);
    if (e->launch_seq - e->fetch_seq == RT_SLOTS) { e->fetch_seq++; e->peeked = false; }   // ring full: the oldest unfetched result is dropped
    int* d_cnt = e->d_counters + 2 * slot;
    cudaStream_t sc_st = e->scan_stream ? e->scan_stream : st;
    // Two streams: the spectrogram of this launch runs on the launch stream while the scan kernels of the
    // previous launch are still busy on the scan stream.  The buffers this launch writes (S[next], part[slot])
    // were last read by the scan of launch i-2, whose completion event is done[slot].
    if (e->launch_seq >= RT_SLOTS && e->scan_stream) CU(cudaStreamWaitEvent(st, e->done[slot], 0));

    rt_engine::EvSet* evs = nullptr;
    if (e->timing_period > 0) e->timing_launches++;
    if (e->timing_period > 0 && ((e->timing_launches - 1) % e->timing_period) == 0) {
        e->timed_launches++;
        if (e->ev_used == e->ev_pool.size()) {
            if (e->ev_pool.size() >= 4096) { int rc = harvest_timing(e); if (rc) return rc; }
            else {
                rt_engine::EvSet s;
                for (auto& ev : s.ev) CU(cudaEventCreate(&ev));
                e->ev_pool.push_back(s);
            }
        }
        evs = &e->ev_pool[e->ev_used++];
        CU(cudaEventRecord(evs->ev[0], st));
    }

    const int next = (e->cur + 1) % RT_SBUFS;
    SpectroArgs sa;
    sa.iq = d_iq; sa.stream_stride = stride; sa.n = e->n; sa.T = e->T;
    sa.bpl = e->bpl; sa.block_bytes = e->block_bytes;
    sa.chunk_segs = e->chunk_segs; sa.n_chunks = e->n_chunks;
    sa.win = e->d_win; sa.tw = e->d_tw; sa.tw1 = e->d_tw1; sa.S = e->d_S[next]; sa.part = e->d_part[slot];
    sa.S_stream_stride = e->s_stride;
    if (e->ci8) launch_spectrogram<true>(e, sa, slot, aligned, st);
    else launch_spectrogram<false>(e, sa, slot, aligned, st);
    CU(cudaGetLastError());
    if (evs) CU(cudaEventRecord(evs->ev[1], st));
    if (e->scan_stream) CU(cudaEventRecord(e->spec_done[slot], st));
    if (!iq_on_device) { CU(cudaEventRecord(e->stage_free[(int)(e->h2d_seq & 1)], st)); e->h2d_seq++; }

    // ---- scan stream: probe, extraction (in launch order; d_work / d_hasprev live here)
    if (e->scan_stream) CU(cudaStreamWaitEvent(sc_st, e->spec_done[slot], 0));
    if (e->hasprev_dirty) {
        for (int u = 0; u < e->n_units; ++u) e->h_hasprev_units[u] = (u % e->bpl) ? 1 : e->h_hasprev[u / e->bpl];
        // pageable source: the driver stages it before returning, so the vector may change right after
        CU(cudaMemcpyAsync(e->d_hasprev, e->h_hasprev_units.data(), e->n_units * sizeof(int), cudaMemcpyHostToDevice, sc_st));
        e->hasprev_dirty = false;
    }
    CU(cudaMemsetAsync(d_cnt, 0, 2 * sizeof(int), sc_st));
    if (evs) CU(cudaEventRecord(evs->ev[2], sc_st));
    if (e->sep_mean) {
        row_mean_kernel<<<dim3((4 * e->n + 127) / 128, e->n_units), 128, 0, sc_st>>>(e->d_part[slot], e->d_avg[slot], e->n, e->n_chunks, e->T, e->part_perm ? 1 : 0);
        CU(cudaGetLastError());
    }
    if (evs) CU(cudaEventRecord(evs->ev[3], sc_st));

    ScanArgs sc;
    sc.S = e->d_S[next]; sc.Sprev = e->d_S[e->cur]; sc.stream_stride = e->s_stride; sc.avg = e->d_avg[slot];
    // the probe kernel takes the row means from the partial sums unless they are already in avg
    sc.part = (e->kind == Spectro::TC256 || e->sep_mean) ? nullptr : e->d_part[slot];
    sc.n_chunks = e->n_chunks; sc.part_perm = e->part_perm ? 1 : 0; sc.thr = e->d_thr; sc.has_prev = e->d_hasprev;
    sc.bpl = e->bpl;
    sc.snr = (float)e->cfg.snr_threshold;
    sc.n = e->n; sc.T = e->T; sc.stride = e->cfg.probe_stride; sc.n_probes = e->n_probes;
    sc.min_cols = e->cfg.min_cols; sc.max_cols = e->cfg.max_cols;
    sc.n_streams_scan = e->n_units;
    sc.widen = ((long long)e->n_units * e->T < 300000) ? 1 : 0;
    sc.work = e->d_work; sc.max_work = e->max_work; sc.counters = d_cnt; sc.rec = e->d_rec[slot]; sc.max_records = e->max_records;
    int rc = e->scan(e, sc, sc_st, evs ? evs->ev[4] : nullptr);
    if (rc != RT_OK) return rc;
    if (evs) CU(cudaEventRecord(evs->ev[5], sc_st));
    e->surveyed[slot] = false;
    if (e->survey) {
        rc = launch_survey(e, e->d_S[next], slot, sc_st);
        if (rc != RT_OK) return rc;
        e->surveyed[slot] = true;
    }
    e->refined[slot] = false;
    if (e->neighbours) {
        rc = launch_neighbours(e, e->d_S[next], e->d_S[e->cur], slot, d_cnt, sc_st);
        if (rc != RT_OK) return rc;
        e->refined[slot] = true;
    }

    CU(cudaEventRecord(e->done[slot], sc_st));
    e->launch_seq++;
    e->cur = next;
    for (auto& h : e->h_hasprev)
        if (!h) { h = 1; e->hasprev_dirty = true; }
    e->launched = true;
    e->acc.launches += 1;
    e->acc.kernels += (e->sep_mean ? 4 : 3) + (e->survey ? 1 : 0) + (e->neighbours ? 1 : 0);
    return RT_OK;
}

int rt_engine_peek(rt_engine* e, int32_t* n_records) {
    if (!e || !n_records) return fail(RT_ERR_INVALID, "null argument");
    if (e->fetch_seq == e->launch_seq) return fail(RT_ERR_STATE, "rt_engine_peek without an unfetched rt_engine_launch");
    CU(cudaSetDevice(e->dev));
    int rc = peek_oldest(e);
    if (rc) return rc;
    *n_records = std::min(e->h_counters[1], e->max_records);
    return RT_OK;
}

int rt_engine_fetch(rt_engine* e, rt_record* out, int32_t max_out, int32_t* n_out) {
    if (!e || !n_out) return fail(RT_ERR_INVALID, "null argument");
    if (e->fetch_seq == e->launch_seq) return fail(RT_ERR_STATE, "rt_engine_fetch without an unfetched rt_engine_launch");
    CU(cudaSetDevice(e->dev));
    int rc = peek_oldest(e);
    if (rc) return rc;
    const int slot = (int)(e->fetch_seq % RT_SLOTS);
    e->fetch_seq++;
    e->peeked = false;
    const int nrec = e->h_counters[1];
    e->last_work_items = e->h_counters[0];
    e->last_records = nrec;
    *n_out = nrec;
    // the survey and the records come back on the copy stream, which waited for done[slot] in peek_oldest; one synchronize for both
    const bool surveyed = e->surveyed[slot];
    e->last_surveyed = false;
    if (surveyed) {
        if (!e->h_survey) CU(cudaMallocHost(&e->h_survey, survey_words(e) * sizeof(uint32_t)));
        CU(cudaMemcpyAsync(e->h_survey, e->d_survey[slot], survey_words(e) * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->copy_stream));
    }
    const int have = std::max(0, std::min(nrec, std::min(e->max_records, out ? max_out : 0)));
    if (have > 0) {
        if ((size_t)have > e->h_rec_cap) {
            if (e->h_rec) CU(cudaFreeHost(e->h_rec));
            e->h_rec = nullptr;
            e->h_rec_cap = std::max<size_t>((size_t)have + have / 2, 4096);
            CU(cudaMallocHost(&e->h_rec, e->h_rec_cap * sizeof(rt_record)));
        }
        CU(cudaMemcpyAsync(e->h_rec, e->d_rec[slot], (size_t)have * sizeof(rt_record), cudaMemcpyDeviceToHost, e->copy_stream));
    }
    // the neighbour bins of the returned records, next to them
    const bool refined = e->refined[slot];
    e->last_refined = false;
    if (refined && have > 0) {
        if ((size_t)have > e->h_nb_cap) {
            if (e->h_nb) CU(cudaFreeHost(e->h_nb));
            e->h_nb = nullptr;
            e->h_nb_cap = std::max<size_t>((size_t)have + have / 2, 4096);
            CU(cudaMallocHost(&e->h_nb, e->h_nb_cap * sizeof(rt_neighbours)));
        }
        CU(cudaMemcpyAsync(e->h_nb, e->d_nb[slot], (size_t)have * sizeof(rt_neighbours), cudaMemcpyDeviceToHost, e->copy_stream));
    }
    if (surveyed || have > 0) CU(cudaStreamSynchronize(e->copy_stream));
    e->last_surveyed = surveyed;
    const auto rec_less = [](const rt_record& x, const rt_record& y) {
        if (x.stream != y.stream) return x.stream < y.stream;
        if (x.fi != y.fi) return x.fi < y.fi;
        return x.start < y.start;
    };
    if (refined) {
        // records and neighbours through one permutation; the records end up in the order the plain sort gives them ((stream,
        // fi, start) is unique: two records of one bin and unit are two runs)
        std::vector<int> perm(have);
        for (int i = 0; i < have; ++i) perm[i] = i;
        std::sort(perm.begin(), perm.end(), [&](int i, int j) { return rec_less(e->h_rec[i], e->h_rec[j]); });
        std::vector<rt_record> rec(e->h_rec, e->h_rec + have);
        e->h_nb_sorted.resize(have);
        const double inv = 1.0 / e->pscale;              // power of two: exact
        for (int i = 0; i < have; ++i) {
            e->h_rec[i] = rec[perm[i]];
            rt_neighbours nb = e->h_nb[perm[i]];
            nb.mean_lo *= inv; nb.mean_hi *= inv;
            nb.row_mean_lo *= (float)inv; nb.row_mean_hi *= (float)inv;
            e->h_nb_sorted[i] = nb;
        }
        e->last_refined = true;
    }
    if (have > 0) {
        if (!refined) std::sort(e->h_rec, e->h_rec + have, rec_less);
        if (e->pscale != 1.f) {
            const float inv = 1.f / e->pscale;           // power of two: exact
            for (int i = 0; i < have; ++i) {
                e->h_rec[i].max_lin *= inv;
                e->h_rec[i].row_mean *= inv;
                e->h_rec[i].mean_lin *= (double)inv;
            }
        }
        std::memcpy(out, e->h_rec, (size_t)have * sizeof(rt_record));
    }
    if (nrec > e->max_records) return fail(RT_ERR_OVERFLOW, "more candidate records than rt_config.max_records (the first max_records were returned)");
    if (nrec > have) return fail(RT_ERR_OVERFLOW, "output buffer smaller than the number of records (the first max_out were returned)");
    return RT_OK;
}

int rt_tc256_tables(const double* window, double sample_rate, uint16_t* bmat_out, double* wc_out, double* pscale_out, int32_t* eligible_out) {
    if (!window || !(sample_rate > 0)) return fail(RT_ERR_INVALID, "null window / bad sample rate");
    double sw2 = 0.0;
    for (int i = 0; i < 256; ++i) sw2 += window[i] * window[i];
    if (!(sw2 > 0)) return fail(RT_ERR_INVALID, "window has no energy");
    const rt::TcTables t = rt::tc_make_tables(window, std::sqrt(1.0 / (sample_rate * sw2)) / 127.5);
    if (bmat_out) std::memcpy(bmat_out, t.bmat.data(), t.bmat.size() * sizeof(uint16_t));
    if (wc_out) { wc_out[0] = t.wc0.x; wc_out[1] = t.wc0.y; wc_out[2] = t.wc1.x; wc_out[3] = t.wc1.y; wc_out[4] = t.wc255.x; wc_out[5] = t.wc255.y; }
    if (pscale_out) *pscale_out = (double)t.pscale;
    if (eligible_out) *eligible_out = t.eligible ? 1 : 0;
    return RT_OK;
}

int rt_engine_last_counts(rt_engine* e, int32_t* work_items, int32_t* records) {
    if (!e) return fail(RT_ERR_INVALID, "null engine");
    if (work_items) *work_items = e->last_work_items;
    if (records) *records = e->last_records;
    return RT_OK;
}

int rt_engine_join(rt_engine* e) {
    if (!e) return fail(RT_ERR_INVALID, "null engine");
    if (e->launch_seq == 0 || !e->scan_stream) return RT_OK;
    CU(cudaSetDevice(e->dev));
    CU(cudaStreamWaitEvent(e->stream, e->done[(int)((e->launch_seq - 1) % RT_SLOTS)], 0));
    return RT_OK;
}

int rt_engine_process(rt_engine* e, const uint8_t* iq, int32_t iq_on_device, size_t stream_stride_bytes,
                      rt_record* out, int32_t max_out, int32_t* n_out) {
    int rc = rt_engine_launch(e, iq, iq_on_device, stream_stride_bytes);
    if (rc != RT_OK) return rc;
    return rt_engine_fetch(e, out, max_out, n_out);
}

int rt_engine_read_spectrogram(rt_engine* e, int32_t stream, float* out) {
    if (!e || !out || stream < 0 || stream >= e->n_units) return fail(RT_ERR_INVALID, "bad argument");
    if (!e->launched) return fail(RT_ERR_STATE, "no launch yet");
    CU(cudaSetDevice(e->dev));
    const size_t cells = (size_t)e->T * e->n;
    const float* src = e->d_S[e->cur] + (size_t)stream * e->s_stride;
    CU(cudaStreamSynchronize(e->stream));
    for (auto& ls : e->lstream) if (ls) CU(cudaStreamSynchronize(ls));
    if (e->scan_stream) CU(cudaStreamSynchronize(e->scan_stream));
    if (e->layout != LAYOUT_LINEAR) {
        if (!e->d_tmp) CU(cudaMalloc(&e->d_tmp, cells * sizeof(float)));
        const unsigned blocks = (unsigned)((cells + 255) / 256);
        if (e->layout == LAYOUT_TILE) untile_kernel<LAYOUT_TILE><<<blocks, 256, 0, e->stream>>>(src, e->d_tmp, (int)cells, 256, 1.f / e->pscale);
        else untile_kernel<LAYOUT_PERM><<<blocks, 256, 0, e->stream>>>(src, e->d_tmp, (int)cells, 256, 1.f);
        CU(cudaGetLastError());
        src = e->d_tmp;
    }
    CU(cudaMemcpyAsync(out, src, cells * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    return RT_OK;
}

int rt_engine_read_row_means(rt_engine* e, int32_t stream, float* out) {
    if (!e || !out || stream < 0 || stream >= e->n_units) return fail(RT_ERR_INVALID, "bad argument");
    if (!e->launched) return fail(RT_ERR_STATE, "no launch yet");
    CU(cudaSetDevice(e->dev));
    for (auto& ls : e->lstream) if (ls) CU(cudaStreamSynchronize(ls));
    if (e->scan_stream) CU(cudaStreamSynchronize(e->scan_stream));      // the row means are written on the scan stream
    CU(cudaMemcpyAsync(out, e->d_avg[(int)((e->launch_seq - 1) % RT_SLOTS)] + (size_t)stream * e->n, e->n * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
    CU(cudaStreamSynchronize(e->stream));
    if (e->pscale != 1.f)
        for (int i = 0; i < e->n; ++i) out[i] *= 1.f / e->pscale;
    return RT_OK;
}

int rt_engine_set_survey(rt_engine* e, int32_t enable) {
    if (!e) return fail(RT_ERR_INVALID, "null engine");
    if (enable) {
        CU(cudaSetDevice(e->dev));
        for (auto& p : e->d_survey)              // every slot: a failed allocation leaves the rest to the next call
            if (!p) CU(cudaMalloc(&p, survey_words(e) * sizeof(uint32_t)));
    }
    e->survey = enable != 0;
    return RT_OK;
}

int rt_engine_read_survey(rt_engine* e, float* noise, float* peak, int32_t* above_cols) {
    if (!e) return fail(RT_ERR_INVALID, "null engine");
    if (!e->last_surveyed) return fail(RT_ERR_INVALID, "the last fetched launch did not survey (rt_engine_set_survey)");
    const size_t cells = (size_t)e->n_units * e->n;
    const float inv = 1.f / e->pscale;                  // power of two: exact
    const float* h_noise = reinterpret_cast<const float*>(e->h_survey);
    for (size_t i = 0; i < cells; ++i) {
        if (noise) noise[i] = h_noise[i] * inv;
        if (peak) { float p; std::memcpy(&p, &e->h_survey[cells + i], sizeof(float)); peak[i] = p * inv; }
    }
    if (above_cols) std::memcpy(above_cols, e->h_survey + 2 * cells, cells * sizeof(int32_t));
    return RT_OK;
}

int rt_engine_set_neighbours(rt_engine* e, int32_t enable) {
    if (!e) return fail(RT_ERR_INVALID, "null engine");
    if (enable) {
        CU(cudaSetDevice(e->dev));
        for (auto& p : e->d_nb)                  // every slot: a failed allocation leaves the rest to the next call
            if (!p) CU(cudaMalloc(&p, (size_t)e->max_records * sizeof(rt_neighbours)));
    }
    e->neighbours = enable != 0;
    return RT_OK;
}

int rt_engine_read_neighbours(rt_engine* e, rt_neighbours* out, int32_t max_out, int32_t* n_out) {
    if (!e || !n_out || (max_out > 0 && !out)) return fail(RT_ERR_INVALID, "null argument");
    if (!e->last_refined) return fail(RT_ERR_INVALID, "the last fetched launch did not compute neighbour bins (rt_engine_set_neighbours)");
    const int have = (int)e->h_nb_sorted.size();
    *n_out = have;
    const int k = std::max(0, std::min(have, max_out));
    if (k > 0) std::memcpy(out, e->h_nb_sorted.data(), (size_t)k * sizeof(rt_neighbours));
    if (have > k) return fail(RT_ERR_OVERFLOW, "output buffer smaller than the number of entries (the first max_out were returned)");
    return RT_OK;
}

int rt_engine_enable_timing(rt_engine* e, int32_t period) {
    if (!e || period < 0) return fail(RT_ERR_INVALID, "null engine / negative period");
    if (period == 0) { int rc = harvest_timing(e); if (rc) return rc; }
    e->timing_period = period;
    return RT_OK;
}

int rt_engine_get_timing(rt_engine* e, rt_timing* out, int32_t reset) {
    if (!e || !out) return fail(RT_ERR_INVALID, "null argument");
    CU(cudaSetDevice(e->dev));
    int rc = harvest_timing(e);
    if (rc) return rc;
    *out = e->acc;
    if (e->timed_launches > 0 && e->timed_launches != e->timing_launches) {
        const double k = (double)e->timing_launches / (double)e->timed_launches;
        out->spectrogram_ms *= k; out->rowmean_ms *= k; out->probe_ms *= k; out->extract_ms *= k;
    }
    if (reset) { e->acc = rt_timing{}; e->timed_launches = 0; e->timing_launches = 0; }
    return RT_OK;
}

}  // extern "C"
