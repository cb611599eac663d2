// spectro_tc256.cuh -- nperseg-256 spectrogram with the first FFT stage on the 5th-generation tensor cores (sm_100a).
//
// Replaces scipy.signal.spectrogram(..., nperseg=256, noverlap=0, return_onesided=False) as called at
// /root/reference/radiotracking/analyze.py:234-241, for windows whose DFT has at most the bins 0 and +-1
// (boxcar, Hann, Hamming = the reference default): for those the detrend is a 3-bin correction.
//
// 256 = 16 x 16 Cooley-Tukey, n = 16 n1 + n2, k = k1 + 16 k2:
//     U[k1][n2] = sum_n1 (b[n] - 128) * c[k1][n],   c[k1][n] = w'[n] exp(-2 pi j k1 n / 256)     (stage 1)
//     X[k1 + 16 k2] = sum_n2 U[k1][n2] W16^{n2 k2}                                               (stage 2)
// Stage 1 absorbs the window AND the inter-stage twiddles into a constant 32x32 real matrix per n2.
// The samples b - 128 are exact in fp16, the matrix is split hi + lo (two fp16 terms = 22 bits), so
// stage 1 is tcgen05.mma.kind::f16 with fp32 accumulation in tensor memory:
//     D_n2[segment][(k1, re|im)] += A_n2[segment][(n1, I|Q)] * B_n2[(k1, re|im)][(n1, I|Q)]      M=64, N=32, K=2x16
// for a half-batch of 64 segments and all 16 n2 (16 x 32 = 512 TMEM columns).  An M=64 accumulator occupies 16 of
// the 32 lanes of every TMEM lane quarter (probed: profiles/r01_tc_probe_tmem_layouts.txt), so TWO half-batches are
// resident at once.  The CTA runs two independent warp groups X and Y (8 warps each, lanes 0-15 / 16-31 of each
// quarter): while one group waits for its tensor-core stage, the other converts or consumes, which keeps both the
// tensor pipe and the fp32 pipe busy without any explicit software pipeline.
// A thread of the consume phase owns two (segment, k1) pairs: it reads their 16 complex U[k1][.] straight from
// tensor memory (tcgen05.ld.16x256b), runs the in-register packed-complex DFT16 of fft_cpk.cuh, applies the detrend
// correction (bins 0, 1, 255 only), squares, accumulates row sums and stores the power cells.
//
// Power cells are stored in a time-tiled layout (TILE): [stream][t / 32][quad][t % 32][4] floats with
// quad = (fi & 15) * 4 + (fi >> 6) and the four floats fi = k1 + 16 * (4 c + e), e = 0..3: a warp (32 segments)
// stores 512 contiguous bytes per instruction, and the scan kernels find 32 consecutive time steps of a bin
// within 512 bytes instead of 32 KB.
//
// All powers carry a factor `pscale` (a power of two chosen so that the fp16 matrix entries are O(1)); the
// engine scales the thresholds by the same factor and the records back, which is exact in binary floating point.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>
#include <vector>

#include "spectro256.cuh"

namespace rt {

struct TcArgs {
    const uint8_t* iq;
    size_t stream_stride;
    int T, n_streams;
    int bps;                   // half-batches (64 segments) per stream
    int total_batches;         // n_streams * bps
    const uint4* bmat;         // [16 n2][hi, lo][2 KB]  UMMA K-major, no swizzle: (n, k) at (n>>3)*512 + (k>>3)*128 + (n&7)*16 + (k&7)*2
    float2 wc0, wc1, wc255;    // scaled DFT of the window at bins 0, 1, 255
    float* S;                  // TILE layout
    size_t S_stream_stride;    // floats per stream = ceil(T/32) * 8192
    float* part;               // [stream][part_slots][256] row sums per warp-group run (FFT bin order)
    int part_slots;
    float* avg;                // [stream][256] row means (nullptr: skip)
    unsigned* ctr;             // [stream] tickets
    int store;                 // 0: no S store (lab)
    int dbg;                   // lab: unused
    unsigned long long* prof;  // lab: per-CTA cycles spent in [convert, mma wait, consume, flush] (nullptr: off)
};

// NG = 1: one warp group of 16 warps, batches of 128 segments (M = 128 accumulator, all TMEM lanes)
// NG = 2: two independent warp groups of 8 warps, half-batches of 64 segments (M = 64 accumulators, 16 lanes of each quarter)
template <int NG>
struct Tc256 {
    static constexpr int THREADS = 512, GROUPS = NG, GROUP_THREADS = THREADS / NG, GROUP_WARPS = 16 / NG, BATCH = 128 / NG;
    static constexpr int A_MAT = BATCH * 64;             // one n2: BATCH rows x 64 B
    static constexpr int OFF_A = 0;
    static constexpr int A_GROUP = 16 * A_MAT + 128;     // + room for the bank skew of the matrix bases
    static constexpr int OFF_B = GROUPS * A_GROUP;
    static constexpr int B_BYTES = 16 * 2 * 2048;
    static constexpr int OFF_SUM = OFF_B + B_BYTES;      // [group][BATCH] u32 segment byte sums
    static constexpr int OFF_BAR = OFF_SUM + 512;        // [group] mbarrier
    static constexpr int OFF_TMEM = OFF_BAR + 16;
    static constexpr int SMEM = OFF_TMEM + 16;
    static constexpr uint32_t IDESC = (1u << 4) | ((32u >> 3) << 17) | ((uint32_t)(BATCH >> 4) << 24);   // f16 x f16 -> f32, K-major A and B, N=32, M=BATCH
};

__host__ __device__ inline uint32_t tc_a_base(int n2, int a_mat) { return (uint32_t)n2 * a_mat + (uint32_t)((n2 >> 1) & 7) * 16; }
// number of warp-group runs that touch stream s and the index of the first one (G = warp groups in the grid)
__host__ __device__ inline int tc_first_run(long long s, long long bps, long long G, long long B) { return (int)(((s * bps + 1) * G + B - 1) / B) - 1; }
__host__ __device__ inline int tc_last_run(long long s, long long bps, long long G, long long B) { return (int)((((s + 1) * bps) * G + B - 1) / B) - 1; }
__host__ __device__ inline size_t tile_cell_off(int t, int fi) {
    return ((size_t)(t >> 5) * 64 + (size_t)((fi & 15) * 4 + (fi >> 6))) * 128 + (size_t)(t & 31) * 4 + ((fi >> 4) & 3);
}

// ---------------------------------------------------------------------------------------------------------
// host: operand image and constants
// ---------------------------------------------------------------------------------------------------------
struct TcTables {
    std::vector<uint16_t> bmat;      // 16 * 2 * 1024 halves
    float2 wc0, wc1, wc255;
    float pscale;                    // power factor 2^(2e)
    bool eligible;                   // window's DFT vanishes outside bins 0, +-1
};

inline uint16_t tc_half_bits(float f) {
    const __half h = __float2half_rn(f);
    uint16_t u;
    memcpy(&u, &h, 2);
    return u;
}
inline float tc_half_val(uint16_t u) {
    __half h;
    memcpy(&h, &u, 2);
    return __half2float(h);
}

// window[n] as scipy returns it; amp = sqrt(1 / (fs * sum w^2)) / 127.5 (cu8) or / 128 (ci8)
inline TcTables tc_make_tables(const double* window, double amp) {
    TcTables t;
    double wmax = 0;
    for (int n = 0; n < 256; ++n) wmax = std::max(wmax, std::fabs(window[n] * amp));
    int e = 0;
    if (wmax > 0) e = -(int)std::floor(std::log2(wmax)) - 1;      // wmax * 2^e in [0.5, 1)
    const double sc = std::ldexp(1.0, e);
    t.pscale = (float)std::ldexp(1.0, 2 * e);
    t.bmat.assign(16 * 2 * 1024, 0);
    for (int n2 = 0; n2 < 16; ++n2)
        for (int k1 = 0; k1 < 16; ++k1)
            for (int n1 = 0; n1 < 16; ++n1) {
                const int n = 16 * n1 + n2;
                const double ang = -2.0 * M_PI * (double)((k1 * n) & 255) / 256.0;
                const double cr = window[n] * amp * sc * std::cos(ang), ci = window[n] * amp * sc * std::sin(ang);
                // D[(k1,re)] = sum xI cr - xQ ci ;  D[(k1,im)] = sum xI ci + xQ cr
                const double val[2][2] = {{cr, -ci}, {ci, cr}};    // [re|im row][I|Q column]
                for (int ri = 0; ri < 2; ++ri)
                    for (int iq = 0; iq < 2; ++iq) {
                        const int nn = 2 * k1 + ri, kk = 2 * n1 + iq;
                        const size_t off = (size_t)(nn >> 3) * 256 + (size_t)(kk >> 3) * 64 + (size_t)(nn & 7) * 8 + (kk & 7);   // in halves
                        const uint16_t hi = tc_half_bits((float)val[ri][iq]);
                        const uint16_t lo = tc_half_bits((float)(val[ri][iq] - (double)tc_half_val(hi)));
                        t.bmat[((size_t)n2 * 2 + 0) * 1024 + off] = hi;
                        t.bmat[((size_t)n2 * 2 + 1) * 1024 + off] = lo;
                    }
            }
    double wr[256], wi[256], big = 0, rest = 0;
    for (int k = 0; k < 256; ++k) {
        double sr = 0, si = 0;
        for (int n = 0; n < 256; ++n) {
            const double ang = -2.0 * M_PI * (double)((k * n) & 255) / 256.0;
            sr += window[n] * std::cos(ang);
            si += window[n] * std::sin(ang);
        }
        wr[k] = sr * amp * sc; wi[k] = si * amp * sc;
        const double m = std::hypot(wr[k], wi[k]);
        if (k == 0 || k == 1 || k == 255) big = std::max(big, m);
        else rest = std::max(rest, m);
    }
    t.wc0 = make_float2((float)wr[0], (float)wi[0]);
    t.wc1 = make_float2((float)wr[1], (float)wi[1]);
    t.wc255 = make_float2((float)wr[255], (float)wi[255]);
    t.eligible = big > 0 && rest <= 1e-11 * big;
    return t;
}

// ---------------------------------------------------------------------------------------------------------
// device
// ---------------------------------------------------------------------------------------------------------
#if defined(__CUDACC__)

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ uint64_t tc_desc(uint32_t smem_addr) {
    // K-major, no swizzle: core matrix = 8 rows x 16 B; LBO (K direction) = 128 B, SBO (row-group direction) = 512 B
    const uint32_t lo = ((smem_addr >> 4) & 0x3fffu) | ((128u >> 4) << 16);
    const uint32_t hi = (512u >> 4) | (1u << 14);          // version 1 (Blackwell), layout type 0
    return ((uint64_t)hi << 32) | lo;
}
__device__ __forceinline__ void tc_mma(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}"
        ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 16 TMEM lanes x 8 columns: thread t receives (lane t/4, columns 2(t%4), 2(t%4)+1) and (lane t/4 + 8, same columns)
__device__ __forceinline__ void tc_ld16x256(uint32_t taddr, unsigned& a0, unsigned& a1, unsigned& b0, unsigned& b1) {
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x1.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a0), "=r"(a1), "=r"(b0), "=r"(b1) : "r"(taddr));
}
// tcgen05.ld is asynchronous: its destination registers are valid after tcgen05.wait::ld.  The registers are
// passed through the wait as in/out operands so that the compiler cannot move a use above it.
__device__ __forceinline__ void tc_wait_ld32(unsigned (&x)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(x[0]), "+r"(x[1]), "+r"(x[2]), "+r"(x[3]), "+r"(x[4]), "+r"(x[5]), "+r"(x[6]), "+r"(x[7]),
                   "+r"(x[8]), "+r"(x[9]), "+r"(x[10]), "+r"(x[11]), "+r"(x[12]), "+r"(x[13]), "+r"(x[14]), "+r"(x[15]),
                   "+r"(x[16]), "+r"(x[17]), "+r"(x[18]), "+r"(x[19]), "+r"(x[20]), "+r"(x[21]), "+r"(x[22]), "+r"(x[23]),
                   "+r"(x[24]), "+r"(x[25]), "+r"(x[26]), "+r"(x[27]), "+r"(x[28]), "+r"(x[29]), "+r"(x[30]), "+r"(x[31])
                 :: "memory");
}
template <int NT>
__device__ __forceinline__ void group_sync(int grp) { asm volatile("bar.sync %0, %1;" ::"r"(1 + grp), "r"(NT) : "memory"); }

// sum of 32 per-lane values over the 8 lanes that share lane & 3; afterwards the lane holds the totals of
// v[base .. base + 3], base = 4 * (lane >> 2), in v[0..3]
__device__ __forceinline__ void octet_transpose_reduce32(float (&v)[32], int lane) {
#define RT_TR_STEP(HALF, BIT)                                                   \
    {                                                                           \
        const bool up = (lane & BIT) != 0;                                      \
        _Pragma("unroll") for (int i = 0; i < HALF; ++i) {                      \
            const float send = up ? v[i] : v[i + HALF];                         \
            const float keep = up ? v[i + HALF] : v[i];                         \
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, BIT);              \
        }                                                                       \
    }
    RT_TR_STEP(16, 16) RT_TR_STEP(8, 8) RT_TR_STEP(4, 4)
#undef RT_TR_STEP
}

// CI8: int8 input, taken as cu8 with the top bit of every byte flipped (sample_format.cuh)
template <int NG, bool CI8 = false>
__global__ void __launch_bounds__(512, 1) spectro_tc256_k(TcArgs a) {
    using C = Tc256<NG>;
    extern __shared__ __align__(128) unsigned char tc_smem[];
    __shared__ unsigned ticket[C::GROUPS];
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
    const int grp = warp / C::GROUP_WARPS, wg = warp % C::GROUP_WARPS, gtid = tid & (C::GROUP_THREADS - 1);
    const uint32_t sm0 = smem_u32(tc_smem);
    uint32_t* segsum = reinterpret_cast<uint32_t*>(tc_smem + C::OFF_SUM) + C::BATCH * grp;
    const uint32_t bar = sm0 + C::OFF_BAR + 8 * grp;
    volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(tc_smem + C::OFF_TMEM);
    const uint32_t a_group = sm0 + C::OFF_A + grp * C::A_GROUP;

    // ---- one-time setup: operand image of the 16 stage-1 matrices, tensor memory, completion barriers
    {
        uint4* dst = reinterpret_cast<uint4*>(tc_smem + C::OFF_B);
        for (int i = tid; i < C::B_BYTES / 16; i += C::THREADS) dst[i] = a.bmat[i];
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(sm0 + C::OFF_TMEM), "r"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(sm0 + C::OFF_BAR) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(sm0 + C::OFF_BAR + 8) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    // this warp group's contiguous range of half-batches ("run"); runs never share state
    const long long G = (long long)gridDim.x * C::GROUPS, Btot = a.total_batches;
    const int run = blockIdx.x * C::GROUPS + grp;
    const int lo_b = (int)((long long)run * Btot / G), hi_b = (int)((long long)(run + 1) * Btot / G);

    // consume-phase role: lane quarter q, lane half hh (NG = 2: the group's half); k1 = 4 (2 jsel + ps) + (lane & 3);
    // two rows (segments) per thread: rowA and rowA + 8
    const int q = wg & 3;
    const int hh = NG == 2 ? grp : ((wg >> 2) & 1), jsel = NG == 2 ? (wg >> 2) : (wg >> 3);
    const uint32_t my_tmem = tmem + ((uint32_t)(32 * q + 16 * hh) << 16) + 16 * jsel;
    const int rowA = (NG == 2 ? 16 * q : 32 * q + 16 * hh) + (lane >> 2);
    // convert-phase role: lane -> (chunk c of 4 n1, sample pair p)
    const int cc = lane >> 3, pp = lane & 7;
    const uint32_t a_dst0 = a_group + tc_a_base(2 * pp, C::A_MAT) + cc * 128;       // + (row >> 3) * 512 + (row & 7) * 16
    const uint32_t a_dst1 = a_group + tc_a_base(2 * pp + 1, C::A_MAT) + cc * 128;

    float acc[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = 0.f;
    unsigned phase = 0;
    int cur_stream = -1;
    long long pt[4] = {0, 0, 0, 0}, pc = clock64();
#define RT_PROF(i) { if (a.prof) { const long long now_ = clock64(); pt[i] += now_ - pc; pc = now_; } }

    auto flush = [&](int s) {
        // row sums of this run over stream s: the 8 lanes sharing a k1, then the four lane quarters
        octet_transpose_reduce32(acc, lane);
        float* red = reinterpret_cast<float*>(tc_smem + C::OFF_A + grp * C::A_GROUP);     // this group's A is idle between half-batches
        group_sync<C::GROUP_THREADS>(grp);
        // lane holds acc index i = 4 * (lane >> 2) + e (e = 0..3) for k1 offset (lane & 3): red[wg][lane & 3][i]
#pragma unroll
        for (int e = 0; e < 4; ++e) red[(wg * 4 + (lane & 3)) * 32 + 4 * (lane >> 2) + e] = acc[e];
        group_sync<C::GROUP_THREADS>(grp);
        const int b_first = tc_first_run(s, a.bps, G, Btot);
        float* pd = a.part + ((size_t)s * a.part_slots + (run - b_first)) * 256;
        {
            // bin fi = k1 + 16 k2; k1 = 4 (2 jsel + ps) + t3; acc index i = 16 ps + k2
            const int fi = gtid & 255, k1 = fi & 15, k2 = fi >> 4, j = k1 >> 2, js = j >> 1, ps = j & 1, t3 = k1 & 3, i = 16 * ps + k2;
            constexpr int WPJ = C::GROUP_WARPS / 2;          // warps per jsel value
            float t = 0.f;
#pragma unroll
            for (int qq = 0; qq < WPJ; ++qq) t += red[((WPJ * js + qq) * 4 + t3) * 32 + i];
            if (gtid < 256) pd[fi] = t;
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) acc[i] = 0.f;
        // row means by the last run of the stream (fixed order over the runs)
        if (a.avg != nullptr) {
            group_sync<C::GROUP_THREADS>(grp);
            if (gtid == 0) {
                __threadfence();
                ticket[grp] = atomicAdd(&a.ctr[s], 1u);
            }
            group_sync<C::GROUP_THREADS>(grp);
            const int n_runs = tc_last_run(s, a.bps, G, Btot) - b_first + 1;
            if (ticket[grp] == (unsigned)(n_runs - 1)) {
                __threadfence();
                if (gtid < 256) {
                    const float* p = a.part + (size_t)s * a.part_slots * 256 + gtid;
                    double t = 0.0;
                    for (int c = 0; c < n_runs; ++c) t += (double)__ldcg(p + (size_t)c * 256);
                    a.avg[(size_t)s * 256 + gtid] = (float)(t / (double)a.T);
                }
                if (gtid == 0) a.ctr[s] = 0;
            }
        }
        group_sync<C::GROUP_THREADS>(grp);
    };

    for (int gb = lo_b; gb < hi_b; ++gb) {
        const int s = gb / a.bps, bi = gb - s * a.bps;
        if (s != cur_stream) {
            if (cur_stream >= 0) flush(cur_stream);
            cur_stream = s;
            RT_PROF(3)
        }
        const int seg0 = bi * C::BATCH;
        const int nseg = min(C::BATCH, a.T - seg0);
        const uint8_t* base = a.iq + (size_t)s * a.stream_stride + (size_t)seg0 * 512;

        // ---------------- convert: uint8 IQ -> fp16 (b - 128, exact) operand tiles, one segment per warp pass
        {
            uint32_t w[8][4];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int row = wg + C::GROUP_WARPS * i;
                const uint32_t* src = reinterpret_cast<const uint32_t*>(base + (size_t)row * 512 + 128 * cc + 4 * pp);
#pragma unroll
                for (int u = 0; u < 4; ++u) w[i][u] = (row < nseg) ? (__ldg(src + 8 * u) ^ (CI8 ? 0x80808080u : 0u)) : 0x80808080u;   // ci8: + 128 per byte
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int row = wg + C::GROUP_WARPS * i;
                uint32_t e0[4], e1[4];
                unsigned sI = 0, sQ = 0;
                const __half2 off = __halves2half2(__ushort_as_half(0x6480), __ushort_as_half(0x6480));   // 1024 + 128
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const uint32_t x = w[i][u];                     // I(2p) Q(2p) I(2p+1) Q(2p+1) of n1 = 4c + u
                    uint32_t h0 = __byte_perm(x, 0x64646464u, 0x4140);   // fp16 pair 1024 + I, 1024 + Q   (sample 2p)
                    uint32_t h1 = __byte_perm(x, 0x64646464u, 0x4342);   //                                 (sample 2p+1)
                    __half2 v0 = __hsub2(*reinterpret_cast<__half2*>(&h0), off);
                    __half2 v1 = __hsub2(*reinterpret_cast<__half2*>(&h1), off);
                    e0[u] = *reinterpret_cast<uint32_t*>(&v0);
                    e1[u] = *reinterpret_cast<uint32_t*>(&v1);
                    sI = __dp4a(x, 0x00010001u, sI);
                    sQ = __dp4a(x, 0x01000100u, sQ);
                }
                const uint32_t roff = (uint32_t)(row >> 3) * 512 + (uint32_t)(row & 7) * 16;
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a_dst0 + roff), "r"(e0[0]), "r"(e0[1]), "r"(e0[2]), "r"(e0[3]) : "memory");
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a_dst1 + roff), "r"(e1[0]), "r"(e1[1]), "r"(e1[2]), "r"(e1[3]) : "memory");
                const unsigned tot = __reduce_add_sync(0xffffffffu, sI | (sQ << 16));   // each total <= 65280
                if (lane == 0) segsum[row] = tot;
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy writes -> tensor-core reads
        if (gb + 1 < hi_b) {
            // the next batch's bytes: one 128-byte line per thread pulled into L2 while this batch is multiplied and consumed
            const int s2 = (gb + 1) / a.bps, bi2 = (gb + 1) - s2 * a.bps;
            const int nseg2 = min(C::BATCH, a.T - bi2 * C::BATCH);
            const uint8_t* nb = a.iq + (size_t)s2 * a.stream_stride + (size_t)bi2 * C::BATCH * 512;
            for (int ln = gtid; ln < nseg2 * 4; ln += C::GROUP_THREADS) asm volatile("prefetch.global.L2 [%0];" ::"l"(nb + (size_t)ln * 128));
        }
        group_sync<C::GROUP_THREADS>(grp);
        RT_PROF(0)

        // ---------------- stage 1 on the tensor cores: 16 n2 x 2 K-steps x (hi, lo), M = 64 rows of this group
        if (wg == 0) {
            if (elect_one()) {
                tc_fence_after();
                const uint32_t d0 = tmem + ((uint32_t)(NG == 2 ? 16 * grp : 0) << 16);
#pragma unroll 1
                for (int n2 = 0; n2 < 16; ++n2) {
                    const uint32_t a_addr = a_group + tc_a_base(n2, C::A_MAT);
                    const uint32_t b_addr = sm0 + C::OFF_B + n2 * 4096;
#pragma unroll
                    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
                        for (int hl = 0; hl < 2; ++hl)
                            tc_mma(d0 + n2 * 32, tc_desc(a_addr + ks * 256), tc_desc(b_addr + hl * 2048 + ks * 256), C::IDESC, (ks | hl) != 0);
                }
                tc_commit(bar);
            }
            __syncwarp();
        }
        mbar_wait(bar, phase);
        phase ^= 1;
        tc_fence_after();
        RT_PROF(1)

        // ---------------- consume: stage 2 in registers, two (segment, k1) pairs per thread and pass
        const unsigned totA = segsum[rowA], totB = segsum[rowA + 8];
        // residual mean after the exact -128: (sum - 32768) / 256, exact in fp32
        const cpk mresA = c_make((float)((int)(totA & 0xffffu) - 32768) * 0.00390625f, (float)((int)(totA >> 16) - 32768) * 0.00390625f);
        const cpk mresB = c_make((float)((int)(totB & 0xffffu) - 32768) * 0.00390625f, (float)((int)(totB >> 16) - 32768) * 0.00390625f);
        const int segA = seg0 + rowA, segB = segA + 8;
#pragma unroll
        for (int ps = 0; ps < 2; ++ps) {
            const int j = 2 * jsel + ps, k1 = 4 * j + (lane & 3);
            cpk vA[16], vB[16];
            {
                unsigned x[32], y[32];
#pragma unroll
                for (int n2 = 0; n2 < 16; ++n2) tc_ld16x256(my_tmem + n2 * 32 + 8 * ps, x[2 * n2], x[2 * n2 + 1], y[2 * n2], y[2 * n2 + 1]);
                tc_wait_ld32(x);
                tc_wait_ld32(y);
#pragma unroll
                for (int n2 = 0; n2 < 16; ++n2) {
                    asm("mov.b64 %0, {%1, %2};" : "=l"(vA[n2].v) : "r"(x[2 * n2]), "r"(x[2 * n2 + 1]));
                    asm("mov.b64 %0, {%1, %2};" : "=l"(vB[n2].v) : "r"(y[2 * n2]), "r"(y[2 * n2 + 1]));
                }
            }
            cdft16(vA);                                  // over n2 -> k2: bin = k1 + 16 k2
            cdft16(vB);
            // detrend='constant': only the bins where the window's DFT lives (0, 1, 255) see the segment mean
            if (j == 0) {
                const float wr = k1 == 0 ? a.wc0.x : (k1 == 1 ? a.wc1.x : 0.f), wi = k1 == 0 ? a.wc0.y : (k1 == 1 ? a.wc1.y : 0.f);
                vA[0] = c_sub(vA[0], c_mul(mresA, wr, wi));
                vB[0] = c_sub(vB[0], c_mul(mresB, wr, wi));
            }
            if (j == 3) {
                const float wr = k1 == 15 ? a.wc255.x : 0.f, wi = k1 == 15 ? a.wc255.y : 0.f;
                vA[15] = c_sub(vA[15], c_mul(mresA, wr, wi));
                vB[15] = c_sub(vB[15], c_mul(mresB, wr, wi));
            }
            float pA[16], pB[16];
#pragma unroll
            for (int k2 = 0; k2 < 16; ++k2) {
                const float ra = c_re(vA[k2]), ia = c_im(vA[k2]), rb = c_re(vB[k2]), ib = c_im(vB[k2]);
                pA[k2] = fmaf(ia, ia, ra * ra);
                pB[k2] = fmaf(ib, ib, rb * rb);
                acc[16 * ps + k2] += pA[k2] + pB[k2];
            }
            if (a.store) {
                float* sbase = a.S + (size_t)s * a.S_stream_stride + (size_t)k1 * 512;
                if (segA < a.T) {
                    float4* dst = reinterpret_cast<float4*>(sbase + (size_t)(segA >> 5) * 8192 + (size_t)(segA & 31) * 4);
#pragma unroll
                    for (int c = 0; c < 4; ++c) dst[32 * c] = make_float4(pA[4 * c], pA[4 * c + 1], pA[4 * c + 2], pA[4 * c + 3]);
                }
                if (segB < a.T) {
                    float4* dst = reinterpret_cast<float4*>(sbase + (size_t)(segB >> 5) * 8192 + (size_t)(segB & 31) * 4);
#pragma unroll
                    for (int c = 0; c < 4; ++c) dst[32 * c] = make_float4(pB[4 * c], pB[4 * c + 1], pB[4 * c + 2], pB[4 * c + 3]);
                }
            }
        }
        tc_fence_before();
        group_sync<C::GROUP_THREADS>(grp);
        RT_PROF(2)
    }
    if (cur_stream >= 0) flush(cur_stream);
    RT_PROF(3)
    if (a.prof && gtid == 0)
        for (int i = 0; i < 4; ++i) a.prof[4 * run + i] = (unsigned long long)pt[i];
#undef RT_PROF

    tc_fence_before();
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512) : "memory");
}


#endif  // __CUDACC__

}  // namespace rt
