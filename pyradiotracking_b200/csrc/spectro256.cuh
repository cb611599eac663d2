// spectro256.cuh -- uint8 IQ -> power spectrogram cells + per-chunk row sums for nperseg == 256 (sm_100a).
//
// Replaces scipy.signal.spectrogram(..., nperseg=256, noverlap=0, return_onesided=False) as called at
// /root/reference/radiotracking/analyze.py:234-241 (detrend='constant', window, FFT, |X|^2 / (fs * sum w^2)).
//
// 16 threads (a half-warp) hold one 256-point FFT as a 16x16 Cooley-Tukey in registers; every complex
// value is one packed register pair (fft_cpk.cuh).  A warp works on 2*NSEG consecutive segments per
// round, fed by a per-warp ring of TMA bulk copies.  The engine instantiates spectro_reg256_v8 (end of this file: v7n with a
// cheaper byte -> float front end); spectro_reg256_v7n and its template switches stay for tools/spectro_lab.cu (variant timing on
// the GPU box; the other losing variants live in tools/spectro256_lab.cuh).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "fft_cpk.cuh"

namespace rt {

struct SpectroArgs {
    const uint8_t* iq;
    size_t stream_stride;
    int n, T, chunk_segs, n_chunks;
    const float* win;      // window * sqrt(1/(fs*sum(w^2))) / full scale of the sample format (127.5 for cu8, sample_format.cuh)
    const float2* tw;      // exp(-2 pi i k / n)
    const float2* tw1 = nullptr;   // spectro_r16: pass-1 twiddles exp(-2 pi i (b i) / n) as [i - 1][b], i = 1..15, b < n / 16
    float* S;              // generic kernel: [stream][T][n]; register kernel: [stream][T][pos(bin)] (see rt_engine.cu)
    size_t S_stream_stride;  // floats per stream
    float* part;           // [stream][chunk][n]   (FFT bin order; spectro_reg256_v7: PERM position order, like its S rows)
    // probe plane (spectro_reg256_v7 only, optional): a dense copy of the rows the probe loop of extract_signals looks at
    // (analyze.py:364, columns k * probe_stride), [stream][n_probes][256] in the order of the S rows, so that the probe
    // kernel reads 1 KB rows instead of one 32-byte sector per cell
    float* probe = nullptr;
    int probe_stride = 1, n_probes = 0;
    // offline replay (rt_config.blocks_per_launch): grid row s is the analyzer unit (stream s / bpl, block s % bpl); the blocks
    // of a stream are consecutive in memory
    int bpl = 1;
    size_t block_bytes = 0;
    __device__ __forceinline__ const uint8_t* unit_base(int s) const {
        return bpl == 1 ? iq + (size_t)s * stream_stride : iq + (size_t)(s / bpl) * stream_stride + (size_t)(s % bpl) * block_bytes;
    }
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void stg128_hint(float4* dst, float4 v, uint64_t pol) {
    asm volatile("st.global.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;"
                 ::"l"(dst), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(pol) : "memory");
}

// ---------------------------------------------------------------------------------------------
// v7: same data flow as spectro_reg256_k<NSEG=1>, hand-tightened non-FMA instruction stream:
//   * warp-uniform TMA issue behind elect.sync (no per-lane address loop, no proxy fence: the
//     WAR hazard generic-read -> async-write is ordered by __syncwarp + the mbarrier itself)
//   * running shared/global offsets instead of per-round index arithmetic
//   * byte sums reduced with two REDUX (warp-wide integer add) instead of a 4-deep shuffle chain
//   * detrend constant without I2F: (2^23 + sum) * 2^-8 == 32768 + sum/256 exactly
//   * inter-pass twiddles as (wr, wi) scalars: the lane swap / sign live in FFMA2 operand modifiers
//   * invalid (ragged-tail) lanes masked by a 0/1 factor in the row-sum FMA instead of a branch
// ---------------------------------------------------------------------------------------------
// LMAP: a segment's 16 threads are the lanes {0-3, 8-11, 16-19, 24-27} (+4 for the warp's second segment) instead of a half-warp, so
// that with the time-pair S layout (TG = 2) each quarter-warp phase of a 128-bit store covers ONE 128-byte line (4 granules x 2 time
// steps) instead of two half lines.  The shared-memory strides change with it: the two segments of a warp must sit 16 banks apart.
template <int WARPS_, int MINB_, bool LMAP_ = false>
struct R256v7T {
    static constexpr int WARPS = WARPS_, THREADS = 32 * WARPS_, STAGES = 4, MINB = MINB_;
    static constexpr bool LMAP = LMAP_;
    static constexpr int RAW_STRIDE = LMAP_ ? 576 : 544, XROW = 36, XTILE = 16 * XROW + (LMAP_ ? 16 : 0);
    static constexpr int STAGE_BYTES = 2 * RAW_STRIDE;                  // two segments per warp per round
    static constexpr int RAW_BYTES = WARPS * STAGES * STAGE_BYTES;
    static constexpr int XCH_BYTES = 2 * WARPS * XTILE * 4;
    static constexpr int RED_BYTES = 2 * WARPS * 256 * 4;
    static constexpr int BAR_OFF = (RAW_BYTES + XCH_BYTES) > RED_BYTES ? (RAW_BYTES + XCH_BYTES) : RED_BYTES;
    static constexpr int TAB_OFF = BAR_OFF + WARPS * STAGES * 8;         // optional constant tables: tw[16][16] float2, win[256]
    static constexpr int SMEM = TAB_OFF + 2048 + 1024;
    static constexpr int SEGS_PER_ROUND = 2 * WARPS;
};
using R256v7 = R256v7T<4, 4>;

__device__ __forceinline__ bool elect_one() {
    unsigned ok;
    asm volatile("{\n.reg .pred p;\nelect.sync _|p, 0xffffffff;\nselp.u32 %0, 1, 0, p;\n}" : "=r"(ok));
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, unsigned parity) {
    asm volatile(
        "{\n.reg .pred p;\n"
        "W: mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@!p bra W;\n}"
        ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_a(uint32_t bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s_a(uint32_t dst, const void* src, unsigned bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_g2s_hint_a(uint32_t dst, const void* src, unsigned bytes, uint32_t bar, uint64_t pol) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(pol) : "memory");
}
__device__ __forceinline__ unsigned lds_u16(uint32_t addr) {
    unsigned short v;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint4 lds_128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ void lds_2x64(uint32_t addr, unsigned long long& a, unsigned long long& b) {
    asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "r"(addr));
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void lds_2f32(uint32_t addr, float& a, float& b) {
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(a), "=f"(b) : "r"(addr));
}
__device__ __forceinline__ void sts_64(uint32_t addr, unsigned long long v) {
    asm volatile("st.shared.b64 [%0], %1;" ::"r"(addr), "l"(v) : "memory");
}

// per-lane partial byte sums (I in the low half, Q in the high half) of this lane's 32 bytes of a segment
__device__ __forceinline__ void lane_byte_sums(uint32_t addr, unsigned& sI, unsigned& sQ) {
    const uint4 q0 = lds_128(addr), q1 = lds_128(addr + 256);
    sI = __dp4a(q0.x, 0x00010001u, 0u); sQ = __dp4a(q0.x, 0x01000100u, 0u);
    sI = __dp4a(q0.y, 0x00010001u, sI); sQ = __dp4a(q0.y, 0x01000100u, sQ);
    sI = __dp4a(q0.z, 0x00010001u, sI); sQ = __dp4a(q0.z, 0x01000100u, sQ);
    sI = __dp4a(q0.w, 0x00010001u, sI); sQ = __dp4a(q0.w, 0x01000100u, sQ);
    sI = __dp4a(q1.x, 0x00010001u, sI); sQ = __dp4a(q1.x, 0x01000100u, sQ);
    sI = __dp4a(q1.y, 0x00010001u, sI); sQ = __dp4a(q1.y, 0x01000100u, sQ);
    sI = __dp4a(q1.z, 0x00010001u, sI); sQ = __dp4a(q1.z, 0x01000100u, sQ);
    sI = __dp4a(q1.w, 0x00010001u, sI); sQ = __dp4a(q1.w, 0x01000100u, sQ);
}

// the same sums on the ALU pipe (LOP3 / PRMT field extraction + IADD3) instead of 16 dp4a, which cost two FMA-pipe
// slots each: the kernel is FMA-pipe bound and its ALU pipe is 20 % busy
__device__ __forceinline__ void lane_byte_sums_alu(uint32_t addr, unsigned& sI, unsigned& sQ) {
    const uint4 q0 = lds_128(addr), q1 = lds_128(addr + 256);
    const unsigned m = 0x00ff00ffu;
    // 16-bit fields (even sample | odd sample << 16); eight words of <= 255 each stay below 2^16
    const unsigned aI = (q0.x & m) + (q0.y & m) + (q0.z & m);
    const unsigned bI = (q0.w & m) + (q1.x & m) + (q1.y & m);
    const unsigned cI = (q1.z & m) + (q1.w & m);
    const unsigned aQ = __byte_perm(q0.x, 0, 0x4341) + __byte_perm(q0.y, 0, 0x4341) + __byte_perm(q0.z, 0, 0x4341);
    const unsigned bQ = __byte_perm(q0.w, 0, 0x4341) + __byte_perm(q1.x, 0, 0x4341) + __byte_perm(q1.y, 0, 0x4341);
    const unsigned cQ = __byte_perm(q1.z, 0, 0x4341) + __byte_perm(q1.w, 0, 0x4341);
    const unsigned tI = aI + bI + cI, tQ = aQ + bQ + cQ;
    sI = (tI & 0xffffu) + (tI >> 16);
    sQ = (tQ & 0xffffu) + (tQ >> 16);
}

// T64: time-blocked S layout [t / 64][position / 8][t % 64][position % 8] instead of [t][position]: the 64 time steps of a group
// of 8 row positions are 2 KB of contiguous memory, so the scan kernels' walks along time read consecutive sectors (whole
// 128-byte lines, open DRAM rows) instead of one sector out of every 1 KB row.
// TG (time group, 1 / 2 / 4 / 8): S layout [t / TG][position / 4][t % TG][position % 4] -- the 16-byte granule (4 bins) of TG consecutive
// time steps lie side by side, so a walk along time (the extraction kernel) finds 2 cells per 32-byte sector at TG = 2, 4 per 64
// bytes at TG = 4, 8 per 128-byte line at TG = 8 instead of one sector per cell.  TG = 2 costs this kernel nothing: the two half-warps
// of a warp hold time steps t and t + 1, and a store instruction of the warp is 512 contiguous bytes.  TG > 2 deals groups of TG
// consecutive segments to a warp (TG / 2 rounds per group) so that the sectors of a group are completed by one warp within microseconds.
template <bool STORE, bool HINT, bool TWS, bool WINS, bool ALUSUM, bool PROBE = false, int T64 = 0, bool PIN = false, bool PACC = false, class C = R256v7, int TG = 1>
__device__ __forceinline__ void spectro_reg256_v7_body(const SpectroArgs& a) {
    static_assert(TG == 1 || TG == 2 || TG == 4 || TG == 8, "time group");
    static_assert(TG == 1 || (!PROBE && T64 == 0), "probe plane / time-blocked lab layouts are TG = 1 only");
    constexpr int RPG = TG > 2 ? TG / 2 : 1;              // rounds per group of TG segments
    constexpr int GSEGS = C::WARPS * (TG > 2 ? TG : 2);    // segments the CTA covers per RPG rounds
    // segment (of half-warp 0) of round `it` of this warp, relative to its first one
    auto seg_rel = [](int it) { return TG > 2 ? (it / RPG) * GSEGS + 2 * (it % RPG) : it * C::SEGS_PER_ROUND; };
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int h = C::LMAP ? (lane >> 2) & 1 : lane >> 4;                              // which of the warp's two segments
    const int j = C::LMAP ? (lane & 3) | ((lane >> 3) << 2) : lane & 15;              // thread of the 16 x 16 FFT
    const int hwi = 2 * (tid >> 5) + h;                                               // segment slot of the CTA
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);          // warp-uniform for the compiler
    const int s = blockIdx.y;
    const int seg0 = blockIdx.x * a.chunk_segs;
    const int seg1 = min(a.T, seg0 + a.chunk_segs);
    const int first = seg0 + (TG > 2 ? TG : 2) * warp;
    int n_it;                                                                        // warp-uniform
    if (TG > 2) {
        const int R = seg1 - 1 - first;                   // rounds whose first segment exists
        n_it = R < 0 ? 0 : (R / GSEGS) * RPG + min(RPG, (R % GSEGS) / 2 + 1);
    } else {
        n_it = (seg1 - first + C::SEGS_PER_ROUND - 1) / C::SEGS_PER_ROUND;
    }

    const uint32_t sm0 = smem_u32(dyn_smem);
    const uint32_t wraw = sm0 + warp * (C::STAGES * C::STAGE_BYTES);
    const uint32_t wbar = sm0 + C::BAR_OFF + warp * (C::STAGES * 8);
    const uint32_t xt = sm0 + C::RAW_BYTES + hwi * (C::XTILE * 4);
    const uint32_t my_u16 = wraw + h * C::RAW_STRIDE + 2 * j;        // + stage offset + 32*n1
    const uint32_t my_sum = wraw + h * C::RAW_STRIDE + 16 * j;       // + stage offset (+256)
    uint32_t xt_st = xt + 8 * j;                                      // + k1 * XROW * 4
    uint32_t xt_ld = xt + j * (C::XROW * 4);                          // + 16 * c
    uint32_t my_u16_ = my_u16, my_sum_ = my_sum;
    if (PIN) {
        // opaque to the compiler: without this ptxas re-derives these four addresses from SR_TID.X in every round
        // (S2R -> SHF -> IMAD -> IADD3 in front of the round's first LDS)
        asm volatile("" : "+r"(my_u16_), "+r"(my_sum_), "+r"(xt_st), "+r"(xt_ld));
    }
    int h16 = 16 * h;                                                 // shift of this half-warp's field in the REDUX sums
    if (PIN) asm volatile("" : "+r"(h16));
    // global source of the segment pair of round `it`: base + (first + 8*it) * 512
    const uint8_t* gsrc = a.unit_base(s) + (size_t)first * 512;
    const int last_seg = seg1 - 1;

    uint64_t pol_in = 0, pol_out = 0;
    if (HINT) { pol_in = policy_evict_first(); pol_out = PIN ? policy_evict_first() : policy_evict_last(); }   // v7h (HINT + PIN): S stores evict-first (streaming)
    auto issue = [&](int itx, int st) {                              // executed by one elected lane
        const int sg = first + seg_rel(itx);
        const uint8_t* p0 = gsrc + (size_t)seg_rel(itx) * 512;
        const uint8_t* p1 = (sg + 1 <= last_seg) ? p0 + 512 : p0;   // ragged tail: copy the same segment twice
        const uint32_t bar = wbar + 8 * st, dst = wraw + st * C::STAGE_BYTES;
        mbar_expect_tx_a(bar, 1024);
        if (HINT) {
            bulk_g2s_hint_a(dst, p0, 512, bar, pol_in);
            bulk_g2s_hint_a(dst + C::RAW_STRIDE, p1, 512, bar, pol_in);
        } else {
            bulk_g2s_a(dst, p0, 512, bar);
            bulk_g2s_a(dst + C::RAW_STRIDE, p1, 512, bar);
        }
    };

    if (elect_one()) {
#pragma unroll
        for (int st = 0; st < C::STAGES; ++st)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(wbar + 8 * st) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#pragma unroll
        for (int st = 0; st < C::STAGES; ++st)
            if (st < n_it) issue(st, st);
    }

    // per-thread constants: window at samples 16*n1 + j, inter-pass twiddles W256^{j*k1}
    // (in registers, or -- TWS / WINS -- in a shared-memory table to buy a fifth / sixth resident CTA)
    float wj[16], twr[16], twi[16], acc[16];
    cpk acc2[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) acc2[c] = c_make(0.f, 0.f);
    const uint32_t tab_tw = sm0 + C::TAB_OFF + 8 * j, tab_win = sm0 + C::TAB_OFF + 2048 + 4 * j;
    if (TWS || WINS) {
        float2* ttw = reinterpret_cast<float2*>(dyn_smem + C::TAB_OFF);
        float* twin = reinterpret_cast<float*>(dyn_smem + C::TAB_OFF + 2048);
        for (int i = tid; i < 256; i += C::THREADS) {
            ttw[i] = a.tw[((i & 15) * (i >> 4)) & 255];      // [k1][j]
            twin[i] = a.win[i];                              // [n1][j]
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        wj[i] = a.win[16 * i + j];
        const float2 t = a.tw[(j * i) & 255];
        twr[i] = t.x;
        twi[i] = t.y;
        acc[i] = 0.f;
    }
    __syncwarp();                                   // barriers initialised before anyone polls them

    // segment byte sums -> detrend constant (32768 + mean_I, 32768 + mean_Q), exact in fp32
    auto detrend_of = [&](uint32_t addr) {
        unsigned sI, sQ;
        if (ALUSUM) lane_byte_sums_alu(addr, sI, sQ);
        else lane_byte_sums(addr, sI, sQ);
        // warp-wide REDUX: half-warp 0 in the low 16 bits, half-warp 1 in the high 16 (each total < 2^16)
        const unsigned tI = __reduce_add_sync(0xffffffffu, sI << h16);
        const unsigned tQ = __reduce_add_sync(0xffffffffu, sQ << h16);
        const unsigned mI = (tI >> h16) & 0xffffu, mQ = (tQ >> h16) & 0xffffu;
        return c_scale(c_make(__uint_as_float(0x4B000000u | mI), __uint_as_float(0x4B000000u | mQ)), 0.00390625f);
    };

    cpk cm = c_make(0.f, 0.f);
    if (n_it > 0) {
        mbar_wait(wbar, 0);
        cm = detrend_of(my_sum_);
    }
    // TG = 1: row (first + h), 4 j floats in; TG = 2: row pair first / 2 (first is even), granule j of 8 floats, half h of it
    float* sdst = a.S + (size_t)s * a.S_stream_stride + (TG == 2 ? (size_t)first * 256 + 8 * j + 4 * h : (size_t)(first + h) * 256 + 4 * j);   // += 8 * 256 floats per round
    float* const sbaseTG = a.S + (size_t)s * a.S_stream_stride + (4 * TG) * j;                // TG > 2: + (seg / TG) * 256 TG + (seg % TG) * 4
    // T64 = positions per block (8 or 32): [t / 64][pos / T64][t % 64][pos % T64]; this thread's positions are 64 c + 4 j ...
    float* const sbase64 = a.S + (size_t)s * a.S_stream_stride + (T64 ? ((4 * j) / (T64 ? T64 : 1)) * (64 * T64) + (4 * j) % (T64 ? T64 : 1) : 0);
    uint32_t st_off = 0, st_bar = wbar;
    unsigned phase = 0;
    const uint8_t* g_next = gsrc + (size_t)seg_rel(C::STAGES) * 512;               // source of the next round to be issued
    int sg_next = first + seg_rel(C::STAGES);
    int seg = first + h;
    // probe plane: seg = pq * probe_stride + prem, kept incrementally (seg advances by SEGS_PER_ROUND per round)
    int pq = 0, prem = 0;
    if (PROBE) { pq = seg / a.probe_stride; prem = seg - pq * a.probe_stride; }

    for (int it = 0; it < n_it; ++it) {
        // uint8 -> float (0x4700bb00 is 32768 + b, no I2F), detrend (scipy detrend='constant'); window folded below
        cpk v[16];
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) {
            const unsigned u = lds_u16(my_u16_ + st_off + 32 * n1);
            const cpk f = c_make(__uint_as_float(__byte_perm(u, 0x47000000u, 0x7604)),
                                 __uint_as_float(__byte_perm(u, 0x47000000u, 0x7614)));
            v[n1] = c_sub(f, cm);
        }
        // this stage's bytes are in registers: refill it with the segments STAGES rounds ahead
        __syncwarp();
        if (it + C::STAGES < n_it) {
            if (PIN) {
                // running source pointer / ring slot instead of re-deriving both from the round number (uniform datapath)
                if (elect_one()) {
                    const uint8_t* p1 = (sg_next + 1 <= last_seg) ? g_next + 512 : g_next;
                    mbar_expect_tx_a(st_bar, 1024);
                    bulk_g2s_a(wraw + st_off, g_next, 512, st_bar);
                    bulk_g2s_a(wraw + st_off + C::RAW_STRIDE, p1, 512, st_bar);
                }
            } else if (elect_one()) issue(it + C::STAGES, it % C::STAGES);
        }
        if (TG > 2) {
            const int d = seg_rel(it + C::STAGES + 1) - seg_rel(it + C::STAGES);
            g_next += d * 512;
            sg_next += d;
        } else {
            g_next += C::SEGS_PER_ROUND * 512;
            sg_next += C::SEGS_PER_ROUND;
        }
        // advance to the next stage; its byte sums overlap the butterflies below
        st_off += C::STAGE_BYTES; st_bar += 8;
        if (st_off == C::STAGES * C::STAGE_BYTES) { st_off = 0; st_bar = wbar; phase ^= 1; }
        cpk cm_next = cm;
        if (it + 1 < n_it) {
            mbar_wait(st_bar, phase);
            cm_next = detrend_of(my_sum_ + st_off);
        }

        if (WINS) {
#pragma unroll
            for (int i = 0; i < 16; ++i) wj[i] = lds_f32(tab_win + 64 * i);
        }
        cdft16_win(v, wj);                          // over n1 -> k1, for column n2 = j
        // inter-pass twiddles, then the 16x16 transpose through shared memory
        sts_64(xt_st, v[0].v);
#pragma unroll
        for (int k1 = 1; k1 < 16; ++k1) {
            float wr = twr[k1], wi = twi[k1];
            if (TWS) lds_2f32(tab_tw + 128 * k1, wr, wi);
            sts_64(xt_st + k1 * (C::XROW * 4), c_mul(v[k1], wr, wi).v);
        }
        __syncwarp();
#pragma unroll
        for (int c = 0; c < 8; ++c) lds_2x64(xt_ld + 16 * c, v[2 * c].v, v[2 * c + 1].v);
        // (the tile is rewritten only after the next round's __syncwarp)
        cdft16(v);                                  // over n2 -> k2, for k1 = j: bin = j + 16*k2
        const bool valid = seg <= last_seg;
        const float m = valid ? 1.f : 0.f;
        float p[16];
#pragma unroll
        for (int k2 = 0; k2 < 16; ++k2) {
            const float re = c_re(v[k2]), im = c_im(v[k2]);
            p[k2] = fmaf(im, im, re * re);
            if (!PACC) acc[k2] = fmaf(p[k2], m, acc[k2]);
        }
        if (PACC) {                                 // row sums as 8 packed FMAs instead of 16 scalar ones (same lanes, half the issue slots)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc2[c] = c_fma_s(c_make(p[2 * c], p[2 * c + 1]), m, acc2[c]);
        }
        if (STORE) {
            if (valid) {
                float4* dst = T64 ? reinterpret_cast<float4*>(sbase64 + ((size_t)(seg >> 6) << 14) + (seg & 63) * T64)
                            : TG > 2 ? reinterpret_cast<float4*>(sbaseTG + (size_t)(seg / TG) * (256 * TG) + (seg % TG) * 4)
                                     : reinterpret_cast<float4*>(sdst);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float4 o = make_float4(p[4 * c], p[4 * c + 1], p[4 * c + 2], p[4 * c + 3]);
                    if (HINT) stg128_hint(dst + 16 * c, o, pol_out);
                    else dst[(T64 ? 1024 : 16 * TG) * c] = o;     // 64 positions further (T64: 64 * 64 floats in either blocked layout)
                }
            }
            sdst += C::SEGS_PER_ROUND * 256;
            if (PROBE) {
                if (valid && prem == 0) {
                    float4* dst = reinterpret_cast<float4*>(a.probe + ((size_t)s * a.n_probes + pq) * 256 + 4 * j);
#pragma unroll
                    for (int c = 0; c < 4; ++c) dst[16 * c] = make_float4(p[4 * c], p[4 * c + 1], p[4 * c + 2], p[4 * c + 3]);
                }
                prem += C::SEGS_PER_ROUND;
                while (prem >= a.probe_stride) { prem -= a.probe_stride; ++pq; }
            }
        }
        seg += TG > 2 ? seg_rel(it + 1) - seg_rel(it) : C::SEGS_PER_ROUND;
        cm = cm_next;
    }

    // chunk row sums: fixed-order reduction over the half-warps, written in FFT bin order (fi = j + 16*k2)
    __syncthreads();
    float* red = reinterpret_cast<float*>(dyn_smem);
    const int hw = hwi;
#pragma unroll
    for (int k2 = 0; k2 < 16; ++k2) red[hw * 256 + 16 * k2 + j] = PACC ? ((k2 & 1) ? c_im(acc2[k2 >> 1]) : c_re(acc2[k2 >> 1])) : acc[k2];
    __syncthreads();
    // written in the order of the S rows (PERM position, see rt_engine.cu) so that the probe kernel reads both coalesced
    float* pd = a.part + ((size_t)s * a.n_chunks + blockIdx.x) * 256;
    for (int fi = tid; fi < 256; fi += C::THREADS) {
        float t = 0.f;
#pragma unroll
        for (int hh = 0; hh < 2 * C::WARPS; ++hh) t += red[hh * 256 + fi];
        pd[((fi >> 6) << 6) | ((fi & 15) << 2) | ((fi >> 4) & 3)] = t;
    }
}

// addresses pinned in registers (see PIN in spectro_reg256_v7_body)
template <bool STORE, int TG = 1, bool LMAP = false>
__global__ void __launch_bounds__(R256v7::THREADS, 4) spectro_reg256_v7n(SpectroArgs a) {
    spectro_reg256_v7_body<STORE, false, false, false, false, false, 0, true, false, R256v7T<4, 4, LMAP>, TG>(a);
}


// ---------------------------------------------------------------------------------------------
// v8 (round 2, session 3) -- the engine's nperseg-256 kernel.  The data flow of v7n (LMAP lane mapping, TG = 1 | 2 time grouping of
// S, pinned addresses, running TMA source pointer) with a cheaper front end:
//   * bytes -> fp16 pair with ONE PRMT per complex sample (0x6400 | b = 1024 + b in fp16, I in the low half, Q in the high half);
//     the mixed-precision add of sm_100 (PTX add.rn.f32.f16, SASS FHADD: one FMA-pipe cycle, tools/ubench_mix3.cu) widens to fp32
//     and subtracts 1024 + mean in one instruction per component -- bit for bit the value v7n's PRMT x 2 + FADD2 produced
//     (b - sum / 256 is exact in fp32);
//   * the segment's byte sums come from those 16 packed words the thread already holds: eight 3-input integer adds give
//     sum(I) + 65536 sum(Q) of the thread's samples, one REDUX per segment of the warp adds the 16 threads -- instead of a second pass
//     over the raw bytes (2 LDS.128 + 16 dp4a, which are two FMA-pipe cycles each, + 2 REDUX and the field shifts).
// S and the row sums are bit-identical to v7n's; 112 registers; back to back 170 -> 161 us at configs[1] (153 us without the S stores).
// Measured and dropped (profiles/r02_v8_lab.txt): loads / sums of round it + 1 issued at the end of round it (128 registers, 165 us),
// a tree instead of a chain of integer adds, the PRMT constant pinned in a register, packed row-sum FMAs, L2 eviction hints on the
// TMA loads and / or the S stores -- all within +-0.5 us; integer detrend + I2F (a non-FMA pipe) instead of FHADD: 32 FMA-pipe cycles
// less but 56 instructions more per round, 168 us -- issue slots and the FMA pipe bind together.
// ---------------------------------------------------------------------------------------------
template <bool STORE, int TG, bool CI8 = false, class C = R256v7T<4, 4, true>>
__device__ __forceinline__ void spectro_reg256_v8_body(const SpectroArgs& a) {
    static_assert(TG == 1 || TG == 2, "time group");
    static_assert(C::LMAP, "v8 uses the LMAP lane mapping");
    extern __shared__ __align__(16) unsigned char dyn_smem[];
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int h = (lane >> 2) & 1;                                    // which of the warp's two segments
    const int j = (lane & 3) | ((lane >> 3) << 2);                    // thread of the 16 x 16 FFT
    const int hwi = 2 * (tid >> 5) + h;                               // segment slot of the CTA
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);          // warp-uniform for the compiler
    const int s = blockIdx.y;
    const int seg0 = blockIdx.x * a.chunk_segs;
    const int seg1 = min(a.T, seg0 + a.chunk_segs);
    const int first = seg0 + 2 * warp;
    const int n_it = (seg1 - first + C::SEGS_PER_ROUND - 1) / C::SEGS_PER_ROUND;   // warp-uniform

    const uint32_t sm0 = smem_u32(dyn_smem);
    const uint32_t wraw = sm0 + warp * (C::STAGES * C::STAGE_BYTES);
    const uint32_t wbar = sm0 + C::BAR_OFF + warp * (C::STAGES * 8);
    const uint32_t xt = sm0 + C::RAW_BYTES + hwi * (C::XTILE * 4);
    uint32_t my_u16 = wraw + h * C::RAW_STRIDE + 2 * j;               // + stage offset + 32 * n1
    uint32_t xt_st = xt + 8 * j;                                      // + k1 * XROW * 4
    uint32_t xt_ld = xt + j * (C::XROW * 4);                          // + 16 * c
    int hsel = h;
    asm volatile("" : "+r"(my_u16), "+r"(xt_st), "+r"(xt_ld), "+r"(hsel));   // opaque: ptxas otherwise re-derives them from SR_TID.X every round
    const uint8_t* gsrc = a.unit_base(s) + (size_t)first * 512;     // segment pair of round it: + it * SEGS_PER_ROUND * 512
    const int last_seg = seg1 - 1;

    if (elect_one()) {
#pragma unroll
        for (int st = 0; st < C::STAGES; ++st)
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(wbar + 8 * st) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#pragma unroll
        for (int st = 0; st < C::STAGES; ++st)
            if (st < n_it) {
                const uint8_t* p0 = gsrc + (size_t)st * (C::SEGS_PER_ROUND * 512);
                const uint8_t* p1 = (first + st * C::SEGS_PER_ROUND + 1 <= last_seg) ? p0 + 512 : p0;   // ragged tail: the same segment twice
                const uint32_t bar = wbar + 8 * st, dst = wraw + st * C::STAGE_BYTES;
                mbar_expect_tx_a(bar, 1024);
                bulk_g2s_a(dst, p0, 512, bar);
                bulk_g2s_a(dst + C::RAW_STRIDE, p1, 512, bar);
            }
    }

    // per-thread constants: window at samples 16 * n1 + j, inter-pass twiddles W256^{j * k1}
    float wj[16], twr[16], twi[16], acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        wj[i] = a.win[16 * i + j];
        const float2 t = a.tw[(j * i) & 255];
        twr[i] = t.x;
        twi[i] = t.y;
        acc[i] = 0.f;
    }
    __syncwarp();                                   // barriers initialised before anyone polls them

    if (n_it > 0) mbar_wait(wbar, 0);
    // TG = 1: row (first + h), floats 4 j ...; TG = 2: row pair first / 2 (first is even), granule j of 8 floats, half h of it
    float* sdst = a.S + (size_t)s * a.S_stream_stride + (TG == 2 ? (size_t)first * 256 + 8 * j + 4 * h : (size_t)(first + h) * 256 + 4 * j);   // += 8 * 256 floats per round
    uint32_t st_off = 0, st_bar = wbar;
    unsigned phase = 0;
    const uint8_t* g_next = gsrc + (size_t)C::STAGES * (C::SEGS_PER_ROUND * 512);   // source of the next round to be issued
    int sg_next = first + C::STAGES * C::SEGS_PER_ROUND;
    int seg = first + h;

    for (int it = 0; it < n_it; ++it) {
        // this thread's 16 samples as fp16 pairs (1024 + I) | (1024 + Q) << 16, and the segment's byte sums from the same words
        // (ci8: one LOP3 per sample turns the int8 pair into the cu8 pair v + 128, sample_format.cuh)
        unsigned hv[16];
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) hv[n1] = __byte_perm(lds_u16(my_u16 + st_off + 32 * n1) ^ (CI8 ? 0x8080u : 0u), 0x64646464u, 0x5140);
        unsigned t = 0;
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) t += hv[n1];
        t -= 0x40064000u;                           // 16 x 0x64006400 mod 2^32: t = sum I + 65536 sum Q over this thread's 16 samples
        const unsigned r0 = __reduce_add_sync(0xffffffffu, hsel ? 0u : t), r1 = __reduce_add_sync(0xffffffffu, hsel ? t : 0u);
        const unsigned tot = hsel ? r1 : r0;        // the segment's byte sums (each < 2^16)
        // (2^23 + sum) * -2^-8 + 31744 = -(1024 + sum / 256), exact: scipy's detrend='constant' on the raw bytes
        const cpk nc = c_fma_s(c_make(__uint_as_float(0x4B000000u | (tot & 0xffffu)), __uint_as_float(0x4B000000u | (tot >> 16))), -0.00390625f, c_make(31744.f, 31744.f));
        const float ncI = c_re(nc), ncQ = c_im(nc);
        cpk v[16];
#pragma unroll
        for (int n1 = 0; n1 < 16; ++n1) {
            float re, im;
            asm("add.rn.f32.f16 %0, %1, %2;" : "=f"(re) : "h"((unsigned short)(hv[n1] & 0xffffu)), "f"(ncI));
            asm("add.rn.f32.f16 %0, %1, %2;" : "=f"(im) : "h"((unsigned short)(hv[n1] >> 16)), "f"(ncQ));
            v[n1] = c_make(re, im);
        }
        // this stage's bytes are in registers: refill it with the segments STAGES rounds ahead
        __syncwarp();
        if (it + C::STAGES < n_it) {
            if (elect_one()) {
                const uint8_t* p1 = (sg_next + 1 <= last_seg) ? g_next + 512 : g_next;
                mbar_expect_tx_a(st_bar, 1024);
                bulk_g2s_a(wraw + st_off, g_next, 512, st_bar);
                bulk_g2s_a(wraw + st_off + C::RAW_STRIDE, p1, 512, st_bar);
            }
        }
        g_next += C::SEGS_PER_ROUND * 512;
        sg_next += C::SEGS_PER_ROUND;
        st_off += C::STAGE_BYTES; st_bar += 8;
        if (st_off == C::STAGES * C::STAGE_BYTES) { st_off = 0; st_bar = wbar; phase ^= 1; }
        if (it + 1 < n_it) mbar_wait(st_bar, phase);                 // (rarely blocks: the copy was issued three rounds ago)

        cdft16_win(v, wj);                          // over n1 -> k1, for column n2 = j
        // inter-pass twiddles, then the 16 x 16 transpose through shared memory
        sts_64(xt_st, v[0].v);
#pragma unroll
        for (int k1 = 1; k1 < 16; ++k1) sts_64(xt_st + k1 * (C::XROW * 4), c_mul(v[k1], twr[k1], twi[k1]).v);
        __syncwarp();
#pragma unroll
        for (int c = 0; c < 8; ++c) lds_2x64(xt_ld + 16 * c, v[2 * c].v, v[2 * c + 1].v);
        // (the tile is rewritten only after the next round's __syncwarp)
        cdft16(v);                                  // over n2 -> k2, for k1 = j: bin = j + 16 * k2
        const bool valid = seg <= last_seg;
        const float m = valid ? 1.f : 0.f;
        float p[16];
#pragma unroll
        for (int k2 = 0; k2 < 16; ++k2) {
            const float re = c_re(v[k2]), im = c_im(v[k2]);
            p[k2] = fmaf(im, im, re * re);
            acc[k2] = fmaf(p[k2], m, acc[k2]);
        }
        if (STORE) {
            if (valid) {
                float4* dst = reinterpret_cast<float4*>(sdst);
#pragma unroll
                for (int c = 0; c < 4; ++c) dst[16 * TG * c] = make_float4(p[4 * c], p[4 * c + 1], p[4 * c + 2], p[4 * c + 3]);   // 64 positions further
            }
            sdst += C::SEGS_PER_ROUND * 256;
        }
        seg += C::SEGS_PER_ROUND;
    }

    // chunk row sums: fixed-order reduction over the CTA's segment slots, written in the order of the S rows (PERM position)
    __syncthreads();
    float* red = reinterpret_cast<float*>(dyn_smem);
#pragma unroll
    for (int k2 = 0; k2 < 16; ++k2) red[hwi * 256 + 16 * k2 + j] = acc[k2];
    __syncthreads();
    float* pd = a.part + ((size_t)s * a.n_chunks + blockIdx.x) * 256;
    for (int fi = tid; fi < 256; fi += C::THREADS) {
        float t = 0.f;
#pragma unroll
        for (int hh = 0; hh < 2 * C::WARPS; ++hh) t += red[hh * 256 + fi];
        pd[((fi >> 6) << 6) | ((fi & 15) << 2) | ((fi >> 4) & 3)] = t;
    }
}

template <bool STORE, int TG = 2, bool CI8 = false>
__global__ void __launch_bounds__(R256v7::THREADS, 4) spectro_reg256_v8(SpectroArgs a) {
    spectro_reg256_v8_body<STORE, TG, CI8>(a);
}

}  // namespace rt
