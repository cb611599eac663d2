// spectro_r16.cuh -- uint8 IQ -> power spectrogram cells + per-chunk row sums for nperseg 1024 and 4096 (sm_100a):
// BASELINE.json configs[2], the wideband single stream.
//
// Replaces scipy.signal.spectrogram(..., nperseg=N, noverlap=0, return_onesided=False) as called at
// /root/reference/radiotracking/analyze.py:234-241 (detrend='constant', window, FFT, |X|^2 / (fs * sum w^2)).
//
// Self-sorting (Stockham, decimation in frequency) FFT with radix-16 passes: a team of N/16 threads owns one segment,
// every thread runs one packed-complex DFT16 (fft_cpk.cuh, 72 FFMA2-class instructions) per pass and the passes
// exchange through ONE padded shared-memory buffer (read 16 values -> barrier -> write 16 values):
//     N = 4096 = 16 * 16 * 16   three radix-16 passes, team = 256 threads = the CTA
//     N = 1024 = 16 * 16 * 4    two radix-16 passes + one radix-4 pass, team = 64 threads, four segments per CTA
// The first pass takes its inputs straight from the TMA-staged raw bytes (no initial shared-memory write) and the
// last pass leaves thread b with the bins b + (N/R) i in registers (no final write): |X|^2, row sums and the
// coalesced stores to S[stream][t][bin] (LINEAR layout) follow directly.
// Raw segments arrive through a two-deep ring of TMA bulk copies per team (cp.async.bulk + mbarrier).
//
// Round 2 (ncu: profiles/r02_r16_*.ncu_summary.txt -- 807 instructions per thread and segment, a quarter of them index
// arithmetic; 2.2-way bank conflicts on the twiddle loads; top stall short_scoreboard on the twiddle multiplies):
//   * every shared-memory address of a thread is one of five per-thread bases plus a COMPILE-TIME offset (the padded
//     exchange indices are affine in the unrolled loop index), held as 32-bit shared addresses;
//   * the pass twiddles live in per-pass tables laid out [i][thread] (pass 1) and [i][thread / 16] (pass 2): consecutive
//     lanes read consecutive 8-byte entries (no bank conflicts) instead of gathering W_N^{b i} out of one table of N entries;
//   * the window is folded into the first butterfly layer (cdft16_win); byte -> float: one PRMT per sample (fp16 pair) + two FHADD;
//   * the segment's byte sums go through per-warp slots (double-buffered) instead of shared-memory atomics: one team
//     barrier less per segment and no reset.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "spectro256.cuh"

namespace rt {

template <int N>
struct R16Cfg {
    static_assert(N == 1024 || N == 4096, "radix-16 Stockham kernel: nperseg 1024 or 4096");
    static constexpr int THREADS = 256;
    static constexpr int BT = N / 16;                       // threads per team = radix-16 butterflies per pass
    static constexpr int TEAMS = THREADS / BT;              // segments in flight per CTA
    static constexpr int TW = BT / 32;                      // warps per team
    static constexpr int LAST_R = N == 4096 ? 16 : 4;       // radix of the last pass
    static constexpr int PADN = N + N / 16;                 // float2 entries of one exchange buffer (index + index/16)
    // Measured variants (profiles/r02_r16_variants.txt): N = 1024 runs best with THREE CTAs per SM (84 registers, 16 bytes of
    // spills, 60 KB of shared memory each; step 81.0 -> 72.5 us: eight more independent teams per SM hide the exchange
    // latencies, and the scan kernels of the previous launch find room beside them); N = 4096 (84 KB per CTA) stays at two.
    // Keeping the pass-1 twiddles in registers instead (128 registers, no table loads) did not pay: 77.5 / 86.6 us.
    static constexpr int CTAS_PER_SM = N == 1024 ? 3 : 2;
    static constexpr int MAXR = N == 1024 ? 84 : 104;
    static constexpr int OFF_TW1 = 0;                       // float2[15][BT]      W_N^{b i},       i = 1..15
    static constexpr int OFF_TW2 = OFF_TW1 + 15 * BT * 8;   // float2[15][BT/16]   W_N^{16 p i},    i = 1..15
    static constexpr int OFF_X = OFF_TW2 + 15 * (BT / 16) * 8;           // [TEAMS][PADN] float2 (16-byte aligned)
    static constexpr int OFF_RAW = OFF_X + TEAMS * PADN * 8;             // [TEAMS][2][2N] bytes
    static constexpr int OFF_SUM = OFF_RAW + TEAMS * 2 * 2 * N;          // [TEAMS][2][TW] uint2 (sum I, sum Q) per warp
    static constexpr int OFF_BAR = OFF_SUM + TEAMS * 2 * TW * 8;         // [TEAMS][2] mbarrier
    static constexpr int SMEM = OFF_BAR + TEAMS * 16;
    static_assert(OFF_X % 16 == 0 && OFF_RAW % 16 == 0 && OFF_SUM % 16 == 0 && OFF_BAR % 8 == 0, "alignment");
};

__device__ __forceinline__ int r16_pad(int idx) { return idx + (idx >> 4); }

__device__ __forceinline__ cpk r16_lds(uint32_t addr) {
    cpk v;
    asm volatile("ld.shared.b64 %0, [%1];" : "=l"(v.v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void r16_lds_tw(uint32_t addr, float& wr, float& wi) {
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(wr), "=f"(wi) : "r"(addr));
}

// CI8: int8 input, taken as cu8 with the top bit of every byte flipped (sample_format.cuh)
template <int N, bool CI8 = false>
__global__ void __maxnreg__(R16Cfg<N>::MAXR) spectro_r16_k(SpectroArgs a) {
    using C = R16Cfg<N>;
    constexpr int BT = C::BT, M1 = N / 16, M2 = N / 256;
    extern __shared__ __align__(16) unsigned char r16_smem[];
    const int tid = threadIdx.x, lane = tid & 31;
    const int team = tid / BT, b = tid % BT;                  // b = butterfly index of this thread in every radix-16 pass
    const int wt = b >> 5;                                    // warp of the team
    const uint32_t sm0 = smem_u32(r16_smem);
    const uint32_t xb = sm0 + C::OFF_X + team * (C::PADN * 8);
    const uint32_t rawb = sm0 + C::OFF_RAW + team * (4 * N);
    const uint32_t sumb = sm0 + C::OFF_SUM + team * (2 * C::TW * 8);
    const uint32_t bar0 = sm0 + C::OFF_BAR + team * 16;

    const int s = blockIdx.y;
    const uint8_t* base = a.unit_base(s);
    // segments are dealt round-robin over the (CTA, team) pairs of the stream: one twiddle-table load per CTA,
    // balanced work for any T; this team's segments: first, first + step, ...
    const int step = a.n_chunks * C::TEAMS;
    const int first = blockIdx.x * C::TEAMS + team;
    const int seg1 = a.T;
    const int n_it = first < seg1 ? (seg1 - first + step - 1) / step : 0;

    {   // per-pass twiddle tables, [i][thread] and [i][thread / 16]: conflict-free reads
        float2* tw1 = reinterpret_cast<float2*>(r16_smem + C::OFF_TW1);
        float2* tw2 = reinterpret_cast<float2*>(r16_smem + C::OFF_TW2);
        for (int e = tid; e < 15 * BT; e += C::THREADS) tw1[e] = a.tw1[e];     // [i - 1][b], prepared by the engine
        for (int e = tid; e < 15 * (BT / 16); e += C::THREADS) {
            const int i = e / (BT / 16) + 1, p = e % (BT / 16);
            tw2[e] = a.tw[(16 * p * i) & (N - 1)];
        }
    }
    if (b == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0) : "memory");
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar0 + 8) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    auto team_sync = [&]() { asm volatile("bar.sync %0, %1;" ::"r"(1 + team), "r"(BT) : "memory"); };
    auto issue = [&](int it) {                                // one thread of the team: TMA copy of segment `it` into ring slot it & 1
        const uint32_t bar = bar0 + 8 * (it & 1);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx_a(bar, 2 * N);
        bulk_g2s_a(rawb + (it & 1) * 2 * N, base + (size_t)(first + it * step) * (2 * N), 2 * N, bar);
    };
    if (b == 0 && n_it > 0) issue(0);

    // per-thread shared-memory bases; everything else is a compile-time offset
    const int p2 = b >> 4, q2 = b & 15;
    uint32_t a_raw = rawb + 2 * b;                            // first-pass sample i: + i * (2 M1)   (+ ring slot)
    uint32_t a_st1 = xb + 8 * (17 * b);                       // pass 1 store i:  pad(16 b + i)            = 17 b + i
    uint32_t a_ld2 = xb + 8 * (q2 + 17 * p2);                 // pass 2 load i:   pad(q + 16 (p + M2 i))   = q + 17 p + 17 M2 i
    uint32_t a_st2 = xb + 8 * (q2 + 272 * p2);                // pass 2 store i:  pad(q + 16 (16 p + i))   = q + 272 p + 17 i
    uint32_t a_ld3 = xb + 8 * (b + (b >> 4));                 // last pass load:  pad(b + 64 u + 256 i)    = b + (b >> 4) + 68 u + 272 i
    uint32_t a_tw1 = sm0 + C::OFF_TW1 + 8 * b;                // + (i - 1) * BT * 8
    uint32_t a_tw2 = sm0 + C::OFF_TW2 + 8 * p2;               // + (i - 1) * (BT / 16) * 8
    // opaque to the compiler, so that they stay in registers instead of being re-derived from SR_TID in every segment
    asm volatile("" : "+r"(a_raw), "+r"(a_st1), "+r"(a_ld2), "+r"(a_st2), "+r"(a_ld3), "+r"(a_tw1), "+r"(a_tw2));

    // window of this thread's 16 first-pass samples (index b + M1 i), constant over the segments
    float wj[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) wj[i] = a.win[b + M1 * i];
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;

    for (int it = 0; it < n_it; ++it) {
        const int seg = first + it * step;
        if (b == 0 && it + 1 < n_it) issue(it + 1);            // slot (it+1)&1 was last read two iterations ago
        mbar_wait(bar0 + 8 * (it & 1), (it >> 1) & 1);
        const uint32_t rb = a_raw + (it & 1) * (2 * N);
        const uint32_t sb = sumb + (it & 1) * (C::TW * 8);

        // ---- gather the 16 first-pass inputs, byte sums for the detrend (exact integers)
        // (like spectro_reg256_v8) one PRMT per sample builds the fp16 pair (1024 + I) | (1024 + Q) << 16; the integer sum of the 16
        // packed words minus 16 x 0x64006400 is sum I + 65536 sum Q of this thread's samples
        unsigned u[16];
        unsigned packed = 0;
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            u[i] = __byte_perm(lds_u16(rb + i * (2 * M1)) ^ (CI8 ? 0x8080u : 0u), 0x64646464u, 0x5140);
            packed += u[i];
        }
        packed -= 0x40064000u;                                 // I in the low half, Q in the high half (each <= 16 * 255)
        const unsigned sI = __reduce_add_sync(0xffffffffu, packed & 0xffffu);
        const unsigned sQ = __reduce_add_sync(0xffffffffu, packed >> 16);
        if (lane == 0) asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(sb + 8 * wt), "r"(sI), "r"(sQ) : "memory");
        team_sync();
        unsigned tI = 0, tQ = 0;
#pragma unroll
        for (int w2 = 0; w2 < C::TW; w2 += 2) {                // every thread adds the team's per-warp sums (broadcast reads)
            const uint4 q = lds_128(sb + 8 * w2);
            tI += q.x + q.z;
            tQ += q.y + q.w;
        }
        // mean = sum / N is exact in fp32 (sum < 2^24, N a power of two), so are -(1024 + mean) and (1024 + byte) - (1024 + mean);
        // add.rn.f32.f16 (SASS FHADD) widens the fp16 half and subtracts in one instruction
        const float ncI = fmaf((float)tI, -1.f / N, -1024.f), ncQ = fmaf((float)tQ, -1.f / N, -1024.f);
        cpk v[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            float re, im;
            asm("add.rn.f32.f16 %0, %1, %2;" : "=f"(re) : "h"((unsigned short)(u[i] & 0xffffu)), "f"(ncI));
            asm("add.rn.f32.f16 %0, %1, %2;" : "=f"(im) : "h"((unsigned short)(u[i] >> 16)), "f"(ncQ));
            v[i] = c_make(re, im);
        }

        // ---- pass 1: ncur = N, stride 1: p = b, q = 0; y[16 b + i] = W_N^{b i} DFT16(w x)[i]
        cdft16_win(v, wj);
        sts_64(a_st1, v[0].v);
#pragma unroll
        for (int i = 1; i < 16; ++i) {
            float wr, wi;
            r16_lds_tw(a_tw1 + (i - 1) * (BT * 8), wr, wi);
            sts_64(a_st1 + 8 * i, c_mul(v[i], wr, wi).v);
        }
        team_sync();
        // ---- pass 2: ncur = N/16, stride 16: p = b / 16, q = b % 16
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = r16_lds(a_ld2 + i * (17 * M2 * 8));
        team_sync();
        cdft16(v);
        sts_64(a_st2, v[0].v);
#pragma unroll
        for (int i = 1; i < 16; ++i) {
            float wr, wi;
            r16_lds_tw(a_tw2 + (i - 1) * ((BT / 16) * 8), wr, wi);
            sts_64(a_st2 + i * (17 * 8), c_mul(v[i], wr, wi).v);
        }
        team_sync();
        // ---- last pass: stride N / R, p = 0: X[k = q + (N/R) i] = DFT_R(x[q + (N/R) i])[i]; outputs stay in registers
        const bool valid = seg < seg1;
        float* dst = a.S + (size_t)s * a.S_stream_stride + (size_t)seg * N + b;
        if (N == 4096) {
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = r16_lds(a_ld3 + i * (272 * 8));
            cdft16(v);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float re = c_re(v[i]), im = c_im(v[i]);
                const float pw = fmaf(im, im, re * re);
                acc[i] += pw;
                if (valid) dst[256 * i] = pw;
            }
        } else {
            // 256 radix-4 butterflies per segment, 4 per thread: q = b + 64 u
#pragma unroll
            for (int uu = 0; uu < 4; ++uu) {
                cpk x0 = r16_lds(a_ld3 + uu * (68 * 8)), x1 = r16_lds(a_ld3 + uu * (68 * 8) + 272 * 8);
                cpk x2 = r16_lds(a_ld3 + uu * (68 * 8) + 2 * 272 * 8), x3 = r16_lds(a_ld3 + uu * (68 * 8) + 3 * 272 * 8);
                cdft4(x0, x1, x2, x3);
                const cpk o[4] = {x0, x1, x2, x3};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const float re = c_re(o[i]), im = c_im(o[i]);
                    const float pw = fmaf(im, im, re * re);
                    acc[4 * uu + i] += pw;
                    if (valid) dst[64 * uu + 256 * i] = pw;
                }
            }
        }
        team_sync();                                            // the exchange buffer is rewritten by the next segment's pass 1
    }

    // ---- chunk row sums: teams added in fixed order, written in FFT bin order
    __syncthreads();
    float* red = reinterpret_cast<float*>(r16_smem + C::OFF_X);        // [TEAMS][N]
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const int fi = N == 4096 ? (b + 256 * i) : ((b + 64 * (i >> 2)) + 256 * (i & 3));
        red[team * N + fi] = acc[i];
    }
    __syncthreads();
    float* pd = a.part + ((size_t)s * a.n_chunks + blockIdx.x) * N;
    for (int fi = tid; fi < N; fi += C::THREADS) {
        float t = 0.f;
#pragma unroll
        for (int tm = 0; tm < C::TEAMS; ++tm) t += red[tm * N + fi];
        pd[fi] = t;
    }
}

}  // namespace rt
