/*
 * rt_fbank.h -- C ABI of the polyphase FFT filter bank of librtb200.so: every channel of a uniform grid across the whole band.
 *
 * The down-converter of rt_ddc.h computes each channel on its own, at C L / D complex x real multiply-adds per input sample.
 * For the one channel plan that covers a band without gaps -- channels fs / (2 D) apart -- the filter bank computes the same
 * channels with about L real x complex multiply-adds and one C-point FFT per D input samples.  The DDC stays the way to get
 * arbitrary channel offsets.
 *
 * Conventions as in rt_engine.h and rt_ddc.h: plain C types, RT_OK / RT_ERR_* return codes, rt_last_error() for the message
 * of the last failure, one host thread per handle, no CPU fallback.
 *
 * Definition (normative).  The output is EXACTLY the quantity of rt_ddc.h for this channel plan:
 *   - C = 2 D grid channels, D a power of two in [RT_FBANK_MIN_DECIMATION, RT_FBANK_MAX_DECIMATION];
 *   - channel k, -(D - 1) <= k <= D - 1, at the offset k fs / (2 D), with the rt_ddc phase increment
 *     inc_k = ((k mod C) 2^32) / C, which is exact because C divides 2^32;
 *   - the channel that straddles +-fs / 2 (k = D) is left out (it does not lie inside the input band);
 *   - so 2 D - 1 output rows per input, in ascending frequency: channel k is row k + D - 1.
 * With inc_k, the rt_ddc definition becomes, for the output time n = n0 + m D and the global input index j,
 *
 *     y_k[m] = sum_{r=0}^{C-1} exp(-2 pi i k r / C) u_r[m],      u_r[m] = sum_{j = r (mod C), 0 <= n - j < L} h[n - j] x[j]
 *
 * i.e. polyphase partial sums (L real x complex products per output frame in all) and one C-point forward DFT.  There is no
 * mixer: the phase is the global index j mod C, kept in uint32 arithmetic, so rt_fbank_reset_input(first_sample) and every
 * split of the samples into calls behave exactly as in the DDC.  Samples before n0 come from a per-input device history of the
 * last L - 1 normalised samples, zero after rt_fbank_create and rt_fbank_reset_input.
 *
 * Determinism: u_r sums its terms in one fixed order (n - j ascending), and the FFT is one fixed sequence of radix-2 steps,
 * whatever tile, block, call or batch an output is computed in.  Splitting the same samples into other calls, block counts
 * or batches gives bit-identical outputs.
 *
 * Accuracy: fp32 on the CUDA cores; the taps are rounded to fp32 once, the FFT twiddles are rounded to fp32 once from float64.
 * The error of an output is bounded by a few units of 2^-24 * (sqrt(L / C) + log2 C) times sum_k |h[k]| * max |x|: like the
 * DDC's it is relative to the FULL-BAND amplitude of the input, not to the channel's own signal (about 1e-6 of it at most; the
 * tests assert 1e-5 * sum |h| * max |x|, the DDC's bound).
 *
 * Limits: L odd, 1 <= L <= 16 D + 1 (the default design has 8 D + 1 taps); block_samples a multiple of D;
 * n_inputs * (2 D - 1) <= 2^30; n_inputs <= 65535.
 */
#ifndef RT_FBANK_H
#define RT_FBANK_H

#include <stddef.h>
#include <stdint.h>

#include "rt_engine.h"

#ifdef __cplusplus
extern "C" {
#endif

#define RT_FBANK_ABI_VERSION 1
#define RT_FBANK_MIN_DECIMATION 4
#define RT_FBANK_MAX_DECIMATION 512
#define RT_FBANK_MAX_TAPS(D) (16 * (D) + 1)

typedef struct rt_fbank_config {
    int32_t abi_version;        /* RT_FBANK_ABI_VERSION */
    int32_t cuda_device;        /* ordinal */
    int32_t n_inputs;           /* wideband streams (>= 1, <= 65535), all in one format */
    int32_t decimation;         /* D, a power of two in [RT_FBANK_MIN_DECIMATION, RT_FBANK_MAX_DECIMATION]; C = 2 D */
    int64_t block_samples;      /* complex input samples per block, a multiple of decimation */
    int32_t n_taps;             /* L, odd, 1 ... RT_FBANK_MAX_TAPS(D) */
    int32_t sample_format;      /* RT_SAMPLE_* of the input */
    int32_t reserved;           /* zero */
    double sample_rate;         /* input rate (informational: the definition above is in samples) */
    const double *taps;         /* h[0 .. L-1], real */
} rt_fbank_config;

typedef struct rt_fbank rt_fbank;

/* RT_ERR_INVALID, before any device is touched, for D that is not a power of two in range, an even or oversized L, a block
 * that is not a multiple of D, an unknown sample_format, a wrong abi_version or a non-zero reserved; RT_ERR_CUDA without a
 * device. */
int rt_fbank_create(const rt_fbank_config *cfg, rt_fbank **out);
/* Waits for the last run, then frees everything. */
void rt_fbank_destroy(rt_fbank *f);

/* Restart input `input` at the global sample index first_sample: its history becomes zero and the next run's first sample has
 * the index first_sample.  Takes effect at the next rt_fbank_run, in that run's stream order. */
int rt_fbank_reset_input(rt_fbank *f, int32_t input, int64_t first_sample);

/*
 * One call, with the contract of rt_ddc_run: `blocks` (>= 1) consecutive blocks of block_samples interleaved I,Q samples per
 * input, input i at iq + i * in_stride_bytes, on the device (iq_on_device != 0, aligned like in_stride_bytes to one complex
 * sample) or on the host (pinned or pageable; copied in with cudaMemcpy2DAsync on `cuda_stream`).
 * Writes cf32 (float I, Q) rows [input][2 D - 1][blocks * block_samples / D]: row (i * (2 D - 1) + k + D - 1) at
 * out + (i * (2 D - 1) + k + D - 1) * out_stride_bytes, a device pointer aligned to 8 bytes.  This is the input layout of an
 * rt_engine with RT_SAMPLE_CF32, n_streams = n_inputs * (2 D - 1) and blocks_per_launch = blocks.
 * Everything is enqueued on cuda_stream and ordered after the previous run of this handle, whichever stream that was on.
 */
int rt_fbank_run(rt_fbank *f, void *cuda_stream, const void *iq, int32_t iq_on_device, size_t in_stride_bytes, int32_t blocks,
                 void *out, size_t out_stride_bytes);

#ifdef __cplusplus
}
#endif
#endif /* RT_FBANK_H */
