/*
 * rt_ddc.h -- C ABI of the wideband down-converter (DDC) of librtb200.so.
 *
 * A wideband recording (Airspy / SDRplay / USRP ci16_le, HackRF ci8, GNU Radio cf32_le, RTL-SDR cu8 at 2.5-20 MS/s) covers a
 * whole tag band.  The DDC cuts it into "virtual SDR channels": complex baseband streams at fs / D, each centred on its own
 * frequency, which the detection engine (rt_engine.h) then analyses exactly as it analyses one RTL-SDR.  The output is written
 * in the engine's RT_SAMPLE_CF32 layout, so a DDC output is an ordinary device-resident engine input.
 *
 * Conventions as in rt_engine.h: plain C types, RT_OK / RT_ERR_* return codes, rt_last_error() for the message of the last
 * failure, one host thread per handle, no CPU fallback.
 *
 * Definition (normative; tests/ddc_oracle.py restates it in float64).  Input i is a stream x_i of normalised complex samples
 * (the table of rt_engine.h: cu8 b / 127.5 - 1, ci8 v / 128, ci16 v / 32768, cf32 as stored) with a global sample index n.
 * Channel c has the phase increment inc_c (cycles per input sample times 2^32).  For the output sample m of a call whose first
 * input sample has the index n0:
 *
 *     y_c[m] = exp(-2 pi i ((inc_c (n0 + m D)) mod 2^32) / 2^32) * sum_{k=0}^{L-1} g_c[k] x[n0 + m D - k],
 *     g_c[k] = h[k] exp(+2 pi i ((inc_c k) mod 2^32) / 2^32)
 *
 * i.e. mix channel c to baseband, filter with the real taps h, keep every D-th sample.  The phase is exact integer arithmetic:
 * it does not drift over any length of recording.  Samples before n0 come from a per-input device history of the last L - 1
 * normalised samples, zero after rt_ddc_create and rt_ddc_reset_input (the zero state of scipy's lfilter).
 *
 * Determinism: every output sums its L terms in one fixed order (by k mod D, then k / D), whatever tile, block, call or batch
 * it is computed in.  Splitting the same samples into other calls, block counts or batches gives bit-identical outputs.
 *
 * Accuracy: fp32 on the CUDA cores (the taps g_c are rounded to fp32 once, on the host).  The error of an output is bounded by
 * a few units of 2^-24 * sqrt(L) times sum_k |h[k]| * max |x|: it is relative to the FULL-BAND amplitude of the input, not to
 * the channel's own signal.  A weak channel beside a much stronger out-of-channel signal therefore has an error floor
 * proportional to that strong signal (about 1e-7 of it in amplitude, -140 dB in power, at L = 513).
 */
#ifndef RT_DDC_H
#define RT_DDC_H

#include <stddef.h>
#include <stdint.h>

#include "rt_engine.h"

#ifdef __cplusplus
extern "C" {
#endif

#define RT_DDC_ABI_VERSION 1
#define RT_DDC_MAX_TAPS 2049          /* L: odd, 1 ... 2049 (the default design of 8 D + 1 taps up to D = 256) */
#define RT_DDC_MAX_DECIMATION 1024    /* D: 2 ... 1024 */

typedef struct rt_ddc_config {
    int32_t abi_version;        /* RT_DDC_ABI_VERSION */
    int32_t cuda_device;        /* ordinal */
    int32_t n_inputs;           /* wideband streams (>= 1, <= 65535), all in one format and sharing one channel plan */
    int32_t n_channels;         /* channels per input (>= 1) */
    int64_t block_samples;      /* complex input samples per block, a multiple of decimation */
    int32_t decimation;         /* D, 2 ... RT_DDC_MAX_DECIMATION */
    int32_t n_taps;             /* L, odd, 1 ... RT_DDC_MAX_TAPS */
    int32_t sample_format;      /* RT_SAMPLE_* of the input */
    int32_t reserved;           /* zero */
    double sample_rate;         /* input rate (informational: the definition above is in samples) */
    const double *taps;         /* h[0 .. L-1], real */
    const uint32_t *phase_inc;  /* inc_c for c = 0 .. n_channels-1 */
} rt_ddc_config;

typedef struct rt_ddc rt_ddc;

/* RT_ERR_INVALID for an even or oversized L, D outside 2 ... RT_DDC_MAX_DECIMATION, a block that is not a multiple of D, an
 * unknown sample_format or a wrong abi_version; RT_ERR_CUDA without a device. */
int rt_ddc_create(const rt_ddc_config *cfg, rt_ddc **out);
/* Waits for the last run, then frees everything. */
void rt_ddc_destroy(rt_ddc *d);

/* Restart input `input` at the global sample index first_sample: its history becomes zero and the next run's first sample has
 * the index first_sample.  Takes effect at the next rt_ddc_run, in that run's stream order. */
int rt_ddc_reset_input(rt_ddc *d, int32_t input, int64_t first_sample);

/*
 * One call: `blocks` (>= 1) consecutive blocks of block_samples interleaved I,Q samples per input, input i starting at
 * iq + i * in_stride_bytes.  iq_on_device != 0: a device pointer, aligned like in_stride_bytes to one complex sample; otherwise
 * a host pointer (pinned or pageable) that is copied in with cudaMemcpy2DAsync on `cuda_stream` (a pinned buffer must stay
 * unchanged until the stream has reached this call).
 * Writes cf32 (float I, Q) rows [input][channel][blocks * block_samples / D]: row (i * n_channels + c) at
 * out + (i * n_channels + c) * out_stride_bytes, a device pointer aligned to 8 bytes.  This is the input layout of an
 * rt_engine with RT_SAMPLE_CF32, n_streams = n_inputs * n_channels and blocks_per_launch = blocks.
 * Everything is enqueued on cuda_stream (a cudaStream_t; 0 is the legacy default stream) and ordered after the previous run of
 * this handle, whichever stream that was on.
 */
int rt_ddc_run(rt_ddc *d, void *cuda_stream, const void *iq, int32_t iq_on_device, size_t in_stride_bytes, int32_t blocks,
               void *out, size_t out_stride_bytes);

/*
 * DC and IQ-imbalance correction (default off).  A zero-IF receiver (HackRF, bladeRF 1, uncorrected GNU Radio captures) forms
 * I and Q in two analog paths whose gain and phase differ slightly, so every signal at offset +f has a mirror image at -f,
 * typically 25-40 dB down, and a DC spike at 0 Hz.  With the correction on, the filter runs on y instead of x (normative;
 * tests/iq_oracle.py restates it in float64).  For input i and each block b of block_samples samples -- the handle's own
 * block, whatever `blocks` a call carries -- with x the normalised samples of that block:
 *
 *     m = mean(x)      p = mean(|x - m|^2)      c = mean((x - m)^2)
 *     w = -c / (p + sqrt(p^2 - |c|^2))  (w = 0 when p = 0)      y = (x - m) + w conj(x - m)
 *
 * Each block's samples get that block's own m and w.  mean(y^2) = c + 2 w p + w^2 conj(c) = 0: the block comes out proper,
 * which removes the image; a proper block (c = 0) only loses its DC.  A frequency-flat gain / phase imbalance is undone up to a
 * complex gain.  A frequency-dependent imbalance (I and Q filters that differ across the band) is only partly corrected: one
 * w per block is the best flat correction, not a per-frequency one.  The history carried into the next run holds y, so
 * switching the correction on or off in the middle of a recording changes only how later samples enter the filter.
 *
 * The moments are exact int64 sums of the elements for cu8, ci8 and ci16, and float64 sums of fixed 16384-sample tiles for
 * cf32, in an order that does not depend on the call, the batch or the grid; m and w are formed in float64 and rounded to fp32
 * once.  So every split of the same samples into calls, block counts or batches still gives bit-identical outputs.
 *
 * Accuracy with the correction on: the bound of the definition above holds for the quantity computed from y, with max |x|
 * replaced by max |y| of the corrected samples (|y| <= (1 + |w|) |x - m|); the fp32 rounding of m and w adds at most a few
 * units of 2^-24 (|m| + |w| max |x - m|) per sample, inside the same bound.
 *
 * Limit: block_samples <= 2^30 while the correction is on.
 */

/* enable != 0: correct every block from the next rt_ddc_run on, in that run's stream order (like rt_ddc_reset_input); 0: stop.
 * RT_ERR_INVALID when block_samples exceeds 2^30. */
int rt_ddc_set_iq_correction(rt_ddc *d, int32_t enable);
/* Test hook: m and w of (input, block) of the last run, out = {m.re, m.im, w.re, w.im} (fp32, as the kernels apply them).
 * Waits for that run.  RT_ERR_INVALID when the last run did not correct, or for an index outside it. */
int rt_ddc_read_iq_correction(rt_ddc *d, int32_t input, int32_t block, float out[4]);

#ifdef __cplusplus
}
#endif
#endif /* RT_DDC_H */
