/*
 * rt_engine.h -- C ABI of the B200 detection engine (librtb200.so).
 *
 * The reference (Nature40/pyradiotracking) is pure Python and has no FFI for this
 * path; its boundary is the class radiotracking.analyze.SignalAnalyzer
 * (radiotracking/analyze.py:20).  The entry points below are what a binding for the
 * inside of SignalAnalyzer.process_samples (analyze.py:192-268) needs; each one names
 * the reference lines it replaces.  The Python side of the binding (ctypes) is
 * pyradiotracking_b200/engine.py; INTEGRATION.md shows the stub a maintainer of the
 * reference would add.
 *
 * Conventions: plain C types only; every function returns RT_OK (0) or a negative
 * RT_ERR_* code and never throws; rt_last_error() returns a thread-local message for
 * the last failure.  A handle is NOT thread-safe: one host thread per engine, like the
 * reference's one-process-per-SDR model (radiotracking/__main__.py:94-130).
 * There is no CPU fallback: without a CUDA device rt_engine_create fails.
 */
#ifndef RT_ENGINE_H
#define RT_ENGINE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RT_ABI_VERSION 2

enum {
    RT_OK = 0,
    RT_ERR_INVALID = -1,      /* bad argument / unsupported configuration */
    RT_ERR_CUDA = -2,         /* CUDA runtime error, no device, wrong architecture */
    RT_ERR_OVERFLOW = -3,     /* more candidate records than max_records (or than the caller's buffer): the first ones are
                                 still returned and *n_out says how many there were; none are lost silently */
    RT_ERR_STATE = -4         /* call order violated (fetch without launch, ...) */
};

/* fft_impl selector: which spectrogram kernel runs (tests compare them). */
enum {
    RT_FFT_AUTO = 0,      /* nperseg 256: RT_FFT_REG256; 1024 / 4096: radix-16 Stockham kernel (spectro_r16.cuh); otherwise RT_FFT_GENERIC.
                           * RT_SAMPLE_CI16 / RT_SAMPLE_CF32: always RT_FFT_GENERIC */
    RT_FFT_GENERIC = 1,   /* shared-memory Stockham FFT, any power-of-two nperseg */
    RT_FFT_REG256 = 2,    /* nperseg 256: 16x16 FFT in registers (packed fp32x2), TMA-fed */
    RT_FFT_TC256 = 3      /* nperseg 256, boxcar/hann/hamming: first FFT stage on the tensor cores (tcgen05, fp16 x split-fp16 -> fp32).
                           * Optional and slower than the default.  Accuracy limit: the bytes are centred at the constant 128 and the
                           * rest of the segment mean is removed from the bins 0 and +-1 afterwards, so captures whose DC offset is far
                           * from 128 (tens of LSB) lose precision in exactly those three bins (tests/test_gpu_parity.py, extreme byte
                           * patterns); the default kernels subtract the exact mean per sample and have no such limit. */
};

/* sample_format: the element type of the interleaved I,Q input, named after the SigMF datatypes.  The spectrogram is that of the
 * normalised complex samples below; the thresholds apply to them (calibration_db absorbs the receiver's gain).
 *   format           element         normalised sample   bytes per complex sample   kernels
 *   RT_SAMPLE_CU8    uint8 I, Q      b / 127.5 - 1       2                          every RT_FFT_* (pyrtlsdr, RTL-SDR)
 *   RT_SAMPLE_CI8    int8 I, Q       v / 128             2                          every RT_FFT_* (v ^ 0x80 is a cu8 byte)
 *   RT_SAMPLE_CI16   int16 LE I, Q   v / 32768           4                          RT_FFT_GENERIC (RT_FFT_AUTO picks it)
 *   RT_SAMPLE_CF32   float32 LE I, Q x as stored         8                          RT_FFT_GENERIC (RT_FFT_AUTO picks it)
 * RT_FFT_REG256 and RT_FFT_TC256 with RT_SAMPLE_CI16 / RT_SAMPLE_CF32 are rejected by rt_engine_create.
 * Accuracy limit of RT_SAMPLE_CF32: the segment mean is an fp32 sum (fixed order: per thread, then a shuffle tree, then the
 * warps in order) whose error is at most about (nperseg / 256 + 13) * 2^-24 * max|x|.  Where the DC offset dominates, the
 * centred samples x - mean are exact (Sterbenz), so that error is one constant per segment, which the window carries into the
 * bins where its DFT lives (bin 0, and +-1 for hann / hamming).  A capture with a DC offset D far above its signals loses
 * precision in those bins only: an absolute error of up to about 1.7e-6 * D (nperseg 4096; 8.3e-7 * D at 256) per sample */
enum {
    RT_SAMPLE_CU8 = 0,
    RT_SAMPLE_CI8 = 1,
    RT_SAMPLE_CI16 = 2,
    RT_SAMPLE_CF32 = 3
};

/* scan_schedule: where the scan kernels (row mean, probe, extraction) of a launch run. */
enum {
    RT_SCAN_AUTO = 0,     /* RT_SCAN_LEAN for nperseg 256 launches of >= 500 k segments, otherwise RT_SCAN_OVERLAP */
    RT_SCAN_SERIAL = 1,   /* on the launch stream, after the spectrogram (no overlap with the next launch) */
    RT_SCAN_OVERLAP = 2,  /* full-size scan kernels on an engine-internal high-priority stream */
    RT_SCAN_LEAN = 3      /* 32-register scan kernels that fit BESIDE the resident spectrogram CTAs of the next launch */
};

/*
 * Engine configuration = the analysis keys of SignalAnalyzer.__init__
 * (analyze.py:62-129), already converted by the host the way the reference does it in
 * float64 (analyze.py:113-116), for a batch of `n_streams` independent analyzers
 * (one per SDR / recorded channel) that share sample rate and FFT settings.
 */
typedef struct rt_config {
    int32_t abi_version;        /* RT_ABI_VERSION */
    int32_t cuda_device;        /* ordinal */
    int32_t n_streams;          /* analyzers in the batch (>= 1) */
    int32_t nperseg;            /* fft_nperseg: power of two in [8, 4096] */
    int64_t block_samples;      /* sdr_callback_length: complex samples per stream per call (analyze.py:108-109) */
    double sample_rate;         /* fs */
    const double *window;       /* nperseg values, as scipy get_window(fft_window, nperseg) returns them */
    const double *signal_threshold; /* [n_streams] linear: 10**((signal_threshold_dbw + calibration_db)/10) (analyze.py:115) */
    double snr_threshold;       /* linear: 10**(snr_threshold_db/10) (analyze.py:116) */
    int32_t probe_stride;       /* max(1, int(signal_min_duration / (times[1]-times[0]))), float64 on the host (analyze.py:354,364) */
    int32_t min_cols;           /* coarse duration gate in spectrogram columns; the exact float64 test */
    int32_t max_cols;           /*   (analyze.py:419-433) is applied by the host on the returned records */
    int32_t max_records;        /* capacity of one call's record list; 0 = sized for the worst case (one record per probe
                                   column of every bin, capped at 4 Mi records), so that a noisy band cannot overflow it */
    int32_t fft_impl;           /* RT_FFT_* */
    int32_t scan_schedule;      /* RT_SCAN_* */
    int32_t launch_streams;     /* 0 = auto; 1 = spectrogram kernels on the launch stream itself; 2 = consecutive launches
                                   alternate between two internal streams (launch i+1 fills the SMs while launch i drains) */
    int32_t chunk_segs;         /* nperseg 256: segments per CTA, a multiple of 8; 0 = auto (64 / 128 / 192 by block length) */
    int32_t blocks_per_launch;  /* offline replay: this many CONSECUTIVE callback blocks of every stream per launch (>= 1).
                                   Block b of stream s is the analyzer unit s * blocks_per_launch + b: it has its own row
                                   means and records, and its carry (analyze.py:383-398) is block b-1 of the same launch,
                                   or the last block of the previous launch for b = 0.
                                   With nperseg 256 and blocks_per_launch > 1, the register kernel needs block_samples to be
                                   a multiple of 8 (16-byte aligned blocks): otherwise RT_FFT_AUTO runs the generic kernel and
                                   RT_FFT_REG256 is rejected by rt_engine_create */
    int32_t sample_format;      /* RT_SAMPLE_* (0 = RT_SAMPLE_CU8: uint8 bytes, as before this field existed) */
    int32_t reserved[2];        /* zero */
} rt_config;

/*
 * One candidate detection = one maximal run of above-threshold cells that the
 * reference's strided probe would visit (analyze.py:364-417), with the statistics
 * of analyze.py:436-447 in linear units.  Columns index the current block's
 * spectrogram; start < 0 reaches into the previous block (analyze.py:383-398).
 * The host turns records into Signal objects (analyze.py:419-450).
 */
typedef struct rt_record {
    int32_t stream;     /* analyzer unit: stream index * blocks_per_launch + block index within the launch */
    int32_t fi;         /* frequency bin, FFT order (no fftshift) */
    int32_t start;      /* first column of the statistics window (inclusive) */
    int32_t end;        /* last column + 1 */
    float max_lin;      /* np.max(data) */
    float row_mean;     /* freq_avg = np.mean(spectrogram[fi]) of the current block (analyze.py:374-375) */
    double mean_lin;    /* np.mean(data) */
    double std_db;      /* np.std(10*log10(data)) */
} rt_record;

typedef struct rt_engine rt_engine;

/* Per-launch device timings accumulated while timing is enabled (milliseconds).  The kernels of every `period`-th launch
 * (rt_engine_enable_timing) are bracketed by CUDA events and the sums are scaled to all `launches`. */
typedef struct rt_timing {
    double spectrogram_ms;  /* uint8 IQ -> power cells + row sums (the dominant kernel) */
    double rowmean_ms;
    double probe_ms;
    double extract_ms;
    int64_t launches;       /* engine launches accumulated */
    int64_t kernels;        /* CUDA kernels launched by those */
} rt_timing;

const char *rt_last_error(void);
int rt_abi_version(void);
/* Number of CUDA devices visible, or a negative RT_ERR_CUDA. */
int rt_device_count(void);

/* Replaces SignalAnalyzer.__init__'s analysis setup (analyze.py:108-129). */
int rt_engine_create(const rt_config *cfg, rt_engine **out);
void rt_engine_destroy(rt_engine *e);

/* Launch on this CUDA stream (cudaStream_t) instead of the engine's own.  Work queued on it before a launch orders that
 * launch; work on any other stream does not (rt_engine_wait_stream). */
int rt_engine_set_stream(rt_engine *e, void *cuda_stream);

/* Forget the carry of one stream (= a restarted analyzer: _spectrogram_last = None, analyze.py:128). */
int rt_engine_reset_stream(rt_engine *e, int32_t stream);

/*
 * One callback for every stream of the batch (analyze.py:234-248 without the shadow
 * filter): `iq` holds, for every stream, blocks_per_launch consecutive blocks of block_samples
 * interleaved I,Q samples in rt_config.sample_format (bytes_per_sample * block_samples bytes each, RT_SAMPLE_*),
 * stream s starting at iq + s*stream_stride_bytes.  iq_on_device != 0: `iq` is a device pointer (no copy), aligned, like
 * stream_stride_bytes, to one complex sample (2, 4 or 8 bytes); otherwise a host pointer (pinned or pageable) that is copied in.
 * Blocks until done.  Records come back sorted by (stream, fi, start).
 * On RT_ERR_OVERFLOW *n_out is the number that would have been needed and `out` holds the first
 * min(max_out, max_records) of them.
 */
int rt_engine_process(rt_engine *e, const uint8_t *iq, int32_t iq_on_device, size_t stream_stride_bytes,
                      rt_record *out, int32_t max_out, int32_t *n_out);

/* The same in two halves: enqueue only (asynchronous; `iq` -- host or device -- must stay valid and unchanged until the
 * fetch or an rt_engine_join: the kernels run on engine-internal streams that are ordered AFTER the work already queued on
 * the launch stream, but work queued on the launch stream later is not ordered after them) ... */
int rt_engine_launch(rt_engine *e, const uint8_t *iq, int32_t iq_on_device, size_t stream_stride_bytes);
/* ... then wait for the OLDEST unfetched launch, copy back and sort its records.  Two launches may be in
 * flight (launch i+1 can be queued before fetch i); a third launch drops the oldest unfetched result. */
int rt_engine_fetch(rt_engine *e, rt_record *out, int32_t max_out, int32_t *n_out);
/* Wait for the oldest unfetched launch WITHOUT consuming it: *n_records = the records rt_engine_fetch will return
 * (callers size their buffer with it). */
int rt_engine_peek(rt_engine *e, int32_t *n_records);

/*
 * The spectrogram kernels of consecutive launches alternate between two engine-internal streams and the scan kernels (row
 * mean, probe, extraction) run on a third, so that launch i+1 overlaps the tail and the scan of launch i.
 * rt_engine_join makes the launch stream (the engine's own or the
 * one given to rt_engine_set_stream) wait for everything launched so far, e.g. before the caller records an
 * event on it or reuses a device-resident `iq` buffer from another stream.  rt_engine_fetch does not need it.
 */
int rt_engine_join(rt_engine *e);

/*
 * The other direction: the next launch is ordered after all work queued on `cuda_stream` (a cudaStream_t; also
 * cudaStreamLegacy / cudaStreamPerThread) so far, e.g. the kernel or copy that produces a device-resident `iq`.  The
 * engine's streams are non-blocking: without this (or the producer being the stream given to rt_engine_set_stream) a
 * launch may read `iq` before it is written.  An event is recorded on `cuda_stream` and the launch stream waits for it;
 * the engine-internal streams fork from the launch stream and inherit the wait.
 */
int rt_engine_wait_stream(rt_engine *e, void *cuda_stream);

/* Counters of the last fetched launch: probe hits handed to the extraction kernel, and records emitted. */
int rt_engine_last_counts(rt_engine *e, int32_t *work_items, int32_t *records);

/* Spectrogram geometry: *T = block_samples / nperseg columns per block.  *n_streams counts analyzer units
 * (streams * blocks_per_launch). */
int rt_engine_shape(const rt_engine *e, int32_t *n_streams, int32_t *nperseg, int32_t *T);

/*
 * Parity hooks (tests only): the power spectrogram of the last launch for one stream,
 * as float32 [T][nperseg] (time-major, bins in FFT order), i.e. scipy's Sxx transposed
 * (analyze.py:234-241); and the row means [nperseg] (analyze.py:375).
 */
int rt_engine_read_spectrogram(rt_engine *e, int32_t stream, float *out_T_by_nperseg);
int rt_engine_read_row_means(rt_engine *e, int32_t stream, float *out_nperseg);

/*
 * Band survey: what the band looked like in each analyzed block, for choosing signal_threshold_dbw and calibration_db and for
 * spotting interferers.  Off by default; with it off no survey work is enqueued.  For analyzer unit u of a launch with T columns,
 * bin fi in FFT order, the launch's power cells S[fi, t] and its row means avg = mean_t S[fi, :] (the record's row_mean),
 * thr[u] = rt_config.signal_threshold of u's stream and snr = rt_config.snr_threshold, exactly as the scan uses them:
 *     noise[u][fi]      = avg                                                   (linear)
 *     peak[u][fi]       = max_t S[fi, t]                                        (linear)
 *     above_cols[u][fi] = #{ t < T : !(S[fi,t] < thr[u]) && !(S[fi,t] / avg < snr) }
 * all over the current block's columns only (no carry).  above_cols uses the scan's fp32 predicate (predicate.h), so it agrees
 * with what the detection saw.  On RT_FFT_TC256 the power scale the kernels carry is undone (a power of two: exact).  The values
 * are the same bits run after run, and for a unit alone or inside a batch.  Cost: one more read of the spectrogram per launch,
 * on the scan stream after the extraction kernel; the peek and fetch of a surveyed launch wait for it.
 */
/* Survey the launches from the next one on (enable != 0) or stop. */
int rt_engine_set_survey(rt_engine *e, int32_t enable);
/* The survey of the last fetched launch, each [units][nperseg] (units = n_streams * blocks_per_launch; bins in FFT order); a
 * null pointer skips that array.  RT_ERR_INVALID when that launch did not survey. */
int rt_engine_read_survey(rt_engine *e, float *noise, float *peak, int32_t *above_cols);

/*
 * Neighbour bins: what a carrier estimate finer than one FFT bin needs (pyradiotracking_b200/finefreq.py).  Off by default; with
 * it off nothing is enqueued.  For a record (stream = unit u, fi, start, end) of a launch with T columns and n = nperseg, its
 * cells in bin b are exactly those the record's mean_lin averages in bin fi:
 *     start >= 0:  S_u[b][start .. end-1]
 *     start <  0:  prev_u[b][T+start .. T-1]  and  S_u[b][0 .. end-1]
 * where prev_u is unit u - 1 of the same launch, or for u % blocks_per_launch == 0 the last block of u's stream in the previous
 * launch (the extraction's carry).  With lo = (fi - 1) mod n and hi = (fi + 1) mod n:
 *     mean_lo / mean_hi         = the mean of those end - start cells in bin lo / hi (float64 sum of the fp32 cells)
 *     row_mean_lo / row_mean_hi = the current block's row means avg[u][lo] / avg[u][hi] (as rt_record.row_mean)
 * On RT_FFT_TC256 the power scale is undone (a power of two: exact).  The values are the same bits run after run, and for a unit
 * alone or inside a batch.  Cost: 2 (end - start) scattered cells per record, one kernel on the scan stream after the
 * extraction kernel (and the survey); the peek and fetch of such a launch wait for it.
 */
typedef struct rt_neighbours {
    double mean_lo, mean_hi;
    float row_mean_lo, row_mean_hi;
} rt_neighbours;    /* 24 bytes */
/* Compute them for the launches from the next one on (enable != 0) or stop; allocates max_records entries for every result slot
 * that lacks them. */
int rt_engine_set_neighbours(rt_engine *e, int32_t enable);
/* Entry i belongs to record i of the last rt_engine_fetch, in its order; *n_out = the records that fetch returned (also after an
 * RT_ERR_OVERFLOW fetch).  RT_ERR_INVALID when that launch did not compute them; RT_ERR_OVERFLOW when max_out < *n_out (the first
 * max_out are written). */
int rt_engine_read_neighbours(rt_engine *e, rt_neighbours *out, int32_t max_out, int32_t *n_out);

/*
 * Parity hook (tests only, no GPU needed): the constant operands of the RT_FFT_TC256 kernel for a 256-point window
 * (as scipy returns it): the 16 stage-1 matrices as two fp16 terms in the tensor-core operand layout
 * (bmat_out: 16 * 2 * 1024 halves, element (n, k) of matrix (n2, hi|lo) at ((n2*2 + hl)*1024 + (n>>3)*256 + (k>>3)*64 + (n&7)*8 + (k&7)),
 * n = 2*k1 + re|im, k = 2*n1 + I|Q), the scaled window DFT at the bins 0, 1, 255 (wc_out: 3 complex), the power-of-two
 * power scale, and whether the window qualifies (its DFT vanishes outside the bins 0 and +-1).
 */
int rt_tc256_tables(const double *window, double sample_rate, uint16_t *bmat_out, double *wc_out, double *pscale_out, int32_t *eligible_out);

/* CUDA-event timing of the individual kernels (bench.py roofline): period = 0 switches it off, k >= 1 brackets the kernels
 * of every k-th launch (two event records between consecutive spectrogram kernels cost ~5 us of launch gap). */
int rt_engine_enable_timing(rt_engine *e, int32_t period);
int rt_engine_get_timing(rt_engine *e, rt_timing *out, int32_t reset);

#ifdef __cplusplus
}
#endif
#endif /* RT_ENGINE_H */
