"""Band survey on the B200 (pytest -m gpu): include/rt_engine.h, rt_engine_set_survey.

  against the float64 oracle on every spectrogram kernel and layout (generic, register / PERM, tensor-core / TILE, radix-16 at
  1024 and 4096), every sample format, blocks_per_launch 1 and 4 with ragged blocks; and bit for bit against the GPU's own cells
  records byte-identical with the survey on and off at configs[1] size, and the same Signals behind the filter bank
  the stream contract: two launches in flight, toggling between launches, a read after an unsurveyed launch, a unit alone and
  inside a batch, repeated runs
  wideband: a tone where the float64 arithmetic puts it in the stitched full-band survey, the stitched grid, the DDC's channel
  surveys against the filter bank's
"""
import datetime

import numpy as np
import pytest

from oracle import restatement as R
from pyradiotracking_b200 import engine as E
from pyradiotracking_b200 import synth
from pyradiotracking_b200 import wideband as W
from pyradiotracking_b200.analyze import BatchAnalyzer
from tests import format_oracle as FO
from tests import parity

pytestmark = pytest.mark.gpu

T0 = datetime.datetime(2026, 9, 9, 9, 9, 9)


def _kw(fs, block, nperseg, window="hamming"):
    return dict(device="0", calibration_db=0.0, sample_rate=fs, center_freq=150_150_000, fft_nperseg=nperseg, fft_window=window,
                signal_min_duration_ms=8.0, signal_max_duration_ms=40.0, signal_threshold_dbw=-90.0, snr_threshold_db=5.0,
                sdr_callback_length=block)


def _capture(fmt, fs, block, nperseg, nb, stream=1):
    """[nb, 2 block] elements of `fmt`: noise and tone bursts (tests/test_gpu_formats.py's recipe)."""
    amp = (6.0, 20.0) if nperseg >= 2048 else (10.0, 30.0)
    w = synth.Workload(97, f"survey-{nperseg}-{fs}-{block}", fs, block, nperseg=nperseg, amp_lsb=amp)
    return synth.make_stream_format(w, fmt, stream, nb)


def _check_unit(P, S64, S32_T, rowmean32, noise, peak, above):
    """One unit's survey: bit for bit against the GPU's own cells and row means, and within the parity bounds of the float64
    oracle's S (FFT order, [n, T])."""
    S32 = S32_T.T
    thr32, snr32 = np.float32(P.signal_threshold), np.float32(P.snr_threshold)
    assert np.array_equal(noise, rowmean32)
    assert np.array_equal(peak, S32.max(axis=1))
    with np.errstate(divide="ignore", invalid="ignore"):
        pred = ~(S32 < thr32) & ~(S32 / noise[:, None] < snr32)          # fp32, correctly rounded: the scan's predicate
    assert np.array_equal(above, pred.sum(axis=1).astype(np.int32))

    n = S64.shape[0]
    avg = S64.mean(axis=1)
    assert np.max(np.abs(noise - avg) / avg) <= 2e-5
    pk = S64.max(axis=1)
    arg = S64.argmax(axis=1)
    deep = (S64 < S64.max(axis=0, keepdims=True) * 10 ** (-parity.DEEP_DB / 10))[np.arange(n), arg]
    big = pk >= 1e-2 * P.signal_threshold
    rel = np.abs(peak - pk) / pk
    assert np.all(rel[big] <= np.where(deep, parity.DEEP_RTOL, parity.POWER_RTOL)[big]), float(rel[big].max())
    ab = (~(S64 < P.signal_threshold) & ~(S64 / avg[:, None] < P.snr_threshold)).sum(axis=1)
    eff = np.maximum(P.signal_threshold, P.snr_threshold * avg)
    near = (np.abs(S64 / eff[:, None] - 1.0) <= parity.NEAR_THRESHOLD).sum(axis=1)
    assert np.all(np.abs(above.astype(np.int64) - ab) <= near)
    return int(ab.sum())


ORACLE_CASES = [  # fmt, nperseg, fs, block, impl, blocks per launch, window
    ("cu8", 256, 300_000, 300_000, E.FFT_GENERIC, 1, "hamming"),
    ("cu8", 256, 300_000, 300_000, E.FFT_AUTO, 1, "hamming"),          # register kernel, PERM
    ("ci8", 256, 300_000, 300_000, E.FFT_TC256, 1, "hamming"),         # tensor-core kernel, TILE, power scale
    ("ci8", 1024, 2_400_000, 2_400_000, E.FFT_AUTO, 1, "hann"),        # radix-16
    ("cu8", 4096, 2_400_000, 2_400_000, E.FFT_AUTO, 1, "hann"),        # radix-16
    ("ci16_le", 256, 300_000, 300_000, E.FFT_AUTO, 1, "hamming"),      # generic
    ("cf32_le", 2048, 2_400_000, 2_400_000, E.FFT_AUTO, 1, "hamming"),
    ("cu8", 256, 300_000, 75_104, E.FFT_AUTO, 4, "hamming"),           # register kernel, 293.375 columns per block
    ("ci16_le", 1024, 2_400_000, 600_100, E.FFT_AUTO, 4, "hann"),      # generic, ragged
]


@pytest.mark.parametrize("fmt,nperseg,fs,block,impl,bpl,window", ORACLE_CASES, ids=lambda v: str(v))
def test_survey_matches_the_oracle(fmt, nperseg, fs, block, impl, bpl, window):
    launches = 2
    cap = _capture(fmt, fs, block, nperseg, launches * bpl)
    kw = _kw(fs, block, nperseg, window)
    P = parity.oracle_params(kw)
    ba = BatchAnalyzer(**parity.batch_kwargs(kw, fft_impl=impl, sample_format=fmt, blocks_per_launch=bpl, survey=True))
    dt = datetime.timedelta(seconds=block / fs)
    n_above = 0
    try:
        eng = ba.engine
        for k in range(launches):
            rec = eng.process(cap[k * bpl:(k + 1) * bpl].reshape(1, -1))
            noise, peak, above = eng.read_survey()
            surveys = ba.last_survey()
            for b in range(bpl):
                u = b
                _, _, S64 = R.spectrogram(FO.decode_samples(cap[k * bpl + b], fmt), fs, P.fft_window, nperseg)
                n_above += _check_unit(P, S64, eng.read_spectrogram(u), eng.read_row_means(u), noise[u], peak[u], above[u])
            # the BandSurvey is in the units of the Signals of the same block
            sigs = ba.finalize(rec, [T0 + k * bpl * dt])
            for u, (ss, keys) in enumerate(sigs):
                sv = surveys[u]
                assert sv.device == "0" and np.all(np.diff(sv.freqs) > 0)
                for s, (fi, start, _) in zip(ss, keys):
                    j = (fi + nperseg // 2) % nperseg
                    assert sv.freqs[j] == s.frequency and sv.noise_dbw[j] == s.noise
                    if start >= 0:                 # a run of this block only: its peak is one of the block's cells
                        assert sv.peak_dbw[j] >= s.max
                assert np.array_equal(sv.occupancy, np.fft.fftshift(above[u]) / ba.plan.T)
    finally:
        ba.close()
    assert n_above > 0


def _c2_analyzer(survey, **extra):
    w = synth.C2
    return BatchAnalyzer(devices=[str(i) for i in range(w.n_streams)], calibration_db=[0.0] * w.n_streams, sample_rate=w.sample_rate,
                         center_freq=w.center_freq, fft_nperseg=w.nperseg, fft_window="hamming",
                         signal_min_duration_ms=w.signal_min_duration_ms, signal_max_duration_ms=w.signal_max_duration_ms,
                         signal_threshold_dbw=w.signal_threshold_dbw, snr_threshold_db=w.snr_threshold_db,
                         sdr_callback_length=w.block_samples, survey=survey, **extra)


def test_survey_leaves_the_records_of_configs1_unchanged():
    w = synth.C2
    data = synth.make_batch(w, range(w.n_streams), 2)
    recs = {}
    for survey in (False, True):
        ba = _c2_analyzer(survey)
        try:
            eng = ba.engine
            eng.launch(data[0])
            eng.launch(data[1])                    # two launches in flight, as the benchmark runs them
            out = [eng.fetch().tobytes(), eng.fetch().tobytes()]
            recs[survey] = out
            if survey:                             # the lean schedule's survey, against the GPU's own cells
                noise, peak, above = eng.read_survey()
                for u in (0, w.n_streams - 1):
                    S32 = eng.read_spectrogram(u).T
                    assert np.array_equal(noise[u], eng.read_row_means(u))
                    assert np.array_equal(peak[u], S32.max(axis=1))
                    thr, snr = np.float32(ba.signal_threshold[u]), np.float32(ba.snr_threshold)
                    assert np.array_equal(above[u], (~(S32 < thr) & ~(S32 / noise[u][:, None] < snr)).sum(axis=1))
        finally:
            ba.close()
    assert recs[True] == recs[False] and all(len(r) > 0 for r in recs[True])


def _small(n_streams=3, impl=E.FFT_AUTO):
    kw = _kw(300_000, 300_000, 256)
    return BatchAnalyzer(**parity.batch_kwargs(kw, devices=[str(i) for i in range(n_streams)], calibration=[0.0] * n_streams,
                                               fft_impl=impl))


def test_survey_stream_contract():
    blocks = [np.stack([_capture("cu8", 300_000, 300_000, 256, 1, stream=10 * k + s)[0] for s in range(3)]) for k in range(3)]
    ref = []
    for blk in blocks:                              # every block alone: no carry enters the survey
        ba = _small()
        try:
            ba.engine.set_survey(True)
            ba.engine.process(blk)
            ref.append(ba.engine.read_survey())
        finally:
            ba.close()
    same = lambda a, b: all(np.array_equal(x, y) for x, y in zip(a, b))
    ba = _small()
    try:
        eng = ba.engine
        with pytest.raises(E.EngineError) as ei:   # nothing fetched yet
            eng.read_survey()
        assert ei.value.code == E.RT_ERR_INVALID
        eng.set_survey(True)
        eng.launch(blocks[0])
        eng.launch(blocks[1])                      # two launches in flight, each with its own survey
        eng.fetch()
        assert same(eng.read_survey(), ref[0])
        eng.fetch()
        assert same(eng.read_survey(), ref[1])
        eng.set_survey(False)                      # takes effect at the next launch
        eng.launch(blocks[2])
        eng.set_survey(True)
        eng.launch(blocks[0])
        eng.fetch()
        with pytest.raises(E.EngineError) as ei:
            eng.read_survey()
        assert ei.value.code == E.RT_ERR_INVALID
        eng.fetch()
        assert same(eng.read_survey(), ref[0])
        assert not same(ref[0], ref[1])
    finally:
        ba.close()


@pytest.mark.parametrize("impl", [E.FFT_GENERIC, E.FFT_AUTO])
def test_a_unit_alone_and_in_a_batch_gives_the_same_bits(impl):
    blk = np.stack([_capture("cu8", 300_000, 300_000, 256, 1, stream=40 + s)[0] for s in range(4)])

    def survey(rows):
        ba = _small(len(rows), impl)
        try:
            ba.engine.set_survey(True)
            ba.engine.process(rows)
            return ba.engine.read_survey()
        finally:
            ba.close()

    batch, alone, again = survey(blk), survey(blk[2:3]), survey(blk)      # in a batch, alone, and the batch once more
    for x, y, z in zip(batch, alone, again):
        assert np.array_equal(x[2], y[0]) and np.array_equal(x, z)


# ---------------------------------------------------------------------------------------------------------------------------
# wideband
# ---------------------------------------------------------------------------------------------------------------------------
FS, D, NPERSEG, CF = 20_000_000, 64, 256, 150_000_000


def _wide_keys(block, thr=-90.0):
    return dict(fft_nperseg=NPERSEG, fft_window="hamming", signal_min_duration_ms=8.0, signal_max_duration_ms=40.0,
                signal_threshold_dbw=thr, snr_threshold_db=5.0, sdr_callback_length=block)


def _wide_capture(block, nb, seed, sigma=0.02, tones=((1317, 0.02), (-6000, 0.01), (200, 0.01)), pulsed=True):
    """ci16_le: complex noise of `sigma` per component plus tones at (multiple of fs / (D nperseg), amplitude), on for 20 ms of
    every 100 ms (pulsed) or continuous."""
    rng = np.random.default_rng(seed)
    t = np.arange(nb * block)
    x = sigma * (rng.normal(size=t.size) + 1j * rng.normal(size=t.size))
    bw = FS / (D * NPERSEG)
    on = ((t + rng.integers(0, FS // 10)) % (FS // 10) < FS // 50) if pulsed else 1.0
    for m, a in tones:
        x += on * a * np.exp(2j * np.pi * (m * bw / FS) * t + 1j * rng.uniform(0, 2 * np.pi))
    return synth.quantise(x, "ci16_le")


def test_full_band_survey_puts_a_tone_where_float64_predicts_it():
    block, m, amp = 2_000_000, 1317, 0.25
    raw = _wide_capture(block, 2, 5, sigma=0.0, tones=((m, amp),), pulsed=False)
    wa = W.WidebandAnalyzer.full_band(devices=["rx"], calibration_db=[0.0], sample_rate=FS, center_freq=CF, decimation=D,
                                      sample_format="ci16_le", survey=True, **_wide_keys(block))
    try:
        for b in range(2):
            wa.process_blocks(raw[b * 2 * block:(b + 1) * 2 * block][None, :], [T0])
            (sv,) = wa.band_survey()
            half, bw, edge = NPERSEG // 2, FS / (D * NPERSEG), FS / 2 - FS / (4 * D)
            assert sv.device == "rx" and len(sv.freqs) == (2 * D - 1) * half
            assert abs(sv.freqs[0] - (CF - edge)) < 1e-6 and abs(sv.freqs[-1] + bw - (CF + edge)) < 1e-6
            assert np.all(np.abs(np.diff(sv.freqs) - bw) < 1e-6)
            # channel c = k + D - 1 with k the nearest grid channel, bin m - k n / 2 of its central half
            k = int(np.rint(m / half))
            idx = (k + D - 1) * half + (m - k * half) + NPERSEG // 4
            assert int(np.argmax(sv.peak_dbw)) == idx
            assert abs(sv.freqs[idx] - (CF + m * bw)) < 1e-6
            win = R.resolve_window("hamming", NPERSEG)
            expect = 10 * np.log10(amp ** 2 * win.sum() ** 2 / (FS / D * (win ** 2).sum()))
            assert abs(sv.peak_dbw[idx] - expect) <= 0.07 + 0.01, (sv.peak_dbw[idx], expect)
            # the channels' surveys, for comparison: the stitched bin is channel c's own
            chans = wa.last_survey()[0]
            assert chans[k + D - 1].peak_dbw[m - k * half + NPERSEG // 2] == sv.peak_dbw[idx]
    finally:
        wa.close()


def test_ddc_channel_surveys_match_the_filter_bank():
    block, nb = 2_000_000, 2
    raw = _wide_capture(block, nb, 7)
    fb = W.WidebandAnalyzer.full_band(devices=["rx"], calibration_db=[1.5], sample_rate=FS, center_freq=CF, decimation=D,
                                      sample_format="ci16_le", survey=True, **_wide_keys(block))
    ddc = W.WidebandAnalyzer(devices=["rx"], calibration_db=[1.5], sample_rate=FS, center_freq=CF, offsets_hz=W.grid_offsets(FS, D),
                             decimation=D, taps=fb.ddc.taps, sample_format="ci16_le", survey=True, **_wide_keys(block))
    try:
        with pytest.raises(ValueError):
            ddc.band_survey()
        n_busy = 0
        for b in range(nb):
            blk = raw[b * 2 * block:(b + 1) * 2 * block][None, :]
            fb.process_blocks(blk, [T0])
            ddc.process_blocks(blk, [T0])
            for a, c in zip(fb.last_survey()[0], ddc.last_survey()[0]):
                assert a.device == c.device and np.array_equal(a.freqs, c.freqs)
                for f in ("noise_dbw", "peak_dbw"):
                    la, lc = 10 ** (getattr(a, f) / 10), 10 ** (getattr(c, f) / 10)
                    assert np.all(np.abs(la - lc) <= 1e-3 * lc), f
                assert np.all(np.abs(a.occupancy - c.occupancy) * fb.channels.plan.T <= 1)
                n_busy += int(np.count_nonzero(a.occupancy))
    finally:
        fb.close()
        ddc.close()
    assert n_busy > 0


def test_survey_leaves_the_full_band_signals_unchanged():
    block, nb = 2_000_000, 2
    raw = _wide_capture(block, nb, 11)
    dt = datetime.timedelta(seconds=block / FS)
    got = {}
    for survey in (False, True):
        wa = W.WidebandAnalyzer.full_band(devices=["rx"], calibration_db=[0.0], sample_rate=FS, center_freq=CF, decimation=D,
                                          sample_format="ci16_le", survey=survey, **_wide_keys(block))
        try:
            out = []
            for b in range(nb):
                (chans,) = wa.process_blocks(raw[b * 2 * block:(b + 1) * 2 * block][None, :], [T0 + b * dt])
                # every channel's candidate keys and all of its Signals' fields, before the shadow filter
                out.append([(keys, [s.as_list for s in sigs]) for _, sigs, keys in chans])
            got[survey] = out
        finally:
            wa.close()
    assert got[True] == got[False]
    assert sum(len(keys) for blk in got[True] for keys, _ in blk) > 0
