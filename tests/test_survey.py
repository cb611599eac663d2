"""Band survey on the host (no GPU): the conversions to Signal conventions, the full-band stitching, replay's regrouping and the
error paths, with the engine stubbed."""
import ctypes
import datetime

import numpy as np
import pytest

from pyradiotracking_b200 import engine as E
from pyradiotracking_b200 import replay as RP
from pyradiotracking_b200 import wideband as W
from pyradiotracking_b200.analyze import BatchAnalyzer
from pyradiotracking_b200.survey import BandSurvey, stitch


class _StubEngine:
    def __init__(self, noise, peak, above):
        self.arrays = (noise, peak, above)

    def read_survey(self):
        return self.arrays


def _analyzer(devices, cal, fs, cf, nperseg, block, bpl=1):
    return BatchAnalyzer(devices=devices, calibration_db=cal, sample_rate=fs, center_freq=cf, fft_nperseg=nperseg,
                         fft_window="hamming", signal_min_duration_ms=8.0, signal_max_duration_ms=40.0, signal_threshold_dbw=-90.0,
                         snr_threshold_db=5.0, sdr_callback_length=block, blocks_per_launch=bpl, survey=True)


def _stub(ba, seed=0):
    rng = np.random.default_rng(seed)
    shape = (ba.n_units, ba.fft_nperseg)
    noise = rng.uniform(1e-11, 1e-9, shape).astype(np.float32)
    peak = (noise * rng.uniform(1, 100, shape)).astype(np.float32)
    above = rng.integers(0, ba.plan.T + 1, shape).astype(np.int32)
    ba._engine = _StubEngine(noise, peak, above)
    return noise, peak, above


@pytest.mark.parametrize("cf", [150_150_000, [150_100_000, 150_175_000.5]])
def test_unit_surveys_follow_the_signal_conventions(cf):
    ba = _analyzer(["a", "b"], [0.0, 2.5], 300_000, cf, 256, 300_000, bpl=3)
    noise, peak, above = _stub(ba)
    sv = ba.last_survey()
    assert [s.device for s in sv] == ["a"] * 3 + ["b"] * 3          # stream-major, block-minor
    # the finaliser's own arithmetic on records carrying these values at every bin
    fi = np.arange(256)
    for u in range(6):
        rec = np.zeros(256, dtype=E.RECORD_DTYPE)
        rec["stream"], rec["fi"], rec["start"], rec["end"] = u, fi, 10, 20
        rec["max_lin"], rec["row_mean"], rec["mean_lin"] = peak[u], noise[u], noise[u]
        fin = ba.finalize_arrays(rec)
        j = (fi + 128) % 256                                         # fftshifted position of bin fi
        assert np.array_equal(sv[u].freqs[j], fin.frequency)
        assert np.array_equal(sv[u].noise_dbw[j], fin.noise)
        assert np.array_equal(sv[u].peak_dbw[j], fin.max)
        assert np.array_equal(sv[u].occupancy[j], above[u] / ba.plan.T)
        assert np.all(np.diff(sv[u].freqs) > 0)


def _full_band_stub(D, nperseg, n_inputs=2, bpl=2, fs=20_000_000, cf=150_000_000, front=W.FilterBank):
    """A WidebandAnalyzer over the full_band grid whose channel analyzer reads a stubbed engine: noise = 1 + unit * 1000 + fi."""
    wa = W.WidebandAnalyzer.__new__(W.WidebandAnalyzer)
    wa.ddc = front.__new__(front)
    wa.devices = [f"rx{i}" for i in range(n_inputs)]
    wa.n_streams, wa.n_channels, wa.blocks_per_launch = n_inputs, 2 * D - 1, bpl
    C = wa.n_channels
    block = D * nperseg * 4
    wa.channels = _analyzer([f"{d}:{c}" for d in wa.devices for c in range(C)], [0.5] * (n_inputs * C), fs // D,
                            W.channel_center_freqs(cf, W.grid_offsets(fs, D)) * n_inputs, nperseg, block // D, bpl)
    units = n_inputs * C * bpl
    noise = (1 + 1000 * np.arange(units)[:, None] + np.arange(nperseg)[None, :]).astype(np.float32)
    wa.channels._engine = _StubEngine(noise, noise * 2, np.zeros_like(noise, dtype=np.int32))
    return wa


@pytest.mark.parametrize("D,nperseg", [(4, 8), (64, 256), (8, 4096)])
def test_full_band_stitching(D, nperseg):
    fs, cf, bpl = 20_000_000, 150_000_000, 2
    wa = _full_band_stub(D, nperseg, bpl=bpl)
    chans = wa.last_survey()
    st = wa.band_survey()
    assert len(st) == len(chans) == 2 * bpl and [s.device for s in st] == ["rx0", "rx0", "rx1", "rx1"]
    bw, edge, half = fs / (D * nperseg), fs / 2 - fs / (4 * D), nperseg // 2
    for u, s in enumerate(st):
        assert len(s.freqs) == (2 * D - 1) * half
        assert s.freqs[0] == pytest.approx(cf - edge, abs=1e-6) and s.freqs[-1] + bw == pytest.approx(cf + edge, abs=1e-6)
        assert np.allclose(np.diff(s.freqs), bw, rtol=0, atol=1e-6)           # uniform, ascending, no gap, no overlap
        i, b = divmod(u, bpl)
        for c in range(2 * D - 1):
            piece = slice(c * half, (c + 1) * half)
            ch = chans[u][c]
            assert np.array_equal(s.freqs[piece], ch.freqs[nperseg // 4: 3 * nperseg // 4])   # the channel's own float64 values
            k = np.arange(-nperseg // 4, nperseg // 4)                         # central half of channel c, bins k
            unit = (i * (2 * D - 1) + c) * bpl + b
            assert np.allclose(10 ** (s.noise_dbw[piece] / 10), 1 + 1000 * unit + k % nperseg, rtol=1e-12, atol=0)
            assert np.array_equal(s.peak_dbw[piece], ch.peak_dbw[nperseg // 4: 3 * nperseg // 4])


def test_band_survey_needs_the_full_band_grid():
    wa = _full_band_stub(4, 8, front=W.Channelizer)
    assert len(wa.last_survey()) == 4
    with pytest.raises(ValueError):
        wa.band_survey()
    with pytest.raises(ValueError):
        stitch("x", [BandSurvey("x", *(np.zeros(6),) * 4)])


def test_replay_hands_the_surveys_of_each_block(tmp_path):
    B, n_streams, block = 3, 2, 64

    class Stub:
        sample_rate, block_samples, blocks_per_launch, sample_format = 1000, block, B, "cu8"

        def __init__(self):
            self.n_streams, self.launches = n_streams, 0

        def submit(self, iq):
            self.launches += 1

        def collect(self, ts):
            return [("res", self.launches, u) for u in range(n_streams * B)]

        def last_survey(self):
            return [("survey", self.launches, u) for u in range(n_streams * B)]

    paths = []
    for s in range(n_streams):
        p = tmp_path / f"s{s}.cu8"
        np.zeros(2 * block * 7, np.uint8).tofile(p)                    # 7 blocks: the last group of 3 is ragged
        paths.append(str(p))
    got, blocks = {}, []
    an = Stub()
    n = RP.replay(paths, an, datetime.datetime(2026, 1, 1), on_block=lambda b, r: blocks.append((b, r)),
                  on_survey=lambda b, s: got.__setitem__(b, s), pinned=False)
    assert n == 7 and sorted(got) == list(range(7))
    for b, res in blocks:
        sv = got[b]
        assert [x[2] for x in sv] == [r[2] for r in res] == [s * B + b % B for s in range(n_streams)]
        assert [x[1] for x in sv] == [r[1] for r in res]                # from the same collect


def test_survey_entry_points_reject_a_null_engine():
    lib = E.load_library()
    assert lib.rt_engine_set_survey(None, 1) == E.RT_ERR_INVALID
    assert lib.rt_engine_read_survey(None, None, None, None) == E.RT_ERR_INVALID
    eng = E.Engine.__new__(E.Engine)
    eng._lib, eng._h, eng.n_units, eng.nperseg = lib, ctypes.c_void_p(), 1, 8
    with pytest.raises(E.EngineError) as ei:
        eng.read_survey()
    assert ei.value.code == E.RT_ERR_INVALID
    with pytest.raises(E.EngineError):
        eng.set_survey(True)
