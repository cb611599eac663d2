"""CPU checks of the wideband down-converter's host side (pyradiotracking_b200/wideband.py, include/rt_ddc.h): the float64
oracle against a textbook formulation, the helpers, the validation, the library's exports, and per-device centre frequencies."""
import ctypes
import datetime
import os
import re

import numpy as np
import pytest

from oracle import restatement as R
from pyradiotracking_b200 import build as B
from pyradiotracking_b200 import engine as E
from pyradiotracking_b200 import wideband as W
from pyradiotracking_b200.analyze import BatchAnalyzer
from tests import ddc_oracle as DO
from tests import format_oracle as FO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _raw(fmt, n, rng):
    dt = FO.SAMPLE_FORMATS[fmt][0]
    if fmt == "cf32_le":
        return rng.normal(0, 0.3, 2 * n).astype(dt)
    info = np.iinfo(dt)
    return rng.integers(info.min, info.max + 1, 2 * n).astype(dt)


def _textbook(x, h, inc, D, n0, hist):
    """Mix to baseband (x[n] exp(-2 pi i f n), f = inc / 2^32), np.convolve with h, keep every D-th sample."""
    L = len(h)
    xx = np.concatenate([hist, x])
    n = np.arange(n0 - (L - 1), n0 + len(x), dtype=object)
    mixed = xx * np.exp(-2j * np.pi * DO.phase_turns(inc, n))
    conv = np.convolve(mixed, h)
    return conv[L - 1: L - 1 + len(x)][::D][: len(x) // D]


@pytest.mark.parametrize("fmt", ["cu8", "ci8", "ci16_le", "cf32_le"])
def test_oracle_equals_mix_convolve_decimate(fmt):
    rng = np.random.default_rng(7 + len(fmt))
    for D, L, n0 in ((4, 33, (1 << 40) - 17), (8, 65, 3 * 10 ** 10 + 5), (5, 7, 0), (3, 1, 12345)):
        x = FO.decode_samples(_raw(fmt, 40 * D + 3, rng), fmt)
        h = rng.normal(0, 1, L)
        incs = [int(v) for v in rng.integers(0, 1 << 32, 3)] + [0, (1 << 32) - 1]
        hist = FO.decode_samples(_raw(fmt, L - 1, rng), fmt)
        y = DO.ddc(x, h, incs, D, n0, hist)
        assert y.shape == (len(incs), len(x) // D)
        for c, inc in enumerate(incs):
            want = _textbook(x, h, inc, D, n0, hist)
            assert np.max(np.abs(y[c] - want)) <= 1e-12 * max(1.0, np.max(np.abs(want))), (D, L, c)
    # zero history is the default, and the history continues a stream: two halves equal the whole
    x = FO.decode_samples(_raw(fmt, 64 * 8, rng), fmt)
    h = rng.normal(0, 1, 17)
    whole = DO.ddc(x, h, [12345678], 8, n0=1 << 40)
    first = DO.ddc(x[:256], h, [12345678], 8, n0=1 << 40)
    second = DO.ddc(x[256:], h, [12345678], 8, n0=(1 << 40) + 256, history=x[256 - 16:256])
    assert np.max(np.abs(np.concatenate([first, second], axis=1) - whole)) <= 1e-12


def test_phase_increment_timestamp_and_frequency_helpers():
    fs = 20_000_000
    inc = W.phase_increment([0.0, fs / 4, -fs / 4, -fs / 2, 1.0, 2_345_678.9], fs)
    assert inc.dtype == np.uint32
    assert inc.tolist() == [0, 1 << 30, 3 << 30, 1 << 31, round(2 ** 32 / fs), round(2_345_678.9 / fs * 2 ** 32)]
    # the increment is the offset to within half a unit of 2^-32 fs (0.0023 Hz at 20 MS/s)
    assert abs((int(inc[5]) / 2 ** 32) * fs - 2_345_678.9) <= fs / 2 ** 33
    t = datetime.datetime(2026, 3, 1, 12, 0, 0, 123456)
    assert W.channel_ts(t, 513, fs) == t - datetime.timedelta(seconds=512 / (2 * fs))
    assert W.channel_ts(t, 513, 2_400_000) == t - datetime.timedelta(microseconds=107)
    assert W.channel_ts(t, 1, fs) == t
    assert W.channel_center_freqs(150_150_000, [0, -1_250_000, 2_500_000.5]) == [150_150_000, 148_900_000, 152_650_000.5]
    h = W.default_taps(8)
    assert len(h) == 65 and abs(h.sum() - 1.0) < 1e-12 and np.allclose(h, h[::-1])


def test_channelizer_and_wideband_analyzer_reject_bad_plans():
    fs, block = 2_400_000, 2_400_000
    bad = [
        dict(decimation=1),                                         # D < 2
        dict(decimation=7),                                         # fs % D
        dict(block_samples=2_400_004, decimation=8),                # block % D
        dict(offsets_hz=[1_100_000.0]),                             # 1.1 MHz + 150 kHz half-width > 1.2 MHz
        dict(offsets_hz=[0.0, -1_050_001.0]),
        dict(taps=np.ones(64)),                                     # even
        dict(taps=np.ones(W.MAX_TAPS + 2)),                         # oversized
        dict(taps=np.ones((3, 3))),
        dict(decimation=2048, offsets_hz=[0.0]),
    ]
    for extra in bad:
        kw = dict(sample_rate=fs, block_samples=block, offsets_hz=[0.0, 500_000.0], decimation=8)
        kw.update(extra)
        with pytest.raises(ValueError):
            W.Channelizer(**kw)
    base = dict(devices=["0"], calibration_db=[0.0], sample_rate=fs, center_freq=150_000_000, offsets_hz=[0.0], decimation=8,
                fft_nperseg=256, fft_window="hamming", signal_min_duration_ms=8, signal_max_duration_ms=40,
                signal_threshold_dbw=-90, snr_threshold_db=5)
    with pytest.raises(ValueError):
        W.WidebandAnalyzer(**dict(base, sdr_callback_length=8 * 511))     # 511 channel samples: one segment of 256
    with pytest.raises(ValueError):
        W.WidebandAnalyzer(**dict(base, calibration_db=[0.0, 1.0]))
    with pytest.raises(ValueError):
        W.WidebandAnalyzer(**dict(base, offsets_hz=[1_150_000.0]))


def test_library_exports_the_ddc_header_and_validates_before_touching_a_device():
    B.build()
    lib = W._load()
    hdr = open(os.path.join(ROOT, "include", "rt_ddc.h")).read()
    declared = set(re.findall(r"^(?:int|void)\s+(rt_[a-z0-9_]+)\s*\(", hdr, re.M))
    assert declared == set(W.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    assert ctypes.sizeof(W.RtDdcConfig) == 64
    h = np.ones(33)
    inc = np.zeros(2, np.uint32)

    def create(**kw):
        cfg = dict(abi_version=W.RT_DDC_ABI_VERSION, cuda_device=0, n_inputs=1, n_channels=2, block_samples=4096, decimation=8,
                   n_taps=33, sample_format=E.SAMPLE_CI16, reserved=0, sample_rate=1e6,
                   taps=h.ctypes.data_as(ctypes.POINTER(ctypes.c_double)), phase_inc=inc.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)))
        cfg.update(kw)
        out = ctypes.c_void_p()
        rc = lib.rt_ddc_create(ctypes.byref(W.RtDdcConfig(**cfg)), ctypes.byref(out))
        if rc == E.RT_OK:
            lib.rt_ddc_destroy(out)
        return rc, lib.rt_last_error().decode()

    for kw, word in ((dict(n_taps=32), "n_taps"), (dict(n_taps=W.MAX_TAPS + 2), "n_taps"), (dict(decimation=1), "decimation"),
                     (dict(decimation=W.MAX_DECIMATION + 1), "decimation"), (dict(block_samples=4100), "block_samples"),
                     (dict(sample_format=4), "sample_format"), (dict(abi_version=99), "abi_version"), (dict(reserved=1), "reserved")):
        rc, msg = create(**kw)
        assert rc == E.RT_ERR_INVALID and word in msg, (kw, msg)


def test_per_device_center_freq_gives_the_oracle_frequencies():
    fs, n = 300_000, 256
    offsets = [0, -1_250_000, 2_500_000.5]
    cfs = W.channel_center_freqs(150_150_000, offsets)
    kw = dict(devices=["a:0", "a:1", "a:2"], calibration_db=[0.0] * 3, sample_rate=fs, fft_nperseg=n, fft_window="hamming",
              signal_min_duration_ms=8, signal_max_duration_ms=40, signal_threshold_dbw=-90, snr_threshold_db=5)
    rec = np.zeros(9, dtype=E.RECORD_DTYPE)
    rec["stream"] = np.repeat(np.arange(3), 3)
    rec["fi"] = [0, 17, 255] * 3
    rec["start"], rec["end"], rec["max_lin"], rec["row_mean"], rec["mean_lin"] = 3, 40, 1e-6, 1e-9, 1e-7
    freqs = np.fft.fftfreq(n, 1 / fs)
    ba = BatchAnalyzer(center_freq=cfs, **kw)
    fin = ba.finalize_arrays(rec)
    for s, fi, f in zip(fin.stream, fin.fi, fin.frequency):
        P = R.Params.make(sample_rate=fs, center_freq=cfs[s])
        assert f == float(freqs[fi] + P.center_freq)                        # the oracle's expression, bit for bit
    # a scalar behaves as before; a wrong count is refused
    one = BatchAnalyzer(center_freq=150_150_000, **kw).finalize_arrays(rec)
    assert one.frequency.tolist() == (freqs[rec["fi"]] + 150_150_000).tolist()
    with pytest.raises(ValueError):
        BatchAnalyzer(center_freq=cfs[:2], **kw)
