"""CPU checks of the polyphase FFT filter bank's host side (include/rt_fbank.h, wideband.FilterBank, WidebandAnalyzer.full_band):
the polyphase + FFT form against the down-converter's float64 oracle, the grid helpers, the validation and the library's
exports."""
import ctypes
import os
import re

import numpy as np
import pytest

from pyradiotracking_b200 import build as B
from pyradiotracking_b200 import engine as E
from pyradiotracking_b200 import wideband as W
from tests import ddc_oracle as DO
from tests import fbank_oracle as FBO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("D", [4, 8, 64])
def test_polyphase_fft_form_equals_the_ddc_oracle_on_the_grid(D):
    rng = np.random.default_rng(D)
    C = 2 * D
    inc = W.grid_phase_increment(D).tolist()
    for L in (1, 7, 8 * D + 1, 16 * D + 1):
        h = rng.normal(0, 1, L)
        for n0 in (0, 7 * C, 3 * C + 5, (1 << 32) - 5, (1 << 32) - C, 3 * 10 ** 10 + 1):
            x = rng.normal(size=24 * D + 3) + 1j * rng.normal(size=24 * D + 3)
            hist = rng.normal(size=L - 1) + 1j * rng.normal(size=L - 1)
            want = DO.ddc(x, h, inc, D, n0, hist)
            got = FBO.fbank(x, h, D, n0, hist, chunk=7)
            assert got.shape == want.shape == (2 * D - 1, len(x) // D)
            scale = np.abs(h).sum() * np.abs(np.concatenate([hist, x])).max()
            assert np.abs(got - want).max() <= 1e-13 * scale, (D, L, n0, np.abs(got - want).max() / scale)


def test_grid_helpers():
    fs, D = 20_000_000, 64
    off = W.grid_offsets(fs, D)
    assert len(off) == 127 and off[0] == -63 * 156_250.0 and off[63] == 0.0 and off[-1] == 63 * 156_250.0
    # the grid's increments are the DDC's phase_increment of the same offsets, exactly
    assert W.grid_phase_increment(D).tolist() == W.phase_increment(off, fs).tolist()
    assert W.grid_phase_increment(4).tolist() == [(k % 8) << 29 for k in range(-3, 4)]
    assert W.FBANK_MIN_DECIMATION == 4 and W.FBANK_MAX_DECIMATION == 512


def test_filter_bank_and_full_band_reject_bad_plans():
    fs, block = 2_400_000, 2_400_000
    bad = [
        dict(decimation=2),                                         # below 4
        dict(decimation=6),                                         # not a power of two
        dict(decimation=1024, sample_rate=1024 * 3000, block_samples=1024 * 3000),
        dict(decimation=16, sample_rate=2_400_008),                 # fs % D
        dict(block_samples=2_400_004),                              # block % D
        dict(taps=np.ones(64)),                                     # even
        dict(taps=np.ones(16 * 8 + 3)),                             # more than 16 D + 1
        dict(taps=np.ones((3, 3))),
        dict(taps=np.r_[np.ones(6), np.inf]),
        dict(blocks_per_launch=0),
        dict(n_inputs=0),
        dict(n_inputs=65536),
        dict(sample_format="cs8x"),
    ]
    for extra in bad:
        kw = dict(sample_rate=fs, block_samples=block, decimation=8)
        kw.update(extra)
        with pytest.raises(ValueError):
            W.FilterBank(**kw)
    base = dict(devices=["0"], calibration_db=[0.0], sample_rate=fs, center_freq=150_000_000, decimation=8, fft_nperseg=256,
                fft_window="hamming", signal_min_duration_ms=8, signal_max_duration_ms=40, signal_threshold_dbw=-90,
                snr_threshold_db=5)
    for extra in (dict(sdr_callback_length=8 * 511),                # 511 channel samples: one segment of 256
                  dict(calibration_db=[0.0, 1.0]),
                  dict(decimation=12),
                  # 65 inputs * 1023 channels = 66495 analyzer units: more than the engine's 65535
                  dict(devices=[str(i) for i in range(65)], calibration_db=[0.0] * 65, sample_rate=512 * 4000, decimation=512,
                       fft_nperseg=256),
                  dict(devices=[str(i) for i in range(3)], calibration_db=[0.0] * 3, decimation=256, sample_rate=256 * 10_000,
                       fft_nperseg=256, sdr_callback_length=256 * 10_000, blocks_per_launch=86)):   # 3 * 511 * 86 > 65535
        with pytest.raises(ValueError):
            W.WidebandAnalyzer.full_band(**dict(base, **extra))


def test_library_exports_the_fbank_header_and_validates_before_touching_a_device():
    B.build()
    lib = W._load()
    hdr = open(os.path.join(ROOT, "include", "rt_fbank.h")).read()
    declared = set(re.findall(r"^(?:int|void)\s+(rt_[a-z0-9_]+)\s*\(", hdr, re.M))
    assert declared == set(W.FBANK_EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    # abi_version .. decimation (16) + block_samples (8) + n_taps, sample_format, reserved (12) + padding (4) + sample_rate,
    # taps (16)
    assert ctypes.sizeof(W.RtFbankConfig) == 56
    assert re.search(r"#define RT_FBANK_ABI_VERSION (\d+)", hdr).group(1) == str(W.RT_FBANK_ABI_VERSION)
    assert re.search(r"#define RT_FBANK_MIN_DECIMATION (\d+)", hdr).group(1) == str(W.FBANK_MIN_DECIMATION)
    assert re.search(r"#define RT_FBANK_MAX_DECIMATION (\d+)", hdr).group(1) == str(W.FBANK_MAX_DECIMATION)
    h = np.ones(33)

    def create(**kw):
        cfg = dict(abi_version=W.RT_FBANK_ABI_VERSION, cuda_device=0, n_inputs=1, decimation=8, block_samples=4096, n_taps=33,
                   sample_format=E.SAMPLE_CI16, reserved=0, sample_rate=1e6, taps=h.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
        cfg.update(kw)
        out = ctypes.c_void_p()
        rc = lib.rt_fbank_create(ctypes.byref(W.RtFbankConfig(**cfg)), ctypes.byref(out))
        if rc == E.RT_OK:
            lib.rt_fbank_destroy(out)
        return rc, lib.rt_last_error().decode()

    for kw, word in ((dict(n_taps=32), "n_taps"), (dict(n_taps=16 * 8 + 3), "n_taps"), (dict(decimation=2), "decimation"),
                     (dict(decimation=12), "decimation"), (dict(decimation=1024, block_samples=8192), "decimation"),
                     (dict(block_samples=4100), "block_samples"), (dict(sample_format=4), "sample_format"),
                     (dict(abi_version=99), "abi_version"), (dict(reserved=1), "reserved"), (dict(n_inputs=0), "n_inputs")):
        rc, msg = create(**kw)
        assert rc == E.RT_ERR_INVALID and word in msg, (kw, msg)
