"""Input sample formats on the CPU: the float64 decoding of tests/format_oracle.py against scipy, the synthetic captures per
format, the capture reader (element sizes, tails, SigMF metadata) and the checks of the binding that need no GPU."""
import json

import numpy as np
import pytest

from oracle import restatement as R
from pyradiotracking_b200 import engine as E
from pyradiotracking_b200 import synth
from pyradiotracking_b200.replay import CaptureReader, sigmf_sample_format
from tests import format_oracle as FO

FORMATS = ["cu8", "ci8", "ci16_le", "cf32_le"]
ELEMENT = {"cu8": np.uint8, "ci8": np.int8, "ci16_le": np.int16, "cf32_le": np.float32}


def test_decode_samples_follows_the_normalisation_table():
    raw = {"cu8": np.array([0, 255, 128, 127], np.uint8), "ci8": np.array([-128, 127, 0, -1], np.int8),
           "ci16_le": np.array([-32768, 32767, 0, -1], "<i2"), "cf32_le": np.array([-1.5, 0.25, 0.0, -1e-3], "<f4")}
    want = {"cu8": [-1 + 1j, 128 / 127.5 - 1 + (127 / 127.5 - 1) * 1j], "ci8": [-1 + 127 / 128 * 1j, -1j / 128],
            "ci16_le": [-1 + 32767 / 32768 * 1j, -1j / 32768], "cf32_le": [-1.5 + 0.25j, -1j * float(np.float32(1e-3))]}
    for fmt in FORMATS:
        x = FO.decode_samples(raw[fmt], fmt)
        assert x.dtype == np.complex128 and x.shape == (2,)
        np.testing.assert_array_equal(x, np.array(want[fmt]))
        np.testing.assert_array_equal(FO.decode_samples(raw[fmt].view(np.uint8), fmt), x)      # the bytes of a recording
    np.testing.assert_array_equal(FO.decode_samples(raw["cu8"], "cu8"), R.bytes_to_iq(raw["cu8"]))


def test_sample_oracle_on_decoded_cu8_equals_the_byte_oracle():
    """The format oracle's entry for decoded samples gives what the restatement gives for the same bytes, block by block."""
    import datetime

    cap = synth.make_stream(synth.C1, 0, 2)
    P = R.Params.make()
    a, b = R.OracleAnalyzer(P), FO.SampleOracle(P)
    t0 = datetime.datetime(2026, 1, 1)
    for blk in cap:
        fa, ta, Sa, founda, kepta = a.process_block(blk, t0)
        fb, tb, Sb, foundb, keptb = b.process_samples(FO.decode_samples(blk, "cu8"), t0)
        assert np.array_equal(Sa, Sb) and founda == foundb and kepta == keptb
    assert len(founda) > 0


@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("nperseg,window", [(256, "hamming"), (1024, "hann"), (64, ("kaiser", 6.0))])
def test_decoded_spectrogram_matches_scipy(fmt, nperseg, window):
    scipy_signal = pytest.importorskip("scipy.signal")
    raw = synth.make_stream_format(synth.C1, fmt, 5, 1)[0][: 2 * 40_000]
    x = FO.decode_samples(raw, fmt)
    f0, t0, s0 = scipy_signal.spectrogram(x, fs=300000, window=window, nperseg=nperseg, noverlap=0, return_onesided=False)
    f1, t1, s1 = R.spectrogram(x, 300000, window, nperseg)
    assert np.array_equal(f0, f1) and np.array_equal(t0, t1)
    np.testing.assert_allclose(s1, s0, rtol=1e-9)


def test_synthetic_formats_carry_one_signal():
    """Every format quantises the same complex signal: the decoded samples agree to the coarser format's step."""
    ref = FO.decode_samples(synth.make_stream_format(synth.C1, "cf32_le", 3, 1), "cf32_le")
    for fmt, step in (("cu8", 1 / 127.5), ("ci8", 1 / 128), ("ci16_le", 1 / 32768)):
        raw = synth.make_stream_format(synth.C1, fmt, 3, 1)
        assert raw.dtype == ELEMENT[fmt] and raw.shape == (1, 2 * synth.C1.block_samples)
        x = FO.decode_samples(raw, fmt)
        assert np.max(np.abs((x - ref).view(np.float64))) <= 0.5 * step + 1e-6
    with pytest.raises(ValueError):
        synth.make_stream_format(synth.C1, "ci12", 3, 1)


def _write(tmp_path, arrays, meta=None):
    paths = []
    for i, a in enumerate(arrays):
        p = tmp_path / f"chan{i}.sigmf-data"
        a.tofile(p)
        if meta is not None:
            (tmp_path / f"chan{i}.sigmf-meta").write_text(json.dumps({"global": {"core:datatype": meta[i]}}))
        paths.append(str(p))
    return paths


@pytest.mark.parametrize("fmt", FORMATS)
def test_reader_reads_elements_of_the_format_and_drops_the_tail(tmp_path, fmt):
    rng = np.random.default_rng(3)
    N = 700
    dt = ELEMENT[fmt]
    a = rng.integers(-100, 100, 2 * N * 4, dtype=np.int64).astype(dt)
    b = rng.integers(-100, 100, 2 * N * 6, dtype=np.int64).astype(dt)
    ba = np.concatenate([a.view(np.uint8), np.full(dt(0).itemsize * 2 * N - 1, 7, np.uint8)])   # a tail one byte short of a block
    paths = _write(tmp_path, [ba, b])
    r = CaptureReader(paths, N, n_buffers=3, pinned=False, sample_format=fmt)
    assert r.n_blocks == 4 and r.block_bytes == 2 * N * dt(0).itemsize
    seen = []
    for k, blk in r:
        assert blk.dtype == dt and blk.shape == (2, 2 * N)
        assert np.array_equal(blk[0], a[2 * N * k: 2 * N * (k + 1)]) and np.array_equal(blk[1], b[2 * N * k: 2 * N * (k + 1)])
        seen.append(k)
    assert seen == list(range(4))
    got = [(k, blk.copy()) for k, blk in CaptureReader(paths, N, pinned=False, blocks_per_read=3, sample_format=fmt)]
    assert [k for k, _ in got] == [0, 3]
    assert got[1][1].shape == (2, 3 * 2 * N) and not got[1][1][:, 2 * N:].any()        # last group: one block and zero padding


def test_reader_takes_the_format_from_sigmf_metadata(tmp_path):
    x = np.arange(2 * 100 * 3, dtype="<i2")
    paths = _write(tmp_path, [x, x], meta=["ci16_le", "ci16_le"])
    assert sigmf_sample_format(paths[0]) == "ci16_le"
    r = CaptureReader(paths, 100, pinned=False)
    assert r.sample_format == "ci16_le" and r.n_blocks == 3
    assert all(blk.dtype == np.int16 for _, blk in r)
    assert CaptureReader(paths, 100, pinned=False, sample_format="ci16_le").n_blocks == 3
    with pytest.raises(ValueError, match="SigMF"):
        CaptureReader(paths, 100, pinned=False, sample_format="cu8")                    # metadata contradicts the caller
    paths = _write(tmp_path, [x, x], meta=["ci16_le", "cf32_le"])
    with pytest.raises(ValueError):
        CaptureReader(paths, 100, pinned=False)                                        # files disagree
    for bad in ("ci16_be", "rf32_le", "cu16_le", None):
        paths = _write(tmp_path, [x], meta=[bad])
        with pytest.raises(ValueError, match="core:datatype"):
            CaptureReader(paths, 100, pinned=False)
    plain = tmp_path / "plain.bin"
    x.tofile(plain)
    assert sigmf_sample_format(str(plain)) is None
    assert CaptureReader([str(plain)], 100, pinned=False).sample_format == "cu8"
    with pytest.raises(ValueError):
        CaptureReader([str(plain)], 100, pinned=False, sample_format="sc16")


class _Cai:
    """A CuPy / Numba style device array (only the interface is read)."""

    def __init__(self, shape, typestr, strides=None, ptr=0x10000):
        self.__cuda_array_interface__ = dict(shape=shape, typestr=typestr, data=(ptr, False), version=3, strides=strides)


def test_device_pointer_checks_element_type_and_row_bytes():
    i16, c64, f32 = ("int16",), ("float32", "complex64"), ("float32",)
    assert E._device_pointer(_Cai((3, 200), "<i2"), 3, 400, i16) == (0x10000, 400)
    assert E._device_pointer(_Cai((3, 100), "<c8"), 3, 800, c64) == (0x10000, 800)
    assert E._device_pointer(_Cai((3, 200), "<f4", strides=(1024, 4)), 3, 800, c64) == (0x10000, 1024)
    assert E._device_pointer(_Cai((400,), "|u1"), 1, 400) == (0x10000, 400)
    with pytest.raises(TypeError):
        E._device_pointer(_Cai((3, 200), "|u1"), 3, 400, i16)
    with pytest.raises(TypeError):
        E._device_pointer(_Cai((3, 200), ">i2"), 3, 400, i16)                         # big-endian
    with pytest.raises(TypeError):
        E._device_pointer(_Cai((3, 200), "<i2"), 3, 400, f32)
    with pytest.raises(ValueError):
        E._device_pointer(_Cai((3, 199), "<i2"), 3, 400, i16)                         # a row is checked in bytes
    with pytest.raises(ValueError):
        E._device_pointer(_Cai((3, 200), "<i2", strides=(400, 4)), 3, 400, i16)      # not dense
    assert E._device_pointer(np.zeros(4), 1, 32) is None                              # host memory


def test_sample_format_names_and_codes():
    assert [E.sample_format_name(f) for f in FORMATS] == FORMATS
    assert [E.sample_format_name(E.SAMPLE_FORMATS[f][0]) for f in FORMATS] == FORMATS
    assert E.RtConfig.sample_format.offset == E.RtConfig.blocks_per_launch.offset + 4        # rt_config.reserved[0] of ABI 2
    assert E.RtConfig.reserved.offset == E.RtConfig.sample_format.offset + 4 and E.RtConfig.reserved.size == 8
    for bad in ("ci12", 4, -1, "CU8"):
        with pytest.raises(ValueError):
            E.sample_format_name(bad)


def test_batch_analyzer_validates_the_format():
    from pyradiotracking_b200.analyze import BatchAnalyzer

    kw = dict(devices=["0"], calibration_db=[0.0], sample_rate=300000, center_freq=150_150_000, fft_nperseg=256,
              fft_window="hamming", signal_min_duration_ms=8, signal_max_duration_ms=40, signal_threshold_dbw=-90.0,
              snr_threshold_db=5.0)
    assert BatchAnalyzer(**kw).sample_format == "cu8"
    assert BatchAnalyzer(**kw, sample_format="cf32_le").sample_format == "cf32_le"
    with pytest.raises(ValueError, match="sample_format"):
        BatchAnalyzer(**kw, sample_format="sc16")
