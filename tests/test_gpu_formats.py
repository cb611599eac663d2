"""Input sample formats (ci8, ci16_le, cf32_le) on the B200 (pytest -m gpu), against the float64 oracle on the decoded samples.

  every kernel that serves a format: ci8 on the generic, register, tensor-core and radix-16 kernels; ci16_le / cf32_le on the
  generic kernel at nperseg 8, 256, 2048 and 4096 (RT_FFT_AUTO picks it for them)
  blocks_per_launch > 1, two launches in flight and a ragged block length; device tensors; replay of files; rejected
  combinations; and a GNU Radio (gr-osmosdr) cf32 recording of RTL-SDR bytes against the cu8 path on the original bytes
"""
import datetime
import json
import math
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import restatement as R
from pyradiotracking_b200 import engine as E
from pyradiotracking_b200 import synth
from pyradiotracking_b200.analyze import BatchAnalyzer
from pyradiotracking_b200.replay import CaptureReader, replay
from tests import format_oracle as FO
from tests import parity

pytestmark = pytest.mark.gpu

T0 = datetime.datetime(2026, 6, 6, 6, 6, 6)


def _kw(fs, block, nperseg, window="hamming", calibration_db=0.0):
    return dict(device="0", calibration_db=calibration_db, sample_rate=fs, center_freq=150_150_000, fft_nperseg=nperseg,
                fft_window=window, signal_min_duration_ms=8.0, signal_max_duration_ms=40.0, signal_threshold_dbw=-90.0,
                snr_threshold_db=5.0, sdr_callback_length=block)


def _capture(fmt, fs, block, nperseg, nb, stream=1):
    """[nb, 2 block] elements of `fmt`: noise and tone bursts (one straddling every block boundary) quantised to the format."""
    # bursts of 10-30 LSB; 6-20 LSB from nperseg 2048 on, where louder tones push the float32 floor of the cells 50 dB under them
    # (parity.DEEP_RTOL) to the limit in every format, cu8 included
    amp = (6.0, 20.0) if nperseg >= 2048 else (10.0, 30.0)
    w = synth.Workload(91, f"formats-{nperseg}-{fs}-{block}", fs, block, nperseg=nperseg, amp_lsb=amp)
    return synth.make_stream_format(w, fmt, stream, nb)


def _ts(kw, b):
    return parity.block_ts(T0, b, kw["sdr_callback_length"], kw["sample_rate"])


def _oracle(kw, cap, fmt):
    """[(S, last, found)] of the float64 oracle on the decoded samples of every block."""
    P = parity.oracle_params(kw)
    ora = FO.SampleOracle(P)
    out = []
    for b in range(len(cap)):
        last = ora.last
        _, _, S, found, _ = ora.process_samples(FO.decode_samples(cap[b], fmt), _ts(kw, b))
        out.append((S, last, found))
    return P, out


def _run_vs_oracle(kw, cap, fmt, impl, tag, want=None, **extra):
    """One stream block by block through BatchAnalyzer: records and spectrogram against the oracle; -> totals, carried
    records, the raw records of every block."""
    P, want = want if want is not None else _oracle(kw, cap, fmt)
    ba = BatchAnalyzer(**parity.batch_kwargs(kw, fft_impl=impl, sample_format=fmt, **extra))
    tot = dict(oracle=0, gpu=0, near_threshold_mismatch=0)
    carried, recs = 0, []
    try:
        for b, (S, last, found) in enumerate(want):
            rec = ba.engine.process(cap[b][None, :])
            recs.append(rec.tobytes())
            sigs, keys = ba.finalize(rec, [_ts(kw, b)])[0]
            st = parity.compare_block(P, S, last, found, sigs, keys)
            parity.compare_spectrogram(P, S, ba.engine.read_spectrogram(0), ba.engine.read_row_means(0), tag=f"{tag}/b{b}")
            for k in tot:
                tot[k] += st[k]
            carried += sum(1 for k in keys if k[1] < 0)
    finally:
        ba.close()
    return tot, carried, recs


# ---------------------------------------------------------------------------------------------------------------------------
# every format on every kernel that serves it
# ---------------------------------------------------------------------------------------------------------------------------
CI8_CASES = [  # nperseg, fs, block, blocks, window, impls
    (256, 300_000, 300_000, 3, "hamming", [E.FFT_GENERIC, E.FFT_AUTO, E.FFT_TC256]),     # AUTO: register kernel
    (1024, 2_400_000, 2_400_000, 3, "hann", [E.FFT_GENERIC, E.FFT_AUTO]),              # AUTO: radix-16 kernel
    (4096, 2_400_000, 2_400_000, 3, "hann", [E.FFT_AUTO]),
]
WIDE_CASES = [  # nperseg, fs, block, blocks, window
    (8, 300_000, 300_000, 3, "hamming"),
    (256, 300_000, 300_000, 3, "hamming"),
    (2048, 2_400_000, 2_400_000, 3, "hamming"),
    (4096, 2_400_000, 2_400_000, 3, "hann"),
]


@pytest.mark.parametrize("nperseg,fs,block,nb,window,impls", CI8_CASES, ids=lambda v: str(v) if not isinstance(v, list) else "")
def test_ci8_on_every_kernel_matches_the_oracle(nperseg, fs, block, nb, window, impls):
    cap = _capture("ci8", fs, block, nperseg, nb)
    kw = _kw(fs, block, nperseg, window)
    want = _oracle(kw, cap, "ci8")
    for impl in impls:
        tot, carried, _ = _run_vs_oracle(kw, cap, "ci8", impl, tag=f"formats/ci8/n{nperseg}/impl{impl}", want=want)
        assert tot["gpu"] >= 5 and carried >= 1, (impl, tot)


@pytest.mark.parametrize("fmt", ["ci16_le", "cf32_le"])
@pytest.mark.parametrize("nperseg,fs,block,nb,window", WIDE_CASES, ids=str)
def test_wide_formats_match_the_oracle(fmt, nperseg, fs, block, nb, window):
    cap = _capture(fmt, fs, block, nperseg, nb)
    kw = _kw(fs, block, nperseg, window)
    want = _oracle(kw, cap, fmt)
    tot, carried, recs = _run_vs_oracle(kw, cap, fmt, E.FFT_GENERIC, tag=f"formats/{fmt}/n{nperseg}", want=want)
    assert tot["gpu"] >= 5 and carried >= 1, tot
    if nperseg in (256, 4096):       # RT_FFT_AUTO runs the generic kernel for 16-bit and float samples: the same records
        _, _, auto = _run_vs_oracle(kw, cap, fmt, E.FFT_AUTO, tag=f"formats/{fmt}/n{nperseg}/auto", want=want)
        assert auto == recs


# ---------------------------------------------------------------------------------------------------------------------------
# blocks_per_launch, two launches in flight, ragged blocks; device inputs
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["ci16_le", "cf32_le"])
@pytest.mark.parametrize("block,B", [(300_000, 2), (250_123, 3)])
def test_blocks_per_launch_equals_block_by_block(fmt, block, B):
    fs, nperseg, nb = 300_000, 256, 6
    caps = [_capture(fmt, fs, block, nperseg, nb, stream=s) for s in (2, 3)]               # two streams, [nb, 2 block] each
    kw = _kw(fs, block, nperseg)
    P, want = _oracle(kw, caps[0], fmt)
    one = BatchAnalyzer(**parity.batch_kwargs(kw, devices=["0", "1"], calibration=[0.0, 0.0], sample_format=fmt))
    many = BatchAnalyzer(**parity.batch_kwargs(kw, devices=["0", "1"], calibration=[0.0, 0.0], sample_format=fmt, blocks_per_launch=B))
    try:
        ref = []
        for b in range(nb):
            rec = one.engine.process(np.stack([c[b] for c in caps]))
            ref.append([rec[rec["stream"] == s] for s in range(2)])
            sigs, keys = one.finalize(rec[rec["stream"] == 0], [_ts(kw, b), _ts(kw, b)])[0]
            S, last, found = want[b]
            parity.compare_block(P, S, last, found, sigs, keys)
        groups = [np.stack([c[g:g + B].reshape(-1) for c in caps]) for g in range(0, nb, B)]
        n, pending = 0, []

        def check(gi):
            nonlocal n
            rec = many.engine.fetch()
            for s in range(2):
                for k in range(B):
                    r = rec[rec["stream"] == s * B + k].copy()
                    r["stream"] = s
                    assert r.tobytes() == ref[gi * B + k][s].tobytes(), (gi, s, k)
                    n += len(r)

        for gi, g in enumerate(groups):                                                    # two launches in flight
            many.engine.launch(g)
            pending.append(gi)
            if len(pending) == 2:
                check(pending.pop(0))
        while pending:
            check(pending.pop(0))
        assert n > 10
    finally:
        one.close()
        many.close()


@pytest.mark.parametrize("fmt", ["ci8", "ci16_le", "cf32_le"])
def test_device_tensors_equal_host_arrays(fmt):
    torch = pytest.importorskip("torch")
    fs, block, nperseg = 300_000, 300_000, 256
    cap = _capture(fmt, fs, block, nperseg, 1)
    host = np.ascontiguousarray(np.stack([cap[0], cap[0][::-1]]))                          # two streams
    kw = _kw(fs, block, nperseg)
    ba = BatchAnalyzer(**parity.batch_kwargs(kw, devices=["0", "1"], calibration=[0.0, 0.0], sample_format=fmt))
    try:
        want = ba.engine.process(host)
        assert len(want) > 0
        inputs = [torch.from_numpy(host).cuda()]                                           # int8 / int16 / float32
        if fmt == "cf32_le":
            inputs += [torch.from_numpy(host.view(np.complex64)).cuda(), host.view(np.complex64)]
        for x in inputs:
            ba.reset_stream(0)
            ba.reset_stream(1)
            assert ba.engine.process(x).tobytes() == want.tobytes(), type(x)
    finally:
        ba.close()


# ---------------------------------------------------------------------------------------------------------------------------
# replay of recordings
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["ci16_le", "cf32_le"])
def test_replay_of_files_equals_feeding_the_blocks(tmp_path, fmt):
    fs = block = 300_000
    nb = 4
    caps = [_capture(fmt, fs, block, 256, nb, stream=10 + i) for i in range(2)]
    tails = [np.zeros(5, caps[0].dtype), np.zeros(2 * block - 1, caps[0].dtype)]
    paths = []
    for i, (c, t) in enumerate(zip(caps, tails)):
        p = tmp_path / f"chan{i}.sigmf-data"
        np.concatenate([c.reshape(-1), t]).tofile(p)
        (tmp_path / f"chan{i}.sigmf-meta").write_text(json.dumps({"global": {"core:datatype": fmt}}))
        paths.append(str(p))
    kw = _kw(fs, block, 256)
    dt = datetime.timedelta(seconds=block / fs)
    a = BatchAnalyzer(**parity.batch_kwargs(kw, devices=["0", "1"], calibration=[0.0, 0.0], sample_format=fmt))
    b = BatchAnalyzer(**parity.batch_kwargs(kw, devices=["0", "1"], calibration=[0.0, 0.0], sample_format=fmt))
    try:
        got = {}
        assert replay(paths, a, T0, on_block=lambda k, res: got.__setitem__(k, res)) == nb
        total = 0
        for k in range(nb):
            want = b.process_blocks(np.stack([c[k] for c in caps]), [T0 + k * dt] * 2)
            for s in range(2):
                assert [(x.ts, x.frequency, x.duration, x.max) for x in got[k][s][0]] == [(x.ts, x.frequency, x.duration, x.max) for x in want[s][0]]
                assert got[k][s][1] == len(want[s][1])
                total += len(want[s][0])
        assert total > 0
    finally:
        a.close()
        b.close()


def test_gr_osmosdr_cf32_recording_of_rtl_bytes_matches_the_cu8_path(tmp_path):
    """GNU Radio's osmosdr source maps RTL-SDR bytes to (b - 127.4) / 128 and a file sink stores them as cf32.  Those samples are
    127.5 / 128 times pyrtlsdr's b / 127.5 - 1 plus a constant the detrend removes, so with calibration_db = 20 log10(127.5 / 128)
    the Signals of the recording are those of the cu8 path on the original bytes (dB fields to parity.DB_ATOL, runs exact unless
    near a threshold).  Only `noise` (the row mean in dBW, which the reference does not calibrate) keeps the scale: it is
    calibration_db lower."""
    fs = block = 300_000
    nb = 3
    u8 = synth.make_stream(synth.Workload(92, "osmosdr", fs, block, amp_lsb=(10.0, 30.0)), 1, nb)
    cf = ((u8.astype(np.float64) - 127.4) / 128.0).astype("<f4")
    path = tmp_path / "rtl.sigmf-data"
    cf.tofile(path)
    (tmp_path / "rtl.sigmf-meta").write_text(json.dumps({"global": {"core:datatype": "cf32_le"}}))
    kw = _kw(fs, block, 256)
    P, want = _oracle(kw, u8, "cu8")                                                          # the cu8 story: the oracle on the bytes
    cal = 20 * math.log10(127.5 / 128.0)
    ba8 = BatchAnalyzer(**parity.batch_kwargs(kw))
    baf = BatchAnalyzer(**parity.batch_kwargs(kw, calibration=[cal], sample_format="cf32_le"))
    reader = CaptureReader([str(path)], block, pinned=False)
    assert reader.sample_format == "cf32_le"
    try:
        n = 0
        for k, blk in reader:
            S, last, found = want[k]
            _, sigs8, keys8 = ba8.process_blocks(u8[k][None, :], [_ts(kw, k)])[0]
            _, sigsf, keysf = baf.process_blocks(blk, [_ts(kw, k)])[0]
            parity.compare_block(P, S, last, found, sigs8, keys8)
            unscaled = [SimpleNamespace(**{f: getattr(x, f) for f in ("ts", "duration", "frequency", "max", "avg", "std", "snr")},
                                        noise=x.noise - cal) for x in sigsf]
            st = parity.compare_block(P, S, last, found, unscaled, keysf)
            n += st["gpu"]
        assert n >= 5
    finally:
        ba8.close()
        baf.close()


# ---------------------------------------------------------------------------------------------------------------------------
# rejected combinations
# ---------------------------------------------------------------------------------------------------------------------------
def test_bad_combinations_are_rejected():
    torch = pytest.importorskip("torch")
    block, n = 300_000, 256
    base = dict(n_streams=1, block_samples=block, nperseg=n, window=np.hamming(n), sample_rate=300_000.0, signal_threshold=1e-9,
                snr_threshold=3.0, probe_stride=9, min_cols=8, max_cols=50)
    for fmt, impl in (("ci16_le", E.FFT_REG256), ("cf32_le", E.FFT_REG256), ("ci16_le", E.FFT_TC256), ("cf32_le", E.FFT_TC256)):
        with pytest.raises(E.EngineError) as ei:
            E.Engine(**base, fft_impl=impl, sample_format=fmt)
        assert ei.value.code == E.RT_ERR_INVALID
    for code in (4, -1, 1 << 20):
        with pytest.raises(E.EngineError) as ei:
            E.Engine(**base, sample_format=code)                                             # unknown rt_config.sample_format
        assert ei.value.code == E.RT_ERR_INVALID and "sample_format" in str(ei.value)
    with pytest.raises(ValueError):
        E.Engine(**base, sample_format="ci12")
    with E.Engine(**base, sample_format="ci16_le") as eng:
        with pytest.raises(TypeError):
            eng.launch(np.zeros((1, 2 * block), np.uint8))
        with pytest.raises(TypeError):
            eng.launch(torch.zeros((1, 2 * block), dtype=torch.uint8, device="cuda"))
        with pytest.raises(TypeError):
            eng.launch(np.zeros((1, 2 * block), np.float32))
        with pytest.raises(ValueError):
            eng.launch(np.zeros((1, block), np.int16))                                    # half a block
        assert len(eng.process(torch.zeros((1, 2 * block), dtype=torch.int16, device="cuda"))) == 0
    with E.Engine(**base, sample_format="cf32_le") as eng:
        with pytest.raises(TypeError):
            eng.launch(np.zeros((1, 2 * block), np.float64))
        with pytest.raises(TypeError):
            eng.launch(np.zeros((1, block), np.complex128))
        t = torch.zeros(2 * block + 1, dtype=torch.float32, device="cuda")[1:]              # 4-byte aligned: half a complex sample off
        with pytest.raises(E.EngineError) as ei:
            eng.launch(t)
        assert ei.value.code == E.RT_ERR_INVALID
        assert len(eng.process(torch.zeros(block, dtype=torch.complex64, device="cuda"))) == 0
    with E.Engine(**base, sample_format="ci8") as eng:
        with pytest.raises(TypeError):
            eng.launch(np.zeros((1, 2 * block), np.uint8))
