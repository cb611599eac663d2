"""CUDA path vs oracle vs reference fixtures, on the B200 (pytest -m gpu).  Everything goes through
the C ABI (pyradiotracking_b200/engine.py -> librtb200.so)."""
import datetime

import numpy as np
import pytest

from oracle import restatement as R
from oracle.cases import BY_NAME, CASES, sha256
from pyradiotracking_b200 import engine as E
from pyradiotracking_b200 import synth
from pyradiotracking_b200.analyze import BatchAnalyzer, SignalAnalyzer
from tests import golden_io, parity

pytestmark = pytest.mark.gpu


def _impls(nperseg, window="hamming"):
    if nperseg in (1024, 4096):
        return [E.FFT_GENERIC, E.FFT_AUTO]           # AUTO = radix-16 Stockham kernel (spectro_r16.cuh)
    if nperseg != 256:
        return [E.FFT_GENERIC]
    impls = [E.FFT_GENERIC, E.FFT_REG256]
    if window in ("hamming", "hann", "boxcar"):      # windows whose DFT lives in the bins 0 and +-1
        impls.append(E.FFT_TC256)                    # tensor-core stage 1 (tcgen05)
    return impls


@pytest.mark.parametrize("case", CASES, ids=lambda c: c.name)
def test_case_matches_oracle_and_fixture(case):
    g = golden_io.load(case.name)
    kw = g.meta["analyzer"]
    cap = case.capture()
    assert sha256(cap) == g.meta["input_sha256"]
    P = parity.oracle_params(kw)
    for impl in _impls(kw["fft_nperseg"], kw["fft_window"] if isinstance(kw["fft_window"], str) else None):
        ora = R.OracleAnalyzer(P)
        ba = BatchAnalyzer(**parity.batch_kwargs(kw, fft_impl=impl))
        try:
            last = None
            totals = dict(oracle=0, gpu=0, near_threshold_mismatch=0)
            for b, gb in enumerate(g.blocks):
                ts0 = parity.block_ts(g.t0, b, kw["sdr_callback_length"], kw["sample_rate"])
                freqs, times, S, found, kept = ora.process_block(cap[b], ts0)
                filtered, sigs, keys = ba.process_blocks(cap[b][None, :], [ts0])[0]
                stats = parity.compare_block(P, S, last, found, sigs, keys)
                parity.compare_spectrogram(P, S, ba.engine.read_spectrogram(0), ba.engine.read_row_means(0), tag=f"{case.name}/impl{impl}/b{b}")
                for k in totals:
                    totals[k] += stats[k]
                if stats["near_threshold_mismatch"] == 0:
                    # identical candidate lists => the shadow filter must keep the same ones, and the
                    # reference fixture must agree field by field
                    assert [(s.ts, s.frequency) for s in filtered] == [(d.ts, d.frequency) for d in kept]
                    assert [golden_io.us(s.ts - golden_io.EPOCH) for s in sigs] == gb.ts_us.tolist()
                    assert [golden_io.us(s.duration) for s in sigs] == gb.dur_us.tolist()
                    assert [s.frequency for s in sigs] == gb.freq.tolist()
                    if len(sigs):
                        got = np.array([[s.max, s.avg, s.std, s.noise, s.snr] for s in sigs])
                        np.testing.assert_allclose(got, gb.stats, rtol=0, atol=parity.DB_ATOL)
                    kept_ids = {id(s) for s in filtered}
                    assert [id(s) in kept_ids for s in sigs] == gb.kept.tolist()
                last = S
            assert totals["gpu"] > 0
            assert totals["near_threshold_mismatch"] == 0        # no fixture has a run that close to a threshold
        finally:
            ba.close()


class _Q:
    def __init__(self):
        self.items = []

    def put(self, x):
        self.items.append(x)


class _V:
    value = 0.0


@pytest.mark.parametrize("name", ["c1_default_300k", "calib_hann_ragged", "tiny_T64"])
def test_signal_analyzer_callback_matches_reference_queue(name):
    """The drop-in class, driven like pyrtlsdr drives the reference: queue content == reference fixture."""
    case = BY_NAME[name]
    g = golden_io.load(name)
    kw = dict(g.meta["analyzer"])
    if isinstance(kw["fft_window"], list):
        kw["fft_window"] = tuple(kw["fft_window"])
    cap = case.capture()
    q = _Q()
    an = SignalAnalyzer(signal_queue=q, last_data_ts=_V(), **kw)
    assert an._spectrogram_last is None
    an.sdr = type("S", (), {"cancel_read_async": lambda self: None})()
    bl = datetime.timedelta(seconds=kw["sdr_callback_length"] / kw["sample_rate"])
    try:
        for b, gb in enumerate(g.blocks):
            an._now = lambda b=b: g.t0 + b * bl
            before = len(q.items)
            if b % 2:
                an.process_samples(synth.bytes_to_iq(cap[b]), None)       # reference-compatible complex entry
            else:
                an.process_bytes(cap[b], None)                            # raw-byte entry
            sigs = [m for m in q.items[before:] if isinstance(m, an.Signal)]
            assert [golden_io.us(s.ts - golden_io.EPOCH) for s in sigs] == gb.ts_us[gb.kept].tolist()
            assert [s.frequency for s in sigs] == gb.freq[gb.kept].tolist()
            assert [golden_io.us(s.duration) for s in sigs] == gb.dur_us[gb.kept].tolist()
            assert all(s.device == kw["device"] for s in sigs)
            if len(sigs):
                got = np.array([[s.max, s.avg, s.std, s.noise, s.snr] for s in sigs])
                np.testing.assert_allclose(got, gb.stats[gb.kept], rtol=0, atol=parity.DB_ATOL)
        # the reference's side state (analyze.py:268): the last block's spectrogram, (nperseg, T) float64
        last = an._spectrogram_last
        _, _, S = R.spectrogram(R.bytes_to_iq(cap[len(g.blocks) - 1]), kw["sample_rate"], kw["fft_window"], kw["fft_nperseg"])
        assert last.shape == S.shape and last.dtype == np.float64
        big = S >= 1e-2 * an.signal_threshold
        assert np.max(np.abs(last[big] - S[big]) / S[big]) <= parity.DEEP_RTOL
        states = [m for m in q.items if isinstance(m, an.StateMessage)]
        assert [m.state.name for m in states][:2] == ["STARTED", "RUNNING"]
    finally:
        an.batch.close()


def test_batch_of_streams_equals_single_streams():
    """Streams are independent: a batch with per-stream calibration == each stream alone == oracle."""
    w = synth.C1
    n, nb = 5, 3
    cal = [0.0, 1.5, -2.0, 3.25, 0.5]
    cap = synth.make_batch(w, list(range(n)), nb)                   # [nb, n, 2N]
    kw = BY_NAME["c1_default_300k"].analyzer_kwargs()
    ba = BatchAnalyzer(**parity.batch_kwargs(kw, devices=[str(i) for i in range(n)], calibration=cal))
    oras = [R.OracleAnalyzer(parity.oracle_params(dict(kw, device=str(i), calibration_db=cal[i]))) for i in range(n)]
    t0 = datetime.datetime(2026, 2, 2, 2, 2, 2)
    try:
        lasts = [None] * n
        for b in range(nb):
            ts0 = [parity.block_ts(t0, b, w.block_samples, w.sample_rate)] * n
            res = ba.process_blocks(cap[b], ts0)
            for i in range(n):
                freqs, times, S, found, kept = oras[i].process_block(cap[b, i], ts0[i])
                stats = parity.compare_block(oras[i].P, S, lasts[i], found, res[i][1], res[i][2])
                assert stats["near_threshold_mismatch"] == 0
                assert [(s.ts, s.frequency, s.device) for s in res[i][0]] == [(d.ts, d.frequency, str(i)) for d in kept]
                lasts[i] = S
    finally:
        ba.close()


def test_device_resident_input_equals_host_input():
    torch = pytest.importorskip("torch")
    w = synth.C1
    cap = synth.make_batch(w, [0, 1], 2)
    kw = BY_NAME["c1_default_300k"].analyzer_kwargs()
    a = BatchAnalyzer(**parity.batch_kwargs(kw, devices=["0", "1"], calibration=[0.0, 0.0]))
    b = BatchAnalyzer(**parity.batch_kwargs(kw, devices=["0", "1"], calibration=[0.0, 0.0]))
    try:
        for blk in cap:
            ra = a.engine.process(blk)
            rb = b.engine.process(torch.from_numpy(blk).cuda())
            assert ra.tobytes() == rb.tobytes() and len(ra) > 0
    finally:
        a.close()
        b.close()


def test_reset_stream_drops_the_carry():
    case = BY_NAME["c1_default_300k"]
    kw = case.analyzer_kwargs()
    cap = case.capture()
    ba = BatchAnalyzer(**parity.batch_kwargs(kw))
    try:
        ba.engine.process(cap[0][None, :])
        with_carry = ba.engine.process(cap[1][None, :])
        ba.reset_stream(0)
        without = ba.engine.process(cap[1][None, :])
        assert (with_carry["start"] < 0).any() and not (without["start"] < 0).any()
    finally:
        ba.close()


def test_engine_rejects_bad_configuration():
    win = np.ones(100)
    with pytest.raises(E.EngineError):
        E.Engine(n_streams=1, block_samples=1000, nperseg=100, window=win, sample_rate=1e5, signal_threshold=1e-9,
                 snr_threshold=3.0, probe_stride=1, min_cols=0, max_cols=10)
    with pytest.raises(E.EngineError):
        E.Engine(n_streams=1, block_samples=300, nperseg=256, window=np.ones(256), sample_rate=1e5,
                 signal_threshold=1e-9, snr_threshold=3.0, probe_stride=1, min_cols=0, max_cols=10)
    with pytest.raises(E.EngineError):       # register kernel, several blocks per launch, blocks not a multiple of 16 bytes
        E.Engine(n_streams=1, block_samples=250_123, nperseg=256, window=np.hamming(256), sample_rate=3e5, signal_threshold=1e-9,
                 snr_threshold=3.0, probe_stride=1, min_cols=0, max_cols=10, fft_impl=E.FFT_REG256, blocks_per_launch=2)
    with pytest.raises(IndexError):          # one-column block: analyze.py:354
        BatchAnalyzer(**parity.batch_kwargs(dict(BY_NAME["c1_default_300k"].analyzer_kwargs(), sdr_callback_length=300)))


@pytest.mark.parametrize("impl", [E.FFT_AUTO, E.FFT_GENERIC, E.FFT_TC256], ids=["reg256", "generic", "tc256"])
@pytest.mark.parametrize("launch_streams", [1, 2])
def test_two_blocks_in_flight_equal_sequential_calls(impl, launch_streams):
    """submit(i+1) before collect(i) (results ring of the engine) == process_blocks one by one -- for every spectrogram kernel
    and with ONE stream: the launches then overlap on the two launch streams (a grid smaller than the GPU), which is where the
    tensor-core kernel's per-stream ticket counters must not be shared between launches."""
    case = BY_NAME["c1_default_300k"]
    kw = case.analyzer_kwargs()
    cap = case.capture()
    t0 = datetime.datetime(2026, 6, 6, 6, 6, 6)
    a = BatchAnalyzer(**parity.batch_kwargs(kw, fft_impl=impl, launch_streams=launch_streams))
    b = BatchAnalyzer(**parity.batch_kwargs(kw, fft_impl=impl, launch_streams=launch_streams))
    try:
        want = [a.process_blocks(cap[i][None, :], [t0])[0][0] for i in range(4)]
        for rep in range(3):                                          # several rounds: a stale ticket would show up later
            got = []
            b.reset_stream(0)
            b.submit(cap[0][None, :])
            for i in range(4):
                if i + 1 < 4:
                    b.submit(cap[i + 1][None, :])
                got.append(b.collect([t0])[0][0])
            assert [[(s.ts, s.frequency, s.max, s.noise) for s in blk] for blk in got] == [[(s.ts, s.frequency, s.max, s.noise) for s in blk] for blk in want]
        assert sum(len(x) for x in got) > 0
        with pytest.raises(E.EngineError):
            b.engine.fetch()                 # nothing left in flight
    finally:
        a.close()
        b.close()


def test_record_overflow_returns_the_first_records_and_says_so():
    """rt_config.max_records smaller than what a dense block produces: the first max_records come back (sorted), the engine reports
    how many were dropped, the next launch is unaffected; the default capacity (worst case) never overflows."""
    case = BY_NAME["c5_dense_loud_300k"]
    kw = case.analyzer_kwargs()
    cap = case.capture()
    full = BatchAnalyzer(**parity.batch_kwargs(kw))
    small = BatchAnalyzer(**parity.batch_kwargs(kw, max_records=64))
    try:
        want = full.engine.process(cap[0][None, :])
        assert len(want) > 64 and full.engine.truncated == 0
        got = small.engine.process(cap[0][None, :])
        assert len(got) == 64 and small.engine.truncated == len(want) - 64
        keys = {(int(r["fi"]), int(r["start"]), int(r["end"])) for r in want}
        assert all((int(r["fi"]), int(r["start"]), int(r["end"])) in keys for r in got)
        lib, n = E.load_library(), __import__("ctypes").c_int32(0)
        small.engine.launch(cap[0][None, :])
        buf = np.empty(8, dtype=E.RECORD_DTYPE)
        rc = lib.rt_engine_fetch(small.engine._h, buf.ctypes.data_as(__import__("ctypes").c_void_p), 8, __import__("ctypes").byref(n))
        assert rc == E.RT_ERR_OVERFLOW and n.value == len(want)
    finally:
        full.close()
        small.close()


def test_device_inputs_are_validated():
    torch = pytest.importorskip("torch")
    kw = BY_NAME["c1_default_300k"].analyzer_kwargs()
    cap = BY_NAME["c1_default_300k"].capture()
    ba = BatchAnalyzer(**parity.batch_kwargs(kw))
    try:
        want = ba.engine.process(cap[0][None, :])
        ba.reset_stream(0)
        got = ba.engine.process(torch.from_numpy(cap[0]).cuda())          # 1-D device tensor: one stream
        assert got.tobytes() == want.tobytes()

        class Cai:                                                        # a CuPy / Numba style object without strides
            def __init__(self, t):
                self.t = t
                self.__cuda_array_interface__ = dict(shape=tuple(t.shape), typestr="|u1", data=(t.data_ptr(), False), version=3, strides=None)

        ba.reset_stream(0)
        got = ba.engine.process(Cai(torch.from_numpy(cap[0]).cuda()))
        assert got.tobytes() == want.tobytes()
        with pytest.raises(ValueError):
            ba.engine.launch(torch.from_numpy(cap[0][:-2]).cuda())        # wrong size: would be read out of bounds
        with pytest.raises(TypeError):
            ba.engine.launch(torch.from_numpy(cap[0]).cuda().to(torch.int16))
    finally:
        ba.close()
    with pytest.raises(ValueError, match="powers of two"):
        BatchAnalyzer(**parity.batch_kwargs(dict(kw, fft_nperseg=300)))


def test_batched_signals_through_the_native_matcher_equal_the_oracle_matcher():
    """SURVEY 8f rank 1 behind the engine: four 'antennas' (streams) hear the same capture with different
    calibration, two more hear another one; the Signals of every block go through SignalMatcher.add_batch in the
    queue order of the batch and must group exactly like the restated reference matcher (oracle/matcher.py)."""
    from oracle import matcher as OM
    from pyradiotracking_b200.match import SignalMatcher

    w = synth.C1
    nb = 3
    a, b = synth.make_stream(w, 0, nb), synth.make_stream(w, 1, nb)
    cap = np.stack([a, a, a, a, b, b], axis=1)                       # [nb, 6, 2N]
    cal = [0.0, 0.5, -0.5, 1.0, 0.0, 0.25]
    devs = [str(i) for i in range(6)]
    kw = BY_NAME["c1_default_300k"].analyzer_kwargs()
    ba = BatchAnalyzer(**parity.batch_kwargs(kw, devices=devs, calibration=cal))
    mk = dict(device=devs, matching_timeout_s=0.5, matching_time_diff_s=0.001, matching_bandwidth_hz=2500.0, matching_duration_diff_ms=2.0)
    q = _Q()
    nat = SignalMatcher(signal_queue=q, **mk)
    ora = OM.OracleMatcher(**mk)
    t0 = datetime.datetime(2026, 4, 4, 4, 4, 4, tzinfo=datetime.timezone.utc)
    try:
        n_sig = 0
        for blk in range(nb):
            ts0 = [parity.block_ts(t0, blk, w.block_samples, w.sample_rate)] * 6
            res = ba.process_blocks(cap[blk], ts0)
            sigs = [s for per in res for s in per[0]]                # queue order: device by device
            for k, s in enumerate(sigs):
                s.idx = n_sig + k
            n_sig += len(sigs)
            nat.add_batch(sigs)
            for s in sigs:
                ora.add(s)
        assert n_sig > 0
        assert OM.groups_as_ids(q.items) == OM.groups_as_ids(ora.emitted)
        assert OM.groups_as_ids(nat._matched) == OM.groups_as_ids(ora._matched)
        sizes = [len(g._sigs) for g in q.items + nat._matched]
        assert max(sizes) >= 4                                       # the four antennas of capture `a` were grouped
    finally:
        ba.close()
        nat.close()


@pytest.mark.parametrize("knobs", [dict(scan_schedule=E.SCAN_SERIAL), dict(scan_schedule=E.SCAN_OVERLAP), dict(scan_schedule=E.SCAN_LEAN),
                                   dict(scan_schedule=E.SCAN_LEAN, launch_streams=1), dict(scan_schedule=E.SCAN_OVERLAP, launch_streams=1),
                                   dict(chunk_segs=0)],
                         ids=["serial", "overlap", "lean", "lean-one-launch-stream", "overlap-one-launch-stream", "auto"])
@pytest.mark.parametrize("name", ["c1_default_300k", "c5_dense_300k", "c2_stream_2400k", "c3a_20M_n1024"])
def test_scan_schedules_give_the_same_records(name, knobs):
    """rt_config.scan_schedule / launch_streams change WHERE and WHEN the scan kernels run (launch stream, scan stream, lean
    32-register variants beside the next spectrogram), not what they find: same records, bit for bit."""
    case = BY_NAME[name]
    g = golden_io.load(case.name)
    kw = g.meta["analyzer"]
    cap = case.capture()

    def run(**extra):
        ba = BatchAnalyzer(**parity.batch_kwargs(kw, fft_impl=E.FFT_AUTO, **extra))
        out = []
        try:
            for b in range(len(g.blocks)):
                ts0 = parity.block_ts(g.t0, b, kw["sdr_callback_length"], kw["sample_rate"])
                filtered, sigs, keys = ba.process_blocks(cap[b][None, :], [ts0])[0]
                out.append((keys, [(s.ts, s.frequency, s.duration, s.max, s.avg, s.std, s.noise, s.snr) for s in sigs]))
        finally:
            ba.close()
        return out

    want = run(scan_schedule=E.SCAN_SERIAL, launch_streams=1)
    got = run(**knobs)
    assert sum(len(k) for k, _ in want) > 0
    assert got == want


@pytest.mark.parametrize("thr_dbw,snr_db,min_ms,max_ms", [(-95.0, 3.0, 4.0, 20.0), (-88.0, 8.0, 8.0, 40.0), (-92.0, 0.5, 2.0, 60.0),
                                                          (-90.0, 5.0, 15.0, 25.0), (-97.0, 2.0, 1.0, 10.0)])
@pytest.mark.parametrize("name", ["c1_default_300k", "c5_dense_300k"])
def test_detection_parameters_sweep_against_the_oracle(name, thr_dbw, snr_db, min_ms, max_ms):
    """Other thresholds / duration limits than the fixtures were generated with: other probe strides (1 ... 17 columns), chain
    lengths and duration gates through the same kernels; the oracle (pinned by the fixtures) is the checker."""
    case = BY_NAME[name]
    g = golden_io.load(case.name)
    kw = dict(g.meta["analyzer"])
    kw.update(signal_threshold_dbw=thr_dbw, snr_threshold_db=snr_db, signal_min_duration_ms=min_ms, signal_max_duration_ms=max_ms)
    cap = case.capture()
    P = parity.oracle_params(kw)
    ora = R.OracleAnalyzer(P)
    ba = BatchAnalyzer(**parity.batch_kwargs(kw))
    try:
        last = None
        totals = dict(oracle=0, gpu=0, near_threshold_mismatch=0)
        for b in range(min(4, len(g.blocks))):
            ts0 = parity.block_ts(g.t0, b, kw["sdr_callback_length"], kw["sample_rate"])
            freqs, times, S, found, kept = ora.process_block(cap[b], ts0)
            filtered, sigs, keys = ba.process_blocks(cap[b][None, :], [ts0])[0]
            stats = parity.compare_block(P, S, last, found, sigs, keys)
            for k in totals:
                totals[k] += stats[k]
            if stats["near_threshold_mismatch"] == 0:
                assert [(s.ts, s.frequency) for s in filtered] == [(d.ts, d.frequency) for d in kept]
            last = S
        assert totals["near_threshold_mismatch"] <= max(2, totals["oracle"] // 50)
    finally:
        ba.close()


def _extreme_blocks(n_samples, rng):
    """Byte patterns at the edges of the uint8 -> float front ends (fp16 pair + widening add, packed integer byte sums)."""
    full = rng.integers(0, 256, 2 * n_samples).astype(np.uint8)                  # full-scale uniform bytes
    hi = np.full(2 * n_samples, 255, np.uint8)                                    # the largest byte sums ...
    hi[rng.integers(0, 2 * n_samples, n_samples // 8)] = 254                      # ... with a little structure left after the detrend
    split = np.empty(2 * n_samples, np.uint8)                                     # I near the top, Q near the bottom: the two sum fields stay apart
    split[0::2] = 255 - rng.integers(0, 3, n_samples)
    split[1::2] = rng.integers(0, 3, n_samples)
    t = np.arange(n_samples)
    off = np.clip(np.rint(30 + 4 * rng.standard_normal(2 * n_samples)), 0, 255).astype(np.uint8)   # DC far from 127.5, sigma of 4 LSB
    tone = 20 * np.exp(2j * np.pi * 0.173 * t)
    off[0::2] = np.clip(off[0::2] + np.rint(tone.real), 0, 255).astype(np.uint8)
    off[1::2] = np.clip(off[1::2] + np.rint(tone.imag), 0, 255).astype(np.uint8)
    return dict(full_scale=full, all_high=hi, split_iq=split, dc_offset_tone=off)


@pytest.mark.parametrize("nperseg", [8, 32, 128, 256, 1024, 2048, 4096])
def test_extreme_byte_patterns_match_the_float64_spectrogram(nperseg):
    fs, n_samples = 2_400_000, 64 * 4096 + 77                                     # ragged tail: the last partial segment is dropped
    rng = np.random.default_rng(20261018)
    blocks = _extreme_blocks(n_samples, rng)
    kw = dict(devices=["0"], calibration_db=[0.0], sample_rate=fs, center_freq=150_000_000, fft_nperseg=nperseg, fft_window="hamming",
              signal_min_duration_ms=8, signal_max_duration_ms=40, signal_threshold_dbw=-90.0, snr_threshold_db=5.0, cuda_device=0,
              sdr_callback_length=n_samples)
    t0 = datetime.datetime(2026, 1, 1)
    for impl in _impls(nperseg, "hamming"):
        ba = BatchAnalyzer(**kw, fft_impl=impl)
        try:
            for name, u8 in blocks.items():
                if impl == E.FFT_TC256 and name != "full_scale":
                    # the optional tensor-core kernel centres the bytes at the CONSTANT 128 and removes the rest of the mean from the
                    # bins 0 and +-1 afterwards (DESIGN 5.2): with a DC offset far from 128 those three bins cancel catastrophically
                    # (measured 5e-2 on all_high).  Documented limit of fft_impl = RT_FFT_TC256, not of the default kernels.
                    continue
                _, _, S = R.spectrogram(R.bytes_to_iq(u8), fs, "hamming", nperseg)
                ba.process_blocks(u8[None, :], [t0])
                got = ba.engine.read_spectrogram(0).T.astype(np.float64)
                assert got.shape == S.shape
                with np.errstate(divide="ignore", invalid="ignore"):
                    rel = np.where(S > 0, np.abs(got - S) / S, 0.0)
                colmax = S.max(axis=0, keepdims=True)
                main = (S >= colmax * 1e-5) & (S > 0)                                        # within 50 dB of the segment's peak (tests/parity.py DEEP_DB)
                print(f"extreme[{nperseg}/impl{impl}/{name}]: max rel {rel[main].max():.2e} (main), {rel.max():.2e} (all)")
                assert rel[main].max() <= parity.POWER_RTOL, (name, impl, float(rel[main].max()))
                rm = ba.engine.read_row_means(0).astype(np.float64)
                assert np.max(np.abs(rm - S.mean(axis=1)) / S.mean(axis=1)) <= 2e-5
        finally:
            ba.close()
