"""CPU-only checks of the host layer: the C-ABI library builds, loads and exports what
include/rt_engine.h declares; host float64 logic (plan, finaliser, shadow filter) vs the oracle;
the register-FFT data flow emulated on the CPU vs numpy."""
import datetime
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import restatement as R
from pyradiotracking_b200 import build as B
from pyradiotracking_b200 import engine as E
from pyradiotracking_b200 import messages, synth
from pyradiotracking_b200.analyze import BatchAnalyzer, DetectionPlan, iq_to_bytes, shadow_mask

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_builds_loads_and_exports_header_symbols():
    B.build()
    lib = E.load_library()
    hdr = open(os.path.join(ROOT, "include", "rt_engine.h")).read() + open(os.path.join(ROOT, "include", "rt_matcher.h")).read()
    declared = set(re.findall(r"\b(rt_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(E.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.rt_abi_version() == E.RT_ABI_VERSION
    assert E.RECORD_DTYPE.itemsize == 40


def test_no_cpu_fallback_without_device():
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(E.EngineError):
        E.Engine(n_streams=1, block_samples=300000, nperseg=256, window=np.ones(256), sample_rate=3e5,
                 signal_threshold=1e-9, snr_threshold=3.0, probe_stride=9, min_cols=8, max_cols=49)


class _StreamCai:
    """A CuPy / Numba style device array (CUDA Array Interface v3) with an optional `stream` entry."""

    def __init__(self, n=64, ptr=0x10000, **stream):
        self.__cuda_array_interface__ = dict(shape=(1, n), typestr="|u1", data=(ptr, False), version=3, strides=None, **stream)


class _RecordingLib:
    """Stands in for librtb200.so: records the engine calls of the binding."""

    def __init__(self):
        self.calls = []

    def rt_engine_create(self, cfg, h):
        h._obj.value = 0x1000
        return E.RT_OK

    def rt_engine_destroy(self, h):
        self.calls.append(("destroy",))

    def rt_engine_set_stream(self, h, s):
        self.calls.append(("set_stream", s.value or 0))
        return E.RT_OK

    def rt_engine_wait_stream(self, h, s):
        self.calls.append(("wait", s.value or 0))
        return E.RT_OK

    def rt_engine_launch(self, h, iq, on_dev, stride):
        self.calls.append(("launch", on_dev))
        return E.RT_OK

    def rt_engine_peek(self, h, n):
        n._obj.value = 0
        return E.RT_OK

    def rt_engine_fetch(self, h, out, max_out, need):
        need._obj.value = 0
        return E.RT_OK


def test_producer_stream_of_device_inputs(monkeypatch):
    """_producer_stream: a CAI `stream` as given (absent / None: no wait; 1 legacy and 2 per-thread default streams and
    pointers pass through; 0 is forbidden by the interface), and for a torch tensor the current stream of its device."""
    assert E._producer_stream(_StreamCai()) is None
    assert E._producer_stream(_StreamCai(stream=None)) is None
    for s in (1, 2, 0x7F00DEADBEE0):
        assert E._producer_stream(_StreamCai(stream=s)) == s
    with pytest.raises(ValueError, match="stream 0"):
        E._producer_stream(_StreamCai(stream=0))
    assert E._device_pointer(_StreamCai(stream=7), 1, 64) == (0x10000, 64)     # the pointer and stride do not change
    torch = pytest.importorskip("torch")
    asked = []

    class _Stream:
        cuda_stream = 0x5150

    def current_stream(device=None):
        asked.append(device)
        return _Stream()

    class _Tensor:                           # what the binding reads of a CUDA torch.Tensor
        is_cuda, dtype, shape, device = True, "torch.uint8", (1, 64), "cuda:3"

        def data_ptr(self):
            return 0x20000

        def element_size(self):
            return 1

        def stride(self):
            return (64, 1)

    monkeypatch.setattr(torch.cuda, "current_stream", current_stream)
    assert E._device_pointer(_Tensor(), 1, 64) == (0x20000, 64)
    assert E._producer_stream(_Tensor()) == 0x5150
    assert asked == ["cuda:3"]


def test_launch_waits_for_the_producer_and_holds_inputs_until_fetched(monkeypatch):
    """The binding's side of the stream contract, on a stand-in library: a launch waits for its input's producer stream unless
    that is the stream given to set_stream, and every input stays referenced until a fetch returned its launch or a later one
    (also after a third launch dropped the oldest result), and until close()."""
    lib = _RecordingLib()
    monkeypatch.setattr(E, "load_library", lambda: lib)
    eng = E.Engine(n_streams=1, block_samples=32, nperseg=8, window=np.ones(8), sample_rate=3e5, signal_threshold=1e-9,
                   snr_threshold=3.0, probe_stride=1, min_cols=1, max_cols=4)
    xs = [_StreamCai(stream=7), _StreamCai(stream=1), _StreamCai(), _StreamCai(stream=2)]
    for x in xs:
        eng.launch(x)
    assert [c for c in lib.calls if c[0] != "launch"] == [("wait", 7), ("wait", 1), ("wait", 2)]
    assert [id(x) for x in eng._held] == [id(x) for x in xs]       # 4 launches, none fetched: the engine dropped 2 results
    eng.fetch()                                                      # launch 2
    assert [id(x) for x in eng._held] == [id(xs[3])]
    eng.fetch()
    assert eng._held == []
    lib.calls.clear()
    eng.set_stream(7)
    eng.launch(xs[0])                                                # produced on the launch stream: no extra call
    with pytest.raises(ValueError):
        eng.launch(_StreamCai(stream=0))
    host = np.zeros((1, 64), np.uint8)
    eng.launch(host)
    assert lib.calls == [("set_stream", 7), ("launch", 1), ("launch", 0)]
    assert [id(x) for x in eng._held] == [id(xs[0]), id(host)]
    eng.fetch()                                                      # launch 4: launch 5 is still in flight
    assert len(eng._held) == 1
    eng.close()
    assert eng._held == [] and lib.calls[-1] == ("destroy",)


@pytest.mark.parametrize("fs,n,N", [(300000, 256, 300000), (2400000, 256, 2400000), (256000, 256, 256000),
                                    (20000000, 1024, 20000000), (20000000, 4096, 2000000), (300000, 256, 250123)])
def test_plan_matches_scipy_axes_and_reference_stride(fs, n, N):
    plan = DetectionPlan(fs, n, N, 0.008, 0.04)
    f, t, _ = R.spectrogram(np.zeros(N, complex), fs, "boxcar", n)
    assert np.array_equal(plan.freqs, f) and np.array_equal(plan.times, t)
    assert plan.stride == max(1, int(0.008 / (t[1] - t[0])))
    # every (start, end) that passes the float64 duration test also passes the coarse device gate
    for start in (0, 5, -3):
        for end in range(max(start, 0) + 1, min(plan.T, 600)):
            _, dur = plan.duration(start, end)
            if 0.008 <= dur <= 0.04:
                cols = end - start + (1 if start < 0 else 0)
                assert plan.min_cols <= cols <= plan.max_cols


def test_stride_is_74_at_2p4_msps():
    assert DetectionPlan(2400000, 256, 2400000, 0.008, 0.04).stride == 74        # SURVEY.md §7 hard part 3


def test_shadow_mask_equals_reference_loop():
    rng = np.random.default_rng(5)
    t0 = datetime.datetime(2026, 1, 1, tzinfo=datetime.timezone.utc)
    dets = [R.Detection(0, 0, 1, t0 + datetime.timedelta(microseconds=int(rng.integers(0, 200000))), 1.0,
                        datetime.timedelta(microseconds=int(rng.integers(8000, 40000))), float(rng.integers(-90, -60)),
                        0, 0, 0, 0) for _ in range(400)]
    keep_ref = [d for d in dets if R.is_shadow_of(d, dets) is None]
    ts = np.array([(d.ts - t0) // datetime.timedelta(microseconds=1) for d in dets])
    du = np.array([d.duration // datetime.timedelta(microseconds=1) for d in dets])
    mx = np.array([d.max for d in dets])
    keep = [d for d, s in zip(dets, shadow_mask(ts, du, mx)) if not s]
    assert keep == keep_ref and 0 < len(keep) < len(dets)


def test_finaliser_reproduces_oracle_fields_from_exact_records():
    """Feed the finaliser records built from the oracle's float64 spectrogram: every Signal field must
    equal the oracle's (this isolates the host arithmetic from the device arithmetic)."""
    w = synth.C1
    cap = synth.make_stream(w, 2, 2)
    P = R.Params.make(sample_rate=w.sample_rate, calibration_db=1.25)
    ora = R.OracleAnalyzer(P)
    ba = BatchAnalyzer(devices=["0"], calibration_db=[1.25], sample_rate=w.sample_rate, center_freq=w.center_freq,
                       fft_nperseg=256, fft_window="hamming", signal_min_duration_ms=8, signal_max_duration_ms=40,
                       signal_threshold_dbw=-90.0, snr_threshold_db=5.0)
    t0 = datetime.datetime(2026, 4, 4, 4, 4, 4)
    last = None
    for b in range(2):
        _, _, S, found, kept = ora.process_block(cap[b], t0)
        rec = np.zeros(len(found), dtype=E.RECORD_DTYPE)
        for i, d in enumerate(found):
            data = np.concatenate((last[d.fi][d.start:], S[d.fi][:d.end])) if d.start < 0 else S[d.fi][d.start:d.end]
            rec[i] = (0, d.fi, d.start, d.end, data.max(), S[d.fi].mean(), data.mean(), np.std(10 * np.log10(data)))
        sigs, keys = ba.finalize(rec, [t0])[0]
        assert keys == [d.key() for d in found]
        for s, d in zip(sigs, found):
            assert (s.ts, s.frequency, s.duration) == (d.ts, d.frequency, d.duration)
            assert abs(s.max - d.max) < 1e-5 and abs(s.noise - d.noise) < 1e-5     # float32 max / row mean in the record
            assert abs(s.avg - d.avg) < 1e-9 and abs(s.std - d.std) < 1e-9
        assert [(s.ts, s.frequency) for s in ba.filter_shadow_signals(sigs)] == [(d.ts, d.frequency) for d in kept]
        last = S
    assert len(found) > 0


def test_iq_to_bytes_round_trip_and_rejection():
    u8 = synth.make_stream(synth.C1, 0, 1)[0][:4096]
    assert np.array_equal(iq_to_bytes(synth.bytes_to_iq(u8)), u8)
    with pytest.raises(ValueError):
        iq_to_bytes(np.array([0.1234 + 0.5j]))


def test_message_types_mirror_reference_surface():
    s = messages.Signal("0", "2026-01-01T00:00:00+00:00", "150.1e6", 0.02, -60, -62, 1.0, -94, 30)
    assert s.as_dict["Frequency"] == 150.1e6 and s.duration == datetime.timedelta(seconds=0.02)
    assert messages.Signal.header == ["Device", "Time", "Frequency", "Duration", "max (dBW)", "avg (dBW)", "std (dB)", "noise (dBW)", "snr (dB)"]
    m = messages.StateMessage("0", datetime.datetime.now(), 2)
    assert m.state is messages.StateMessage.State.STARTED and m.as_list[2] == 2
    assert abs(messages.from_dB(messages.dB(3.0)) - 3.0) < 1e-12


def test_register_fft_dataflow_on_cpu(tmp_path):
    """spectro_reg256's 16x16 decomposition, emulated with the same header on the host."""
    exe = tmp_path / "hostcheck"
    subprocess.run(["g++", "-O2", "-o", str(exe), os.path.join(ROOT, "tests", "csrc_host_check.cpp")], check=True)
    rng = np.random.default_rng(3)
    for trial in range(6):
        raw = synth.make_stream(synth.C1, 40 + trial, 1)[0][trial * 512: trial * 512 + 512].copy()
        if trial == 3:
            raw = rng.integers(0, 256, 512).astype(np.uint8)           # full-scale bytes
        if trial == 4:
            raw[:] = 255                                               # largest byte sums (the packed fields must not overflow)
            raw[7] = 0                                                 # (one sample off the constant, so that the spectrum is not all zero)
        if trial == 5:
            raw[0::2] = 255                                            # I at full scale, Q at zero: the two sum fields stay apart
            raw[1::2] = 0
            raw[9] = 3
        win = R.resolve_window("hamming", 256).astype(np.float32)
        out = subprocess.run([str(exe)], input=raw.tobytes() + win.tobytes(), capture_output=True, check=True).stdout
        got = np.frombuffer(out, np.float32).astype(np.float64)
        x = raw[0::2].astype(float) + 1j * raw[1::2].astype(float)
        ref = np.abs(np.fft.fft((x - x.mean()) * win.astype(float))) ** 2
        assert np.max(np.abs(got - ref) / ref.max()) < 1e-6
        big = ref > 1e-3 * ref.max()
        assert np.max(np.abs(got[big] - ref[big]) / ref[big]) < 2e-5


def test_timedelta_us_matches_cpython_rounding():
    from pyradiotracking_b200.analyze import timedelta_us

    rng = np.random.default_rng(0)
    x = np.concatenate([rng.uniform(-2, 2, 20000), rng.integers(-2000000, 2000000, 5000) / 1e6 + rng.choice([0, 5e-7, -5e-7], 5000),
                        np.arange(-3000, 3000) * 0.0000005])
    want = [(lambda td: (td.days * 86400 + td.seconds) * 1000000 + td.microseconds)(datetime.timedelta(seconds=float(v))) for v in x]
    assert timedelta_us(x).tolist() == want


# ---------------------------------------------------------------------------------------------------------
# tensor-core spectrogram path (csrc/spectro_tc256.cuh): the shipped operand tables + the kernel's algebra on the CPU
# ---------------------------------------------------------------------------------------------------------
def _tc_matrices(bmat):
    """[16 n2, 2 hi|lo, 32 n, 32 k] float64 from the operand image (core-matrix layout of the header comment)."""
    n, k = np.meshgrid(np.arange(32), np.arange(32), indexing="ij")
    off = (n >> 3) * 256 + (k >> 3) * 64 + (n & 7) * 8 + (k & 7)
    return bmat.view(np.float16)[:, :, off].astype(np.float64)


@pytest.mark.parametrize("window", ["hamming", "hann", "boxcar"])
def test_tensor_core_tables_and_stage_algebra_on_cpu(window):
    fs = 2_400_000
    w = R.resolve_window(window, 256)
    bmat, wc, pscale, eligible = E.tc256_tables(w, fs)
    assert eligible and pscale > 0 and np.log2(pscale) == int(np.log2(pscale))
    B = _tc_matrices(bmat)                                   # hi and lo terms
    amp = np.sqrt(1.0 / (fs * np.sum(w * w))) / 127.5
    sc = np.sqrt(pscale)
    # (1) hi + lo reproduces  w'[n] e^{-2 pi j k1 n / 256}  to ~2^-22: D[(k1,re)] = sum xI cr - xQ ci, D[(k1,im)] = sum xI ci + xQ cr
    for n2 in (0, 5, 15):
        nn = 16 * np.arange(16) + n2
        c = (w[nn] * amp * sc)[None, :] * np.exp(-2j * np.pi * np.outer(np.arange(16), nn) / 256.0)     # [k1, n1]
        want = np.empty((32, 32))
        want[0::2, 0::2], want[0::2, 1::2] = c.real, -c.imag
        want[1::2, 0::2], want[1::2, 1::2] = c.imag, c.real
        got = B[n2, 0] + B[n2, 1]
        assert np.max(np.abs(got - want)) <= 2.0 ** -21 * np.max(np.abs(want))
        assert np.max(np.abs(B[n2, 1])) <= 2.0 ** -11 * np.max(np.abs(B[n2, 0]))
    # (2) the kernel's algebra in float32 accumulation: stage 1 (exact bytes x split matrix), DFT16 over n2, 3-bin detrend
    cap = synth.make_stream(synth.C2, 3, 1)[0][: 512 * 40].reshape(40, 256, 2).astype(np.int64)
    cap[7] += 9                                              # a segment with a DC offset
    cap = np.clip(cap, 0, 255)
    x = (cap - 128).astype(np.float32)                       # exact in fp16
    A = x.reshape(40, 16, 16, 2).transpose(0, 2, 1, 3).reshape(40, 16, 32)      # [seg, n2, (n1, iq)]
    U = np.zeros((40, 16, 32), np.float32)
    for hl in (0, 1):
        U += np.einsum("snk,nmk->snm", A, B[:, hl].astype(np.float32), dtype=np.float32)
    Uc = (U[:, :, 0::2] + 1j * U[:, :, 1::2]).astype(np.complex64)              # [seg, n2, k1]
    X = np.fft.fft(Uc, axis=1)                                                  # over n2 -> k2: bin = k1 + 16 k2
    Xk = np.empty((40, 256), np.complex128)
    for k1 in range(16):
        Xk[:, k1 + 16 * np.arange(16)] = X[:, :, k1]
    m = (cap.sum(axis=1) - 32768) / 256.0                                        # residual mean, exact
    mres = m[:, 0] + 1j * m[:, 1]
    for k, c in zip((0, 1, 255), wc):
        Xk[:, k] -= mres * c
    got = (np.abs(Xk) ** 2) / pscale
    iq = synth.bytes_to_iq(cap.astype(np.uint8).reshape(-1))
    _, _, S = R.spectrogram(iq, fs, window, 256)
    ref = S.T
    big = ref >= 1e-4 * ref.max(axis=1, keepdims=True)      # within 40 dB of the column maximum: fp32 accumulation floor
    assert np.max(np.abs(got[big] - ref[big]) / ref[big]) < 5e-5
    # windows whose DFT leaks beyond the bins 0, +-1 are refused
    assert not E.tc256_tables(R.resolve_window(("kaiser", 8.0), 256), fs)[3]
    assert not E.tc256_tables(R.resolve_window("blackman", 256), fs)[3]


@pytest.mark.parametrize("N", [1024, 4096])
def test_radix16_stockham_index_algebra_on_cpu(N):
    """The pass structure of csrc/spectro_r16.cuh (read/write indices, twiddles, last pass in registers) vs numpy."""
    rng = np.random.default_rng(N)
    x = rng.standard_normal(N) + 1j * rng.standard_normal(N)
    tw = np.exp(-2j * np.pi * np.arange(N) / N)
    i16 = np.arange(16)
    F16 = np.exp(-2j * np.pi * np.outer(i16, i16) / 16)
    BT, M1, M2 = N // 16, N // 16, N // 256
    X = np.zeros(N, complex)
    for b in range(BT):                                      # pass 1: inputs b + M1 i -> y[16 b + i] * W_N^{b i}
        v = F16 @ x[b + M1 * i16]
        X[16 * b + i16] = v * tw[(b * i16) % N]
    Y = np.zeros(N, complex)
    for b in range(BT):                                      # pass 2: p = b / 16, q = b % 16
        p, q = b >> 4, b & 15
        v = F16 @ X[q + 16 * (p + M2 * i16)]
        Y[q + 16 * (16 * p + i16)] = v * tw[(16 * p * i16) % N]
    out = np.zeros(N, complex)
    if N == 4096:
        for b in range(256):
            out[b + 256 * i16] = F16 @ Y[b + 256 * i16]
    else:
        F4 = np.exp(-2j * np.pi * np.outer(np.arange(4), np.arange(4)) / 4)
        for q in range(256):
            out[q + 256 * np.arange(4)] = F4 @ Y[q + 256 * np.arange(4)]
    assert np.max(np.abs(out - np.fft.fft(x))) < 1e-9 * N


def test_cheap_predicate_equals_exact_predicate_on_cpu(tmp_path):
    """csrc/predicate.h: the 3-instruction predicate of the scan kernels takes the decision of the exact one
    (analyze.py:370-379) for every float, also within a few ulp of the thresholds and for degenerate row means."""
    exe = tmp_path / "pred_host_check"
    subprocess.run(["g++", "-O2", "-o", str(exe), os.path.join(ROOT, "tests", "pred_host_check.cpp")], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    assert int(out[0]) > 10_000_000 and int(out[1]) == 0


def test_shadow_sweep_equals_the_pairwise_definition_with_ties():
    """The O(S log S) shadow filter against the pairwise definition (analyze.py:283-313) on random lists with equal start times,
    zero durations, touching intervals and equal loudness; and a whole batch evaluated in one pass == unit by unit."""
    from pyradiotracking_b200.analyze import _UNIT_GAP_US

    def pairwise(ts, du, mx):
        te = ts + du
        return np.array([bool((((ts[i] <= te) & (te[i] >= ts)) & (mx > mx[i])).any()) for i in range(len(ts))], dtype=bool)

    rng = np.random.default_rng(11)
    for _ in range(300):
        n = int(rng.integers(0, 70))
        ts = rng.integers(0, 120, n) * 1000
        du = rng.integers(0, 40, n) * 1000
        mx = np.round(rng.normal(-70, 3, n), 0)
        assert np.array_equal(shadow_mask(ts, du, mx), pairwise(ts, du, mx))
    unit = np.sort(rng.integers(0, 5, 400))
    ts = rng.integers(0, 900_000, 400)
    du = rng.integers(8000, 40000, 400)
    mx = rng.normal(-70, 4, 400)
    whole = shadow_mask(ts + unit * _UNIT_GAP_US, du, mx)
    for u in range(5):
        m = unit == u
        assert np.array_equal(whole[m], pairwise(ts[m], du[m], mx[m]))


def test_c_shadow_filter_per_unit_equals_the_pairwise_definition():
    """csrc/rt_pyfinal.c shadow_units (what finalize_arrays runs): rows sorted by unit, every unit on its own, == the pairwise
    definition of analyze.py:283-313 with ties, zero durations and touching intervals; a unit beyond its size limit is refused
    (return 1, output untouched) so that the caller takes the numpy sweep."""
    from pyradiotracking_b200 import _rtfinal

    def pairwise(unit, ts, du, mx):
        te = ts + du
        return np.array([bool(((unit == unit[i]) & (ts[i] <= te) & (te[i] >= ts) & (mx > mx[i])).any()) for i in range(len(ts))], dtype=bool)

    rng = np.random.default_rng(23)
    for trial in range(200):
        n = int(rng.integers(0, 300))
        unit = np.sort(rng.integers(0, int(rng.integers(1, 9)), n)).astype(np.int64)
        scale = int(rng.choice([1, 1000]))
        ts = (rng.integers(0, 60, n) * scale).astype(np.int64)
        du = (rng.integers(0, 25, n) * int(rng.choice([1, 700]))).astype(np.int64)
        mx = np.round(rng.normal(-70, 3, n), int(rng.integers(0, 3)))
        out = np.zeros(n, dtype=bool)
        assert _rtfinal.shadow_units(unit, ts, du, mx, out.view(np.uint8)) == 0
        assert np.array_equal(out, pairwise(unit, ts, du, mx)), trial
    n = 8193
    out = np.ones(n, dtype=bool)
    z = np.zeros(n, dtype=np.int64)
    assert _rtfinal.shadow_units(z, z, z, np.zeros(n), out.view(np.uint8)) == 1 and out.all()


def test_unit_timestamps_and_parity_counters():
    """blocks_per_launch: unit u = stream * B + block starts `block` callback lengths after the launch (the reference's `_ts +=
    buffer_len_dt`, analyze.py:221); and oracle/check.py (the bench's parity gate) counts an identical result as identical."""
    from oracle import check as C

    w = synth.C1
    ba = BatchAnalyzer(devices=["a", "b"], calibration_db=[0.0, 1.0], sample_rate=w.sample_rate, center_freq=w.center_freq,
                       fft_nperseg=256, fft_window="hamming", signal_min_duration_ms=8, signal_max_duration_ms=40,
                       signal_threshold_dbw=-90.0, snr_threshold_db=5.0, blocks_per_launch=3)
    t0 = datetime.datetime(2026, 1, 1)
    uts = ba.unit_ts([t0, t0 + datetime.timedelta(seconds=5)])
    ts, step = t0, datetime.timedelta(seconds=w.block_samples / w.sample_rate)
    for b in range(3):
        assert uts[b] == ts and uts[3 + b] == ts + datetime.timedelta(seconds=5)
        ts += step
    with pytest.raises(ValueError, match="powers of two"):
        BatchAnalyzer(devices=["a"], calibration_db=[0.0], sample_rate=300000, center_freq=0, fft_nperseg=250, fft_window="hamming",
                      signal_min_duration_ms=8, signal_max_duration_ms=40, signal_threshold_dbw=-90.0, snr_threshold_db=5.0)
    P = R.Params.make(sample_rate=w.sample_rate)
    ora = R.OracleAnalyzer(P)
    cap = synth.make_stream(w, 0, 1)
    _, _, S, found, kept = ora.process_block(cap[0], t0)
    tot = C.new_totals()
    C.add_block(tot, P, S, None, found, kept, list(found), [d.key() for d in found], list(kept), S.T.astype(np.float32), S.mean(axis=1).astype(np.float32))
    assert C.verdict(tot) and tot["key_mismatches"] == 0 and tot["cells_checked"] > 0
    C.add_block(tot, P, S, None, found, kept, list(found)[1:], [d.key() for d in found][1:], list(kept))
    assert tot["key_mismatches"] == 1 and not C.verdict(tot)
