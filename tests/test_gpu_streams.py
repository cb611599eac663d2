"""The engine's stream contract on the B200 (pytest -m gpu), against the float64 oracle.

  A  producer ordering: a device input still being written by queued work (a spin, then the copy of the real capture over a
     poison capture) on the default stream, a torch side stream, a __cuda_array_interface__ `stream`, the engine's own
     set_stream stream or another one, for every spectrogram kernel, sample format and scan schedule, and pipelined
  B  input lifetime: a device input freed right after `submit` while the engine's reads are still queued
  C  the results ring (a third launch drops the oldest), the parity hooks of every unit while an older launch is unfetched,
     `join`, timing (records unchanged) and set_stream with launches in flight

An engine that does not order its reads after the producer reads valid, stale memory: the poison's records, no fault.
"""
import datetime
import functools

import numpy as np
import pytest

from pyradiotracking_b200 import engine as E
from pyradiotracking_b200 import synth
from pyradiotracking_b200.analyze import BatchAnalyzer
from tests import format_oracle as FO
from tests import parity

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

T0 = datetime.datetime(2026, 7, 7, 7, 7, 7)
FS = BLOCK = 300_000
SPIN_CYCLES = 100_000_000          # torch.cuda._sleep: about 50 ms at the B200's clocks; bounded, queued once per case
REAL, POISON = 1, 2                # synth stream indices of the capture analysed and of the stale one under it
WINDOW = {256: "hamming", 512: "hamming", 1024: "hann"}


def _kw(nperseg):
    # nperseg 1024 at 300 kS/s: at -90 dBW the noise itself crosses the threshold hundreds of times per block, some of them
    # within parity.NEAR_THRESHOLD of it; at -82 dBW no run of these captures is that close, so every run must match
    return dict(device="0", calibration_db=0.0, sample_rate=FS, center_freq=150_150_000, fft_nperseg=nperseg,
                fft_window=WINDOW[nperseg], signal_min_duration_ms=8.0, signal_max_duration_ms=40.0,
                signal_threshold_dbw=-82.0 if nperseg == 1024 else -90.0, snr_threshold_db=5.0, sdr_callback_length=BLOCK)


@functools.lru_cache(maxsize=None)
def _capture(fmt, nperseg, stream, nb):
    """[nb, 2 BLOCK] elements of `fmt`: noise and 10-30 LSB bursts, one straddling every block boundary."""
    w = synth.Workload(93, f"streams-{nperseg}", FS, BLOCK, nperseg=nperseg, amp_lsb=(10.0, 30.0))
    return synth.make_stream_format(w, fmt, stream, nb)


@functools.lru_cache(maxsize=None)
def _oracle(fmt, nperseg, stream, nb):
    """[(S, last, found)] of the float64 oracle on the decoded samples of every block of one stream."""
    ora = FO.SampleOracle(parity.oracle_params(_kw(nperseg)))
    out = []
    for b, blk in enumerate(_capture(fmt, nperseg, stream, nb)):
        last = ora.last
        _, _, S, found, _ = ora.process_samples(FO.decode_samples(blk, fmt), _ts(b))
        out.append((S, last, found))
    return out


def _ts(b):
    return parity.block_ts(T0, b, BLOCK, FS)


def _analyzer(nperseg, fmt="cu8", n_streams=1, **extra):
    kw = _kw(nperseg)
    return BatchAnalyzer(**parity.batch_kwargs(kw, devices=[str(i) for i in range(n_streams)], calibration=[0.0] * n_streams,
                                               sample_format=fmt, **extra))


def _check(ba, rec, nperseg, wants, b0, spectro=False, tag=""):
    """Records of one launch against the oracle: wants[u] = (S, last, found) of analyzer unit u, b0 = the launch's first block.
    -> records the oracle has."""
    P = parity.oracle_params(_kw(nperseg))
    res = ba.finalize(rec, [_ts(b0)] * ba.n_streams)
    n = 0
    for u, (S, last, found) in enumerate(wants):
        sigs, keys = res[u]
        st = parity.compare_block(P, S, last, found, sigs, keys)
        assert st["near_threshold_mismatch"] == 0, (tag, u, st)
        n += st["oracle"]
        if spectro:
            parity.compare_spectrogram(P, S, ba.engine.read_spectrogram(u), ba.engine.read_row_means(u), tag=f"{tag}/u{u}")
    return n


def _dev(blk, complex64=False):
    """One block as a [1, ...] device tensor, written synchronously (pageable source)."""
    x = blk.view(np.complex64) if complex64 else blk
    return torch.from_numpy(np.ascontiguousarray(x[None])).cuda()


class Cai:
    """A CuPy / Numba style device array over a torch tensor (CUDA Array Interface v3)."""

    def __init__(self, t, **stream):
        self.t = t
        cai = dict(shape=tuple(t.shape), typestr=np.dtype(str(t.dtype)[6:]).str, data=(t.data_ptr(), False), version=3, strides=None)
        cai.update(stream)
        self.__cuda_array_interface__ = cai


@pytest.fixture
def delayed():
    """delayed(real, poison, producer) -> a device buffer that holds `poison` now and `real` once `producer` (a torch stream)
    has run a ~50 ms spin; the caller asserts `not producer.query()` right before the engine call."""
    torch.cuda.synchronize()

    def make(real, poison, producer):
        buf = poison.clone()
        torch.cuda.synchronize()                  # the poison is in place, the producer idle
        with torch.cuda.stream(producer):
            torch.cuda._sleep(SPIN_CYCLES)
            buf.copy_(real)
        return buf

    try:
        yield make
    finally:
        torch.cuda.synchronize()                  # no work outlives the test


def _pair(fmt, nperseg, nb, complex64=False):
    """device blocks of the real and the poison capture, and the real capture's oracle; the two must disagree."""
    real, poison = _capture(fmt, nperseg, REAL, nb), _capture(fmt, nperseg, POISON, nb)
    want, other = _oracle(fmt, nperseg, REAL, nb), _oracle(fmt, nperseg, POISON, nb)
    for b in range(nb):
        assert [d.key() for d in want[b][2]] != [d.key() for d in other[b][2]] and want[b][2], b
    return [_dev(x, complex64) for x in real], [_dev(x, complex64) for x in poison], want


# ---------------------------------------------------------------------------------------------------------------------------
# A. producer ordering
# ---------------------------------------------------------------------------------------------------------------------------
A1_CASES = [  # fmt, nperseg, impl, complex64
    ("cu8", 256, E.FFT_AUTO, False),              # register kernel
    ("cu8", 256, E.FFT_TC256, False),
    ("cu8", 1024, E.FFT_AUTO, False),             # radix-16 kernel
    ("cu8", 512, E.FFT_GENERIC, False),
    ("ci8", 256, E.FFT_AUTO, False),
    ("ci16_le", 256, E.FFT_AUTO, False),          # generic kernel
    ("cf32_le", 256, E.FFT_AUTO, False),
    ("cf32_le", 256, E.FFT_AUTO, True),           # complex64 tensor
]


@pytest.mark.parametrize("fmt,nperseg,impl,complex64", A1_CASES, ids=lambda v: str(v))
def test_input_written_on_the_default_stream_is_read_after_it(delayed, fmt, nperseg, impl, complex64):
    nb = 2
    real, poison, want = _pair(fmt, nperseg, nb, complex64)
    default = torch.cuda.default_stream()
    ba = _analyzer(nperseg, fmt, fft_impl=impl)
    try:
        n = 0
        for b in range(nb):                       # block 1 carries from block 0
            buf = delayed(real[b], poison[b], default)
            assert not default.query()
            rec = ba.engine.process(buf)
            n += _check(ba, rec, nperseg, [want[b]], b, spectro=True, tag=f"streams/A1/{fmt}/n{nperseg}/impl{impl}/b{b}")
        assert n >= 2
    finally:
        ba.close()


def test_input_written_on_a_side_stream_is_read_after_it(delayed):
    real, poison, want = _pair("cu8", 256, 2)
    side = torch.cuda.Stream()
    ba = _analyzer(256)
    try:
        for b in range(2):
            buf = delayed(real[b], poison[b], side)
            with torch.cuda.stream(side):
                assert not side.query()
                _check(ba, ba.engine.process(buf), 256, [want[b]], b, tag="streams/A2")
    finally:
        ba.close()


@pytest.mark.parametrize("which", ["producer", "legacy"])
def test_cuda_array_interface_stream_is_waited_for(delayed, which):
    """CAI v3 `stream`: the producer's handle, or 1 (the legacy default stream), with torch's current stream idle."""
    real, poison, want = _pair("cu8", 256, 2)
    side = torch.cuda.Stream()
    producer = side if which == "producer" else torch.cuda.default_stream()
    handle = side.cuda_stream if which == "producer" else 1
    ba = _analyzer(256)
    try:
        for b in range(2):
            buf = delayed(real[b], poison[b], producer)
            assert not producer.query()
            _check(ba, ba.engine.process(Cai(buf, stream=handle)), 256, [want[b]], b, tag=f"streams/A3/{which}")
    finally:
        ba.close()


def test_cuda_array_interface_without_stream_needs_no_wait():
    """`stream` absent or None: the producer has synchronised (the spec's contract); the engine reads the data as it is."""
    real, _, want = _pair("cu8", 256, 2)
    ba = _analyzer(256)
    try:
        for b, extra in enumerate(({}, {"stream": None})):
            torch.cuda.synchronize()
            _check(ba, ba.engine.process(Cai(real[b], **extra)), 256, [want[b]], b, tag=f"streams/A3/{extra}")
        with pytest.raises(ValueError):
            ba.engine.launch(Cai(real[0], stream=0))          # ambiguous: forbidden by the CUDA Array Interface
    finally:
        ba.close()


@pytest.mark.parametrize("schedule,launch_streams", [(E.SCAN_SERIAL, 1), (E.SCAN_OVERLAP, 1), (E.SCAN_OVERLAP, 2), (E.SCAN_LEAN, 2)],
                         ids=["serial-1", "overlap-1", "overlap-2", "lean-2"])
def test_every_schedule_inherits_the_producer_order(delayed, schedule, launch_streams):
    """The spectrogram kernels run on internal streams forked from the launch stream: they must wait for the producer too."""
    real, poison, want = _pair("cu8", 256, 3)
    default = torch.cuda.default_stream()
    ba = _analyzer(256, scan_schedule=schedule, launch_streams=launch_streams)
    try:
        for b in range(3):                        # with two launch streams, consecutive launches alternate between them
            buf = delayed(real[b], poison[b], default)
            assert not default.query()
            _check(ba, ba.engine.process(buf), 256, [want[b]], b, tag=f"streams/A4/{schedule}/{launch_streams}")
    finally:
        ba.close()


def test_engine_on_a_set_stream_waits_for_another_producer(delayed):
    real, poison, want = _pair("cu8", 256, 2)
    eng_stream, producer = torch.cuda.Stream(), torch.cuda.Stream()
    ba = _analyzer(256)
    try:
        ba.engine.set_stream(eng_stream.cuda_stream)
        for b in range(2):
            buf = delayed(real[b], poison[b], producer)
            with torch.cuda.stream(producer):
                assert not producer.query()
                _check(ba, ba.engine.process(buf), 256, [want[b]], b, tag="streams/A5")
    finally:
        ba.close()


def test_pipelined_submit_waits_for_the_input_still_being_written(delayed):
    """submit, submit, collect, collect: the second input is written while the first launch runs."""
    real, poison, want = _pair("cu8", 256, 2)
    default = torch.cuda.default_stream()
    ba = _analyzer(256)
    try:
        first = real[0].clone()
        torch.cuda.synchronize()
        ba.submit(first)
        second = delayed(real[1], poison[1], default)
        assert not default.query()
        ba.submit(second)
        for b in range(2):
            rec = ba.engine.fetch()
            _check(ba, rec, 256, [want[b]], b, tag=f"streams/A6/b{b}")
    finally:
        ba.close()


# ---------------------------------------------------------------------------------------------------------------------------
# B. input lifetime
# ---------------------------------------------------------------------------------------------------------------------------
def test_input_freed_after_submit_is_not_reused_before_it_is_read():
    """submit(tmp); del tmp; a new tensor of the same size written on the default stream must not land in tmp's memory while
    the engine's reads are still queued (its stream runs a spin first).  No empty_cache: the freed block stays mapped."""
    real, poison, want = _pair("cu8", 256, 1)
    eng_stream = torch.cuda.Stream()
    ba = _analyzer(256)
    try:
        ba.engine.set_stream(eng_stream.cuda_stream)
        torch.cuda.synchronize()
        with torch.cuda.stream(eng_stream):
            torch.cuda._sleep(SPIN_CYCLES)
        tmp = real[0].clone()
        ptr = tmp.data_ptr()
        assert not eng_stream.query()
        ba.submit(tmp)
        del tmp
        other = torch.empty_like(real[0])
        other.copy_(poison[0])
        reused = other.data_ptr() == ptr
        rec = ba.engine.fetch()
        try:
            _check(ba, rec, 256, [want[0]], 0, tag="streams/B")
        except AssertionError as e:
            raise AssertionError(f"freed input overwritten (new tensor at the same address: {reused}): {e}") from e
    finally:
        torch.cuda.synchronize()
        ba.close()


# ---------------------------------------------------------------------------------------------------------------------------
# C. ring, hooks, join, timing, set_stream in flight
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("impl", [E.FFT_AUTO, E.FFT_TC256, E.FFT_GENERIC], ids=["reg256", "tc256", "generic"])
@pytest.mark.parametrize("launch_streams", [1, 2])
def test_third_launch_drops_the_oldest_result(impl, launch_streams):
    cap, want = _capture("cu8", 256, REAL, 3), _oracle("cu8", 256, REAL, 3)
    ba = _analyzer(256, fft_impl=impl, launch_streams=launch_streams)
    try:
        for b in range(3):
            ba.submit(cap[b][None, :])
        n = 0
        for b in (1, 2):                          # block 0's result was dropped; block 1 still carried from it
            n += _check(ba, ba.engine.fetch(), 256, [want[b]], b, spectro=(b == 2), tag=f"streams/C1/impl{impl}/ls{launch_streams}/b{b}")
        assert n > 0 and any(d.key()[1] < 0 for d in want[2][2])      # block 2 has a run carried from block 1
        with pytest.raises(E.EngineError) as ei:
            ba.engine.fetch()
        assert ei.value.code == E.RT_ERR_STATE
    finally:
        ba.close()


@pytest.mark.parametrize("nperseg,impl,bpl", [(256, E.FFT_AUTO, 2), (256, E.FFT_GENERIC, 2), (1024, E.FFT_AUTO, 2), (256, E.FFT_TC256, 1)],
                         ids=["perm", "linear", "radix16", "tile"])
def test_parity_hooks_read_the_newest_launch_of_every_unit(nperseg, impl, bpl):
    """read_spectrogram / read_row_means of every analyzer unit while the older of two launches is still unfetched."""
    n_streams, nb = 3, 2 * bpl
    caps = [_capture("cu8", nperseg, s, nb) for s in range(n_streams)]
    wants = [_oracle("cu8", nperseg, s, nb) for s in range(n_streams)]
    ba = _analyzer(nperseg, n_streams=n_streams, fft_impl=impl, blocks_per_launch=bpl)
    try:
        for g in range(2):
            ba.submit(np.stack([c[g * bpl:(g + 1) * bpl].reshape(-1) for c in caps]))
        newest = [wants[s][bpl + k] for s in range(n_streams) for k in range(bpl)]
        P = parity.oracle_params(_kw(nperseg))
        for u, (S, _, _) in enumerate(newest):
            parity.compare_spectrogram(P, S, ba.engine.read_spectrogram(u), ba.engine.read_row_means(u), tag=f"streams/C2/n{nperseg}/impl{impl}/u{u}")
        n = 0
        for g in range(2):
            n += _check(ba, ba.engine.fetch(), nperseg, [wants[s][g * bpl + k] for s in range(n_streams) for k in range(bpl)], g * bpl,
                        tag=f"streams/C2/n{nperseg}/impl{impl}/g{g}")
        assert n > 0
    finally:
        ba.close()


@pytest.mark.parametrize("schedule", [E.SCAN_OVERLAP, E.SCAN_LEAN], ids=["overlap", "lean"])
def test_join_orders_later_work_on_the_launch_stream(schedule):
    """set_stream(S), launch a device buffer, join, then overwrite the buffer on S: the launch saw the original."""
    real, poison, want = _pair("cu8", 256, 1)
    s = torch.cuda.Stream()
    ba = _analyzer(256, scan_schedule=schedule, launch_streams=2)
    try:
        ba.engine.set_stream(s.cuda_stream)
        buf = real[0].clone()
        torch.cuda.synchronize()
        with torch.cuda.stream(s):
            torch.cuda._sleep(SPIN_CYCLES // 10)  # the launch forks from S behind this spin
            ba.submit(buf)
            ba.engine.join()
            buf.copy_(poison[0])
        _check(ba, ba.engine.fetch(), 256, [want[0]], 0, tag=f"streams/C3/{schedule}")
    finally:
        torch.cuda.synchronize()
        ba.close()


def test_timing_does_not_change_the_records():
    nb = 6
    cap, want = _capture("cu8", 256, REAL, nb), _oracle("cu8", 256, REAL, nb)

    def run(period):
        ba = _analyzer(256)
        try:
            if period:
                ba.engine.enable_timing(period)
            out = []
            ba.submit(cap[0][None, :])
            for b in range(nb):                   # two launches in flight
                if b + 1 < nb:
                    ba.submit(cap[b + 1][None, :])
                out.append(ba.engine.fetch())
            return out, (ba.engine.timing() if period else None)
        finally:
            ba.close()

    ref, _ = run(0)
    ba = _analyzer(256)
    try:
        assert sum(_check(ba, r, 256, [want[b]], b) for b, r in enumerate(ref)) > 0
    finally:
        ba.close()
    for period in (1, 3):
        got, tim = run(period)
        assert [r.tobytes() for r in got] == [r.tobytes() for r in ref], period
        assert tim["launches"] == nb and tim["kernels"] in (3 * nb, 4 * nb) and tim["spectrogram_ms"] > 0, (period, tim)


def test_set_stream_with_two_launches_in_flight():
    cap, want = _capture("cu8", 256, REAL, 3), _oracle("cu8", 256, REAL, 3)
    s = torch.cuda.Stream()
    ba = _analyzer(256)
    try:
        ba.submit(cap[0][None, :])
        ba.submit(cap[1][None, :])
        ba.engine.set_stream(s.cuda_stream)
        for b in range(2):
            _check(ba, ba.engine.fetch(), 256, [want[b]], b, tag=f"streams/C5/b{b}")
        ba.submit(cap[2][None, :])                # and the engine goes on on S
        _check(ba, ba.engine.fetch(), 256, [want[2]], 2, spectro=True, tag="streams/C5/b2")
    finally:
        torch.cuda.synchronize()
        ba.close()
