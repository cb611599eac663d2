"""Host side of the detection hot path: the reference's `SignalAnalyzer` interface on top of
the CUDA engine.

* `SignalAnalyzer` keeps the reference constructor keys, the `process_samples(buffer, context)`
  callback and the queue outputs (reference: radiotracking/analyze.py:20-280), so
  `radiotracking/__main__.py:94-130` can start it in place of the reference class.
* `BatchAnalyzer` is the same analysis for many independent streams on one GPU (one engine
  call per block of every stream); `SignalAnalyzer` is a batch of one.

Split of labour (SURVEY.md §7 hard part 3): the device does everything per cell and returns
integer run limits `(fi, start, end)` plus linear statistics; everything that the reference
computes in float64 *per signal* -- `times`, `freqs`, the probe stride, the duration test,
timestamps, dB conversion (analyze.py:354, 419-450) -- is done here with the reference's own
expressions so those fields are bit-identical.
"""
import datetime
import logging
import math
import multiprocessing
import signal as _signal
import sys
import time
from typing import List, NamedTuple, Optional, Sequence, Tuple

import numpy as np

from . import engine as _engine
from .messages import from_dB, message_types

try:
    from . import _rtfinal                  # csrc/rt_pyfinal.c: the Signal-object builder of the finaliser
except ImportError:                         # never built in this tree: build it now (gcc), like engine.load_library does with nvcc
    from . import build as _build

    _build.build_pyfinal()
    from . import _rtfinal

logger = logging.getLogger(__name__)
UTC = datetime.timezone.utc


def resolve_window(window, nperseg: int) -> np.ndarray:
    """What scipy's `_triage_segments` makes of `fft_window` (analyze.py:236): a name or
    `(name, param)` tuple goes through `scipy.signal.get_window` (periodic), an array is used
    verbatim."""
    if isinstance(window, (str, tuple)):
        from scipy.signal import get_window

        return np.asarray(get_window(window, nperseg), dtype=np.float64)
    win = np.asarray(window, dtype=np.float64)
    if win.ndim != 1:
        raise ValueError("window must be 1-D")
    if win.shape[0] != nperseg:
        raise ValueError("window must have length of nperseg")
    return win


class DetectionPlan:
    """Per-configuration float64 constants, computed exactly like scipy / the reference do."""

    def __init__(self, sample_rate: float, nperseg: int, block_samples: int, min_duration_s: float, max_duration_s: float):
        fs = sample_rate
        self.nperseg = nperseg
        self.block_samples = block_samples
        # scipy _spectral_helper: freqs = fftfreq(nfft, 1/fs); time = arange(nperseg/2, N - nperseg/2 + 1, nperseg - noverlap)/fs
        self.freqs = np.fft.fftfreq(nperseg, 1 / fs)
        self.times = np.arange(nperseg / 2, block_samples - nperseg / 2 + 1, nperseg) / float(fs)
        self.T = len(self.times)
        if block_samples > 0 and self.T < 2:
            # one column (or a block shorter than nperseg, which scipy shrinks to one column): analyze.py:354 indexes times[1]
            raise IndexError("index 1 is out of bounds for axis 0 with size 1")
        self.min_duration = min_duration_s
        self.max_duration = max_duration_s
        if self.T >= 2:
            dt = self.times[1] - self.times[0]
            self.min_num = min_duration_s / dt                       # analyze.py:354
            self.stride = max(1, int(self.min_num))                  # analyze.py:364
            # coarse gates for the device (+-1 column of slack around the float64 test below)
            self.min_cols = max(0, int(math.floor(min_duration_s / dt)) - 1)
            self.max_cols = int(math.ceil(max_duration_s / dt)) + 2
        else:
            self.stride, self.min_cols, self.max_cols = 1, 0, 2

    def duration(self, start: int, end: int) -> Tuple[float, float]:
        """(start_dt, duration_s) exactly as analyze.py:419-427."""
        times = self.times
        end_dt = times[end]
        start_dt = -times[-start] if start < 0 else times[start]
        return start_dt, end_dt - start_dt


def _us(td: datetime.timedelta) -> int:
    return (td.days * 86400 + td.seconds) * 1_000_000 + td.microseconds


def timedelta_us(seconds: np.ndarray) -> np.ndarray:
    """int64 microseconds of `datetime.timedelta(seconds=x)` for float64 x, vectorised: CPython splits x with
    modf and rounds the fractional microseconds half-to-even."""
    frac, whole = np.modf(np.asarray(seconds, dtype=np.float64))
    return whole.astype(np.int64) * 1_000_000 + np.rint(frac * 1e6).astype(np.int64)


class Finalized(NamedTuple):
    """Column view of the signals of one engine call (rows sorted by stream, bin, start)."""
    stream: np.ndarray
    fi: np.ndarray
    start: np.ndarray
    end: np.ndarray
    ts_off_us: np.ndarray       # microseconds from the stream's ts_start (analyze.py:434)
    dur_us: np.ndarray
    frequency: np.ndarray
    max: np.ndarray
    avg: np.ndarray
    std: np.ndarray
    noise: np.ndarray
    snr: np.ndarray
    shadow: np.ndarray          # True: dropped by filter_shadow_signals


def shadow_mask(ts_us: np.ndarray, dur_us: np.ndarray, max_dbw: np.ndarray) -> np.ndarray:
    """True where a signal is a shadow (analyze.py:283-313): some signal of the same list overlaps
    it in time (closed intervals, microsecond datetimes) and is strictly louder.  No frequency term.

    The reference compares every pair (O(S^2), 18 ms at S = 900).  Signal j overlaps signal i iff it STARTS inside
    [ts_i, te_i] or its interval CONTAINS ts_i, so the loudest overlapping signal is the maximum of a range-maximum
    query over the start times (sparse table) and of a stabbing query at ts_i (every interval is a chmax update of a
    range of start times, written as two power-of-two blocks and pushed down level by level): O(S log S), vectorised."""
    n = len(ts_us)
    if n < 2:
        return np.zeros(n, dtype=bool)
    ts = np.asarray(ts_us, dtype=np.int64)
    te = ts + np.asarray(dur_us, dtype=np.int64)
    mx = np.asarray(max_dbw, dtype=np.float64)
    order = np.argsort(ts, kind="stable")
    ts_s = ts[order]
    first = np.r_[True, ts_s[1:] != ts_s[:-1]]             # first signal of every distinct start time
    U = ts_s[first]
    lo = np.empty(n, dtype=np.int64)
    lo[order] = np.cumsum(first) - 1                       # lo[i]: index of ts[i] among the sorted distinct start times
    hi = np.searchsorted(U, te, side="right") - 1         # last distinct start time <= te[i] (>= lo[i]: durations are >= 0)
    m = len(U)
    K = int(np.max(hi - lo + 1)).bit_length()             # levels needed: 2^(K-1) <= longest range of start times
    st = np.full((K, m), -np.inf)                         # st[k][u] = max over start times u .. u + 2^k - 1
    st[0] = np.maximum.reduceat(mx[order], np.flatnonzero(first))
    for k in range(1, K):
        h = 1 << (k - 1)
        st[k] = st[k - 1]
        st[k, : m - h] = np.maximum(st[k - 1, : m - h], st[k - 1, h:])
    k = np.frexp((hi - lo + 1).astype(np.float64))[1] - 1     # floor(log2(range length))
    off = hi - (1 << k) + 1
    starts_inside = np.maximum(st[k, lo], st[k, off])
    rt = np.full(K * m, -np.inf)                          # pending chmax updates of the blocks [u, u + 2^k), flattened [k][u]
    cell = np.concatenate((k * m + lo, k * m + off))      # two (overlapping) blocks per interval; grouped maximum per cell
    val = np.concatenate((mx, mx))
    o2 = np.argsort(cell, kind="stable")
    cell_s = cell[o2]
    g = np.flatnonzero(np.r_[True, cell_s[1:] != cell_s[:-1]])
    rt[cell_s[g]] = np.maximum.reduceat(val[o2], g)
    rt = rt.reshape(K, m)
    for kk in range(K - 1, 0, -1):
        h = 1 << (kk - 1)
        np.maximum(rt[kk - 1], rt[kk], out=rt[kk - 1])
        np.maximum(rt[kk - 1, h:], rt[kk, : m - h], out=rt[kk - 1, h:])
    contains_start = rt[0, lo]
    return np.maximum(starts_inside, contains_start) > mx


# time offset between analyzer units when the shadow filter of a whole batch is evaluated in one pass (2^44 us = 203 days:
# further apart than any two signals of one callback, so units never overlap)
_UNIT_GAP_US = 1 << 44


class BatchAnalyzer:
    """`n` independent analyzers (same sample rate / FFT / duration keys, own device name and
    calibration) evaluated together on one GPU."""

    def __init__(self, devices: Sequence[str], calibration_db: Sequence[float], sample_rate: int, center_freq,
                 fft_nperseg: int, fft_window, signal_min_duration_ms: float, signal_max_duration_ms: float,
                 signal_threshold_dbw: float, snr_threshold_db: float, sdr_callback_length: Optional[int] = None,
                 cuda_device: int = 0, max_records: int = 0, fft_impl: int = _engine.FFT_AUTO,
                 scan_schedule: int = _engine.SCAN_AUTO, launch_streams: int = 0, chunk_segs: int = 0,
                 blocks_per_launch: int = 1, sample_format: str = "cu8"):
        """`sample_format`: the SigMF datatype of the input blocks, one of `engine.SAMPLE_FORMATS` (cu8: RTL-SDR bytes, ci8, ci16_le,
        cf32_le); the thresholds apply to the normalised samples (INTEGRATION.md).  `center_freq`: one value for every device, or
        one per device (the channels of a wideband recording, wideband.py); a Signal's frequency is `freqs[fi] + center_freq`."""
        if sample_format not in _engine.SAMPLE_FORMATS:
            raise ValueError(f"sample_format = {sample_format!r}: the B200 engine reads {', '.join(_engine.SAMPLE_FORMATS)} (see INTEGRATION.md)")
        self.sample_format = sample_format
        self.devices = [str(d) for d in devices]
        self.n_streams = len(self.devices)
        self.calibration_db = [float(c) for c in calibration_db]
        if len(self.calibration_db) != self.n_streams:
            raise ValueError("one calibration value per device")
        if not isinstance(fft_nperseg, (int, np.integer)) or fft_nperseg < 8 or fft_nperseg > 4096 or fft_nperseg & (fft_nperseg - 1):
            # scope limit of the CUDA path (scipy takes any length): say so here, not as an EngineError inside the child process
            raise ValueError(f"fft_nperseg = {fft_nperseg}: the B200 engine supports powers of two in [8, 4096] (see INTEGRATION.md)")
        if blocks_per_launch < 1:
            raise ValueError("blocks_per_launch must be >= 1")
        self.sample_rate = sample_rate
        self.center_freq = center_freq
        self._center_freqs = None           # per device, or None: one scalar for all
        if np.ndim(center_freq) != 0:
            self._center_freqs = np.asarray(center_freq)
            if self._center_freqs.shape != (self.n_streams,):
                raise ValueError("center_freq: one value, or one per device")
        self.fft_nperseg = int(fft_nperseg)
        self.fft_window = fft_window
        self.blocks_per_launch = int(blocks_per_launch)
        self.n_units = self.n_streams * self.blocks_per_launch     # analyzer units per launch (stream-major, block-minor)
        self.block_samples = sample_rate if sdr_callback_length is None else sdr_callback_length   # analyze.py:108-109
        self.signal_min_duration = signal_min_duration_ms / 1000                                    # analyze.py:113
        self.signal_max_duration = signal_max_duration_ms / 1000                                    # analyze.py:114
        self.signal_threshold = [from_dB(signal_threshold_dbw + c) for c in self.calibration_db]   # analyze.py:115
        self.snr_threshold = from_dB(snr_threshold_db)                                              # analyze.py:116
        self.plan = DetectionPlan(sample_rate, fft_nperseg, self.block_samples, self.signal_min_duration, self.signal_max_duration)
        self.window = resolve_window(fft_window, fft_nperseg)
        self.cuda_device = cuda_device
        self.max_records = max_records
        self.fft_impl = fft_impl
        self.scan_schedule, self.launch_streams, self.chunk_segs = scan_schedule, launch_streams, chunk_segs
        self.timings = {"fetch_wait_s": 0.0, "finalize_s": 0.0, "build_s": 0.0, "collects": 0}   # host-side split of collect()
        self._engine: Optional[_engine.Engine] = None
        self.last_record_count = 0          # candidate records copied back by the last collect()
        self.Signal, self.StateMessage = message_types()
        # the two known Signal classes only store their arguments (radiotracking/__init__.py:136-170): their instances may be
        # filled directly; any other class is called like the reference calls it
        self._direct = self.Signal.__module__ in ("radiotracking", "pyradiotracking_b200.messages")

    # the engine is created on first use: after a fork, inside the analyzer process
    @property
    def engine(self) -> _engine.Engine:
        if self._engine is None:
            if self.plan.T < 2:
                raise ValueError("block shorter than two FFT segments")
            self._engine = _engine.Engine(
                n_streams=self.n_streams, block_samples=self.block_samples, nperseg=self.fft_nperseg, window=self.window,
                sample_rate=self.sample_rate, signal_threshold=self.signal_threshold, snr_threshold=self.snr_threshold,
                probe_stride=self.plan.stride, min_cols=self.plan.min_cols, max_cols=self.plan.max_cols,
                max_records=self.max_records, cuda_device=self.cuda_device, fft_impl=self.fft_impl,
                scan_schedule=self.scan_schedule, launch_streams=self.launch_streams, chunk_segs=self.chunk_segs,
                blocks_per_launch=self.blocks_per_launch, sample_format=self.sample_format)
        return self._engine

    def close(self):
        if self._engine is not None:
            self._engine.close()
            self._engine = None

    def reset_stream(self, stream: int):
        """Forget the previous block of one stream (a restarted analyzer)."""
        self.engine.reset_stream(stream)

    # -- finaliser: records -> Signal objects ----------------------------------------------------
    def finalize_arrays(self, records: np.ndarray) -> "Finalized":
        """Vectorised analyze.py:419-450 for the candidate records of one engine call (sorted by stream, bin,
        start): exact float64 duration test, timestamps / durations rounded to microseconds exactly like
        `datetime.timedelta(seconds=float)`, dB statistics, and the per-stream shadow mask (analyze.py:283-328)."""
        plan = self.plan
        times = plan.times
        start = records["start"].astype(np.int64)
        end = records["end"].astype(np.int64)
        neg = start < 0
        start_dt = np.where(neg, -times[np.where(neg, -start, 0)], times[np.where(neg, 0, start)])   # :420-425
        duration_s = times[end] - start_dt                                                             # :427
        ok = ~(duration_s < self.signal_min_duration) & ~(duration_s > self.signal_max_duration)       # :429-433
        r = records[ok]
        start_dt, duration_s = start_dt[ok], duration_s[ok]
        stream = r["stream"].astype(np.int64)                   # analyzer unit = stream * blocks_per_launch + block
        cal = np.asarray(self.calibration_db, dtype=np.float64)[stream // self.blocks_per_launch]
        mean = r["mean_lin"].astype(np.float64)
        row = r["row_mean"].astype(np.float64)
        with np.errstate(divide="ignore", invalid="ignore"):
            fin = Finalized(
                stream=stream, fi=r["fi"].astype(np.int64), start=r["start"].astype(np.int64), end=r["end"].astype(np.int64),
                ts_off_us=timedelta_us(start_dt), dur_us=timedelta_us(duration_s),
                frequency=plan.freqs[r["fi"]] + (self.center_freq if self._center_freqs is None else self._center_freqs[stream // self.blocks_per_launch]),
                max=10 * np.log10(r["max_lin"].astype(np.float64)) - cal, avg=10 * np.log10(mean) - cal,
                std=r["std_db"].astype(np.float64), noise=10 * np.log10(row), snr=10 * np.log10(mean / row),
                shadow=np.zeros(len(r), dtype=bool))
        # shadow filter per analyzer unit (signals of one callback share ts_start, so offsets are enough): one pass over the
        # whole batch, the units shifted so far apart in time that they cannot overlap
        if len(r) > 1:
            # per unit in C (exact pairwise pass over the few signals of a callback, csrc/rt_pyfinal.c); a unit with thousands of
            # candidates falls back to the O(S log S) sweep over the whole batch
            cols = [np.ascontiguousarray(c) for c in (fin.stream, fin.ts_off_us, fin.dur_us, fin.max)]
            if _rtfinal.shadow_units(*cols, fin.shadow.view(np.uint8)) != 0:
                fin.shadow[:] = shadow_mask(fin.ts_off_us + fin.stream * _UNIT_GAP_US, fin.dur_us, fin.max)
        return fin

    def unit_ts(self, ts_start: Sequence[datetime.datetime]) -> List[datetime.datetime]:
        """ts_start of every analyzer unit: block b of a launch starts b callback lengths after the stream's first block
        (the reference advances `_ts` by `timedelta(seconds=len(buffer) / sample_rate)` per callback, analyze.py:205,221)."""
        if self.blocks_per_launch == 1:
            return list(ts_start)
        dt = datetime.timedelta(seconds=self.block_samples / self.sample_rate)
        return [t + b * dt for t in ts_start for b in range(self.blocks_per_launch)]

    def build_signals(self, fin: "Finalized", ts_start: Sequence[datetime.datetime], keep: Optional[np.ndarray] = None):
        """Signal objects per analyzer unit, in the reference's emission order (bin, then time), for the rows of
        `fin` selected by `keep` (default: all).  `ts_start`: one per stream (the first block of the launch).

        The objects are built by the C helper `_rtfinal` (csrc/rt_pyfinal.c): `ts = (ts_start + timedelta(start_dt)).astimezone(utc)`
        (analyze.py:434,449) is evaluated as `ts_start.astimezone(utc) + timedelta` per unit, which is the same instant unless
        the local UTC offset changes inside the block -- checked per unit, the plain Python expression is used then."""
        uts = self.unit_ts(ts_start)
        idx = slice(None) if keep is None else np.nonzero(keep)[0]
        cols = [np.ascontiguousarray(c[idx], dtype=np.int64) for c in (fin.stream, fin.ts_off_us, fin.dur_us)]
        cols += [np.ascontiguousarray(c[idx], dtype=np.float64) for c in (fin.frequency, fin.max, fin.avg, fin.std, fin.noise, fin.snr)]
        block = datetime.timedelta(seconds=self.block_samples / self.sample_rate)
        base = [t.astimezone(UTC) for t in uts]
        if all((t + block).astimezone(UTC) - b == block and b - (t - block).astimezone(UTC) == block for t, b in zip(uts, base)):
            devices = self.devices if self.blocks_per_launch == 1 else [d for d in self.devices for _ in range(self.blocks_per_launch)]
            return _rtfinal.build_signals(self.Signal, self._direct, devices, base, *cols)
        out = [[] for _ in range(self.n_units)]                 # a UTC-offset change inside a block: the reference's expression
        Signal, devices, bpl, td = self.Signal, self.devices, self.blocks_per_launch, datetime.timedelta
        for u, off, dur, f, mx, av, sd, no, sn in zip(*[c.tolist() for c in cols]):
            ts = (uts[u] + td(microseconds=off)).astimezone(UTC)
            out[u].append(Signal(devices[u // bpl], ts, f, td(microseconds=dur), mx, av, sd, no, sn))
        return out

    def finalize(self, records: np.ndarray, ts_start: Sequence[datetime.datetime]):
        """-> per analyzer unit `(signals, keys)`: the reference's `extract_signals` output (analyze.py:419-450)
        in its order (bin, then time) and the integer `(fi, start, end)` of each."""
        fin = self.finalize_arrays(records)
        sigs = self.build_signals(fin, ts_start)
        keys = [[] for _ in range(self.n_units)]
        for s, k in zip(fin.stream.tolist(), zip(fin.fi.tolist(), fin.start.tolist(), fin.end.tolist())):
            keys[s].append(k)
        return list(zip(sigs, keys))

    @staticmethod
    def filter_shadow_signals(signals: list) -> list:
        """analyze.py:315-328, vectorised."""
        if len(signals) < 2:
            return list(signals)
        epoch = datetime.datetime(1970, 1, 1, tzinfo=UTC)
        ts = np.array([_us(s.ts - epoch) for s in signals], dtype=np.int64)
        du = np.array([_us(s.duration) for s in signals], dtype=np.int64)
        mx = np.array([s.max for s in signals], dtype=np.float64)
        shadow = shadow_mask(ts, du, mx)
        return [s for s, sh in zip(signals, shadow) if not sh]

    # -- one callback for every stream --------------------------------------------------------------
    def submit(self, iq) -> None:
        """Enqueue one block of every stream (H2D copy if `iq` is a host array, then the kernels); returns at once.
        Up to two submissions may be in flight; results come back in order from `collect`.  A CUDA tensor is read after the work
        queued so far on its device's current stream; `iq` is held until `collect` has returned this submission or a later one."""
        self.engine.launch(iq)

    def collect(self, ts_start: Sequence[datetime.datetime], with_all: bool = False):
        """Wait for the oldest submission.  -> per analyzer unit (= per stream when `blocks_per_launch` is 1; otherwise stream-major,
        block-minor) `(filtered_signals, n_before_filter)`, or with `with_all` `(filtered_signals, all_signals, keys)` like
        `process_blocks`.  `ts_start`: one per stream, the start of the first block of the launch."""
        t0 = time.perf_counter()
        records = self.engine.fetch()
        t1 = time.perf_counter()
        self.last_record_count = len(records)
        fin = self.finalize_arrays(records)
        t2 = time.perf_counter()
        if not with_all:
            kept = self.build_signals(fin, ts_start, ~fin.shadow)
            counts = np.bincount(fin.stream, minlength=self.n_units)
            out = [(kept[u], int(counts[u])) for u in range(self.n_units)]
        else:
            sigs = self.build_signals(fin, ts_start)
            keys = [[] for _ in range(self.n_units)]
            kept = [[] for _ in range(self.n_units)]
            pos = [0] * self.n_units
            for s, sh, k in zip(fin.stream.tolist(), fin.shadow.tolist(), zip(fin.fi.tolist(), fin.start.tolist(), fin.end.tolist())):
                keys[s].append(k)
                if not sh:
                    kept[s].append(sigs[s][pos[s]])      # the very objects of `sigs`, in order
                pos[s] += 1
            out = [(kept[u], sigs[u], keys[u]) for u in range(self.n_units)]
        tm = self.timings
        tm["fetch_wait_s"] += t1 - t0
        tm["finalize_s"] += t2 - t1
        tm["build_s"] += time.perf_counter() - t2
        tm["collects"] += 1
        return out

    def process_blocks(self, iq, ts_start: Sequence[datetime.datetime]):
        """`iq`: `[n_streams, 2*block_samples]` (`[n_streams, blocks_per_launch, 2*block_samples]`) interleaved I,Q elements of
        the analyzer's `sample_format` (uint8, int8, int16 or float32; cf32_le also complex64 with `block_samples` per block) on
        the host, or a CUDA tensor of that shape.  -> per analyzer unit `(filtered_signals, all_signals, keys)`."""
        self.submit(iq)
        return self.collect(ts_start, with_all=True)


def iq_to_bytes(buffer: np.ndarray) -> np.ndarray:
    """Inverse of pyrtlsdr's `packed_bytes_to_iq` (x = b/127.5 - 1): recover the uint8 I/Q bytes the
    SDR delivered from the complex samples handed to `process_samples`.  The kernels consume raw
    bytes; samples that are not on the 8-bit grid cannot have come from an RTL-SDR and are rejected."""
    x = np.ascontiguousarray(buffer, dtype=np.complex128).view(np.float64)
    b = (x + 1.0) * 127.5
    q = np.rint(b)
    if q.size and (np.max(np.abs(b - q)) > 1e-6 or q.min() < 0 or q.max() > 255):
        raise ValueError("samples are not 8-bit RTL-SDR IQ (x = byte/127.5 - 1); use process_bytes with the raw buffer")
    return q.astype(np.uint8)


class SignalAnalyzer(multiprocessing.Process):
    """Drop-in for `radiotracking.analyze.SignalAnalyzer` (analyze.py:20-129): same constructor keys,
    same callback, same queue traffic; the spectrogram and the scans run on the GPU.

    Extra keys (ignored by the reference thanks to its `**kwargs`): `cuda_device`.
    """

    def __init__(self, device: str, calibration_db: float, sample_rate: int, center_freq: int, gain: float,
                 fft_nperseg: int, fft_window, signal_min_duration_ms: float, signal_max_duration_ms: float,
                 signal_threshold_dbw: float, snr_threshold_db: float, verbose: int, sdr_max_restart: int,
                 sdr_timeout_s: int, state_update_s: int, sdr_callback_length: int, signal_queue, last_data_ts,
                 cuda_device: int = 0, **kwargs):
        super().__init__()
        self.device = device
        self.calibration_db = calibration_db
        try:
            self.device_index = int(device)                         # analyze.py:88-91
            logger.info(f"Using '{device}' as device index.")
        except ValueError:
            import rtlsdr                                           # analyze.py:93-99

            try:
                self.device_index = rtlsdr.RtlSdr.get_device_index_by_serial(device)
                logger.info(f"Using '{device}' as serial number (index: {self.device_index}).")
            except rtlsdr.rtlsdr.LibUSBError:
                logger.warning(f"Device '{device}' could was not found, aborting.")
                sys.exit(1)
        self.sample_rate = sample_rate
        self.center_freq = center_freq
        self._center_freqs = None           # per device, or None: one scalar for all
        if np.ndim(center_freq) != 0:
            self._center_freqs = np.asarray(center_freq)
            if self._center_freqs.shape != (self.n_streams,):
                raise ValueError("center_freq: one value, or one per device")
        try:
            self.gain = float(gain)
        except ValueError:
            self.gain = gain
        if sdr_callback_length is None:
            sdr_callback_length = sample_rate
        self.fft_nperseg = fft_nperseg
        self.fft_window = fft_window
        self.signal_min_duration = signal_min_duration_ms / 1000
        self.signal_max_duration = signal_max_duration_ms / 1000
        self.signal_threshold = from_dB(signal_threshold_dbw + calibration_db)
        self.snr_threshold = from_dB(snr_threshold_db)
        self.sdr_callback_length = sdr_callback_length
        self.verbose = verbose
        self.sdr_max_restart = sdr_max_restart
        self.sdr_timeout_s = sdr_timeout_s
        self.state_update_s = state_update_s
        self.signal_queue = signal_queue
        self.last_data_ts = last_data_ts
        self.cuda_device = cuda_device
        self._batch_args = dict(
            devices=[device], calibration_db=[calibration_db], sample_rate=sample_rate, center_freq=center_freq,
            fft_nperseg=fft_nperseg, fft_window=fft_window, signal_min_duration_ms=signal_min_duration_ms,
            signal_max_duration_ms=signal_max_duration_ms, signal_threshold_dbw=signal_threshold_dbw,
            snr_threshold_db=snr_threshold_db, sdr_callback_length=sdr_callback_length, cuda_device=cuda_device,
            fft_impl=kwargs.get("fft_impl", _engine.FFT_AUTO))
        self._batch: Optional[BatchAnalyzer] = None
        self._ts = None
        self._have_last = False         # `_spectrogram_last is not None` (the carry itself lives on the device)
        self._alarm_armed = False
        self.last_state = None
        self.sdr = None
        self._now = datetime.datetime.now
        self.Signal, self.StateMessage = message_types()

    @property
    def batch(self) -> BatchAnalyzer:
        if self._batch is None:
            self._batch = BatchAnalyzer(**self._batch_args)
        return self._batch

    @property
    def _spectrogram_last(self) -> Optional[np.ndarray]:
        """The reference's side state (analyze.py:128,268): the previous block's spectrogram as scipy returns it, float64
        `(fft_nperseg, T)`, or None before the first callback.  The carry the engine uses stays on the device (fp32); this
        copies it back on demand, for callers that inspect it."""
        if not self._have_last:
            return None
        return self.batch.engine.read_spectrogram(0).T.astype(np.float64)

    # -- process entry (analyze.py:131-157) ------------------------------------------------------
    def run(self):
        import rtlsdr

        _signal.signal(_signal.SIGTERM, self.handle_signal)
        _signal.signal(_signal.SIGINT, self.handle_signal)
        logging.basicConfig(level=max(0, logging.WARN - (self.verbose * 10)))
        sdr = rtlsdr.RtlSdr(self.device_index)
        sdr.sample_rate = self.sample_rate
        sdr.center_freq = self.center_freq
        sdr.gain = float(self.gain)
        sdr.set_agc_mode(False)
        self.sdr = sdr
        self.last_state = None
        self.batch.engine                                       # CUDA context is created in this process
        _signal.signal(_signal.SIGALRM, self.handle_signal)
        _signal.alarm(self.sdr_timeout_s)
        self._alarm_armed = True
        # raw bytes: no complex128 round trip (the reference registers process_samples via read_samples_async)
        self.sdr.read_bytes_async(self.process_bytes, 2 * self.sdr_callback_length)

    def handle_signal(self, sig, frame):
        """analyze.py:159-178."""
        if sig == _signal.SIGALRM:
            logger.warning("SDR %s received SIGALRM, last data received %s ago.", self.device,
                           self._now() - self._ts if self._ts else "(no signal yet)")
        elif sig == _signal.SIGTERM:
            logger.warning("SDR %s received SIGTERM, terminating.", self.device)
        elif sig == _signal.SIGINT:
            return
        self.update_state(self._now(), self.StateMessage.State.STOPPED)
        self.sdr.cancel_read_async()

    def update_state(self, ts: datetime.datetime, state):
        """analyze.py:180-190: at most one message per state every `state_update_s`."""
        if self.last_state and self.last_state.state == state:
            if self.last_state.ts + datetime.timedelta(seconds=self.state_update_s) >= ts.astimezone(UTC):
                return
        self.last_state = self.StateMessage(self.device, ts.astimezone(UTC), state)
        self.signal_queue.put(self.last_state)

    # -- the callback (analyze.py:192-268) ---------------------------------------------------------
    def process_samples(self, buffer: np.ndarray, context):
        """Reference-compatible entry: complex samples as pyrtlsdr's `read_samples_async` delivers them."""
        self.process_bytes(iq_to_bytes(buffer), context)

    def process_bytes(self, buffer, context):
        """Fast entry: the raw interleaved uint8 buffer of `read_bytes_async` (valid only during the call;
        it is copied to the device before returning)."""
        raw = np.frombuffer(buffer, dtype=np.uint8) if not isinstance(buffer, np.ndarray) else buffer
        n_samples = raw.shape[0] // 2
        ts_recv = self._now()
        buffer_len_dt = datetime.timedelta(seconds=n_samples / self.sample_rate)
        if self._alarm_armed:
            _signal.alarm(self.sdr_timeout_s)                   # analyze.py:208
        if not self.last_data_ts.value:
            self.update_state(self._now(), self.StateMessage.State.STARTED)
        else:
            self.update_state(ts_recv, self.StateMessage.State.RUNNING)
        self.last_data_ts.value = datetime.datetime.timestamp(ts_recv)
        logger.info(f"SDR {self.device} received data at {self.last_data_ts.value}")

        if not self._ts:                                        # analyze.py:217-221
            self._ts = ts_recv
        else:
            self._ts += buffer_len_dt
        clock_drift = (ts_recv - self._ts).total_seconds()
        if clock_drift > 2 * buffer_len_dt.total_seconds():     # analyze.py:223-229
            logger.warning(f"SDR {self.device} total clock drift ({clock_drift:.5f} s) is larger than two blocks, signal detection is degraded. Terminating...")
            self.update_state(self._now(), self.StateMessage.State.STOPPED)
            self.sdr.cancel_read_async()
        ts_start = self._ts - buffer_len_dt

        if n_samples == 0:                                      # scipy returns empty arrays, extract_signals returns [] (analyze.py:351)
            return
        if n_samples != self.sdr_callback_length:
            # the reference indexes times[-start] of the CURRENT block into the previous one (analyze.py:423);
            # a changing block length is undefined there, and the engine is sized for one length
            raise ValueError(f"callback delivered {n_samples} samples, analyzer is configured for {self.sdr_callback_length}")

        batch = self.batch
        tm0 = dict(batch.timings)
        bench_start = time.time()
        filtered, signals, _ = batch.process_blocks(raw.reshape(1, -1), [ts_start])[0]
        bench_filter = time.time()
        [self.consume_signal(s) for s in filtered]
        bench_consume = time.time()
        self._have_last = True
        tm = batch.timings
        t_device = tm["fetch_wait_s"] - tm0["fetch_wait_s"]             # H2D copy + kernels + D2H of the records
        t_final = (tm["finalize_s"] - tm0["finalize_s"]) + (tm["build_s"] - tm0["build_s"])
        # Same line and fields as analyze.py:254-260 -- including its unit quirk (seconds x 100 printed as "ms") so that anything
        # parsing the reference's log keeps working -- followed by the CUDA path's own split in real milliseconds.
        logger.info(
            f"SDR {self.device} recv {n_samples}, "
            + f"clock drift: {clock_drift:.2f} s, "
            + f"filtered {len(filtered)} / {len(signals)} signals, "
            + f"block len: {(buffer_len_dt.total_seconds())*100:.1f} ms, "
            + f"compute: {(bench_consume-bench_start)*100:.1f} ms, "
            + f"cuda: device {t_device * 1e3:.2f} ms, finalise {t_final * 1e3:.2f} ms"
        )
        # analyze.py:262-267: the spectrogram and the scans are one device step here; "filter" is part of the finaliser
        logger.debug(
            f"timings - spectogram: {t_device*100:.1f} ms, "
            + f"extract: {t_final*100:.1f} ms, "
            + f"filter: {max(0.0, bench_filter - bench_start - t_device - t_final)*100:.1f} ms, "
            + f"consume: {(bench_consume-bench_filter)*100:.1f} ms"
        )

    def consume_signal(self, signal):
        """analyze.py:270-280."""
        logger.debug(f"SDR {self.device} received {signal}")
        self.signal_queue.put(signal)

    # reference static helpers, kept for callers that use them directly (analyze.py:282-328)
    @staticmethod
    def is_shadow_of(sig, signals) -> Optional[int]:
        for i, fsig in enumerate(signals):
            if sig.ts > fsig.ts + fsig.duration or sig.ts + sig.duration < fsig.ts:
                continue
            if fsig.max > sig.max:
                return i
        return None

    def filter_shadow_signals(self, signals):
        return BatchAnalyzer.filter_shadow_signals(signals)
