"""Supervision of a multi-stream engine (SURVEY.md section 8f rank 4).

In the reference every SDR is one `SignalAnalyzer` process with its own life-cycle bookkeeping
(radiotracking/analyze.py:180-231: STARTED / RUNNING / STOPPED `StateMessage`s rate-limited by `state_update_s`, the
`last_data_ts` heartbeat, the drift-free virtual clock `_ts` and the stop on a clock drift of more than two blocks), and
`Runner.check_analyzers` (radiotracking/__main__.py:153-190) restarts analyzers whose heartbeat is older than
`sdr_timeout_s` while their restart budget `sdr_max_restart` lasts.  `MultiStreamAnalyzer` keeps exactly that state per
stream for N analyzers that share one `BatchAnalyzer` / GPU, so a batched engine can sit under the reference's runner
and consumers: the queue sees the same messages per device as N reference processes would have produced.
"""
import datetime
import logging
from typing import List, Optional, Sequence

import numpy as np

from .analyze import UTC, BatchAnalyzer
from .messages import message_types

logger = logging.getLogger(__name__)


class _Value:
    """Stand-in for multiprocessing.Value('d') when the caller does not share the heartbeat with another process."""

    def __init__(self, value: float = 0.0):
        self.value = value


class MultiStreamAnalyzer:
    """N reference analyzers' side state over one batched engine.

    Keys are `SignalAnalyzer`'s (analyze.py:62-83) with `device` / `calibration_db` as lists; `last_data_ts` is a list
    of `multiprocessing.Value('d')`-like objects (one per stream) or None."""

    def __init__(self, device: Sequence[str], calibration_db: Sequence[float], sample_rate: int, center_freq: int,
                 fft_nperseg: int, fft_window, signal_min_duration_ms: float, signal_max_duration_ms: float,
                 signal_threshold_dbw: float, snr_threshold_db: float, sdr_max_restart: int, sdr_timeout_s: int,
                 state_update_s: int, sdr_callback_length: Optional[int], signal_queue, last_data_ts=None,
                 cuda_device: int = 0, **kwargs):
        self.devices = [str(d) for d in device]
        self.n_streams = len(self.devices)
        self.sample_rate = sample_rate
        self.sdr_callback_length = sample_rate if sdr_callback_length is None else sdr_callback_length   # analyze.py:108-109
        self.sdr_timeout_s = sdr_timeout_s
        self.state_update_s = state_update_s
        self.signal_queue = signal_queue
        self.last_data_ts = list(last_data_ts) if last_data_ts is not None else [_Value() for _ in self.devices]
        self.restarts_left = [sdr_max_restart] * self.n_streams       # __main__.py:176-183
        self.batch = BatchAnalyzer(
            devices=self.devices, calibration_db=list(calibration_db), sample_rate=sample_rate, center_freq=center_freq,
            fft_nperseg=fft_nperseg, fft_window=fft_window, signal_min_duration_ms=signal_min_duration_ms,
            signal_max_duration_ms=signal_max_duration_ms, signal_threshold_dbw=signal_threshold_dbw,
            snr_threshold_db=snr_threshold_db, sdr_callback_length=self.sdr_callback_length, cuda_device=cuda_device,
            **{k: v for k, v in kwargs.items() if k in ("fft_impl", "max_records", "survey", "fine_frequency")})
        self.Signal, self.StateMessage = message_types()
        self._ts: List[Optional[datetime.datetime]] = [None] * self.n_streams
        self.last_state: List[object] = [None] * self.n_streams
        self.stopped = [False] * self.n_streams        # cancel_read_async was called for this stream (analyze.py:178,229)
        self._now = datetime.datetime.now

    # -- per-stream pieces of the reference callback ------------------------------------------------
    def update_state(self, s: int, ts: datetime.datetime, state) -> None:
        """analyze.py:180-190: at most one message per state every `state_update_s`."""
        last = self.last_state[s]
        if last and last.state == state:
            if last.ts + datetime.timedelta(seconds=self.state_update_s) >= ts.astimezone(UTC):
                return
        self.last_state[s] = self.StateMessage(self.devices[s], ts.astimezone(UTC), state)
        self.signal_queue.put(self.last_state[s])

    def _clock(self, s: int, ts_recv: datetime.datetime, buffer_len_dt: datetime.timedelta) -> datetime.datetime:
        """analyze.py:204-231 for one stream -> ts_start of its block."""
        if not self.last_data_ts[s].value:
            self.update_state(s, self._now() if ts_recv is None else ts_recv, self.StateMessage.State.STARTED)
        else:
            self.update_state(s, ts_recv, self.StateMessage.State.RUNNING)
        self.last_data_ts[s].value = datetime.datetime.timestamp(ts_recv)
        if not self._ts[s]:
            self._ts[s] = ts_recv
        else:
            self._ts[s] += buffer_len_dt
        clock_drift = (ts_recv - self._ts[s]).total_seconds()
        if clock_drift > 2 * buffer_len_dt.total_seconds():
            logger.warning(f"SDR {self.devices[s]} total clock drift ({clock_drift:.5f} s) is larger than two blocks, signal detection is degraded. Terminating...")
            self.update_state(s, ts_recv, self.StateMessage.State.STOPPED)
            self.stopped[s] = True                      # the reference cancels the read loop; this block is still analysed
        return self._ts[s] - buffer_len_dt

    # -- the batched callback ---------------------------------------------------------------------------
    def process_bytes(self, buffers: np.ndarray, ts_recv: Optional[Sequence[datetime.datetime]] = None) -> List[list]:
        """One callback block of every stream (`[n_streams, 2*sdr_callback_length]` uint8).  `ts_recv[s]` is the wall
        clock at which stream s delivered its block (default: now).  Streams that were stopped are skipped until
        `restart`.  Returns the shadow-filtered Signals per stream; they are also put on the queue, stream by stream,
        each in the reference's order (analyze.py:248-251)."""
        buffers = np.asarray(buffers)
        if buffers.shape != (self.n_streams, 2 * self.sdr_callback_length):
            raise ValueError(f"expected {(self.n_streams, 2 * self.sdr_callback_length)} bytes, got {buffers.shape}")
        now = self._now()
        recv = [now] * self.n_streams if ts_recv is None else list(ts_recv)
        dt = datetime.timedelta(seconds=self.sdr_callback_length / self.sample_rate)
        active = [not st for st in self.stopped]          # streams whose read loop is alive when the block arrives
        ts_start = [recv[s] for s in range(self.n_streams)]
        for s in range(self.n_streams):
            if active[s]:
                ts_start[s] = self._clock(s, recv[s], dt)
        res = self.batch.process_blocks(buffers, ts_start)
        out: List[list] = []
        for s in range(self.n_streams):
            if not active[s]:
                self.batch.reset_stream(s)              # no analyzer is listening: nothing carries over
                out.append([])
                continue
            filtered = res[s][0]
            for sig in filtered:
                self.signal_queue.put(sig)              # consume_signal (analyze.py:270-280)
            out.append(filtered)
        return out

    # -- the runner's check (radiotracking/__main__.py:153-190) -----------------------------------------
    def restart(self, s: int) -> None:
        """What `create_and_start` amounts to for one stream: a fresh analyzer (no carry, no clock, no state)."""
        self.batch.reset_stream(s)
        self._ts[s] = None
        self.last_state[s] = None
        self.last_data_ts[s].value = 0.0
        self.stopped[s] = False
        self.restarts_left[s] -= 1

    def check_streams(self, now: Optional[datetime.datetime] = None) -> bool:
        """Time-out supervision of every stream.  A stream whose heartbeat is older than `sdr_timeout_s`, or that
        stopped itself, gets a STOPPED message stamped with its last heartbeat (__main__.py:171) and is restarted
        while its budget lasts.  Returns False when a stream is dead beyond its restart count (the reference then
        terminates the application, __main__.py:178-181)."""
        now = self._now() if now is None else now
        for s in range(self.n_streams):
            hb = self.last_data_ts[s].value
            if not self.stopped[s]:
                if hb == 0.0:
                    continue                                            # not started yet (__main__.py:161-162)
                if hb > datetime.datetime.timestamp(now) - self.sdr_timeout_s:
                    continue
                logger.warning(f"SDR {self.devices[s]} received last data {datetime.datetime.fromtimestamp(hb)}; timed out.")
                self.signal_queue.put(self.StateMessage(self.devices[s], datetime.datetime.fromtimestamp(hb, tz=UTC), self.StateMessage.State.STOPPED))
                self.stopped[s] = True
            if self.restarts_left[s] <= 0:
                logger.critical(f"SDR {self.devices[s]} is dead and beyond restart count, terminating.")
                return False
            logger.warning(f"Restarting SDR {self.devices[s]}.")
            self.restart(s)
        return True

    def close(self):
        self.batch.close()
