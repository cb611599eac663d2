"""Wideband recordings as narrowband SDR channels: a CUDA down-converter (include/rt_ddc.h) in front of the engine.

A 2.5-20 MS/s receiver (Airspy, SDRplay, USRP, HackRF) covers a whole tag band, but the reference's detection keys are tuned for
an RTL-SDR at 250 kS/s-2.4 MS/s: `signal_threshold_dbw` is compared with density-scaled cells (a tone's cell scales with
1 / bin width) and the duration limits are counted in columns of nperseg / fs.  So the wideband stream is cut into virtual SDR
channels -- complex baseband streams at fs / D centred on `center_freq + offset` -- and every channel is analysed by an unchanged
analyzer unit, exactly as the reference analyses one RTL-SDR (one analyzer per SDR with its own centre frequency, device name
and calibration; the shadow filter per analyzer).

    Channelizer        the ctypes binding of rt_ddc: wideband blocks -> float32 [inputs * channels, 2 * samples / D] on the GPU,
                       for arbitrary channel offsets
    FilterBank         the ctypes binding of rt_fbank (include/rt_fbank.h): the same quantity for every in-band channel of the
                       uniform grid k fs / (2 D), -(D - 1) <= k <= D - 1, from a polyphase FFT filter bank (about L / log2(2 D)
                       times less work than the DDC on that grid)
    WidebandAnalyzer   a Channelizer (or, from `WidebandAnalyzer.full_band`, a FilterBank) plus one cf32 BatchAnalyzer with an
                       analyzer unit per (input, channel); `replay()` drives it like a BatchAnalyzer with one stream per input

`iq_correction=True` (both front ends, default off) removes each wideband block's DC and makes the block proper before the
channel filter (include/rt_ddc.h): the mirror images a zero-IF receiver (HackRF, bladeRF 1) puts at -f of every signal at +f
then no longer reach the channel analyzers as tags that do not exist.

Default channel filter (`default_taps`): `scipy.signal.firwin(8 D + 1, 1 / D, window=("kaiser", 8.0))`, cutoff at the channel
Nyquist frequency fs / (2 D), unit gain at DC.  Its response (scipy.signal.freqz, D = 4, 8, 64 alike): flat within 0.07 dB over
the central half of the channel (|f| <= fs / (4 D)), -6.0 dB at the channel edge, at most -42 dB from 1.5 times the edge on
and at most -83 dB from twice the edge on.  After decimation, everything that folds onto the central half of a channel comes
from 1.5 times the edge or beyond, so the central half is alias-free to 42 dB; tags belong there, and channels that should
cover a band without gaps are spaced fs / (2 D) apart.
"""
import ctypes
import datetime
from typing import Optional, Sequence, Union

import numpy as np

from . import engine as _engine
from .analyze import BatchAnalyzer
from .finefreq import central_half
from .survey import stitch

RT_DDC_ABI_VERSION = 1
MAX_TAPS = 2049           # RT_DDC_MAX_TAPS
MAX_DECIMATION = 1024     # RT_DDC_MAX_DECIMATION
KAISER_BETA = 8.0

# every symbol include/rt_ddc.h declares
EXPORTS = ("rt_ddc_create", "rt_ddc_destroy", "rt_ddc_reset_input", "rt_ddc_run", "rt_ddc_set_iq_correction",
           "rt_ddc_read_iq_correction")

RT_FBANK_ABI_VERSION = 1
FBANK_MIN_DECIMATION = 4     # RT_FBANK_MIN_DECIMATION
FBANK_MAX_DECIMATION = 512   # RT_FBANK_MAX_DECIMATION
MAX_ENGINE_UNITS = 65535     # rt_engine: n_streams * blocks_per_launch

# every symbol include/rt_fbank.h declares
FBANK_EXPORTS = ("rt_fbank_create", "rt_fbank_destroy", "rt_fbank_reset_input", "rt_fbank_run", "rt_fbank_set_iq_correction",
                 "rt_fbank_read_iq_correction")


# the functions of either front end, after its prefix (rt_ddc_, rt_fbank_)
_FRONT_END_FUNCTIONS = ("create", "destroy", "reset_input", "run", "set_iq_correction", "read_iq_correction")


class RtDdcConfig(ctypes.Structure):
    _fields_ = [
        ("abi_version", ctypes.c_int32), ("cuda_device", ctypes.c_int32), ("n_inputs", ctypes.c_int32),
        ("n_channels", ctypes.c_int32), ("block_samples", ctypes.c_int64), ("decimation", ctypes.c_int32),
        ("n_taps", ctypes.c_int32), ("sample_format", ctypes.c_int32), ("reserved", ctypes.c_int32),
        ("sample_rate", ctypes.c_double), ("taps", ctypes.POINTER(ctypes.c_double)),
        ("phase_inc", ctypes.POINTER(ctypes.c_uint32)),
    ]


class RtFbankConfig(ctypes.Structure):
    _fields_ = [
        ("abi_version", ctypes.c_int32), ("cuda_device", ctypes.c_int32), ("n_inputs", ctypes.c_int32),
        ("decimation", ctypes.c_int32), ("block_samples", ctypes.c_int64), ("n_taps", ctypes.c_int32),
        ("sample_format", ctypes.c_int32), ("reserved", ctypes.c_int32), ("sample_rate", ctypes.c_double),
        ("taps", ctypes.POINTER(ctypes.c_double)),
    ]


def _load():
    lib = _engine.load_library()
    if not getattr(lib, "_ddc_types", False):
        for prefix, config in (("rt_ddc", RtDdcConfig), ("rt_fbank", RtFbankConfig)):
            create, destroy, reset, run, set_iq, read_iq = (getattr(lib, f"{prefix}_{name}") for name in _FRONT_END_FUNCTIONS)
            create.argtypes = [ctypes.POINTER(config), ctypes.POINTER(ctypes.c_void_p)]
            destroy.argtypes = [ctypes.c_void_p]
            destroy.restype = None
            reset.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64]
            run.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_size_t, ctypes.c_int32,
                            ctypes.c_void_p, ctypes.c_size_t]
            set_iq.argtypes = [ctypes.c_void_p, ctypes.c_int32]
            read_iq.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.POINTER(ctypes.c_float)]
        lib._ddc_types = True
    return lib


def phase_increment(offset_hz: Union[float, Sequence[float]], sample_rate: float) -> np.ndarray:
    """uint32 phase increment of each channel: round(offset / fs * 2^32) mod 2^32 (cycles per input sample times 2^32)."""
    off = np.atleast_1d(np.asarray(offset_hz, dtype=np.float64))
    return (np.rint(off / float(sample_rate) * 2.0 ** 32).astype(np.int64) % (1 << 32)).astype(np.uint32)


def default_taps(decimation: int) -> np.ndarray:
    """The default channel filter (module docstring): 8 D + 1 Kaiser-window taps, cutoff at the channel Nyquist, unit DC gain."""
    from scipy.signal import firwin

    return firwin(8 * decimation + 1, 1.0 / decimation, window=("kaiser", KAISER_BETA))


def channel_ts(ts_start: datetime.datetime, n_taps: int, sample_rate: float) -> datetime.datetime:
    """Start of a channel block: the wideband block's start minus the filter's centre delay (L - 1) / (2 fs)."""
    return ts_start - datetime.timedelta(seconds=(n_taps - 1) / (2 * sample_rate))


def channel_center_freqs(center_freq, offsets_hz: Sequence[float]) -> list:
    """Centre frequency of every channel: center_freq + offset (float64 when either is a float)."""
    return [center_freq + off for off in offsets_hz]


def grid_offsets(sample_rate: float, decimation: int) -> list:
    """Offsets of the filter bank's channels, in row order: k fs / (2 D) for k = -(D - 1) ... D - 1."""
    D = int(decimation)
    return [k * sample_rate / (2 * D) for k in range(-(D - 1), D)]


def grid_phase_increment(decimation: int) -> np.ndarray:
    """The rt_ddc phase increment of every filter-bank row: ((k mod 2 D) 2^32) / (2 D), exact."""
    D = int(decimation)
    return np.array([((k % (2 * D)) << 32) // (2 * D) for k in range(-(D - 1), D)], dtype=np.uint32)


def _check_taps(h: np.ndarray, max_taps: int) -> None:
    if h.ndim != 1 or len(h) % 2 == 0 or len(h) > max_taps:
        raise ValueError(f"taps: an odd number of real taps up to {max_taps} is needed, got {h.shape}")
    if not np.all(np.isfinite(h)):
        raise ValueError("taps must be finite")


class _WidebandFrontEnd:
    """What Channelizer and FilterBank share: the constructor's common steps, the handle's life cycle and the input / output
    handling of `run`.  A subclass checks its plan, sets `offsets_hz`, `phase_inc` and `n_channels`, calls `__init__` with its
    C prefix and tap limit, and builds its config struct in `_config`."""

    _h = None
    iq_correction = False

    def __init__(self, prefix: str, sample_rate: int, block_samples: int, decimation: int, taps, max_taps: int,
                 sample_format: str, n_inputs: int, cuda_device: int, blocks_per_launch: int, iq_correction: bool):
        h = default_taps(decimation) if taps is None else np.asarray(taps, dtype=np.float64)
        _check_taps(h, max_taps)
        if blocks_per_launch < 1:
            raise ValueError("blocks_per_launch must be >= 1")
        self._set_format(sample_format)
        self.sample_rate, self.block_samples, self.decimation = sample_rate, int(block_samples), decimation
        self.taps = np.ascontiguousarray(h)
        self.n_inputs = int(n_inputs)
        self.blocks_per_launch = int(blocks_per_launch)
        self.cuda_device = cuda_device
        self._lib = _load()
        create, self._destroy, self._reset, self._run, self._set_iq, self._read_iq = (
            getattr(self._lib, f"{prefix}_{name}") for name in _FRONT_END_FUNCTIONS)
        self._h = ctypes.c_void_p()
        _engine._check(create(ctypes.byref(self._config()), ctypes.byref(self._h)))
        if iq_correction:
            self.set_iq_correction(True)

    def _set_format(self, sample_format: str) -> None:
        self.sample_format = _engine.sample_format_name(sample_format)
        code, dtype, self.sample_bytes = _engine.SAMPLE_FORMATS[self.sample_format]
        self._format_code = code
        self._dtypes = (dtype, np.dtype(np.complex64)) if self.sample_format == "cf32_le" else (dtype,)
        self._dtype_names = tuple(d.name for d in self._dtypes)

    @property
    def n_taps(self) -> int:
        return len(self.taps)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._destroy(self._h)            # waits for the last run
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_iq_correction(self, enable: bool) -> None:
        """Turn the per-block DC and IQ-imbalance correction (include/rt_ddc.h) on or off from the next `run` on."""
        _engine._check(self._set_iq(self._h, 1 if enable else 0))
        self.iq_correction = bool(enable)

    def read_iq_correction(self, i: int, block: int):
        """Test hook: `(m, w)` (complex, from the fp32 values the kernels applied) of input `i` and block `block` of the last
        `run`, which must have corrected; waits for that run."""
        out = (ctypes.c_float * 4)()
        _engine._check(self._read_iq(self._h, int(i), int(block), out))
        return complex(out[0], out[1]), complex(out[2], out[3])

    def reset_input(self, i: int, first_sample: int = 0) -> None:
        """Restart input `i` at the global sample index `first_sample`, with a zero filter history (from the next `run`)."""
        _engine._check(self._reset(self._h, int(i), int(first_sample)))

    def run(self, iq, out=None):
        """Channelize `blocks_per_launch` consecutive blocks of every input: `iq` is `[n_inputs, 2 * blocks_per_launch *
        block_samples]` elements of the sample format (cf32_le also complex64 with half as many) on the host (pinned or not) or a
        CUDA tensor / __cuda_array_interface__ object.  -> float32 CUDA tensor `[n_inputs * n_channels, 2 * blocks_per_launch *
        block_samples / D]` (interleaved I, Q; row i * n_channels + c), written by work enqueued on the current torch stream.  A
        device input is read after the work queued on its producer stream (engine._producer_stream); a pinned host input is
        copied asynchronously and must stay unchanged until that stream has reached this call."""
        import torch

        row = self.sample_bytes * self.block_samples * self.blocks_per_launch
        dev = _engine._device_pointer(iq, self.n_inputs, row, self._dtype_names)
        cur = torch.cuda.current_stream(self.cuda_device)
        if dev is not None:
            ptr, stride = dev
            producer = _engine._producer_stream(iq)
            if producer is not None and producer != cur.cuda_stream:
                ev = torch.cuda.Event()
                ev.record(torch.cuda.ExternalStream(producer, device=self.cuda_device))
                cur.wait_event(ev)
            on_dev = 1
        else:
            arr = np.asarray(iq)
            if arr.dtype not in self._dtypes:
                raise TypeError(f"IQ blocks must be {' / '.join(self._dtype_names)} for sample format {self.sample_format}, got {arr.dtype}")
            if arr.ndim == 1:
                arr = arr.reshape(1, -1)
            if arr.ndim != 2 or arr.shape != (self.n_inputs, row // arr.itemsize) or arr.strides[1] != arr.itemsize:
                raise ValueError(f"expected {arr.dtype.name} [{self.n_inputs}, {row // arr.itemsize}], got {arr.shape}")
            ptr, stride, on_dev = int(arr.ctypes.data), int(arr.strides[0]), 0
        m = self.blocks_per_launch * self.block_samples // self.decimation
        if out is None:
            out = torch.empty((self.n_inputs * self.n_channels, 2 * m), dtype=torch.float32, device=f"cuda:{self.cuda_device}")
        elif out.dtype != torch.float32 or tuple(out.shape) != (self.n_inputs * self.n_channels, 2 * m) or out.stride(1) != 1:
            raise ValueError("out must be float32 [n_inputs * n_channels, 2 * samples / D] with contiguous rows")
        _engine._check(self._run(self._h, ctypes.c_void_p(cur.cuda_stream), ctypes.c_void_p(ptr), on_dev, stride,
                                 self.blocks_per_launch, ctypes.c_void_p(out.data_ptr()), out.stride(0) * 4))
        return out


class Channelizer(_WidebandFrontEnd):
    """The down-converter of include/rt_ddc.h for `n_inputs` wideband streams and one channel plan (`offsets_hz`)."""

    def __init__(self, sample_rate: int, block_samples: int, offsets_hz: Sequence[float], decimation: int,
                 taps: Optional[Sequence[float]] = None, sample_format: str = "cu8", n_inputs: int = 1, cuda_device: int = 0,
                 blocks_per_launch: int = 1, iq_correction: bool = False):
        """`taps`: real FIR taps (odd count, at most MAX_TAPS); None: `default_taps(decimation)`.  `iq_correction`: correct
        every block's DC and IQ imbalance before the filter (`set_iq_correction`).  ValueError for a channel plan the
        down-converter cannot produce; the CUDA side checks the rest (engine.EngineError)."""
        fs, D = sample_rate, int(decimation)
        if not 2 <= D <= MAX_DECIMATION:
            raise ValueError(f"decimation = {decimation}: must be in [2, {MAX_DECIMATION}]")
        if fs % D or block_samples % D:
            raise ValueError(f"sample_rate ({fs}) and block_samples ({block_samples}) must be multiples of the decimation {D}")
        off = [float(o) for o in np.atleast_1d(offsets_hz)]
        if not off:
            raise ValueError("no channels")
        for o in off:
            if abs(o) + fs / (2 * D) > fs / 2:
                raise ValueError(f"channel at {o} Hz with half-width {fs / (2 * D)} Hz does not lie inside the input band +-{fs / 2} Hz")
        self.offsets_hz, self.phase_inc, self.n_channels = off, phase_increment(off, fs), len(off)
        super().__init__("rt_ddc", fs, block_samples, D, taps, MAX_TAPS, sample_format, n_inputs, cuda_device, blocks_per_launch,
                         iq_correction)

    def _config(self) -> RtDdcConfig:
        return RtDdcConfig(
            abi_version=RT_DDC_ABI_VERSION, cuda_device=self.cuda_device, n_inputs=self.n_inputs, n_channels=self.n_channels,
            block_samples=self.block_samples, decimation=self.decimation, n_taps=self.n_taps, sample_format=self._format_code,
            reserved=0, sample_rate=float(self.sample_rate), taps=self.taps.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
            phase_inc=self.phase_inc.ctypes.data_as(ctypes.POINTER(ctypes.c_uint32)))


class FilterBank(_WidebandFrontEnd):
    """The polyphase FFT filter bank of include/rt_fbank.h for `n_inputs` wideband streams: every in-band channel of the grid
    k fs / (2 D), -(D - 1) <= k <= D - 1 (`n_channels` = 2 D - 1, row k + D - 1, ascending frequency).  Its output is the
    quantity `Channelizer` computes for `offsets_hz` = `grid_offsets(fs, D)`, at about L / log2(2 D) times less work."""

    def __init__(self, sample_rate: int, block_samples: int, decimation: int, taps: Optional[Sequence[float]] = None,
                 sample_format: str = "cu8", n_inputs: int = 1, cuda_device: int = 0, blocks_per_launch: int = 1,
                 iq_correction: bool = False):
        """`decimation` D: a power of two in [FBANK_MIN_DECIMATION, FBANK_MAX_DECIMATION]; `taps`: real FIR taps (odd count,
        at most 16 D + 1); None: `default_taps(decimation)`; `iq_correction` as for `Channelizer`.  ValueError for a plan the
        filter bank cannot produce; the CUDA side checks the rest (engine.EngineError)."""
        fs, D = sample_rate, int(decimation)
        if not FBANK_MIN_DECIMATION <= D <= FBANK_MAX_DECIMATION or D & (D - 1):
            raise ValueError(f"decimation = {decimation}: must be a power of two in [{FBANK_MIN_DECIMATION}, {FBANK_MAX_DECIMATION}]")
        if fs % D or block_samples % D or block_samples < D:
            raise ValueError(f"sample_rate ({fs}) and block_samples ({block_samples}) must be multiples of the decimation {D}")
        if not 1 <= int(n_inputs) <= 65535 or int(n_inputs) * (2 * D - 1) > 1 << 30:
            raise ValueError(f"n_inputs = {n_inputs}: must be in [1, 65535] with n_inputs * (2 D - 1) <= 2^30")
        self.offsets_hz, self.phase_inc, self.n_channels = grid_offsets(fs, D), grid_phase_increment(D), 2 * D - 1
        super().__init__("rt_fbank", fs, block_samples, D, taps, 16 * D + 1, sample_format, n_inputs, cuda_device, blocks_per_launch,
                         iq_correction)

    def _config(self) -> RtFbankConfig:
        return RtFbankConfig(
            abi_version=RT_FBANK_ABI_VERSION, cuda_device=self.cuda_device, n_inputs=self.n_inputs, decimation=self.decimation,
            block_samples=self.block_samples, n_taps=self.n_taps, sample_format=self._format_code, reserved=0,
            sample_rate=float(self.sample_rate), taps=self.taps.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))


class WidebandAnalyzer:
    """Wideband recordings (`n_streams` inputs) analysed as narrowband SDR channels: a `Channelizer` (the constructor, for
    arbitrary `offsets_hz`) or a `FilterBank` (`full_band`, the whole uniform grid) plus one cf32_le `BatchAnalyzer` with one
    analyzer unit per (input, channel).

    The channel analyzer runs at `sample_rate / decimation` with blocks of `block_samples / decimation`.  Channel c of input i
    is the device `f"{devices[i]}:{c}"` with the calibration of input i and the centre frequency `center_freq + offsets_hz[c]`;
    its blocks start the filter's centre delay earlier than the wideband blocks (`channel_ts`).  `n_streams`, `block_samples`,
    `sample_rate`, `sample_format` and `blocks_per_launch` describe the wideband input, so `replay()` drives this class like a
    `BatchAnalyzer` with one stream per recording.  A tag in the overlap of two channels gives a Signal in each, as two
    overlapping SDRs would; grouping them is the matcher's job."""

    def __init__(self, devices: Sequence[str], calibration_db: Sequence[float], sample_rate: int, center_freq,
                 offsets_hz: Sequence[float], decimation: int, fft_nperseg: int, fft_window, signal_min_duration_ms: float,
                 signal_max_duration_ms: float, signal_threshold_dbw: float, snr_threshold_db: float,
                 sdr_callback_length: Optional[int] = None, taps: Optional[Sequence[float]] = None, sample_format: str = "cu8",
                 cuda_device: int = 0, blocks_per_launch: int = 1, iq_correction: bool = False, **batch_options):
        """`iq_correction`: correct every wideband block's DC and IQ imbalance before the channel filter (`Channelizer`).
        `batch_options`: further `BatchAnalyzer` keys of the channel analyzer (max_records, fft_impl, survey, fine_frequency,
        ...); with `survey=True` every channel is surveyed (`last_survey`), with `fine_frequency=True` every Signal gets a
        carrier estimate (`last_fine_frequencies`)."""
        block = self._check_plan(devices, calibration_db, sample_rate, decimation, fft_nperseg, sdr_callback_length)
        front = Channelizer(sample_rate, block, offsets_hz, int(decimation), taps=taps, sample_format=sample_format,
                            n_inputs=len(self.devices), cuda_device=cuda_device, blocks_per_launch=blocks_per_launch,
                            iq_correction=iq_correction)
        self._attach(front, center_freq, fft_nperseg, fft_window, signal_min_duration_ms, signal_max_duration_ms,
                     signal_threshold_dbw, snr_threshold_db, cuda_device, batch_options)

    @classmethod
    def full_band(cls, devices: Sequence[str], calibration_db: Sequence[float], sample_rate: int, center_freq, decimation: int,
                  fft_nperseg: int, fft_window, signal_min_duration_ms: float, signal_max_duration_ms: float,
                  signal_threshold_dbw: float, snr_threshold_db: float, sdr_callback_length: Optional[int] = None,
                  taps: Optional[Sequence[float]] = None, sample_format: str = "cu8", cuda_device: int = 0,
                  blocks_per_launch: int = 1, iq_correction: bool = False, **batch_options) -> "WidebandAnalyzer":
        """The whole band of every input: a `FilterBank` in front, so channel c (0 ... 2 D - 2) of input i is the device
        `f"{devices[i]}:{c}"` at `center_freq + (c - D + 1) fs / (2 D)`.  Adjacent channels overlap by half their width, so
        every frequency within fs / 2 - fs / (4 D) of the centre lies in the flat central half of some channel.  ValueError
        when the 2 D - 1 channels of every input and block exceed the engine's 65535 analyzer units per launch.
        `iq_correction` and `batch_options` as in the constructor; with `survey=True`, `band_survey` stitches the channels."""
        self = cls.__new__(cls)
        block = self._check_plan(devices, calibration_db, sample_rate, decimation, fft_nperseg, sdr_callback_length)
        D = int(decimation)
        units = len(self.devices) * (2 * D - 1) * int(blocks_per_launch)
        if units > MAX_ENGINE_UNITS:
            raise ValueError(f"{len(self.devices)} inputs * {2 * D - 1} channels * {blocks_per_launch} blocks per launch = {units} "
                             f"analyzer units: more than the engine's {MAX_ENGINE_UNITS}")
        front = FilterBank(sample_rate, block, D, taps=taps, sample_format=sample_format, n_inputs=len(self.devices),
                           cuda_device=cuda_device, blocks_per_launch=blocks_per_launch, iq_correction=iq_correction)
        self._attach(front, center_freq, fft_nperseg, fft_window, signal_min_duration_ms, signal_max_duration_ms,
                     signal_threshold_dbw, snr_threshold_db, cuda_device, batch_options)
        return self

    def _check_plan(self, devices, calibration_db, sample_rate, decimation, fft_nperseg, sdr_callback_length) -> int:
        """Set the devices and calibrations; -> the wideband block length."""
        self.devices = [str(d) for d in devices]
        self.calibration_db = [float(c) for c in calibration_db]
        if len(self.calibration_db) != len(self.devices):
            raise ValueError("one calibration value per device")
        block = sample_rate if sdr_callback_length is None else sdr_callback_length
        D = int(decimation)
        if D >= 1 and block % D == 0 and (block // D) // fft_nperseg < 2:
            raise ValueError(f"a channel block of {block // D} samples holds fewer than two FFT segments of {fft_nperseg}")
        return block

    def _attach(self, front, center_freq, fft_nperseg, fft_window, signal_min_duration_ms, signal_max_duration_ms,
                signal_threshold_dbw, snr_threshold_db, cuda_device, batch_options) -> None:
        """The channel analyzer behind the Channelizer or FilterBank `front` (kept as `self.ddc`)."""
        self.ddc = front
        sample_rate, block, D = front.sample_rate, front.block_samples, front.decimation
        self.n_streams = len(self.devices)
        self.n_channels = self.ddc.n_channels
        self.sample_rate, self.block_samples = sample_rate, block
        self.sample_format = self.ddc.sample_format
        self.blocks_per_launch = self.ddc.blocks_per_launch
        C = self.n_channels
        self.channels = BatchAnalyzer(
            devices=[f"{d}:{c}" for d in self.devices for c in range(C)],
            calibration_db=[cal for cal in self.calibration_db for _ in range(C)],
            sample_rate=sample_rate // D, center_freq=channel_center_freqs(center_freq, self.ddc.offsets_hz) * self.n_streams,
            fft_nperseg=fft_nperseg, fft_window=fft_window, signal_min_duration_ms=signal_min_duration_ms,
            signal_max_duration_ms=signal_max_duration_ms, signal_threshold_dbw=signal_threshold_dbw,
            snr_threshold_db=snr_threshold_db, sdr_callback_length=block // D, cuda_device=cuda_device,
            blocks_per_launch=self.blocks_per_launch, sample_format="cf32_le", **batch_options)
        self._held = []          # wideband inputs of the submissions not collected yet (a pinned buffer is copied asynchronously)

    def close(self):
        self.channels.close()
        self.ddc.close()
        self._held = []

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def reset_stream(self, stream: int, first_sample: int = 0):
        """Restart input `stream` (a new recording): zero filter history, and every channel analyzer without a previous block."""
        self.ddc.reset_input(stream, first_sample)
        for c in range(self.n_channels):
            self.channels.reset_stream(stream * self.n_channels + c)

    def submit(self, iq) -> None:
        """Enqueue the down-conversion and the analysis of `blocks_per_launch` blocks of every input (asynchronous; two
        submissions may be in flight).  `iq` as `Channelizer.run` takes it; it is held until its `collect`."""
        self.channels.submit(self.ddc.run(iq))
        self._held.append(iq)

    def collect(self, ts_start: Sequence[datetime.datetime], with_all: bool = False):
        """Wait for the oldest submission.  `ts_start`: one per input, the start of the first wideband block of the launch.
        -> per input unit (input-major, block-minor, like `BatchAnalyzer.collect`) `(signals, candidates)`: the shadow-filtered
        Signals of all its channels in channel order and their candidate count; with `with_all` the list of the channels'
        `(filtered, all, keys)`."""
        C, B = self.n_channels, self.blocks_per_launch
        cts = [channel_ts(t, self.ddc.n_taps, self.sample_rate) for t in ts_start for _ in range(C)]
        res = self.channels.collect(cts, with_all=with_all)
        self._held.pop(0)
        out = []
        for i in range(self.n_streams):
            for b in range(B):
                per = [res[(i * C + c) * B + b] for c in range(C)]
                out.append(per if with_all else ([s for p in per for s in p[0]], sum(p[1] for p in per)))
        return out

    def last_survey(self) -> list:
        """The band survey of the last collected launch (built with `survey=True`): per input unit (input-major, block-minor,
        like `collect`) the list of its channels' `BandSurvey`s in channel order."""
        C, B = self.n_channels, self.blocks_per_launch
        res = self.channels.last_survey()
        return [[res[(i * C + c) * B + b] for c in range(C)] for i in range(self.n_streams) for b in range(B)]

    def last_fine_frequencies(self, all_signals: bool = False) -> list:
        """The carrier estimates of the last collected launch (built with `fine_frequency=True`): per input unit (input-major,
        block-minor, like `collect`) one float64 array aligned with the Signals `collect` returned for it, its channels'
        concatenated in channel order (with `all_signals`: their `all_signals`), computed at the channel rate fs / D.
        An estimate is kept only where the Signal's bin lies in its channel's flat central half, signed bin k in
        [-n/4, n/4); elsewhere it is NaN.  On the `full_band` grid those halves tile the band without overlap, so a pulse
        found in two overlapping channels gets its estimate from exactly one of them -- except within about two bins of a
        channel centre, where the estimator has none (finefreq.py: the bins next to DC), so such a pulse gets none."""
        C, B, n = self.n_channels, self.blocks_per_launch, self.channels.fft_nperseg
        res = [np.where(central_half(fi, n), f, np.nan) for f, fi in self.channels._fine_units(all_signals)]
        return [np.concatenate([res[(i * C + c) * B + b] for c in range(C)]) for i in range(self.n_streams) for b in range(B)]

    def band_survey(self) -> list:
        """`full_band` only: per input unit (input-major, block-minor) one `BandSurvey` of the whole band, stitched from the flat
        central halves of its channels (`survey.stitch`): a uniform grid of spacing fs / (D nperseg) from
        center_freq - (fs / 2 - fs / (4 D)) up to, not including, center_freq + fs / 2 - fs / (4 D), with the frequencies of the
        channels' Signals.  ValueError for an analyzer on arbitrary channel offsets, whose channels may overlap or leave gaps."""
        if not isinstance(self.ddc, FilterBank):
            raise ValueError("band_survey needs the uniform channel grid of full_band; last_survey gives the channels of this plan")
        B = self.blocks_per_launch
        return [stitch(self.devices[u // B], chans) for u, chans in enumerate(self.last_survey())]

    def process_blocks(self, iq, ts_start: Sequence[datetime.datetime]):
        self.submit(iq)
        return self.collect(ts_start, with_all=True)
