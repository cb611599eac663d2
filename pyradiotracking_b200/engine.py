"""ctypes binding of the C ABI in include/rt_engine.h (librtb200.so, sm_100a CUDA).

This is the thin host layer between `SignalAnalyzer` and the kernels.  There is no
CPU fallback: if the shared library is missing or no CUDA device is present, creating
an `Engine` raises.
"""
import ctypes
import functools
import logging
import os
import sys
from typing import Optional, Sequence, Tuple, Union

import numpy as np

from . import build as _build

RT_OK, RT_ERR_INVALID, RT_ERR_CUDA, RT_ERR_OVERFLOW, RT_ERR_STATE = 0, -1, -2, -3, -4
RT_ABI_VERSION = 2
FFT_AUTO, FFT_GENERIC, FFT_REG256, FFT_TC256 = 0, 1, 2, 3
SCAN_AUTO, SCAN_SERIAL, SCAN_OVERLAP, SCAN_LEAN = 0, 1, 2, 3
SAMPLE_CU8, SAMPLE_CI8, SAMPLE_CI16, SAMPLE_CF32 = 0, 1, 2, 3
RT_SLOTS = 2        # results the engine holds: a third launch without a fetch drops the oldest (include/rt_engine.h)

# rt_config.sample_format by SigMF datatype: (code, element dtype, bytes per complex sample).  The engine analyses the normalised
# samples (cu8: b / 127.5 - 1 as pyrtlsdr delivers them, ci8: v / 128, ci16_le: v / 32768, cf32_le: x); include/rt_engine.h
# has the table and its limits.
SAMPLE_FORMATS = {
    "cu8": (SAMPLE_CU8, np.dtype(np.uint8), 2),
    "ci8": (SAMPLE_CI8, np.dtype(np.int8), 2),
    "ci16_le": (SAMPLE_CI16, np.dtype("<i2"), 4),
    "cf32_le": (SAMPLE_CF32, np.dtype("<f4"), 8),
}
_FORMAT_BY_CODE = {v[0]: k for k, v in SAMPLE_FORMATS.items()}


def sample_format_name(fmt: Union[str, int]) -> str:
    """The SigMF name of a sample format given by name or by rt_config.sample_format code; ValueError if unknown."""
    name = _FORMAT_BY_CODE.get(fmt) if isinstance(fmt, (int, np.integer)) and not isinstance(fmt, bool) else fmt
    if name not in SAMPLE_FORMATS:
        raise ValueError(f"unknown sample format {fmt!r}: expected one of {', '.join(SAMPLE_FORMATS)}")
    return name


logger = logging.getLogger(__name__)

# every symbol include/rt_engine.h declares
EXPORTS = (
    "rt_last_error", "rt_abi_version", "rt_device_count", "rt_engine_create", "rt_engine_destroy",
    "rt_engine_set_stream", "rt_engine_reset_stream", "rt_engine_process", "rt_engine_launch", "rt_engine_fetch", "rt_engine_peek",
    "rt_engine_shape", "rt_engine_read_spectrogram", "rt_engine_read_row_means", "rt_engine_enable_timing",
    "rt_engine_get_timing", "rt_engine_join", "rt_engine_wait_stream", "rt_engine_last_counts", "rt_tc256_tables",
    # include/rt_matcher.h
    "rt_matcher_create", "rt_matcher_destroy", "rt_matcher_add", "rt_matcher_pending", "rt_matcher_drain",
    "rt_matcher_open", "rt_matcher_read_open",
)


class RtConfig(ctypes.Structure):
    _fields_ = [
        ("abi_version", ctypes.c_int32), ("cuda_device", ctypes.c_int32), ("n_streams", ctypes.c_int32),
        ("nperseg", ctypes.c_int32), ("block_samples", ctypes.c_int64), ("sample_rate", ctypes.c_double),
        ("window", ctypes.POINTER(ctypes.c_double)), ("signal_threshold", ctypes.POINTER(ctypes.c_double)),
        ("snr_threshold", ctypes.c_double), ("probe_stride", ctypes.c_int32), ("min_cols", ctypes.c_int32),
        ("max_cols", ctypes.c_int32), ("max_records", ctypes.c_int32), ("fft_impl", ctypes.c_int32),
        ("scan_schedule", ctypes.c_int32), ("launch_streams", ctypes.c_int32), ("chunk_segs", ctypes.c_int32),
        ("blocks_per_launch", ctypes.c_int32), ("sample_format", ctypes.c_int32), ("reserved", ctypes.c_int32 * 2),
    ]


class RtTiming(ctypes.Structure):
    _fields_ = [
        ("spectrogram_ms", ctypes.c_double), ("rowmean_ms", ctypes.c_double), ("probe_ms", ctypes.c_double),
        ("extract_ms", ctypes.c_double), ("launches", ctypes.c_int64), ("kernels", ctypes.c_int64),
    ]


# rt_record, 40 bytes
RECORD_DTYPE = np.dtype([
    ("stream", "<i4"), ("fi", "<i4"), ("start", "<i4"), ("end", "<i4"),
    ("max_lin", "<f4"), ("row_mean", "<f4"), ("mean_lin", "<f8"), ("std_db", "<f8"),
])
assert RECORD_DTYPE.itemsize == 40

_lib = None


class EngineError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"rt_engine error {code}: {msg}")
        self.code = code


def library_path() -> str:
    return _build.LIB


def load_library() -> ctypes.CDLL:
    """dlopen librtb200.so (building it first if it has never been built and nvcc is here)."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        _build.build()          # raises if nvcc is missing: there is nothing to fall back to
    lib = ctypes.CDLL(path)
    lib.rt_last_error.restype = ctypes.c_char_p
    lib.rt_engine_create.argtypes = [ctypes.POINTER(RtConfig), ctypes.POINTER(ctypes.c_void_p)]
    lib.rt_engine_destroy.argtypes = [ctypes.c_void_p]
    lib.rt_engine_destroy.restype = None
    lib.rt_engine_set_stream.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    lib.rt_engine_reset_stream.argtypes = [ctypes.c_void_p, ctypes.c_int32]
    lib.rt_engine_process.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_size_t,
                                      ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32)]
    lib.rt_engine_launch.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.c_size_t]
    lib.rt_engine_fetch.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32)]
    lib.rt_engine_peek.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32)]
    lib.rt_engine_join.argtypes = [ctypes.c_void_p]
    lib.rt_engine_wait_stream.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    lib.rt_tc256_tables.argtypes = [ctypes.c_void_p, ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    lib.rt_engine_last_counts.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int32)]
    lib.rt_engine_shape.argtypes = [ctypes.c_void_p] + [ctypes.POINTER(ctypes.c_int32)] * 3
    lib.rt_engine_read_spectrogram.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p]
    lib.rt_engine_read_row_means.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p]
    lib.rt_engine_enable_timing.argtypes = [ctypes.c_void_p, ctypes.c_int32]
    lib.rt_engine_get_timing.argtypes = [ctypes.c_void_p, ctypes.POINTER(RtTiming), ctypes.c_int32]
    if lib.rt_abi_version() != RT_ABI_VERSION:
        raise ImportError(f"{path}: ABI {lib.rt_abi_version()} != {RT_ABI_VERSION}; rebuild (python -m pyradiotracking_b200.build --force)")
    _lib = lib
    return lib


def _check(rc: int):
    if rc != RT_OK:
        raise EngineError(rc, load_library().rt_last_error().decode("utf-8", "replace"))


def device_count() -> int:
    n = load_library().rt_device_count()
    if n < 0:
        _check(n)
    return n


@functools.lru_cache(maxsize=None)
def _cai_type(typestr: str) -> Tuple[str, int]:
    """(numpy name, itemsize) of a __cuda_array_interface__ typestr; the name is empty for a non-native byte order."""
    dt = np.dtype(typestr)
    return (dt.name if dt.isnative else ""), dt.itemsize


def _producer_stream(obj) -> Optional[int]:
    """The cudaStream_t handle whose queued work a reader of the device object `obj` must wait for: for a torch tensor the
    current stream of its device (0: the legacy default stream), for a __cuda_array_interface__ object its `stream` entry
    (None when absent or None: the producer has synchronised; 1 and 2 are the legacy and per-thread default streams)."""
    if hasattr(obj, "data_ptr") and getattr(obj, "is_cuda", False):      # torch.Tensor: torch is loaded, the binding does not import it
        return sys.modules["torch"].cuda.current_stream(obj.device).cuda_stream
    s = obj.__cuda_array_interface__.get("stream")
    if s is None:
        return None
    if int(s) == 0:         # the CUDA Array Interface (v3) forbids 0: it would not say which default stream is meant
        raise ValueError("__cuda_array_interface__ stream 0 is ambiguous: use 1 (legacy default) or 2 (per-thread default)")
    return int(s)


def _device_pointer(obj, n_rows: int, row_bytes: int, dtypes: Tuple[str, ...] = ("uint8",)) -> Optional[Tuple[int, int]]:
    """(pointer, row stride in bytes) if `obj` lives in device memory, else None.  `obj` must have one of the native-endian
    element types named in `dtypes` (numpy names; default uint8) and hold `n_rows` rows of `row_bytes` contiguous bytes (a 1-D
    object: one row); a wrong size would be read out of bounds."""
    if hasattr(obj, "data_ptr") and getattr(obj, "is_cuda", False):      # torch.Tensor, without importing torch
        if str(obj.dtype)[6:] not in dtypes:                            # "torch.uint8"
            raise TypeError(f"IQ blocks must be {' / '.join(dtypes)}, got {obj.dtype}")
        item = obj.element_size()
        shape, strides = tuple(obj.shape), tuple(int(x) * item for x in obj.stride())
        ptr = int(obj.data_ptr())
    else:
        cai = getattr(obj, "__cuda_array_interface__", None)
        if cai is None:
            return None
        name, item = _cai_type(cai["typestr"])
        if name not in dtypes:
            raise TypeError(f"IQ blocks must be {' / '.join(dtypes)}, got {cai['typestr']}")
        shape = tuple(cai["shape"])
        st = cai.get("strides")
        if st is None:                                                   # C-contiguous: strides in BYTES
            st, acc = [], item
            for d in reversed(shape):
                st.insert(0, acc)
                acc *= d
        strides = tuple(int(x) for x in st)
        ptr = int(cai["data"][0])
    # the trailing axes of a row must be dense; the leading axis is the stream
    if len(shape) == 1:
        shape, strides = (1,) + shape, (shape[0] * strides[0],) + strides
    inner, dense = item, True
    for d, st in zip(reversed(shape[1:]), reversed(strides[1:])):
        dense = dense and (d == 1 or st == inner)
        inner *= d
    if shape[0] != n_rows or inner != row_bytes or not dense:
        raise ValueError(f"expected {' / '.join(dtypes)} [{n_rows}, {row_bytes // item}] on the device, got shape {shape} strides {strides}")
    return ptr, (strides[0] if n_rows > 1 else row_bytes)


class Engine:
    """A batch of `n_streams` analyzers on one GPU (rt_engine handle)."""

    def __init__(self, *, n_streams: int, block_samples: int, nperseg: int, window: np.ndarray, sample_rate: float,
                 signal_threshold: Union[float, Sequence[float]], snr_threshold: float, probe_stride: int,
                 min_cols: int, max_cols: int, max_records: int = 0, cuda_device: int = 0, fft_impl: int = FFT_AUTO,
                 scan_schedule: int = SCAN_AUTO, launch_streams: int = 0, chunk_segs: int = 0, blocks_per_launch: int = 1,
                 sample_format: Union[str, int] = "cu8"):
        """`sample_format`: the SigMF datatype of the input (`SAMPLE_FORMATS`) or an rt_config.sample_format code."""
        self._lib = load_library()
        self._h = ctypes.c_void_p()
        win = np.ascontiguousarray(window, dtype=np.float64)
        if win.shape != (nperseg,):
            raise ValueError("window must have nperseg entries")
        thr = np.ascontiguousarray(np.broadcast_to(np.asarray(signal_threshold, dtype=np.float64), (n_streams,)))
        cfg = RtConfig(
            abi_version=RT_ABI_VERSION, cuda_device=cuda_device, n_streams=n_streams, nperseg=nperseg,
            block_samples=block_samples, sample_rate=float(sample_rate),
            window=win.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
            signal_threshold=thr.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
            snr_threshold=float(snr_threshold), probe_stride=int(probe_stride), min_cols=int(min_cols),
            max_cols=int(max_cols), max_records=int(max_records), fft_impl=int(fft_impl),
            scan_schedule=int(scan_schedule), launch_streams=int(launch_streams), chunk_segs=int(chunk_segs),
            blocks_per_launch=int(blocks_per_launch),
            sample_format=int(sample_format) if isinstance(sample_format, (int, np.integer)) else SAMPLE_FORMATS[sample_format_name(sample_format)][0],
        )
        _check(self._lib.rt_engine_create(ctypes.byref(cfg), ctypes.byref(self._h)))
        self.sample_format = sample_format_name(cfg.sample_format)       # the engine accepted it: a known format
        _, dtype, self.sample_bytes = SAMPLE_FORMATS[self.sample_format]
        # element types a launch accepts: the format's, and complex64 (an I,Q pair of float32) for cf32
        self._dtypes = (dtype, np.dtype(np.complex64)) if self.sample_format == "cf32_le" else (dtype,)
        self._dtype_names = tuple(d.name for d in self._dtypes)
        self.n_streams, self.nperseg, self.block_samples = n_streams, nperseg, block_samples
        self.blocks_per_launch = int(blocks_per_launch)
        self.n_units = n_streams * self.blocks_per_launch      # analyzer units per launch: rt_record.stream counts these
        self.T = block_samples // nperseg
        self.cuda_device = cuda_device
        self.truncated = 0           # records the last fetch could not return (rt_config.max_records exceeded)
        # The inputs (host or device) of the launches no fetch has returned yet, oldest first: the kernels of a launch may still
        # read its input, also after a third launch dropped its result from the engine's ring.  A fetch has waited for its
        # launch's kernels and for every earlier launch's (the scan kernels run in launch order), so it releases them.
        self._held = []
        self._launches = self._fetches = 0    # mirror of the engine's ring: launches made, results fetched or dropped
        self._stream = None                   # the cudaStream_t handle last given to set_stream

    # -- lifetime ---------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._lib.rt_engine_destroy(self._h)          # waits for the engine's streams
            self._h = ctypes.c_void_p()
        self._held = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- data path ----------------------------------------------------------------------------
    def _resolve(self, iq) -> Tuple[int, int, int, Optional[int], object]:
        """(pointer, on device, row stride in bytes, producer stream, object that owns the memory) of one launch's input:
        [n_streams, 2 * block_samples * blocks_per_launch] elements of the engine's sample format (or [n_streams,
        blocks_per_launch, 2 * block_samples]); cf32 also as complex64 with half as many elements per row.  The producer stream
        (`_producer_stream`) is None for host memory."""
        row = self.sample_bytes * self.block_samples * self.blocks_per_launch       # bytes: the consecutive blocks of one stream
        dev = _device_pointer(iq, self.n_streams, row, self._dtype_names)
        if dev is not None:
            return dev[0], 1, dev[1], _producer_stream(iq), iq
        arr = np.asarray(iq)
        if arr.dtype not in self._dtypes:
            raise TypeError(f"IQ blocks must be {' / '.join(self._dtype_names)} for sample format {self.sample_format}, got {arr.dtype}")
        item = arr.itemsize
        if arr.ndim == 3 and arr.shape[1:] == (self.blocks_per_launch, row // self.blocks_per_launch // item) and arr[0].flags.c_contiguous:
            arr = arr.reshape(arr.shape[0], -1) if arr.flags.c_contiguous else np.lib.stride_tricks.as_strided(
                arr, (arr.shape[0], row // item), (arr.strides[0], item))
        if arr.ndim == 1:
            arr = arr.reshape(1, -1)
        if arr.shape != (self.n_streams, row // item) or arr.strides[1] != item:
            raise ValueError(f"expected {arr.dtype.name} [{self.n_streams}, {row // item}], got {arr.shape}")
        return int(arr.ctypes.data), 0, int(arr.strides[0]), None, arr

    def launch(self, iq) -> None:
        """Enqueue one block (`blocks_per_launch` consecutive blocks) for every stream (asynchronous).  A CUDA tensor is read
        after the work queued so far on its device's current stream, a __cuda_array_interface__ object after its `stream`;
        `iq` is held until a fetch has returned this launch or a later one."""
        ptr, on_dev, stride, producer, owner = self._resolve(iq)
        if producer is not None and producer != self._stream:
            _check(self._lib.rt_engine_wait_stream(self._h, ctypes.c_void_p(producer)))
        _check(self._lib.rt_engine_launch(self._h, ctypes.c_void_p(ptr), on_dev, stride))
        self._held.append(owner)
        self._launches += 1
        if self._launches - self._fetches > RT_SLOTS:
            self._fetches += 1            # the engine dropped the oldest unfetched result; its input stays held

    def fetch(self) -> np.ndarray:
        """Wait for the oldest unfetched launch; candidate records sorted by (unit, fi, start).  If the launch produced more
        records than `max_records`, the first ones are returned, `self.truncated` says how many are missing, and an error
        is logged (the reference has no such limit: one noisy band must not take the other streams' detections down)."""
        n = ctypes.c_int32(0)
        _check(self._lib.rt_engine_peek(self._h, ctypes.byref(n)))
        out = np.empty(n.value, dtype=RECORD_DTYPE)
        need = ctypes.c_int32(0)
        rc = self._lib.rt_engine_fetch(self._h, out.ctypes.data_as(ctypes.c_void_p), n.value, ctypes.byref(need))
        self.truncated = 0
        if rc in (RT_OK, RT_ERR_OVERFLOW):              # the launch was consumed: release its input and every older one
            self._fetches += 1
            del self._held[:len(self._held) - (self._launches - self._fetches)]
        if rc == RT_ERR_OVERFLOW:
            self.truncated = need.value - n.value
            logger.error("rt_engine: %d candidate records exceed max_records, %d dropped", need.value, self.truncated)
        else:
            _check(rc)
        return out

    def process(self, iq) -> np.ndarray:
        self.launch(iq)
        return self.fetch()

    def reset_stream(self, stream: int) -> None:
        _check(self._lib.rt_engine_reset_stream(self._h, stream))

    def set_stream(self, cuda_stream: int) -> None:
        """Launch on this cudaStream_t handle.  Inputs produced on it need no extra wait (`launch`)."""
        _check(self._lib.rt_engine_set_stream(self._h, ctypes.c_void_p(cuda_stream)))
        self._stream = int(cuda_stream)

    def last_counts(self) -> tuple:
        """(probe hits handed to the extraction kernel, records emitted) of the last fetched launch."""
        w, r = ctypes.c_int32(0), ctypes.c_int32(0)
        _check(self._lib.rt_engine_last_counts(self._h, ctypes.byref(w), ctypes.byref(r)))
        return w.value, r.value

    def join(self) -> None:
        """Make the launch stream wait for the scan kernels of every launch so far (they run on an
        engine-internal stream, overlapping the next launch's spectrogram)."""
        _check(self._lib.rt_engine_join(self._h))

    # -- parity hooks / timing ------------------------------------------------------------------
    def read_spectrogram(self, stream: int = 0) -> np.ndarray:
        """float32 [T, nperseg] of the last launch (= scipy's Sxx transposed)."""
        if not 0 <= stream < self.n_units:
            raise IndexError("no such analyzer unit")
        out = np.empty((self.T, self.nperseg), dtype=np.float32)
        _check(self._lib.rt_engine_read_spectrogram(self._h, stream, out.ctypes.data_as(ctypes.c_void_p)))
        return out

    def read_row_means(self, stream: int = 0) -> np.ndarray:
        out = np.empty(self.nperseg, dtype=np.float32)
        _check(self._lib.rt_engine_read_row_means(self._h, stream, out.ctypes.data_as(ctypes.c_void_p)))
        return out

    def enable_timing(self, period: int = 4) -> None:
        """Bracket the kernels of every `period`-th launch with CUDA events (0 / False: off)."""
        _check(self._lib.rt_engine_enable_timing(self._h, int(period)))

    def timing(self, reset: bool = False) -> dict:
        t = RtTiming()
        _check(self._lib.rt_engine_get_timing(self._h, ctypes.byref(t), int(reset)))
        return {k: getattr(t, k) for k, _ in RtTiming._fields_}


def tc256_tables(window, sample_rate: float):
    """Constant operands of the tensor-core spectrogram kernel (parity hook, CPU only): (bmat uint16 [16, 2, 1024] in the
    operand layout, wc complex128 [3] for the bins 0 / 1 / 255, pscale, eligible)."""
    lib = load_library()
    w = np.ascontiguousarray(window, dtype=np.float64)
    if w.shape != (256,):
        raise ValueError("the tensor-core kernel is a 256-point kernel")
    bmat = np.zeros((16, 2, 1024), dtype=np.uint16)
    wc = np.zeros(6, dtype=np.float64)
    ps = ctypes.c_double(0.0)
    el = ctypes.c_int32(0)
    _check(lib.rt_tc256_tables(w.ctypes.data_as(ctypes.c_void_p), float(sample_rate), bmat.ctypes.data_as(ctypes.c_void_p),
                               wc.ctypes.data_as(ctypes.c_void_p), ctypes.byref(ps), ctypes.byref(el)))
    return bmat, wc.view(np.complex128), ps.value, bool(el.value)
