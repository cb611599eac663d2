"""Recorded-capture ingest for the batched engine (SURVEY.md section 8f rank 2, BASELINE configs[3]).

The reference ingests only live (`sdr.read_samples_async`, radiotracking/analyze.py:143-157) and has no file reader;
its wire format is what librtlsdr delivers and `rtl_sdr -f ... file.bin` records: interleaved uint8 I,Q bytes ("cu8").
Archives of other receivers hold ci8 (HackRF), ci16_le (Airspy, SDRplay, USRP sc16) or cf32_le (GNU Radio file sinks,
`.cfile`); the reader takes the element type from `sample_format` or from a SigMF `.sigmf-meta` file beside the data
(`core:datatype`).  This module feeds such recordings -- one file per station channel -- to a `BatchAnalyzer`:

    CaptureReader     blocks `[n_streams, 2*block_samples]` elements (or groups of `blocks_per_read` consecutive blocks per
                      stream) out of a ring of (pinned) host buffers, filled by a reader thread so that disk reads overlap
                      the GPU
    replay()          submit / collect with two launches in flight; an analyzer built with `blocks_per_launch = B` gets B
                      consecutive callback blocks of every channel per launch (the carry between them stays inside the
                      engine), which is what makes a batch of slow channels (64 x 300 kS/s) fill the GPU; the results are
                      those of block-by-block replay (the engine's staging ring copies block i+1 while the
                      kernels of block i run, INTEGRATION.md); timestamps follow the reference's drift-free virtual
                      clock: block b starts at t0 + b * block_samples / sample_rate (analyze.py:218-231)

A recording ends like an SDR that is unplugged mid-callback: the incomplete last block is dropped, for every channel
at the length of the shortest one.
"""
import datetime
import os
import queue
import threading
from typing import Callable, Iterator, List, Optional, Sequence

import json

import numpy as np

from .engine import SAMPLE_FORMATS


def _alloc(shape, pinned: bool) -> np.ndarray:
    """Host buffer, page-locked when torch sees a CUDA device (plumbing only: the H2D copies of the engine then run
    at full PCIe speed and asynchronously)."""
    if pinned:
        try:
            import torch

            if torch.cuda.is_available():
                t = torch.empty(shape, dtype=torch.uint8, pin_memory=True)
                arr = t.numpy()
                _alloc.keep.append(t)          # the tensor owns the memory
                return arr
        except ImportError:
            pass
    return np.empty(shape, dtype=np.uint8)


_alloc.keep = []


def sigmf_meta_path(path: str) -> str:
    """The SigMF metadata file that belongs to a data file: `x.sigmf-data` -> `x.sigmf-meta`, any other name -> name + `.sigmf-meta`."""
    stem = path[: -len(".sigmf-data")] if path.endswith(".sigmf-data") else path
    return stem + ".sigmf-meta"


def sigmf_sample_format(path: str) -> Optional[str]:
    """`core:datatype` of the SigMF metadata beside the data file `path`, or None without one.  ValueError for a datatype the
    engine does not read (big-endian, real-valued, or not in `engine.SAMPLE_FORMATS`)."""
    meta = sigmf_meta_path(path)
    if not os.path.exists(meta):
        return None
    with open(meta, "r", encoding="utf-8") as f:
        dt = json.load(f).get("global", {}).get("core:datatype")
    if dt not in SAMPLE_FORMATS:
        raise ValueError(f"{meta}: core:datatype {dt!r} is not one of {', '.join(SAMPLE_FORMATS)}")
    return dt


class CaptureReader:
    """Iterate over the blocks of `paths` (one raw IQ file per stream).

    `sample_format`: the element type of the files (`engine.SAMPLE_FORMATS`); None takes it from the SigMF metadata beside the
    files (all must agree) and reads cu8 without one.  An explicit format that a metadata file contradicts is a ValueError.
    Items are arrays of that element type (views of byte buffers).

    Yields `(block_index, array)`; `array` is a view of one of `n_buffers` ring buffers and stays valid until
    `n_buffers - 1` further blocks have been taken (with the default 4: two blocks in flight in the engine plus the one
    being filled).  With `blocks_per_read = B > 1` an item is a group of B consecutive blocks, `[n_streams, B * 2 * block_samples]`
    (`block_index` = index of its first block); a last, incomplete group is padded with zero bytes (its blocks beyond
    `n_blocks` must be ignored by the consumer)."""

    def __init__(self, paths: Sequence[str], block_samples: int, n_buffers: int = 4, pinned: bool = True,
                 max_blocks: Optional[int] = None, blocks_per_read: int = 1, sample_format: Optional[str] = None):
        if not paths:
            raise ValueError("no capture files")
        if n_buffers < 2:
            raise ValueError("need at least two ring buffers")
        self.paths = list(paths)
        if sample_format is not None and sample_format not in SAMPLE_FORMATS:
            raise ValueError(f"sample_format {sample_format!r} is not one of {', '.join(SAMPLE_FORMATS)}")
        metas = {m for m in (sigmf_sample_format(p) for p in self.paths) if m is not None}
        if len(metas) > 1 or (sample_format is not None and metas and metas != {sample_format}):
            raise ValueError(f"SigMF metadata says {', '.join(sorted(metas))}, expected {sample_format or 'one format for every file'}")
        self.sample_format = sample_format or (metas.pop() if metas else "cu8")
        _, self.dtype, sample_bytes = SAMPLE_FORMATS[self.sample_format]
        self.block_bytes = sample_bytes * int(block_samples)
        sizes = [os.path.getsize(p) for p in self.paths]
        self.n_blocks = min(sizes) // self.block_bytes              # tail dropped
        if max_blocks is not None:
            self.n_blocks = min(self.n_blocks, max_blocks)
        self.n_streams = len(self.paths)
        self.blocks_per_read = max(1, int(blocks_per_read))
        self._bufs = [_alloc((self.n_streams, self.blocks_per_read * self.block_bytes), pinned) for _ in range(n_buffers)]
        self._free: "queue.Queue[int]" = queue.Queue()
        self._full: "queue.Queue" = queue.Queue()
        for i in range(n_buffers):
            self._free.put(i)
        self._thread: Optional[threading.Thread] = None
        self._stop = False

    def _fill(self):
        try:
            files = [open(p, "rb", buffering=0) for p in self.paths]
            try:
                for b in range(0, self.n_blocks, self.blocks_per_read):
                    i = self._free.get()
                    if self._stop:
                        return
                    buf = self._bufs[i]
                    want = min(self.blocks_per_read, self.n_blocks - b) * self.block_bytes
                    if want < buf.shape[1]:
                        buf[:, want:] = 0                        # incomplete last group
                    for s, f in enumerate(files):
                        view = memoryview(buf[s])[:want]
                        got = 0
                        while got < want:                        # raw files may return short reads
                            n = f.readinto(view[got:])
                            if not n:
                                raise IOError(f"{self.paths[s]}: unexpected end of file in block {b}")
                            got += n
                    self._full.put((b, i))
            finally:
                for f in files:
                    f.close()
            self._full.put(None)
        except Exception as exc:        # hand the error to the consumer thread
            self._full.put(exc)

    def __iter__(self) -> Iterator:
        if self._thread is not None:
            raise RuntimeError("a CaptureReader can be iterated once")
        self._thread = threading.Thread(target=self._fill, daemon=True)
        self._thread.start()
        held: List[int] = []
        while True:
            item = self._full.get()
            if item is None:
                break
            if isinstance(item, Exception):
                raise item
            b, i = item
            held.append(i)
            if len(held) == len(self._bufs):                     # the oldest view is no longer needed by contract
                self._free.put(held.pop(0))
            yield b, self._bufs[i].view(self.dtype)
        self._thread.join()

    def close(self):
        self._stop = True
        self._free.put(0)


def replay(paths: Sequence[str], analyzer, t0: datetime.datetime, on_block: Optional[Callable] = None,
           max_blocks: Optional[int] = None, pinned: bool = True, on_survey: Optional[Callable] = None,
           on_fine_frequencies: Optional[Callable] = None) -> int:
    """Run every full block of the recordings through `analyzer` (a `BatchAnalyzer` with one stream per file), read in the
    analyzer's `sample_format` (a SigMF metadata file beside a recording must agree with it).

    `on_block(block_index, per_stream)` receives what `BatchAnalyzer.collect` returns for that block
    (`per_stream[s] = (shadow-filtered Signals, candidates before the filter)`), in block order -- also when the
    analyzer takes several blocks per launch.  `on_survey(block_index, surveys)` (an analyzer built with `survey=True`) receives
    what `analyzer.last_survey()` gives for that block, regrouped per block the same way; `on_fine_frequencies(block_index,
    per_stream)` (an analyzer built with `fine_frequency=True`) what `analyzer.last_fine_frequencies()` gives, aligned with the
    filtered Signals `on_block` received.  Returns the number of blocks processed."""
    if analyzer.n_streams != len(paths):
        raise ValueError("one capture file per analyzer stream")
    B = getattr(analyzer, "blocks_per_launch", 1)
    reader = CaptureReader(paths, analyzer.block_samples, pinned=pinned, max_blocks=max_blocks, blocks_per_read=B,
                           sample_format=getattr(analyzer, "sample_format", "cu8"))
    dt = datetime.timedelta(seconds=analyzer.block_samples / analyzer.sample_rate)
    pending: List[int] = []
    done = 0

    def drain():
        nonlocal done
        b0 = pending.pop(0)
        res = analyzer.collect([t0 + b0 * dt] * analyzer.n_streams)      # per analyzer unit: stream-major, block-minor
        surveys = analyzer.last_survey() if on_survey is not None else None
        fine = analyzer.last_fine_frequencies() if on_fine_frequencies is not None else None
        for k in range(min(B, reader.n_blocks - b0)):                     # (the padding blocks of a last group are ignored)
            if on_block is not None:
                on_block(b0 + k, [res[s * B + k] for s in range(analyzer.n_streams)])
            if on_survey is not None:
                on_survey(b0 + k, [surveys[s * B + k] for s in range(analyzer.n_streams)])
            if on_fine_frequencies is not None:
                on_fine_frequencies(b0 + k, [fine[s * B + k] for s in range(analyzer.n_streams)])
            done += 1

    try:
        for b, block in reader:
            analyzer.submit(block)
            pending.append(b)
            if len(pending) == 2:                                # two launches in flight
                drain()
        while pending:
            drain()
    finally:
        reader.close()
    return done
