"""Float64 restatement of the down-converter (include/rt_ddc.h) for the tests, on `format_oracle.decode_samples`.

TEST INFRASTRUCTURE ONLY: nothing under `pyradiotracking_b200/` imports it.

    y_c[m] = exp(-2 pi i ((inc_c (n0 + m D)) mod 2^32) / 2^32) * sum_{k<L} g_c[k] x[n0 + m D - k],
    g_c[k] = h[k] exp(+2 pi i ((inc_c k) mod 2^32) / 2^32),

with x before the first sample of a stream taken from its history (zero at the start).
"""
from typing import Optional, Sequence

import numpy as np

from tests import format_oracle as FO

_TWO32 = float(1 << 32)


def phase_turns(inc: int, n: np.ndarray) -> np.ndarray:
    """((inc * n) mod 2^32) / 2^32 in exact integer arithmetic, for any integer n (also past 2^40)."""
    n32 = (np.asarray(n, dtype=object) % (1 << 32)).astype(np.uint64)
    return ((np.uint64(int(inc) % (1 << 32)) * n32) % np.uint64(1 << 32)).astype(np.float64) / _TWO32


def complex_taps(h: np.ndarray, inc: int) -> np.ndarray:
    """g[k] = h[k] exp(+2 pi i ((inc k) mod 2^32) / 2^32)."""
    k = np.arange(len(h))
    return np.asarray(h, dtype=np.float64) * np.exp(2j * np.pi * phase_turns(inc, k))


def ddc(x: np.ndarray, h: Sequence[float], phase_inc: Sequence[int], D: int, n0: int = 0,
        history: Optional[np.ndarray] = None, chunk: int = 4096) -> np.ndarray:
    """complex128 [C, len(x) // D]: the channels of the complex samples `x` whose first sample has the index n0; `history`:
    the L - 1 samples before it (default zeros)."""
    h = np.asarray(h, dtype=np.float64)
    L = len(h)
    hist = np.zeros(L - 1, np.complex128) if history is None else np.asarray(history, np.complex128)
    xx = np.concatenate([hist, np.asarray(x, np.complex128)])
    M = len(x) // D
    # row m of the window view: xx[m D .. m D + L - 1] = x[n0 + m D - (L - 1) .. n0 + m D], reversed against g
    win = np.lib.stride_tricks.sliding_window_view(xx, L)[::D][:M]
    G = np.stack([complex_taps(h, inc)[::-1] for inc in phase_inc], axis=1)       # [L, C]
    acc = np.empty((M, len(phase_inc)), np.complex128)
    for a in range(0, M, chunk):
        acc[a:a + chunk] = win[a:a + chunk] @ G
    m = n0 + D * np.arange(M, dtype=object)
    rot = np.stack([np.exp(-2j * np.pi * phase_turns(inc, m)) for inc in phase_inc], axis=0)
    return rot * acc.T


def ddc_raw(raw: np.ndarray, fmt: str, h, phase_inc, D: int, n0: int = 0, history=None) -> np.ndarray:
    """`ddc` of interleaved I,Q elements in the sample format `fmt` (normalised like the engine)."""
    return ddc(FO.decode_samples(raw, fmt), h, phase_inc, D, n0, history)
