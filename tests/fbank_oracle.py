"""Float64 restatement of the polyphase FFT filter bank (include/rt_fbank.h) for the tests.

TEST INFRASTRUCTURE ONLY: nothing under `pyradiotracking_b200/` imports it.

With C = 2 D, the output time n = n0 + m D and the global input index j:

    y_k[m] = sum_{r<C} exp(-2 pi i k r / C) u_r[m],      u_r[m] = sum_{j = r (mod C), 0 <= n - j < L} h[n - j] x[j]

for k = -(D - 1) ... D - 1 (row k + D - 1).  `tests/test_fbank.py` checks that this equals `ddc_oracle.ddc` with the phase
increments inc_k = ((k mod C) 2^32) / C, to float64 rounding; it is the fast form of that oracle for all 2 D - 1 channels.
"""
from typing import Optional

import numpy as np


def fbank(x: np.ndarray, h, D: int, n0: int = 0, history: Optional[np.ndarray] = None, chunk: int = 2048) -> np.ndarray:
    """complex128 [2 D - 1, len(x) // D]: the grid channels of the complex samples `x` whose first sample has the index n0;
    `history`: the L - 1 samples before it (default zeros)."""
    h = np.asarray(h, dtype=np.float64)
    L, C = len(h), 2 * D
    hist = np.zeros(L - 1, np.complex128) if history is None else np.asarray(history, np.complex128)
    xx = np.concatenate([hist, np.asarray(x, np.complex128)])
    M = len(x) // D
    Q = -(-L // C)
    hp = np.zeros(Q * C)
    hp[:L] = h
    # window row m: xx[m D .. m D + L - 1] = x[n - (L - 1) .. n]; reversed, column k holds x[n - k]
    win = np.lib.stride_tricks.sliding_window_view(xx, L)[::D][:M]
    s = np.arange(C)
    rows = np.arange(-(D - 1), D) % C
    y = np.empty((2 * D - 1, M), np.complex128)
    for a in range(0, M, chunk):
        w = np.zeros((min(chunk, M - a), Q * C), np.complex128)
        w[:, :L] = win[a:a + chunk, ::-1]
        v = (w * hp).reshape(-1, Q, C).sum(axis=1)                       # v_s: the taps k = s (mod C)
        m = np.arange(a, a + len(v))
        r = (n0 % C + (m[:, None] * D) - s[None, :]) % C                 # the phase of x[n - s] is its global index mod C
        u = np.zeros_like(v)
        np.put_along_axis(u, r, v, axis=1)
        y[:, a:a + len(v)] = np.fft.fft(u, axis=1)[:, rows].T
    return y
