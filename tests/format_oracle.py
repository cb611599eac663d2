"""Float64 decoding of the input sample formats for the parity tests, on top of the CPU restatement (oracle/restatement.py),
which reads RTL-SDR bytes only.

TEST INFRASTRUCTURE ONLY, like the restatement: nothing under `pyradiotracking_b200/` imports it.  Normalisation (SigMF datatypes,
include/rt_engine.h): cu8 b / 127.5 - 1 (pyrtlsdr), ci8 v / 128, ci16_le v / 32768, cf32_le x as stored.
"""
import datetime

import numpy as np

from oracle import restatement as R

# SigMF datatype -> (element dtype, full scale): the normalised sample is element / full scale (cu8: pyrtlsdr's b / 127.5 - 1)
SAMPLE_FORMATS = {
    "cu8": (np.dtype(np.uint8), 127.5),
    "ci8": (np.dtype(np.int8), 128.0),
    "ci16_le": (np.dtype("<i2"), 32768.0),
    "cf32_le": (np.dtype("<f4"), 1.0),
}


def decode_samples(raw: np.ndarray, fmt: str) -> np.ndarray:
    """complex128 samples of the interleaved I,Q elements `raw` in the sample format `fmt`, in float64.  `raw` may also be
    the bytes of a recording (uint8 for any format)."""
    if fmt == "cu8":
        return R.bytes_to_iq(np.asarray(raw).view(np.uint8))
    dt, scale = SAMPLE_FORMATS[fmt]
    x = np.ascontiguousarray(raw)
    x = x.view(dt) if x.dtype == np.uint8 else x.astype(dt, copy=False)
    iq = x.astype(np.float64).view(np.complex128)
    if scale != 1.0:
        iq /= scale
    return iq


class SampleOracle(R.OracleAnalyzer):
    """`OracleAnalyzer` that also takes already-decoded complex samples (`decode_samples`)."""

    def process_samples(self, x: np.ndarray, ts_start: datetime.datetime):
        """`process_block` for complex samples: -> (freqs, times, S, detections_before_shadow_filter, detections_after)."""
        P = self.P
        freqs, times, S = R.spectrogram(x, P.sample_rate, P.fft_window, P.fft_nperseg)
        fn = R.extract_sequential if self.sequential else R.extract_runs
        found = fn(P, freqs, times, S, self.last, ts_start)
        kept = R.filter_shadow(found)
        self.last = S
        return freqs, times, S, found, kept
