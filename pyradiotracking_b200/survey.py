"""Band survey: what the band looked like in each analyzed block (include/rt_engine.h, `rt_engine_set_survey`).

The detection keys are chosen against the band: `signal_threshold_dbw` a few dB above each SDR's noise floor, `calibration_db` so
that the floors of a station's SDRs agree, and an interferer is a bin that is above the threshold in most columns of every
block.  With `survey=True` (`BatchAnalyzer`, `WidebandAnalyzer`, `MultiStreamAnalyzer`) the engine computes, next to the scan
and from the same power cells, per analyzer unit and bin the row mean, the peak cell and the number of columns that pass the
scan's predicate; this module turns them into `BandSurvey`s in the units of the Signals of the same block, and stitches the
channels of a full-band analyzer (`WidebandAnalyzer.band_survey`) into one spectrum.
"""
from typing import List, NamedTuple, Sequence

import numpy as np


class BandSurvey(NamedTuple):
    """One analyzer unit's block, bins in ascending frequency (fftshifted)."""
    device: str
    freqs: np.ndarray       # absolute Hz: freqs[fi] + center_freq in float64, equal to Signal.frequency at the same bin
    noise_dbw: np.ndarray   # 10 log10(row mean), uncalibrated, like Signal.noise
    peak_dbw: np.ndarray    # 10 log10(peak cell) - calibration_db, like Signal.max
    occupancy: np.ndarray   # fraction of the block's columns above the detection threshold (the scan's predicate)


def unit_surveys(devices: Sequence[str], bin_freqs: np.ndarray, center_freqs, calibration_db, noise: np.ndarray, peak: np.ndarray,
                 above_cols: np.ndarray, T: int) -> List[BandSurvey]:
    """The `BandSurvey`s of units u = 0, 1, ... from the engine's linear values `[units, nperseg]` in FFT order
    (`Engine.read_survey`): `devices`, `center_freqs` and `calibration_db` give one value per unit, `bin_freqs` is the
    analyzer's `fftfreq(nperseg, 1 / fs)` and `T` its columns per block."""
    shift = lambda x: np.fft.fftshift(x, axes=-1)
    cf = np.asarray(center_freqs)
    freqs = shift(bin_freqs[None, :] + cf.reshape(-1, 1))              # element by element the Signal's freqs[fi] + center_freq
    cal = np.asarray(calibration_db, dtype=np.float64)[:, None]
    with np.errstate(divide="ignore"):
        noise_dbw = shift(10 * np.log10(np.asarray(noise).astype(np.float64)))
        peak_dbw = shift(10 * np.log10(np.asarray(peak).astype(np.float64)) - cal)
    occ = shift(np.asarray(above_cols) / T)
    return [BandSurvey(d, *rows) for d, *rows in zip(devices, freqs, noise_dbw, peak_dbw, occ)]


def stitch(device: str, channels: Sequence[BandSurvey]) -> BandSurvey:
    """One spectrum from the surveys of the channels of a uniform grid spaced half a channel apart, in ascending order (the
    filter bank's): channel c gives the bins of its flat central half, k in [-n/4, n/4) for n bins.  Adjacent pieces are
    n/2 bins apart, so they tile the band without gap or overlap."""
    n = len(channels[0].freqs)
    if n % 4 or any(len(c.freqs) != n for c in channels):
        raise ValueError("channels of one length, a multiple of 4, are needed")
    mid = slice(n // 4, 3 * n // 4)          # fftshifted index n/2 + k
    return BandSurvey(device, *(np.concatenate([c[f][mid] for c in channels]) for f in range(1, len(BandSurvey._fields))))
