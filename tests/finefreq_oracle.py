"""Float64 restatement of the neighbour bins (include/rt_engine.h, rt_engine_set_neighbours) and a generator of pulsed tones at
fractional-bin carriers, shared by the CPU and GPU tests of the fine frequency."""
import numpy as np

from pyradiotracking_b200 import engine as E


def neighbours(S: np.ndarray, last, keys) -> np.ndarray:
    """`NEIGHBOURS_DTYPE` entries of the records `keys` = (fi, start, end) of one unit: S [n, T] is its block's power
    spectrogram (FFT order), `last` the block its carry reaches into (or None).  Sums in float64, like analyze.py:436."""
    n = S.shape[0]
    out = np.zeros(len(keys), dtype=E.NEIGHBOURS_DTYPE)
    for i, (fi, start, end) in enumerate(keys):
        for name, b in (("lo", (fi - 1) % n), ("hi", (fi + 1) % n)):
            data = np.concatenate((last[b][start:], S[b][:end])) if start < 0 else S[b][start:end]
            out[i]["mean_" + name] = np.mean(data.astype(np.float64))
            out[i]["row_mean_" + name] = np.mean(S[b].astype(np.float64))
    return out


def pulse_amplitude(snr_db: float, noise_power: float, window: np.ndarray) -> float:
    """Amplitude of a complex tone whose cells in its own bin (tone at the bin centre) stand `snr_db` above the mean noise cell
    of complex noise of total power `noise_power` (density scaling: the noise cell is noise_power / fs, the tone's
    a^2 (sum w)^2 / (fs sum w^2))."""
    return float(np.sqrt(10 ** (snr_db / 10) * noise_power * np.sum(window ** 2) / np.sum(window) ** 2))


def pulsed_tones(n_samples: int, pulses, sigma: float, rng: np.random.Generator) -> np.ndarray:
    """Complex noise of `sigma` per component plus tones: `pulses` = [(first sample, length, carrier in cycles per sample,
    amplitude)], each with a random phase."""
    x = sigma * (rng.normal(size=n_samples) + 1j * rng.normal(size=n_samples))
    for s0, ln, f, a in pulses:
        t = np.arange(s0, s0 + ln)
        x[s0:s0 + ln] += a * np.exp(2j * np.pi * f * t + 1j * rng.uniform(0, 2 * np.pi))
    return x
