"""Deterministic synthetic RTL-SDR captures (uint8 interleaved I,Q,I,Q...).

The reference ships no recorded IQ and no fake SDR backend (SURVEY.md §4), so
every parity test and benchmark in this repo runs on captures made here.  The
recipe follows SURVEY.md §8(d): Gaussian receiver noise of `sigma` LSB per
component plus complex tone bursts `A*exp(2*pi*j*f*t)`, quantised the way an
RTL-SDR delivers them: `clip(round(x + 127.5), 0, 255)`.  Stream `s` of
workload `c` is seeded `1000*c + s` with `numpy.random.default_rng`.
"""
from dataclasses import dataclass, field, replace
from typing import List, Optional, Sequence, Tuple

import numpy as np


@dataclass(frozen=True)
class Workload:
    """One BASELINE.json configuration (sizes per SURVEY.md §8a)."""

    config_id: int
    name: str
    sample_rate: int
    block_samples: int
    nperseg: int = 256
    n_streams: int = 1
    n_blocks: int = 4
    sigma_lsb: float = 1.0
    pulses_per_block: Tuple[int, int] = (5, 5)
    pulse_ms: Tuple[float, float] = (20.0, 20.0)
    amp_lsb: Tuple[float, float] = (6.0, 20.0)
    # used when amp_lsb == (0, 0): peak cell power in dB relative to max(thr, snr*noise density)
    amp_db_over_thr: Tuple[float, float] = (-1.0, 1.0)
    # extra bursts of an exact number of spectrogram columns (duration-test boundaries)
    exact_cols: Tuple[int, ...] = ()
    straddle: bool = True
    center_freq: int = 150_150_000
    signal_threshold_dbw: float = -90.0
    snr_threshold_db: float = 5.0
    signal_min_duration_ms: float = 8.0
    signal_max_duration_ms: float = 40.0

    @property
    def block_bytes(self) -> int:
        return 2 * self.block_samples


# BASELINE.json `configs`, in order.  configs[1] is the one the metric is quoted on.
C1 = Workload(1, "c1-single-300k", 300_000, 300_000, n_blocks=10, sigma_lsb=1.0)
C2 = Workload(
    2, "c2-64x2.4M", 2_400_000, 2_400_000, n_streams=64, n_blocks=4, sigma_lsb=2.8,
    pulses_per_block=(5, 20), pulse_ms=(8.0, 40.0), exact_cols=(75, 375),
)
C3A = Workload(3, "c3a-20M-n1024", 20_000_000, 20_000_000, nperseg=1024, n_blocks=2, sigma_lsb=8.0,
               pulses_per_block=(20, 20), pulse_ms=(8.0, 40.0), amp_lsb=(20.0, 60.0))
C3B = replace(C3A, name="c3b-20M-n4096", nperseg=4096)
C4 = Workload(4, "c4-replay-512x300k", 300_000, 300_000, n_streams=512, n_blocks=60, sigma_lsb=1.0)
C5 = Workload(5, "c5-dense-300k", 300_000, 300_000, n_blocks=3, sigma_lsb=1.0,
              pulses_per_block=(1000, 1000), pulse_ms=(8.0, 40.0), amp_lsb=(0.0, 0.0))
C5B = replace(C5, name="c5-dense-2.4M", sample_rate=2_400_000, block_samples=2_400_000, sigma_lsb=2.8)
# same tag density, bursts 6-14 dB over the threshold: ~1000 detections per block for the shadow filter
C5L = replace(C5, name="c5-dense-loud-300k", amp_db_over_thr=(6.0, 14.0))

WORKLOADS = {w.name: w for w in (C1, C2, C3A, C3B, C4, C5, C5B, C5L)}


def near_threshold_amp(w: Workload, rng: np.random.Generator, n: int) -> np.ndarray:
    """Tone amplitudes [LSB] whose peak spectrogram cell lands `amp_db_over_thr` dB from
    the effective detection threshold max(thr, snr*noise_density) (config 5: +-1 dB)."""
    # Hamming coherent gain 0.54, sum(w^2)/n = 0.3974 (periodic, n >= 64).
    noise_density = 2.0 * (w.sigma_lsb / 127.5) ** 2 / w.sample_rate
    thr = max(10 ** (w.signal_threshold_dbw / 10), 10 ** (w.snr_threshold_db / 10) * noise_density)
    # bin-centred tone: S = (A/127.5)^2 * (0.54 n)^2 / (fs * 0.3974 n)
    gain = (0.54 * w.nperseg) ** 2 / (w.sample_rate * 0.3974 * w.nperseg) / 127.5 ** 2
    a0 = np.sqrt(thr / gain)
    return a0 * 10 ** (rng.uniform(w.amp_db_over_thr[0], w.amp_db_over_thr[1], n) / 20.0)


def make_stream(w: Workload, stream: int = 0, n_blocks: Optional[int] = None, seed: Optional[int] = None) -> np.ndarray:
    """uint8 array `[n_blocks, 2*block_samples]` for one stream of workload `w`.

    Bursts are laid on the continuous timeline so some cross block boundaries
    (the reference re-finds those from the next block, analyze.py:383-398).
    """
    iq = _signal_lsb(w, stream, n_blocks, seed)
    iq += np.float32(127.5)
    np.rint(iq, out=iq)
    np.clip(iq, 0, 255, out=iq)
    return iq.astype(np.uint8).reshape(iq.shape[0] // w.block_samples, 2 * w.block_samples)


def make_stream_format(w: Workload, fmt: str, stream: int = 0, n_blocks: Optional[int] = None, seed: Optional[int] = None) -> np.ndarray:
    """The signal of `make_stream` (noise and bursts in units of 1/127.5) quantised to the sample format `fmt` (a SigMF datatype):
    `[n_blocks, 2*block_samples]` elements whose normalised samples (cu8 b / 127.5 - 1, ci8 v / 128, ci16_le v / 32768,
    cf32_le x) approximate the same complex signal.  cu8 is `make_stream` itself."""
    if fmt == "cu8":
        return make_stream(w, stream, n_blocks, seed)
    x = _signal_lsb(w, stream, n_blocks, seed).astype(np.float64) / 127.5
    if fmt == "ci8":
        q = np.clip(np.rint(x * 128.0), -128, 127).astype(np.int8)
    elif fmt == "ci16_le":
        q = np.clip(np.rint(x * 32768.0), -32768, 32767).astype("<i2")
    elif fmt == "cf32_le":
        q = x.astype("<f4")
    else:
        raise ValueError(f"unknown sample format {fmt!r}")
    return q.reshape(q.shape[0] // w.block_samples, 2 * w.block_samples)


def _signal_lsb(w: Workload, stream: int, n_blocks: Optional[int], seed: Optional[int]) -> np.ndarray:
    """float32 `[n_blocks * block_samples, 2]`: receiver noise plus bursts in 8-bit LSB, before the offset and rounding."""
    nb = w.n_blocks if n_blocks is None else n_blocks
    N = w.block_samples
    M = nb * N
    rng = np.random.default_rng(1000 * w.config_id + stream if seed is None else seed)
    iq = rng.standard_normal((M, 2), dtype=np.float32)
    iq *= np.float32(w.sigma_lsb)

    col = w.nperseg  # samples per spectrogram column
    bursts: List[Tuple[int, int, float, float, float]] = []  # start, length, amp, freq/fs, phase
    for b in range(nb):
        k = int(rng.integers(w.pulses_per_block[0], w.pulses_per_block[1] + 1))
        starts = rng.uniform(0.05, 0.9, k) * N + b * N
        durs = rng.uniform(w.pulse_ms[0], w.pulse_ms[1], k) * 1e-3 * w.sample_rate
        if w.amp_lsb[1] > 0:
            amps = rng.uniform(w.amp_lsb[0], w.amp_lsb[1], k)
        else:
            amps = near_threshold_amp(w, rng, k)
        fr = rng.uniform(-0.45, 0.45, k)
        ph = rng.uniform(0, 2 * np.pi, k)
        for i in range(k):
            bursts.append((int(starts[i]), int(durs[i]), float(amps[i]), float(fr[i]), float(ph[i])))
        for nc in w.exact_cols:
            # column-aligned burst spanning exactly `nc` spectrogram columns
            c0 = int(rng.integers(10, N // col - nc - 10))
            bursts.append((b * N + c0 * col, nc * col, float(rng.uniform(*w.amp_lsb)) if w.amp_lsb[1] > 0 else 10.0,
                           float(rng.uniform(-0.45, 0.45)), 0.0))
        if w.straddle and b + 1 < nb:
            L = int(0.5 * (w.pulse_ms[0] + w.pulse_ms[1]) * 1e-3 * w.sample_rate)
            s0 = (b + 1) * N - int(rng.uniform(0.2, 0.8) * L)
            bursts.append((s0, L, float(max(w.amp_lsb[1], 10.0)), float(rng.uniform(-0.45, 0.45)), 0.0))

    for s0, L, a, f, ph in bursts:
        s0 = max(0, s0)
        e0 = min(M, s0 + L)
        if e0 <= s0:
            continue
        n = np.arange(e0 - s0, dtype=np.float64)
        arg = 2 * np.pi * f * n + ph
        iq[s0:e0, 0] += (a * np.cos(arg)).astype(np.float32)
        iq[s0:e0, 1] += (a * np.sin(arg)).astype(np.float32)
    return iq


def make_batch(w: Workload, streams: Sequence[int], n_blocks: Optional[int] = None) -> np.ndarray:
    """uint8 `[n_blocks, len(streams), 2*block_samples]` (block-major: one engine call per block)."""
    nb = w.n_blocks if n_blocks is None else n_blocks
    out = np.empty((nb, len(streams), 2 * w.block_samples), dtype=np.uint8)
    for i, s in enumerate(streams):
        out[:, i, :] = make_stream(w, s, nb)
    return out


def bytes_to_iq(u8: np.ndarray) -> np.ndarray:
    """The uint8 -> complex128 conversion pyrtlsdr performs before handing samples to
    the callback registered at analyze.py:157 (`packed_bytes_to_iq`: bytes as
    float64 pairs viewed as complex128, `/= 127.5`, `-= (1+1j)`).  pyrtlsdr is
    not vendored in the reference (requirements.txt:1); this restates it."""
    iq = np.ascontiguousarray(u8, dtype=np.uint8).astype(np.float64).view(np.complex128)
    iq /= 127.5
    iq -= 1 + 1j
    return iq


def quantise(x: np.ndarray, fmt: str) -> np.ndarray:
    """Interleaved I,Q elements of the sample format `fmt` (cu8, ci8, ci16_le, cf32_le) whose normalised value is (close to)
    the complex samples x: rounded and clipped to the format's range."""
    v = np.ascontiguousarray(x, np.complex128).view(np.float64)
    if fmt == "cu8":
        return np.clip(np.rint(v * 127.5 + 127.5), 0, 255).astype(np.uint8)
    if fmt == "ci8":
        return np.clip(np.rint(v * 128.0), -128, 127).astype(np.int8)
    if fmt == "ci16_le":
        return np.clip(np.rint(v * 32768.0), -32768, 32767).astype("<i2")
    if fmt == "cf32_le":
        return v.astype("<f4")
    raise ValueError(f"unknown sample format {fmt}")


def zero_if_imbalance(x: np.ndarray, gain_db: float = 0.0, phase_deg: float = 0.0, dc: complex = 0j) -> np.ndarray:
    """What a zero-IF receiver with unequal I and Q paths makes of the complex baseband x: I' = Re x, Q' = g (Im x cos phi +
    Re x sin phi) with g = 10^(gain_db / 20), plus a DC offset.  That is mu x + nu conj(x) + dc with mu = (1 + g e^(i phi)) / 2
    and nu = (1 - g e^(-i phi)) / 2, so a signal at +f leaves a mirror image at -f |mu|^2 / |nu|^2 below it (0.5 dB / 3 deg:
    28 dB; 1 dB / 6 deg: 22 dB)."""
    x = np.asarray(x, np.complex128)
    g, phi = 10.0 ** (gain_db / 20.0), np.deg2rad(phase_deg)
    return x.real + 1j * g * (x.imag * np.cos(phi) + x.real * np.sin(phi)) + dc


def zero_if_capture(x: np.ndarray, fmt: str, gain_db: float = 0.0, phase_deg: float = 0.0, dc: complex = 0j) -> np.ndarray:
    """A synthetic zero-IF recording: `zero_if_imbalance` of x, quantised to `fmt` (ci8 is what a HackRF writes)."""
    return quantise(zero_if_imbalance(x, gain_db, phase_deg, dc), fmt)
