"""CPU checks of the per-block DC and IQ-imbalance correction (include/rt_ddc.h, include/rt_fbank.h): the float64 restatement
(tests/iq_oracle.py) makes every block proper, leaves a proper block alone but for its DC, suppresses the mirror image of a
synthetic zero-IF capture (pyradiotracking_b200.synth.zero_if_imbalance), and the integer moments the kernels sum are the exact
element sums; the binding declares every new symbol of the headers."""
import os
import re

import numpy as np
import pytest

from pyradiotracking_b200 import synth as S
from pyradiotracking_b200 import wideband as W
from tests import format_oracle as FO
from tests import iq_oracle as IQ

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _noise_and_tones(n, bins, amps, sigma, seed):
    """Complex Gaussian noise plus tones on exact FFT bins of an n-point block (so each tone and its image own one bin)."""
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    x = sigma * (rng.normal(size=n) + 1j * rng.normal(size=n))
    for k, a in zip(bins, amps):
        x += a * np.exp(2j * np.pi * (k * t / n + rng.uniform()))
    return x


def _image_db(y, bins):
    """Power of the mirror bin -k below the tone bin k, per tone (dB, positive = below)."""
    Y = np.abs(np.fft.fft(y)) ** 2
    return [10 * np.log10(Y[k % len(y)] / Y[-k % len(y)]) for k in bins]


def test_every_corrected_block_is_proper():
    rng = np.random.default_rng(3)
    block = 4096
    x = S.zero_if_imbalance(rng.normal(size=5 * block) + 1j * rng.normal(size=5 * block), 1.5, 7.0, 0.1 - 0.05j)
    x[block:2 * block] = np.abs(x[block:2 * block]) + 0.2            # nearly real: |c| close to p, |w| close to 1
    y, ms, ws = IQ.correct(x, block)
    for b in range(5):
        yb = y[b * block:(b + 1) * block]
        assert abs(np.sum(yb * yb)) <= 1e-12 * np.sum(np.abs(yb) ** 2), b
        assert abs(yb.mean()) <= 1e-12 * np.abs(yb).max() * (1 + abs(ws[b]))
        assert abs(ws[b]) <= 1.0
    assert abs(ws[1]) > 0.5 and abs(ws[0]) < 0.2


def test_a_proper_block_only_loses_its_dc():
    # dyadic samples whose deviations come in (d, -d, i d, -i d) quadruples: the mean is exact and sum((x - m)^2) = 0 exactly
    rng = np.random.default_rng(5)
    d = (rng.integers(-100, 100, 256) + 1j * rng.integers(-100, 100, 256)) / 128.0
    m0 = 0.25 - 0.375j
    x = m0 + np.concatenate([d, -d, 1j * d, -1j * d])
    assert np.sum((x - x.mean()) ** 2) == 0
    m, w = IQ.coefficients(x)
    assert m == m0 and w == 0
    assert np.array_equal(IQ.apply(x, m, w), x - m0)
    # and a constant block (p = 0) gets w = 0
    m, w = IQ.coefficients(np.full(64, 0.5 + 0.5j))
    assert w == 0 and m == 0.5 + 0.5j


@pytest.mark.parametrize("gain_db,phase_deg", [(0.5, 3.0), (-0.5, -3.0), (0.5, -3.0)])
def test_the_mirror_image_of_a_flat_imbalance_is_suppressed(gain_db, phase_deg):
    n, bins, amps = 1 << 16, (1000, -3217, 12345), (1.0, 0.5, 0.25)
    x = _noise_and_tones(n, bins, amps, 0.003, seed=11)
    img = S.zero_if_imbalance(x, gain_db, phase_deg, dc=0.05 + 0.02j)
    before = _image_db(img, bins)
    y, ms, ws = IQ.correct(img, n)
    after = _image_db(y, bins)
    # about 28 dB for 0.5 dB / 3 deg without the correction (the "~30 dB" of typical zero-IF receivers) ...
    assert all(25.0 < v < 31.0 for v in before), before
    # ... at least 60 dB with it, and the DC is gone
    assert all(v >= 60.0 for v in after), after
    Y = np.abs(np.fft.fft(y)) ** 2
    assert Y[0] < 1e-6 * Y[bins[0]]
    # w undoes mu x + nu conj(x): the corrected block is (mu + w conj(nu)) x up to the noise, with w = -nu / conj(mu)
    g, phi = 10 ** (gain_db / 20), np.deg2rad(phase_deg)
    mu, nu = (1 + g * np.exp(1j * phi)) / 2, (1 - g * np.exp(-1j * phi)) / 2
    assert abs(ws[0] - (-nu / np.conj(mu))) < 2e-3


@pytest.mark.parametrize("fmt", ["cu8", "ci8", "ci16_le"])
def test_integer_moments_are_the_exact_element_sums(fmt):
    rng = np.random.default_rng(len(fmt))
    block = 3000
    x = S.zero_if_imbalance(0.3 * (rng.normal(size=4 * block) + 1j * rng.normal(size=4 * block)), 0.5, 3.0, 0.05 + 0.1j)
    raw = S.quantise(x, fmt)
    sums = IQ.element_sums(raw, fmt, block)
    dt, full = FO.SAMPLE_FORMATS[fmt]
    e = [int(v) - IQ.ELEMENT_BIAS[fmt] for v in raw.view(dt).tolist()]
    xs = FO.decode_samples(raw, fmt)
    for b, s in enumerate(sums):
        i, q = e[2 * b * block:2 * (b + 1) * block:2], e[2 * b * block + 1:2 * (b + 1) * block:2]
        assert s == (sum(i), sum(q), sum(v * v for v in i), sum(v * v for v in q), sum(a * c for a, c in zip(i, q)))
        # the kernels' float64 form from the sums equals the definition on the decoded samples
        scale = 1.0 / full
        m, w = IQ.coefficients_from_sums(s, block, scale, (-1.0 + 128 * scale) if fmt == "cu8" else 0.0)
        m_ref, w_ref = IQ.coefficients(xs[b * block:(b + 1) * block])
        assert abs(m - m_ref) <= 1e-12 and abs(w - w_ref) <= 1e-9, (b, m, m_ref, w, w_ref)
    # the largest block the correction takes (2^30 samples) keeps every int64 sum exact for every integer format
    assert (1 << 30) * 32768 ** 2 < 1 << 63 and (1 << 30) * 32768 * 32768 < 1 << 63


def test_headers_declare_the_correction_functions_and_the_binding_exports_them():
    for hdr, names in (("rt_ddc.h", W.EXPORTS), ("rt_fbank.h", W.FBANK_EXPORTS)):
        text = open(os.path.join(ROOT, "include", hdr)).read()
        declared = set(re.findall(r"^(?:int|void)\s+(rt_[a-z0-9_]+)\s*\(", text, re.M))
        stem = hdr[:-2]
        assert {f"{stem}_set_iq_correction", f"{stem}_read_iq_correction"} <= declared == set(names)
        assert "w = -c / (p + sqrt(p^2 - |c|^2))" in text
