"""The per-block DC and IQ-imbalance correction of the wideband front ends on the B200 (pytest -m gpu): Channelizer and
FilterBank with the correction on against the float64 oracle of the definition (tests/iq_oracle.py) composed with the front
ends' oracles, the coefficients of the test hook, bit-identity across every way of splitting the same work, switching it off
again, and WidebandAnalyzer.full_band on a synthetic zero-IF ci8 recording whose 25 dB mirror image becomes a Signal without
the correction and disappears with it."""
import datetime

import numpy as np
import pytest

from pyradiotracking_b200 import synth as S
from pyradiotracking_b200 import wideband as W
from tests import ddc_oracle as DO
from tests import fbank_oracle as FBO
from tests import format_oracle as FO
from tests import iq_oracle as IQ
from tests import parity

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

T0 = datetime.datetime(2026, 7, 7, 7, 7, 7)


def _zero_if_input(fmt, n, block, seed, fs=1.0, tones=(0.31, -0.12)):
    """Noise and strong tones through a 0.5 dB / 3 deg zero-IF imbalance, with a DC offset that changes from block to block
    (so every block has its own m and w)."""
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    x = 0.15 * (rng.normal(size=n) + 1j * rng.normal(size=n))
    for f in tones:
        x += 0.25 * np.exp(2j * np.pi * f * t + 1j * rng.uniform(0, 2 * np.pi))
    dc = np.repeat(0.05 * (rng.normal(size=-(-n // block)) + 1j * rng.normal(size=-(-n // block))), block)[:n]
    return S.quantise(S.zero_if_imbalance(x / 1.5, 0.5, 3.0) + dc, fmt)


def _run(front, host):
    out = front.run(host)
    torch.cuda.synchronize()
    return out.cpu().numpy().view(np.complex64)


def _make(kind, fs, block, D, taps=None, fmt="ci16_le", n_inputs=1, bpl=1, iq=True):
    if kind == "ddc":
        offsets = [0.0, -0.3 * fs / 2, fs / 2 - fs / (2 * D), 12_345.6]
        return W.Channelizer(fs, block, offsets, D, taps=taps, sample_format=fmt, n_inputs=n_inputs, blocks_per_launch=bpl,
                             iq_correction=iq)
    return W.FilterBank(fs, block, D, taps=taps, sample_format=fmt, n_inputs=n_inputs, blocks_per_launch=bpl, iq_correction=iq)


def _oracle(front, y, n0=0):
    if isinstance(front, W.FilterBank):
        return FBO.fbank(y, front.taps, front.decimation, n0)
    return DO.ddc(y, front.taps, front.phase_inc.tolist(), front.decimation, n0)


# ---------------------------------------------------------------------------------------------------------------------------
# against the oracle
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["ddc", "fbank"])
@pytest.mark.parametrize("fmt", ["cu8", "ci8", "ci16_le", "cf32_le"])
@pytest.mark.parametrize("D", [4, 8, 64])
@pytest.mark.parametrize("L", ["7", "8D+1"])
@pytest.mark.parametrize("short", [False, True], ids=["block37D", "blockD"])
def test_corrected_outputs_match_the_oracle(kind, fmt, D, L, short):
    fs = 1024 * 10_000
    # blocks of 37 D samples, or of D samples (every CTA span straddles many blocks), 3 calls of `bpl` blocks
    block, bpl = (D, 48) if short else (37 * D, 2)
    n_taps = {"7": 7, "8D+1": 8 * D + 1}[L]
    rng = np.random.default_rng(D * 1000 + n_taps)
    taps = None if L == "8D+1" else rng.normal(0, 1, n_taps) / n_taps
    front = _make(kind, fs, block, D, taps=taps, fmt=fmt, n_inputs=2, bpl=bpl)
    n = 3 * bpl * block
    raw = [_zero_if_input(fmt, n, block, 17 + i) for i in range(2)]
    worst = 0.0
    try:
        got = []
        for k in range(3):
            host = np.stack([r[2 * k * bpl * block:2 * (k + 1) * bpl * block] for r in raw])
            got.append(_run(front, host))
        C = front.n_channels
        for i in range(2):
            x = FO.decode_samples(raw[i], fmt)
            y, ms, ws = IQ.correct(x, block)
            want = _oracle(front, y)
            got_i = np.concatenate([g[i * C:(i + 1) * C] for g in got], axis=1)
            scale = np.abs(front.taps).sum() * np.abs(y).max()
            err = np.abs(got_i.astype(np.complex128) - want).max()
            worst = max(worst, err / scale)
            assert err <= 1e-5 * scale, (i, err, 1e-5 * scale)
            # the hook: m and w of the last call's blocks, equal to the oracle's to fp32 rounding
            for b in range(bpl):
                m, w = front.read_iq_correction(i, b)
                mr, wr = ms[2 * bpl + b], ws[2 * bpl + b]
                assert abs(m - mr) <= 4e-7 * (abs(mr) + np.abs(x).max()), (i, b, m, mr)
                assert abs(w - wr) <= 4e-7 * max(abs(wr), 1e-3), (i, b, w, wr)
    finally:
        front.close()
    print(f"iq[{kind}/{fmt}/D{D}/L{len(front.taps)}/block{block}]: worst |y - y_ref| = {worst:.2e} * sum|h| * max|y|")


# ---------------------------------------------------------------------------------------------------------------------------
# bit-identity across splits of the same work, and switching it off
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["ddc", "fbank"])
@pytest.mark.parametrize("fmt", ["ci8", "cf32_le"])
def test_every_split_of_the_work_gives_the_same_bits(kind, fmt):
    fs, D, block, nb = 2_400_000, 8, 8 * 300 + 8 * 37, 12
    raw = [_zero_if_input(fmt, nb * block, block, 40 + i) for i in range(3)]
    rows = lambda r, b0, n: r[2 * b0 * block:2 * (b0 + n) * block]
    outs = {}
    for B in (1, 2, 3, 4, 6):                  # blocks per call (= blocks_per_launch)
        f = _make(kind, fs, block, D, fmt=fmt, n_inputs=3, bpl=B)
        outs[B] = np.concatenate([_run(f, np.stack([rows(r, b0, B) for r in raw])) for b0 in range(0, nb, B)], axis=1)
        f.close()
    for B in (2, 3, 4, 6):
        assert outs[B].tobytes() == outs[1].tobytes(), B
    C = outs[1].shape[0] // 3
    # one input alone vs the middle input of the batch
    alone = _make(kind, fs, block, D, fmt=fmt)
    y = np.concatenate([_run(alone, rows(raw[1], b, 1)[None]) for b in range(nb)], axis=1)
    assert y.tobytes() == outs[1][C:2 * C].tobytes()
    # reset_input vs a fresh object
    n0 = 3 * 10 ** 10 + 3
    alone.reset_input(0, n0)
    again = np.concatenate([_run(alone, rows(raw[1], b, 1)[None]) for b in range(3)], axis=1)
    fresh = _make(kind, fs, block, D, fmt=fmt)
    fresh.reset_input(0, n0)
    first = np.concatenate([_run(fresh, rows(raw[1], b, 1)[None]) for b in range(3)], axis=1)
    assert again.tobytes() == first.tobytes()
    x = FO.decode_samples(rows(raw[1], 0, 3), fmt)
    want = _oracle(fresh, IQ.correct(x, block)[0], n0)
    assert np.abs(first - want).max() <= 1e-5 * np.abs(fresh.taps).sum() * np.abs(x).max() * 2
    alone.close()
    fresh.close()


@pytest.mark.parametrize("kind", ["ddc", "fbank"])
def test_switching_it_off_again_gives_the_uncorrected_bits(kind):
    fs, D, block, fmt = 2_400_000, 8, 8 * 500, "ci16_le"
    raw = _zero_if_input(fmt, 4 * block, block, 77)[None]
    never = _make(kind, fs, block, D, fmt=fmt, bpl=4, iq=False)
    toggled = _make(kind, fs, block, D, fmt=fmt, bpl=4, iq=True)
    used = _make(kind, fs, block, D, fmt=fmt, bpl=4, iq=True)
    try:
        ref = _run(never, raw)
        toggled.set_iq_correction(False)                # on, then off before any run
        assert _run(toggled, raw).tobytes() == ref.tobytes()
        on = _run(used, raw)                            # a corrected run, then off with a restart: the uncorrected bits again
        assert on.tobytes() != ref.tobytes()
        used.set_iq_correction(False)
        used.reset_input(0, 0)
        assert _run(used, raw).tobytes() == ref.tobytes()
        with pytest.raises(Exception):
            used.read_iq_correction(0, 0)               # the last run did not correct
        # on again: the same as a handle that was on all along, after the same restart
        used.set_iq_correction(True)
        used.reset_input(0, 0)
        assert _run(used, raw).tobytes() == on.tobytes()
    finally:
        never.close()
        toggled.close()
        used.close()


# ---------------------------------------------------------------------------------------------------------------------------
# end to end: a zero-IF ci8 recording with a strong pulsed tag and its 25 dB mirror image
# ---------------------------------------------------------------------------------------------------------------------------
E2E = dict(fs=20_000_000, D=64, block=2_000_000, nb=3, nperseg=256, k0=10, fi=20, sigma=0.012, amp=0.5, thr=-90.0,
           gain_db=0.7, phase_deg=4.5, dc=0.03 + 0.02j)


def _zero_if_tag_capture(p, seed=7):
    """Noise plus one 15 ms tone pulse per block at +f0 (bin fi of channel k0), through a 0.7 dB / 4.5 deg imbalance (a
    25.0 dB image at -f0, in channel -k0) with a DC offset, quantised to ci8 (HackRF).  -> (elements, f0)."""
    rng = np.random.default_rng(seed)
    fs, D, block, nb = p["fs"], p["D"], p["block"], p["nb"]
    f0 = p["k0"] * fs / (2 * D) + p["fi"] * fs / (D * p["nperseg"])
    x = p["sigma"] * (rng.normal(size=nb * block) + 1j * rng.normal(size=nb * block))
    dur = int(0.015 * fs)
    for b in range(nb):
        s0 = b * block + block // 3
        t = np.arange(s0, s0 + dur)
        x[s0:s0 + dur] += p["amp"] * np.exp(2j * np.pi * (f0 / fs * t + rng.uniform()))
    return S.zero_if_capture(x, "ci8", p["gain_db"], p["phase_deg"], p["dc"]), f0


def test_full_band_drops_the_mirror_image_of_a_zero_if_recording():
    p = E2E
    fs, D, block, nb, nperseg = p["fs"], p["D"], p["block"], p["nb"], p["nperseg"]
    raw, f0 = _zero_if_tag_capture(p)
    keys = dict(fft_nperseg=nperseg, fft_window="hamming", signal_min_duration_ms=8.0, signal_max_duration_ms=40.0,
                signal_threshold_dbw=p["thr"], snr_threshold_db=5.0, sdr_callback_length=block)
    c_tag, c_img = p["k0"] + D - 1, -p["k0"] + D - 1
    cf = 150_000_000
    got = {}
    for iq in (False, True):
        wa = W.WidebandAnalyzer.full_band(devices=["rx"], calibration_db=[0.0], sample_rate=fs, center_freq=cf, decimation=D,
                                          sample_format="ci8", iq_correction=iq, **keys)
        try:
            per = []
            for b in range(nb):
                ts = T0 + datetime.timedelta(seconds=b * block / fs)
                (per_channel,) = wa.process_blocks(raw[2 * b * block:2 * (b + 1) * block][None], [ts])
                per.append(per_channel)
        finally:
            wa.close()
        got[iq] = per
    sig = lambda per, c: [s for blk in per for s in blk[c][0]]
    # without the correction the image is a Signal at -f0: the test exercises the problem ...
    img = sig(got[False], c_img)
    assert len(img) == nb and all(abs(s.frequency - (cf - f0)) < 2 * fs / (D * nperseg) for s in img), img
    assert len(sig(got[False], c_tag)) == nb
    # ... with it there is none there, and no Signal anywhere but in the tag's channel (and its overlap neighbours)
    assert sig(got[True], c_img) == []
    assert {c for blk in got[True] for c in range(2 * D - 1) if blk[c][0]} <= {c_tag - 1, c_tag, c_tag + 1}

    # the corrected run's Signals and cells equal the float64 detection oracle on the oracle-corrected channels
    x = FO.decode_samples(raw, "ci8")
    y, _, _ = IQ.correct(x, block)
    L = len(W.default_taps(D))
    ych = FBO.fbank(y, W.default_taps(D), D)
    bc = block // D
    tot = dict(oracle=0, gpu=0, near_threshold_mismatch=0)
    for c in range(2 * D - 1):
        kw = dict(device=f"rx:{c}", calibration_db=0.0, sample_rate=fs // D, center_freq=cf + (c - D + 1) * fs / (2 * D),
                  fft_nperseg=nperseg, fft_window="hamming", signal_min_duration_ms=8.0, signal_max_duration_ms=40.0,
                  signal_threshold_dbw=p["thr"], snr_threshold_db=5.0)
        ora = FO.SampleOracle(parity.oracle_params(kw))
        for b in range(nb):
            ts = T0 + datetime.timedelta(seconds=b * block / fs)
            cts = ts - datetime.timedelta(seconds=(L - 1) / (2 * fs))
            last = ora.last
            _, _, Sg, found, _ = ora.process_samples(ych[c, b * bc:(b + 1) * bc], cts)
            filtered, sigs, gkeys = got[True][b][c]
            st = parity.compare_block(ora.P, Sg, last, found, sigs, gkeys)
            for key in tot:
                tot[key] += st[key]
    print(f"iq e2e: image Signals without the correction {len(img)}, with it 0; parity {tot}")
    assert tot["near_threshold_mismatch"] == 0 and tot["gpu"] == tot["oracle"] >= nb, tot
