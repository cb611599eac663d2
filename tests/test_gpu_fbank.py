"""The polyphase FFT filter bank on the B200 (pytest -m gpu): rt_fbank against the down-converter's float64 oracle
(tests/ddc_oracle.py with the grid's phase increments) for every format, bit-identity across every way of splitting the same
work, agreement with the DDC on the same grid, producer-stream ordering, and WidebandAnalyzer.full_band end to end against the
oracle's channels analysed by the float64 detection oracle, and through replay()."""
import datetime
import json

import numpy as np
import pytest

from pyradiotracking_b200 import wideband as W
from pyradiotracking_b200.replay import replay
from tests import ddc_oracle as DO
from tests import fbank_oracle as FBO
from tests import format_oracle as FO
from tests import parity
from tests.test_gpu_ddc import SPIN_CYCLES, Cai, _keys, _quantise

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

T0 = datetime.datetime(2026, 7, 7, 7, 7, 7)


def _random_input(fmt, n, seed, fs=1.0, tones=(0.31,)):
    """Full-range noise plus strong tones (at the given fractions of fs) and a tone on the +-fs / 2 edge: the error bound is
    relative to the full-band amplitude."""
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    x = 0.25 * (rng.normal(size=n) + 1j * rng.normal(size=n)) + 0.3 * np.exp(1j * np.pi * t)
    for f in tones:
        x += 0.3 * np.exp(2j * np.pi * f * t + 1j * rng.uniform(0, 2 * np.pi))
    return _quantise(x / 2.0, fmt)


def _run(fb, host):
    out = fb.run(host)
    torch.cuda.synchronize()
    return out.cpu().numpy().view(np.complex64)


def _bound(h, x):
    return 1e-5 * np.abs(h).sum() * np.abs(x).max()


# ---------------------------------------------------------------------------------------------------------------------------
# against the oracle
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["cu8", "ci8", "ci16_le", "cf32_le"])
@pytest.mark.parametrize("D", [4, 8, 64, 512])
@pytest.mark.parametrize("L", ["1", "7", "8D+1", "16D+1"])
def test_filter_bank_matches_the_ddc_oracle(fmt, D, L):
    fs = 1024 * 10_000
    block = D * (24 if D == 512 else 150) + (0 if D == 512 else D * 7)
    n_taps = {"1": 1, "7": 7, "8D+1": 8 * D + 1, "16D+1": 16 * D + 1}[L]
    rng = np.random.default_rng(D * 1000 + n_taps)
    taps = None if L == "8D+1" else rng.normal(0, 1, n_taps) / n_taps
    fb = W.FilterBank(fs, block, D, taps=taps, sample_format=fmt, n_inputs=2, blocks_per_launch=2)
    h = fb.taps
    assert len(h) == n_taps and fb.n_channels == 2 * D - 1
    raw = [_random_input(fmt, 3 * 2 * block, 17 + i, tones=(0.31, -0.5 + 1 / (4 * D), 1 / (4 * D))) for i in range(2)]
    worst = 0.0
    try:
        got = []
        for k in range(3):
            host = np.stack([r[k * 4 * block:(k + 1) * 4 * block] for r in raw])
            got.append(_run(fb, host))
        C = fb.n_channels
        for i in range(2):
            x = FO.decode_samples(raw[i], fmt)
            want = DO.ddc(x, h, fb.phase_inc.tolist(), D)
            y = np.concatenate([g[i * C:(i + 1) * C] for g in got], axis=1)
            err = np.abs(y.astype(np.complex128) - want).max()
            worst = max(worst, err / (np.abs(h).sum() * np.abs(x).max()))
            assert err <= _bound(h, x), (i, err, _bound(h, x))
    finally:
        fb.close()
    print(f"fbank[{fmt}/D{D}/L{len(h)}]: worst |y - y_ref| = {worst:.2e} * sum|h| * max|x|")


# ---------------------------------------------------------------------------------------------------------------------------
# bit-identity across splits of the same work
# ---------------------------------------------------------------------------------------------------------------------------
def test_every_split_of_the_work_gives_the_same_bits():
    fs, D, block, fmt, nb = 2_400_000, 8, 8 * 1000 + 8 * 37, "ci16_le", 12
    C = 2 * D - 1
    raw = [_random_input(fmt, nb * block, 40 + i, tones=(0.139,)) for i in range(3)]
    rows = lambda r, b0, n: r[2 * b0 * block:2 * (b0 + n) * block]
    outs = {}
    for B in (1, 2, 3, 4, 6, 12):               # blocks per call (= blocks_per_launch), and one call on the concatenation
        fb = W.FilterBank(fs, block, D, sample_format=fmt, n_inputs=3, blocks_per_launch=B)
        outs[B] = np.concatenate([_run(fb, np.stack([rows(r, b0, B) for r in raw])) for b0 in range(0, nb, B)], axis=1)
        fb.close()
    for B in (2, 3, 4, 6, 12):
        assert outs[B].tobytes() == outs[1].tobytes(), B
    # one input alone vs the middle input of the batch
    alone = W.FilterBank(fs, block, D, sample_format=fmt, n_inputs=1)
    y = np.concatenate([_run(alone, rows(raw[1], b, 1)[None]) for b in range(nb)], axis=1)
    assert y.tobytes() == outs[1][C:2 * C].tobytes()
    # reset_input vs a fresh object; first_sample = 3e10 + 3 (not a multiple of C) vs the oracle at the same n0
    n0 = 3 * 10 ** 10 + 3
    alone.reset_input(0, n0)
    again = np.concatenate([_run(alone, rows(raw[1], b, 1)[None]) for b in range(2)], axis=1)
    fresh = W.FilterBank(fs, block, D, sample_format=fmt, n_inputs=1)
    fresh.reset_input(0, n0)
    first = np.concatenate([_run(fresh, rows(raw[1], b, 1)[None]) for b in range(2)], axis=1)
    assert again.tobytes() == first.tobytes()
    x = FO.decode_samples(rows(raw[1], 0, 2), fmt)
    want = DO.ddc(x, fresh.taps, fresh.phase_inc.tolist(), D, n0=n0)
    assert np.abs(first - want).max() <= _bound(fresh.taps, x)
    # the rotation is not that of n0 = 0
    assert np.abs(first[D] - y[D, :first.shape[1]]).max() > 1e-3
    alone.close()
    fresh.close()


def test_filter_bank_agrees_with_the_ddc_on_the_same_grid():
    fs, D, block = 20_000_000, 64, 64 * 3000
    for fmt in ("ci16_le", "cf32_le"):
        raw = np.stack([_random_input(fmt, 2 * block, 90 + i, tones=(0.2, -0.41)) for i in range(2)])
        fb = W.FilterBank(fs, block, D, sample_format=fmt, n_inputs=2, blocks_per_launch=2)
        ch = W.Channelizer(fs, block, fb.offsets_hz, D, taps=fb.taps, sample_format=fmt, n_inputs=2, blocks_per_launch=2)
        try:
            assert ch.phase_inc.tolist() == fb.phase_inc.tolist()
            a, b = _run(fb, raw), _run(ch, raw)
            x = FO.decode_samples(raw, fmt)
            assert np.abs(a.astype(np.complex128) - b).max() <= _bound(fb.taps, x), fmt
        finally:
            fb.close()
            ch.close()


def test_device_inputs_of_every_kind_equal_host_input():
    fs, D, block = 2_400_000, 8, 8 * 2000
    for fmt in ("cu8", "ci8", "ci16_le", "cf32_le"):
        raw = np.stack([_random_input(fmt, block, 60 + i) for i in range(2)])
        outs = []
        for x in ([raw, torch.from_numpy(raw).cuda()]
                  + ([torch.from_numpy(raw.view(np.complex64)).cuda(), raw.view(np.complex64)] if fmt == "cf32_le" else [])):
            fb = W.FilterBank(fs, block, D, sample_format=fmt, n_inputs=2)
            outs.append(_run(fb, x).tobytes())
            fb.close()
        assert all(o == outs[0] for o in outs), fmt


# ---------------------------------------------------------------------------------------------------------------------------
# producer ordering (the pattern of tests/test_gpu_streams.py: a spin, then the copy of the real input over a poison input)
# ---------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("how", ["current_stream", "cai_stream"])
def test_input_still_being_written_on_a_side_stream(how):
    fs, D, block, fmt = 2_400_000, 8, 8 * 4000, "ci16_le"
    real = _random_input(fmt, block, 71, tones=(0.08,))[None]
    poison = _random_input(fmt, block, 72, tones=(-0.2,))[None]
    fb = W.FilterBank(fs, block, D, sample_format=fmt)
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    try:
        src = torch.from_numpy(real).cuda()
        buf = torch.from_numpy(poison).cuda()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            torch.cuda._sleep(SPIN_CYCLES)
            buf.copy_(src)
        assert not side.query()
        if how == "current_stream":
            with torch.cuda.stream(side):
                out = fb.run(buf)
        else:
            out = fb.run(Cai(buf, stream=side.cuda_stream))
        torch.cuda.synchronize()
        y = out.cpu().numpy().view(np.complex64)
        x = FO.decode_samples(real[0], fmt)
        want = DO.ddc(x, fb.taps, fb.phase_inc.tolist(), D)
        assert np.abs(y - want).max() <= _bound(fb.taps, x)
    finally:
        torch.cuda.synchronize()
        fb.close()


# ---------------------------------------------------------------------------------------------------------------------------
# end to end: wideband captures with tone pulses across the whole band
# ---------------------------------------------------------------------------------------------------------------------------
def _capture_grid(fmt, fs, D, block, nb, nperseg, sigma, amp, seed):
    """Wideband noise and tone pulses of 10-30 ms on the channels' common bin grid (bin width fs / (D nperseg); channel k is
    centred on bin k nperseg / 2), two per channel k and block, each in the central half of channel k and at least 4 bins from
    its centre (the segment-mean detrend removes a tone at DC, as in the reference): one of them sits on the
    upper edge of that half -- in the overlap with channel k + 1 -- on every third channel, and the outermost channels reach to
    fs / 2 - fs / (4 D).  Amplitudes within 3 dB of each other; one pulse straddles the first block boundary.
    -> (elements [nb * 2 * block], pulses [(absolute bin, first sample, last sample + 1)])."""
    rng = np.random.default_rng(seed)
    n = nb * block
    x = sigma * (rng.normal(size=n) + 1j * rng.normal(size=n))
    bw = fs / (D * nperseg)
    half, quarter = nperseg // 2, nperseg // 4
    pulses = []
    for k in range(-(D - 1), D):
        fis = rng.permutation(np.r_[-quarter + 4:-3, 4:quarter - 4])[:2 * nb]         # not at DC: the detrend removes it
        for b in range(nb):
            for p in range(2):
                dur = int(rng.uniform(0.010, 0.030) * fs)
                if b == 0 and p == 0 and k == 0:
                    s0 = block - dur // 2                                      # straddles the first block boundary
                else:
                    lo = b * block + (p * block) // 2
                    s0 = int(rng.integers(lo + block // 40, lo + block // 2 - dur - block // 40))
                fi = int(fis[2 * b + p])
                if p == 1 and k % 3 == 0 and k < D - 1:
                    fi = quarter                                                # the overlap with channel k + 1
                if p == 0 and abs(k) == D - 1:
                    fi = int(np.sign(k)) * (quarter - 2)                        # the outer edge of the band
                g = k * half + fi
                t = np.arange(s0, s0 + dur)
                a = amp * 10 ** (rng.uniform(-1.5, 1.5) / 20)
                x[s0:s0 + dur] += a * np.exp(2j * np.pi * (g * bw / fs * t + rng.uniform()))
                pulses.append((g, s0, s0 + dur))
    return _quantise(x, fmt), pulses


E2E_CASES = [  # fmt, fs, D, block, sigma (normalised), tone amplitude, threshold dBW (the pulses stand clear of the threshold,
    # so each is detected whole in its own channel; a pulse within a few dB of it may break into pieces in the oracle too)
    ("cu8", 2_400_000, 8, 2_400_000, 3 / 127.5, 0.05, -85.0),
    ("ci16_le", 20_000_000, 64, 2_000_000, 0.002, 0.004, -110.0),
    ("cf32_le", 20_000_000, 64, 2_000_000, 0.002, 0.004, -110.0),
]


@pytest.mark.parametrize("fmt,fs,D,block,sigma,amp,thr", E2E_CASES, ids=lambda v: str(v) if isinstance(v, str) else "")
def test_full_band_matches_the_oracle_channels(fmt, fs, D, block, sigma, amp, thr):
    nb, nperseg, cf = 3, 256, 150_000_000
    raw, pulses = _capture_grid(fmt, fs, D, block, nb, nperseg, sigma, amp, seed=fs // 1000 + len(fmt))
    keys = _keys(fs, D, nperseg, thr, block)
    wa = W.WidebandAnalyzer.full_band(devices=["rx"], calibration_db=[0.0], sample_rate=fs, center_freq=cf, decimation=D,
                                      sample_format=fmt, **keys)
    C, L, fs_ch, bc = wa.n_channels, wa.ddc.n_taps, fs // D, block // D
    assert C == 2 * D - 1 and isinstance(wa.ddc, W.FilterBank)
    half, quarter = nperseg // 2, nperseg // 4
    x = FO.decode_samples(raw, fmt)
    ych = FBO.fbank(x, wa.ddc.taps, D)                                           # the oracle's channels, [C, nb * bc]
    spot = [0, D - 1, C - 1]                                                      # ... equal to the DDC oracle's
    want = DO.ddc(x, wa.ddc.taps, wa.ddc.phase_inc[spot].tolist(), D)
    assert np.abs(ych[spot] - want).max() <= 1e-12 * np.abs(wa.ddc.taps).sum() * np.abs(x).max()
    oracles = []
    for c in range(C):
        kw = dict(device=f"rx:{c}", calibration_db=0.0, sample_rate=fs_ch, center_freq=cf + (c - D + 1) * fs / (2 * D),
                  fft_nperseg=nperseg, fft_window="hamming", signal_min_duration_ms=8.0, signal_max_duration_ms=40.0,
                  signal_threshold_dbw=thr, snr_threshold_db=5.0)
        oracles.append(FO.SampleOracle(parity.oracle_params(kw)))
    tot = dict(oracle=0, gpu=0, near_threshold_mismatch=0)
    carried = 0
    found_pulses = set()
    T = bc // nperseg
    delay = (L - 1) / 2                                                           # filter delay, input samples
    try:
        for b in range(nb):
            ts = T0 + datetime.timedelta(seconds=b * block / fs)
            (per_channel,) = wa.process_blocks(raw[2 * b * block:2 * (b + 1) * block][None], [ts])
            cts = ts - datetime.timedelta(seconds=(L - 1) / (2 * fs))
            for c in range(C):
                k = c - (D - 1)
                ora = oracles[c]
                last = ora.last
                _, _, S, found, _ = ora.process_samples(ych[c, b * bc:(b + 1) * bc], cts)
                filtered, sigs, gkeys = per_channel[c]
                st = parity.compare_block(ora.P, S, last, found, sigs, gkeys)
                if c in spot:
                    parity.compare_spectrogram(ora.P, S, wa.channels.engine.read_spectrogram(c),
                                               wa.channels.engine.read_row_means(c), tag=f"fbank/{fmt}/c{c}/b{b}")
                assert all(s.device == f"rx:{c}" for s in sigs)
                for key in tot:
                    tot[key] += st[key]
                carried += sum(1 for g in gkeys if g[1] < 0)
                # the synthesized truth in the columns of this channel block (pulse edges delayed by the filter), at its bin in
                # this channel, modulo nperseg (an alias far outside the channel lands on the same bin)
                truth = []
                for i, (g, s0, s1) in enumerate(pulses):
                    fi = g - k * half
                    if abs(fi) >= nperseg:
                        continue
                    a = (s0 + delay) / D - b * bc
                    e = (s1 + delay) / D - b * bc
                    if e <= 0 or a >= bc:
                        continue
                    truth.append((i, fi % nperseg, int(np.floor(a / nperseg)), min(T, int(np.ceil(e / nperseg))),
                                  a >= 0 and e <= bc and abs(fi) <= quarter))
                near = lambda f, tf: min((f - tf) % nperseg, (tf - f) % nperseg) <= 1
                # every detection lies within a pulse (in a channel's transition band a pulse is attenuated towards the
                # threshold, and noise may split its run into pieces)
                for fi, start, end in gkeys:
                    assert any(near(fi, tf) and max(start, -T) >= max(ts_, -T) - 1 and end <= te + 1
                               for _, tf, ts_, te, _ in truth), (c, b, (fi, start, end), [t for t in truth if near(fi, t[1])])
                for i, tf, ts_, te, central in truth:
                    if central and any(near(fi, tf) and abs(start - ts_) <= 1 and abs(end - te) <= 1 for fi, start, end in gkeys):
                        found_pulses.add(i)
    finally:
        wa.close()
    # every pulse that lies inside a block is found in a channel whose central half holds it
    inside = {i for i, (g, s0, s1) in enumerate(pulses)
              if any(0 <= (s0 + delay) / D - b * bc and (s1 + delay) / D - b * bc <= bc for b in range(nb))}
    print(f"fbank e2e[{fmt}]: {tot}, carried {carried}, pulses found {len(found_pulses & inside)} / {len(inside)}")
    assert inside - found_pulses == set(), sorted(inside - found_pulses)[:10]
    assert tot["near_threshold_mismatch"] == 0 and carried >= 1, (tot, carried)


@pytest.mark.parametrize("B", [1, 4])
def test_replay_through_full_band_equals_submit_collect(tmp_path, B):
    fmt, fs, D, block, nb = "ci16_le", 2_400_000, 8, 480_000, 6
    keys = _keys(fs, D, 256, -85.0, block)
    paths, caps = [], []
    for i in range(2):
        raw, _ = _capture_grid(fmt, fs, D, block, nb, 256, 3 / 32768 * 64, 0.03, seed=500 + i)
        caps.append(raw)
        p = tmp_path / f"wide{i}.sigmf-data"
        np.concatenate([raw, np.zeros(7, raw.dtype)]).tofile(p)
        (tmp_path / f"wide{i}.sigmf-meta").write_text(json.dumps({"global": {"core:datatype": fmt}}))
        paths.append(str(p))
    mk = lambda bpl: W.WidebandAnalyzer.full_band(devices=["a", "b"], calibration_db=[0.0, 1.5], sample_rate=fs,
                                                  center_freq=150_000_000, decimation=D, sample_format=fmt,
                                                  blocks_per_launch=bpl, **keys)
    a, ref = mk(B), mk(1)
    dt = datetime.timedelta(seconds=block / fs)
    try:
        got = {}
        assert replay(paths, a, T0, on_block=lambda k, res: got.__setitem__(k, res)) == nb
        total = 0
        pending = []
        for k in range(nb):                                  # two submissions in flight
            ref.submit(np.stack([c[2 * k * block:2 * (k + 1) * block] for c in caps]))
            pending.append(k)
            if len(pending) == 2 or k == nb - 1:
                while pending:
                    kk = pending.pop(0)
                    want = ref.collect([T0 + kk * dt] * 2)
                    for s in range(2):
                        g, w = got[kk][s], want[s]
                        assert [(x.device, x.ts, x.frequency, x.duration, x.max) for x in g[0]] == \
                               [(x.device, x.ts, x.frequency, x.duration, x.max) for x in w[0]], (kk, s)
                        assert g[1] == w[1]
                        total += len(w[0])
        assert total >= nb * 2
    finally:
        a.close()
        ref.close()
