"""The wideband down-converter on the B200 (pytest -m gpu): rt_ddc against the float64 oracle (tests/ddc_oracle.py) for every
format, bit-identity across every way of splitting the same work, producer-stream ordering, and WidebandAnalyzer end to end
against the oracle's channels analysed by the float64 detection oracle, and through replay()."""
import datetime
import json

import numpy as np
import pytest

from pyradiotracking_b200 import wideband as W
from pyradiotracking_b200.replay import replay
from tests import ddc_oracle as DO
from tests import format_oracle as FO
from tests import parity

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

T0 = datetime.datetime(2026, 7, 7, 7, 7, 7)


def _quantise(x: np.ndarray, fmt: str) -> np.ndarray:
    """Interleaved I,Q elements of `fmt` whose normalised value is (close to) the complex samples x."""
    v = np.ascontiguousarray(x, np.complex128).view(np.float64)
    if fmt == "cu8":
        return np.clip(np.rint(v * 127.5 + 127.5), 0, 255).astype(np.uint8)
    if fmt == "ci8":
        return np.clip(np.rint(v * 128.0), -128, 127).astype(np.int8)
    if fmt == "ci16_le":
        return np.clip(np.rint(v * 32768.0), -32768, 32767).astype("<i2")
    return v.astype("<f4")


def _random_input(fmt, n, seed, tone_hz=0.0, fs=1.0):
    """Full-range noise plus a strong tone: the error bound is relative to the full-band amplitude."""
    rng = np.random.default_rng(seed)
    t = np.arange(n)
    x = 0.25 * (rng.normal(size=n) + 1j * rng.normal(size=n)) + 0.4 * np.exp(2j * np.pi * tone_hz / fs * t)
    return _quantise(x / 1.5, fmt)


def _run(ch, host):
    out = ch.run(host)
    torch.cuda.synchronize()
    return out.cpu().numpy().view(np.complex64)


# ---------------------------------------------------------------------------------------------------------------------------
# against the oracle
# ---------------------------------------------------------------------------------------------------------------------------
ORACLE_CASES = [  # D, L (None: default 8 D + 1)
    (4, None), (4, 7), (8, None), (8, 257), (64, None), (64, 129), (64, 1025),
]


@pytest.mark.parametrize("fmt", ["cu8", "ci8", "ci16_le", "cf32_le"])
@pytest.mark.parametrize("D,L", ORACLE_CASES, ids=str)
def test_ddc_matches_the_oracle(fmt, D, L):
    fs = 64 * 40_000
    block = D * 600
    offsets = [0.0, -0.3 * fs / 2, fs / 2 - fs / (2 * D), -(fs / 2 - fs / (2 * D)), 12_345.6]      # 0, negative, both band edges
    rng = np.random.default_rng(D * 1000 + (L or 0))
    taps = None if L is None else rng.normal(0, 1, L) / L
    ch = W.Channelizer(fs, block, offsets, D, taps=taps, sample_format=fmt, n_inputs=2, blocks_per_launch=2)
    h = ch.taps
    raw = [_random_input(fmt, 3 * 2 * block, 17 + i, tone_hz=0.31 * fs, fs=fs) for i in range(2)]
    worst = 0.0
    try:
        got = []
        for k in range(3):
            host = np.stack([r[k * 4 * block:(k + 1) * 4 * block] for r in raw])
            got.append(_run(ch, host))
        for i in range(2):
            x = FO.decode_samples(raw[i], fmt)
            want = DO.ddc(x, h, ch.phase_inc.tolist(), D)
            y = np.concatenate([g[i * len(offsets):(i + 1) * len(offsets)] for g in got], axis=1)
            bound = 1e-5 * np.abs(h).sum() * np.abs(x).max()
            err = np.abs(y.astype(np.complex128) - want).max()
            worst = max(worst, err / (np.abs(h).sum() * np.abs(x).max()))
            assert err <= bound, (i, err, bound)
    finally:
        ch.close()
    print(f"ddc[{fmt}/D{D}/L{len(h)}]: worst |y - y_ref| = {worst:.2e} * sum|h| * max|x|")


# ---------------------------------------------------------------------------------------------------------------------------
# bit-identity across splits of the same work
# ---------------------------------------------------------------------------------------------------------------------------
def test_every_split_of_the_work_gives_the_same_bits():
    fs, D, block, fmt = 2_400_000, 8, 8 * 1000 + 8 * 37, "ci16_le"
    offsets = [0.0, -600_000.0, 1_000_000.0]
    C = len(offsets)
    raw = [_random_input(fmt, 6 * block, 40 + i, tone_hz=333_333.0, fs=fs) for i in range(3)]
    rows = lambda r, b0, nb: r[2 * b0 * block:2 * (b0 + nb) * block]
    outs = {}
    for B in (1, 2, 3, 6):                                   # blocks = 1, 2, 3 per call, and one call on the concatenation
        ch = W.Channelizer(fs, block, offsets, D, sample_format=fmt, n_inputs=3, blocks_per_launch=B)
        outs[B] = np.concatenate([_run(ch, np.stack([rows(r, b0, B) for r in raw])) for b0 in range(0, 6, B)], axis=1)
        ch.close()
    for B in (2, 3, 6):
        assert outs[B].tobytes() == outs[1].tobytes(), B
    # one input alone vs the middle input of the batch
    alone = W.Channelizer(fs, block, offsets, D, sample_format=fmt, n_inputs=1)
    y = np.concatenate([_run(alone, rows(raw[1], b, 1)[None]) for b in range(6)], axis=1)
    assert y.tobytes() == outs[1][C:2 * C].tobytes()
    # reset_input vs a fresh object; first_sample = 3e10 vs the oracle at the same n0
    n0 = 3 * 10 ** 10
    alone.reset_input(0, n0)
    again = np.concatenate([_run(alone, rows(raw[1], b, 1)[None]) for b in range(2)], axis=1)
    fresh = W.Channelizer(fs, block, offsets, D, sample_format=fmt, n_inputs=1)
    fresh.reset_input(0, n0)
    first = np.concatenate([_run(fresh, rows(raw[1], b, 1)[None]) for b in range(2)], axis=1)
    assert again.tobytes() == first.tobytes()
    x = FO.decode_samples(rows(raw[1], 0, 2), fmt)
    want = DO.ddc(x, fresh.taps, fresh.phase_inc.tolist(), D, n0=n0)
    assert np.abs(first - want).max() <= 1e-5 * np.abs(fresh.taps).sum() * np.abs(x).max()
    # the rotation is not that of n0 = 0 (3e10 * inc is not a multiple of 2^32 here)
    assert np.abs(first[2] - y[2, :first.shape[1]]).max() > 1e-3
    alone.close()
    fresh.close()


def test_device_inputs_of_every_kind_equal_host_input():
    fs, D, block = 2_400_000, 8, 8 * 2000
    for fmt in ("cu8", "ci8", "ci16_le", "cf32_le"):
        raw = np.stack([_random_input(fmt, block, 60 + i, tone_hz=100_000.0, fs=fs) for i in range(2)])
        outs = []
        for x in ([raw, torch.from_numpy(raw).cuda()]
                  + ([torch.from_numpy(raw.view(np.complex64)).cuda(), raw.view(np.complex64)] if fmt == "cf32_le" else [])):
            ch = W.Channelizer(fs, block, [0.0, 300_000.0], D, sample_format=fmt, n_inputs=2)
            outs.append(_run(ch, x).tobytes())
            ch.close()
        assert all(o == outs[0] for o in outs), fmt


# ---------------------------------------------------------------------------------------------------------------------------
# producer ordering (the pattern of tests/test_gpu_streams.py: a spin, then the copy of the real input over a poison input)
# ---------------------------------------------------------------------------------------------------------------------------
SPIN_CYCLES = 100_000_000


class Cai:
    def __init__(self, t, **stream):
        self.t = t
        self.__cuda_array_interface__ = dict(shape=tuple(t.shape), typestr=np.dtype(str(t.dtype)[6:]).str,
                                             data=(t.data_ptr(), False), version=3, strides=None, **stream)


@pytest.mark.parametrize("how", ["current_stream", "cai_stream"])
def test_input_still_being_written_on_a_side_stream(how):
    fs, D, block, fmt = 2_400_000, 8, 8 * 4000, "ci16_le"
    real = _random_input(fmt, block, 71, tone_hz=200_000.0, fs=fs)[None]
    poison = _random_input(fmt, block, 72, tone_hz=-500_000.0, fs=fs)[None]
    ch = W.Channelizer(fs, block, [0.0, 200_000.0], D, sample_format=fmt)
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
                out = ch.run(buf)
        else:
            out = ch.run(Cai(buf, stream=side.cuda_stream))
        torch.cuda.synchronize()
        y = out.cpu().numpy().view(np.complex64)
        x = FO.decode_samples(real[0], fmt)
        want = DO.ddc(x, ch.taps, ch.phase_inc.tolist(), D)
        assert np.abs(y - want).max() <= 1e-5 * np.abs(ch.taps).sum() * np.abs(x).max()
    finally:
        torch.cuda.synchronize()
        ch.close()


# ---------------------------------------------------------------------------------------------------------------------------
# end to end: wideband captures with tone pulses in several channels
# ---------------------------------------------------------------------------------------------------------------------------
def _keys(fs, D, nperseg, thr_dbw, block):
    return dict(fft_nperseg=nperseg, fft_window="hamming", signal_min_duration_ms=8.0, signal_max_duration_ms=40.0,
                signal_threshold_dbw=thr_dbw, snr_threshold_db=5.0, sdr_callback_length=block)


def _capture(fmt, fs, D, block, nb, offsets, nperseg, sigma, amp, seed):
    """Wideband noise and bin-centred tone pulses of 10-30 ms (inside the 8-40 ms limits after the filter's smear): two per
    channel and block, in distinct bins of the central half of the channel, amplitudes within 3 dB of each other (neighbours within 30 dB), one pulse straddling the first block
    boundary.  -> (elements [nb * 2 * block], pulses [(channel, bin, first sample, last sample + 1)])."""
    rng = np.random.default_rng(seed)
    n = nb * block
    x = sigma * (rng.normal(size=n) + 1j * rng.normal(size=n))
    fs_ch = fs // D
    pulses = []
    for c, off in enumerate(offsets):
        bins = rng.permutation(np.r_[4:nperseg // 4 - 4, -nperseg // 4 + 4:-4])[:2 * nb]
        for b in range(nb):
            for p in range(2):
                dur = int(rng.uniform(0.010, 0.030) * fs)
                if b == 0 and p == 0 and c == 0:
                    s0 = block - dur // 2                                      # straddles the first block boundary
                else:
                    lo = b * block + (p * block) // 2
                    s0 = int(rng.integers(lo + block // 40, lo + block // 2 - dur - block // 40))
                fi = int(bins[2 * b + p])
                f = off + fi * fs_ch / nperseg
                t = np.arange(s0, s0 + dur)
                a = amp * 10 ** (rng.uniform(-1.5, 1.5) / 20)
                x[s0:s0 + dur] += a * np.exp(2j * np.pi * (f / fs * t + rng.uniform()))
                pulses.append((c, fi % nperseg, s0, s0 + dur))
    return _quantise(x, fmt), pulses


E2E_CASES = [  # fmt, fs, D, block, offsets, sigma (normalised), tone amplitude, threshold dBW
    ("cu8", 2_400_000, 8, 2_400_000, [0.0, -600_000.0, 300_000.0, 900_000.0], 3 / 127.5, 0.05, -85.0),
    ("ci16_le", 20_000_000, 64, 4_000_000, [-9_843_750.0, -2_500_000.0, 0.0, 312_500.0, 6_100_000.0], 0.002, 0.0025, -110.0),
    ("cf32_le", 20_000_000, 64, 4_000_000, [-5_000_000.0, 156_250.0, 9_843_750.0], 0.002, 0.0025, -110.0),
]


@pytest.mark.parametrize("fmt,fs,D,block,offsets,sigma,amp,thr", E2E_CASES, ids=lambda v: str(v) if isinstance(v, str) else "")
def test_wideband_analyzer_matches_the_oracle_channels(fmt, fs, D, block, offsets, sigma, amp, thr):
    nb, nperseg, cf = 3, 256, 150_000_000
    raw, pulses = _capture(fmt, fs, D, block, nb, offsets, nperseg, sigma, amp, seed=fs // 1000 + len(fmt))
    keys = _keys(fs, D, nperseg, thr, block)
    wa = W.WidebandAnalyzer(devices=["rx"], calibration_db=[0.0], sample_rate=fs, center_freq=cf, offsets_hz=offsets,
                            decimation=D, sample_format=fmt, **keys)
    C, L, fs_ch, bc = len(offsets), wa.ddc.n_taps, fs // D, block // D
    x = FO.decode_samples(raw, fmt)
    ych = DO.ddc(x, wa.ddc.taps, wa.ddc.phase_inc.tolist(), D)                     # the oracle's channels, [C, nb * bc]
    oracles = []
    for c in range(C):
        kw = dict(device=f"rx:{c}", calibration_db=0.0, sample_rate=fs_ch, center_freq=cf + offsets[c], fft_nperseg=nperseg,
                  fft_window="hamming", signal_min_duration_ms=8.0, signal_max_duration_ms=40.0, signal_threshold_dbw=thr,
                  snr_threshold_db=5.0)
        oracles.append(FO.SampleOracle(parity.oracle_params(kw)))
    tot = dict(oracle=0, gpu=0, near_threshold_mismatch=0)
    carried = 0
    T = bc // nperseg
    delay = (L - 1) / 2                                                           # filter delay, input samples
    try:
        for b in range(nb):
            ts = T0 + datetime.timedelta(seconds=b * block / fs)
            (per_channel,) = wa.process_blocks(raw[2 * b * block:2 * (b + 1) * block][None], [ts])
            cts = ts - datetime.timedelta(seconds=(L - 1) / (2 * fs))
            for c in range(C):
                ora = oracles[c]
                last = ora.last
                _, _, S, found, _ = ora.process_samples(ych[c, b * bc:(b + 1) * bc], cts)
                filtered, sigs, gkeys = per_channel[c]
                st = parity.compare_block(ora.P, S, last, found, sigs, gkeys)
                parity.compare_spectrogram(ora.P, S, wa.channels.engine.read_spectrogram(c), wa.channels.engine.read_row_means(c),
                                           tag=f"ddc/{fmt}/c{c}/b{b}")
                assert all(s.device == f"rx:{c}" for s in sigs)
                for k in tot:
                    tot[k] += st[k]
                carried += sum(1 for k in gkeys if k[1] < 0)
                # the synthesized truth, in the columns of this channel block (pulse edges delayed by the filter)
                truth = []
                for pc, fi, s0, s1 in pulses:
                    if pc != c:
                        continue
                    a = (s0 + delay) / D - b * bc
                    e = (s1 + delay) / D - b * bc
                    if e <= 0 or a >= bc:
                        continue
                    truth.append((fi, int(np.floor(a / nperseg)), min(T, int(np.ceil(e / nperseg))), a >= 0 and e <= bc))
                for fi, start, end in gkeys:
                    assert any(abs(fi - tf) <= 1 and abs(max(start, -T) - max(ts_, -T)) <= 1 and abs(end - te) <= 1
                               for tf, ts_, te, _ in truth), (c, b, (fi, start, end), truth)
                for tf, ts_, te, inside in truth:
                    if inside:
                        assert any(abs(fi - tf) <= 1 and abs(start - ts_) <= 1 and abs(end - te) <= 1 for fi, start, end in gkeys), (c, b, tf, ts_, te, gkeys)
    finally:
        wa.close()
    print(f"ddc e2e[{fmt}]: {tot}, carried {carried}")
    assert tot["near_threshold_mismatch"] == 0 and tot["gpu"] >= 2 * C * nb - 2 and carried >= 1, (tot, carried)


@pytest.mark.parametrize("B", [1, 4])
def test_replay_through_the_wideband_analyzer_equals_submit_collect(tmp_path, B):
    fmt, fs, D, block, nb = "ci16_le", 2_400_000, 8, 480_000, 6
    offsets = [0.0, -600_000.0, 450_000.0]
    keys = _keys(fs, D, 256, -85.0, block)
    paths, caps = [], []
    for i in range(2):
        raw, _ = _capture(fmt, fs, D, block, nb, offsets, 256, 3 / 32768 * 64, 0.03, seed=500 + i)
        caps.append(raw)
        p = tmp_path / f"wide{i}.sigmf-data"
        np.concatenate([raw, np.zeros(7, raw.dtype)]).tofile(p)
        (tmp_path / f"wide{i}.sigmf-meta").write_text(json.dumps({"global": {"core:datatype": fmt}}))
        paths.append(str(p))
    mk = lambda bpl: W.WidebandAnalyzer(devices=["a", "b"], calibration_db=[0.0, 1.5], sample_rate=fs, center_freq=150_000_000,
                                        offsets_hz=offsets, decimation=D, sample_format=fmt, blocks_per_launch=bpl, **keys)
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
