"""Fine frequency on the host (no GPU): the estimator against the exact model, the window rule, synthetic pulses through the
float64 oracle's spectrogram and records, the alignment with the Signals (engine stubbed), replay's regrouping and the wideband
flat-half rule."""
import datetime

import numpy as np
import pytest
import scipy.signal as ss
from scipy.optimize import brentq

from oracle import restatement as R
from pyradiotracking_b200 import engine as E
from pyradiotracking_b200 import replay as RP
from pyradiotracking_b200 import wideband as W
from pyradiotracking_b200.analyze import BatchAnalyzer
from pyradiotracking_b200.finefreq import FineFrequency, fine_frequencies
from tests import finefreq_oracle as FO

# The windows fine_frequency accepts, and the bins next to DC where it gives no estimate (finefreq.py's docstring)
WINDOWS = ["hamming", "hann", "blackman", ("kaiser", 8.0)]
REJECTED = ["boxcar", "flattop", "triang", ("kaiser", 4.0), ("tukey", 0.5)]


def documented_nan_bins(window, n):
    extra = [-2, 2] if window == "hamming" and n >= 256 else []
    return sorted([-1, 0, 1] + extra)


def model_powers(w, k, d):
    """g_{k-1}, g_{k+1} at bin positions k + d (arrays): the detrended, windowed tone through an n-point DFT, in float64."""
    n = len(w)
    m = np.arange(n)
    s = np.exp(2j * np.pi * np.outer(np.asarray(k) + np.asarray(d), m) / n)
    s -= s.mean(axis=1, keepdims=True)
    return [np.abs(np.sum(s * w * np.exp(-2j * np.pi * np.outer(b, m) / n), axis=1)) ** 2 for b in (np.asarray(k) - 1, np.asarray(k) + 1)]


@pytest.mark.parametrize("window", WINDOWS, ids=str)
@pytest.mark.parametrize("n", [16, 256, 4096])
def test_model_powers_are_inverted_in_every_bin(window, n):
    w = ss.get_window(window, n)
    est = FineFrequency(w)
    assert est.nan_bins.tolist() == documented_nan_bins(window, n)
    ds = np.array([-0.93, -0.5, -0.21, 0.0, 0.37, 0.5, 0.88]) if n < 4096 else np.array([-0.71, 0.0, 0.43])
    ks = np.arange(-n // 2, n // 2)
    kk, dd = np.repeat(ks, len(ds)), np.tile(ds, len(ks))
    p_lo, p_hi = model_powers(w, kk, dd)
    got = est.offsets(kk % n, p_lo, p_hi)
    nan = np.isin(kk, est.nan_bins) | (kk == -n // 2) | (kk == n // 2 - 1)
    assert np.all(np.isnan(got[nan]))
    assert np.all(np.abs(got[~nan] - dd[~nan]) <= 1e-6), float(np.nanmax(np.abs(got[~nan] - dd[~nan])))


@pytest.mark.parametrize("window", WINDOWS, ids=str)
def test_the_inversion_agrees_with_a_bracketed_root_finder(window):
    n = 256
    w = ss.get_window(window, n)
    est = FineFrequency(w)
    rng = np.random.default_rng(3)
    k = rng.integers(3, 120, 40) * rng.choice([-1, 1], 40)
    rho = rng.uniform(-3, 3, 40)
    got = est.offsets(k % n, np.ones(40), np.exp(rho))

    def ratio(kv, d):
        lo, hi = model_powers(w, np.array([kv]), np.array([d]))
        return float(np.log(hi[0] / lo[0]))

    for kv, r, g in zip(k, rho, got):
        ref = brentq(lambda d: ratio(kv, d) - r, -1 + 1e-9, 1 - 1e-9, xtol=1e-14)
        assert abs(g - ref) <= 1e-6


@pytest.mark.parametrize("window", REJECTED, ids=str)
def test_windows_without_an_invertible_ratio_are_rejected(window):
    kw = dict(devices=["0"], calibration_db=[0.0], sample_rate=300_000, center_freq=150_150_000, fft_nperseg=256,
              fft_window=window, signal_min_duration_ms=8.0, signal_max_duration_ms=40.0, signal_threshold_dbw=-90.0,
              snr_threshold_db=5.0)
    BatchAnalyzer(**kw)
    with pytest.raises(ValueError):
        BatchAnalyzer(fine_frequency=True, **kw)


def test_noise_and_band_edges_give_no_estimate():
    est = FineFrequency(ss.get_window("hamming", 256))
    got = est.offsets(np.array([40, 40, 40, 128, 127, 129]), np.array([0.0, 1.0, -1.0, 1.0, 1.0, 1.0]),
                      np.array([1.0, 0.0, 1.0, 1.0, 1.0, 1.0]))
    assert np.all(np.isnan(got[:5])) and np.isfinite(got[5])         # fi 129 = k -127: its neighbours stay inside
    # beyond the ratio the window can produce over the bin: blackman's response does not vanish at two bins
    b = FineFrequency(ss.get_window("blackman", 256))
    assert np.isnan(b.offsets(np.array([40]), np.array([1.0]), np.array([1e6]))[0])


# ---------------------------------------------------------------------------------------------------------------------------
# synthetic pulses through the oracle's spectrogram and records
# ---------------------------------------------------------------------------------------------------------------------------
FS, N = 300_000, 256


def simulate(snr_db, seed, n_blocks=4, block=60_000, window="hamming"):
    """Errors (bins) of the estimates of 20 ms pulses at random fractional-bin carriers, found by the oracle's extraction
    (records with their edge columns, carries into the previous block included)."""
    rng = np.random.default_rng(seed)
    win = R.resolve_window(window, N)
    sigma = 0.01
    amp = FO.pulse_amplitude(snr_db, 2 * sigma ** 2, win)
    pulses, truth = [], []
    ln = int(0.02 * FS)
    for b in range(n_blocks):
        bins = rng.choice(np.r_[-120:-8:4, 8:120:4], 6, replace=False)     # at least four bins apart
        for j in range(6):                    # six pulses per block; one straddles the block start
            k, d = int(bins[j]), rng.uniform(-0.5, 0.5)
            s0 = b * block - ln // 2 if (j == 0 and b > 0) else b * block + int(rng.integers(0, block - ln))
            pulses.append((s0, ln, (k + d) / N, amp))
            truth.append((s0, k, d))
    x = FO.pulsed_tones(n_blocks * block, pulses, sigma, rng)
    P = R.Params.make(sample_rate=FS, fft_nperseg=N, fft_window=window,
                      signal_threshold_dbw=10 * np.log10(2 * sigma ** 2 / FS) + 3.0, snr_threshold_db=5.0)
    est = FineFrequency(win)
    errs, last = [], None
    for b in range(n_blocks):
        freqs, times, S = R.spectrogram(x[b * block:(b + 1) * block], FS, window, N)
        found = R.extract_runs(P, freqs, times, S, last, datetime.datetime(2026, 1, 1))
        keys = [d.key() for d in found]
        nb = FO.neighbours(S, last, keys)
        fine = fine_frequencies(est, [d.frequency for d in found], [k[0] for k in keys], nb, FS)
        for s0, k, d in truth:
            c0, c1 = (s0 - b * block) / N, (s0 + ln - b * block) / N       # the pulse in this block's columns
            for det, f in zip(found, fine):
                if det.fi == k % N and det.start < c1 and det.end > c0 and det.start >= c0 - 2 and det.end <= c1 + 2:
                    errs.append((f - det.frequency) / (FS / N) - d)
        last = S
    return np.array(errs)


# bounds measured with this generator (hamming, nperseg 256), 24 pulses per seed: at 20 dB, seeds 1-6, rms 0.016-0.028 bin and
# max 0.037-0.093 bin; at 10 dB, seeds 5-7, rms 0.11-0.14 and max 0.26-0.31 (1-2 pulses without an estimate)
ERR_20DB_MAX, ERR_20DB_RMS = 0.12, 0.035
ERR_10DB_MAX, ERR_10DB_RMS = 0.45, 0.2


@pytest.mark.parametrize("seed", [1, 6])
def test_pulses_at_20_db(seed):
    e = simulate(20.0, seed)
    assert len(e) >= 20 and np.all(np.isfinite(e))
    assert np.max(np.abs(e)) <= ERR_20DB_MAX and np.sqrt(np.mean(e ** 2)) <= ERR_20DB_RMS, (np.max(np.abs(e)), np.sqrt(np.mean(e ** 2)))


@pytest.mark.parametrize("seed", [5, 7])
def test_pulses_at_10_db(seed):
    e = simulate(10.0, seed)
    e = e[np.isfinite(e)]
    assert len(e) >= 10
    assert np.max(np.abs(e)) <= ERR_10DB_MAX and np.sqrt(np.mean(e ** 2)) <= ERR_10DB_RMS, (np.max(np.abs(e)), np.sqrt(np.mean(e ** 2)))


@pytest.mark.parametrize("window", WINDOWS, ids=str)
def test_a_tone_on_every_column_of_its_record_is_exact(window):
    """No noise, the tone on exactly the record's columns: every cell of the record but its leading not-above one holds the
    model power, so P+ / P- is the model ratio."""
    block, d, k = 40 * N, 0.3141, 37
    x = np.zeros(block, complex)
    x[10 * N: 30 * N] = np.exp(2j * np.pi * (k + d) / N * np.arange(20 * N))
    P = R.Params.make(sample_rate=FS, fft_nperseg=N, fft_window=window, signal_threshold_dbw=-120.0, snr_threshold_db=2.0)
    freqs, times, S = R.spectrogram(x, FS, window, N)
    found = R.extract_runs(P, freqs, times, S, None, datetime.datetime(2026, 1, 1))
    det = [f for f in found if f.fi == k]
    assert len(det) == 1 and det[0].key() == (k, 9, 30)
    est = FineFrequency(R.resolve_window(window, N))
    fine = fine_frequencies(est, [det[0].frequency], [k], FO.neighbours(S, None, [det[0].key()]), FS)
    assert abs((fine[0] - det[0].frequency) / (FS / N) - d) <= 1e-6


# ---------------------------------------------------------------------------------------------------------------------------
# alignment with the Signals (engine stubbed)
# ---------------------------------------------------------------------------------------------------------------------------
class _StubEngine:
    def __init__(self, rec, nb):
        self.rec, self.nb = rec, nb

    def fetch(self):
        return self.rec

    def read_neighbours(self):
        return self.nb


def _analyzer(bpl, n_streams=2, **extra):
    return BatchAnalyzer(devices=[f"d{i}" for i in range(n_streams)], calibration_db=[0.0, 1.5][:n_streams], sample_rate=FS,
                         center_freq=150_150_000, fft_nperseg=N, fft_window="hamming", signal_min_duration_ms=8.0,
                         signal_max_duration_ms=40.0, signal_threshold_dbw=-90.0, snr_threshold_db=5.0,
                         sdr_callback_length=FS // 4, blocks_per_launch=bpl, fine_frequency=True, **extra)


def _records(ba, seed):
    """Candidate records of every unit: some fail the duration test (2 or 70 columns), overlapping louder ones shadow others."""
    rng = np.random.default_rng(seed)
    rows = []
    for u in range(ba.n_units):
        for fi in rng.choice(np.r_[5:120, 136:250], 12, replace=False):
            start = int(rng.integers(-20, 200))
            ln = int(rng.choice([2, 20, 30, 70]))
            rows.append((u, fi, start, min(start + ln, ba.plan.T - 1)))
    rec = np.zeros(len(rows), dtype=E.RECORD_DTYPE)
    rec["stream"], rec["fi"], rec["start"], rec["end"] = np.array(rows).T
    rec["max_lin"] = rng.uniform(1e-8, 1e-6, len(rows))
    rec["row_mean"] = rec["mean_lin"] = 1e-9
    rec["std_db"] = 1.0
    rec = rec[np.lexsort((rec["start"], rec["fi"], rec["stream"]))]
    nb = np.zeros(len(rec), dtype=E.NEIGHBOURS_DTYPE)
    nb["mean_lo"], nb["mean_hi"] = 2e-9, 1e-9 + rng.uniform(0.1, 10, len(rec)) * 1e-9    # a distinct estimate per record
    nb["row_mean_lo"] = nb["row_mean_hi"] = 1e-9
    return rec, nb


@pytest.mark.parametrize("bpl", [1, 4])
def test_fine_frequencies_follow_the_signals(bpl):
    ba = _analyzer(bpl)
    rec, nb = _records(ba, bpl)
    ba._engine = _StubEngine(rec, nb)
    expect = fine_frequencies(ba.fine, ba.plan.freqs[rec["fi"]] + 150_150_000, rec["fi"], nb, FS)
    by_key = {(int(r["stream"]), int(r["fi"]), int(r["start"]), int(r["end"])): f for r, f in zip(rec, expect)}
    ts = [datetime.datetime(2026, 1, 1)] * ba.n_streams
    res = ba.collect(ts, with_all=True)
    fine_all, fine_kept = ba.last_fine_frequencies(all_signals=True), ba.last_fine_frequencies()
    n_dropped = n_shadow = 0
    for u, (kept, sigs, keys) in enumerate(res):
        assert len(fine_all[u]) == len(sigs) == len(keys) and len(fine_kept[u]) == len(kept)
        n_dropped += int(np.sum(rec["stream"] == u)) - len(sigs)
        n_shadow += len(sigs) - len(kept)
        for s, k, f in zip(sigs, keys, fine_all[u]):
            assert f == by_key[(u,) + tuple(k)] and abs(f - s.frequency) < FS / N
        pos = [next(i for i, s in enumerate(sigs) if s is k) for k in kept]
        assert np.array_equal(fine_kept[u], fine_all[u][pos])
    assert n_dropped > 0 and n_shadow > 0
    # the plain collect gives the same filtered arrays
    ba.collect(ts)
    assert all(np.array_equal(a, b) for a, b in zip(ba.last_fine_frequencies(), fine_kept))


def test_without_fine_frequency_there_is_nothing_to_read():
    ba = BatchAnalyzer(devices=["0"], calibration_db=[0.0], sample_rate=FS, center_freq=0, fft_nperseg=N, fft_window="hamming",
                       signal_min_duration_ms=8.0, signal_max_duration_ms=40.0, signal_threshold_dbw=-90.0, snr_threshold_db=5.0)
    with pytest.raises(ValueError):
        ba.last_fine_frequencies()


def test_replay_hands_the_fine_frequencies_of_each_block(tmp_path):
    B, n_streams, block = 3, 2, 64

    class Stub:
        sample_rate, block_samples, blocks_per_launch, sample_format = 1000, block, B, "cu8"

        def __init__(self):
            self.n_streams, self.launches = n_streams, 0

        def submit(self, iq):
            self.launches += 1

        def collect(self, ts):
            return [("res", self.launches, u) for u in range(n_streams * B)]

        def last_fine_frequencies(self):
            return [("fine", self.launches, u) for u in range(n_streams * B)]

    paths = []
    for s in range(n_streams):
        p = tmp_path / f"s{s}.cu8"
        np.zeros(2 * block * 7, np.uint8).tofile(p)
        paths.append(str(p))
    got, blocks = {}, []
    n = RP.replay(paths, Stub(), datetime.datetime(2026, 1, 1), on_block=lambda b, r: blocks.append((b, r)),
                  on_fine_frequencies=lambda b, f: got.__setitem__(b, f), pinned=False)
    assert n == 7 and sorted(got) == list(range(7))
    for b, res in blocks:
        assert [x[2] for x in got[b]] == [r[2] for r in res] == [s * B + b % B for s in range(n_streams)]
        assert [x[1] for x in got[b]] == [r[1] for r in res]


# ---------------------------------------------------------------------------------------------------------------------------
# wideband
# ---------------------------------------------------------------------------------------------------------------------------
def test_wideband_keeps_the_estimates_of_the_flat_central_half():
    D, n, n_inputs, bpl, fs, cf = 4, 256, 2, 2, 2_400_000, 150_000_000
    C = 2 * D - 1
    wa = W.WidebandAnalyzer.__new__(W.WidebandAnalyzer)
    wa.ddc = W.FilterBank.__new__(W.FilterBank)
    wa.ddc.taps, wa.sample_rate = W.default_taps(D), fs
    wa.devices = [f"rx{i}" for i in range(n_inputs)]
    wa.n_streams, wa.n_channels, wa.blocks_per_launch = n_inputs, C, bpl
    ch_fs = fs // D
    wa.channels = BatchAnalyzer(devices=[f"{d}:{c}" for d in wa.devices for c in range(C)], calibration_db=[0.0] * (n_inputs * C),
                                sample_rate=ch_fs, center_freq=W.channel_center_freqs(cf, W.grid_offsets(fs, D)) * n_inputs,
                                fft_nperseg=n, fft_window="hamming", signal_min_duration_ms=8.0, signal_max_duration_ms=40.0,
                                signal_threshold_dbw=-90.0, snr_threshold_db=5.0, sdr_callback_length=ch_fs // 4,
                                blocks_per_launch=bpl, fine_frequency=True)
    units = n_inputs * C * bpl
    fis = np.array([3, 40, 63, 64, 100, 127, 128, 150, 192, 193, 250])        # k = 3 ... -6: both sides of +-n/4
    rec = np.zeros(units * len(fis), dtype=E.RECORD_DTYPE)
    rec["stream"] = np.repeat(np.arange(units), len(fis))
    rec["fi"] = np.tile(fis, units)
    rec["start"], rec["end"] = 10, 30
    rec["max_lin"], rec["row_mean"], rec["mean_lin"], rec["std_db"] = 1e-6, 1e-9, 1e-8, 1.0
    nb = np.zeros(len(rec), dtype=E.NEIGHBOURS_DTYPE)
    nb["mean_lo"], nb["mean_hi"], nb["row_mean_lo"], nb["row_mean_hi"] = 2e-9, 4e-9, 1e-9, 1e-9
    wa.channels._engine = _StubEngine(rec, nb)
    wa._held = [None]
    ts = [datetime.datetime(2026, 1, 1)] * n_inputs
    res = wa.collect(ts, with_all=True)
    got = wa.last_fine_frequencies(all_signals=True)
    row = float(np.float32(1e-9))
    d = wa.channels.fine.offsets(fis, np.full(len(fis), 2e-9 - row), np.full(len(fis), 4e-9 - row))
    k = np.where(fis >= n // 2, fis - n, fis)
    half = (k >= -n // 4) & (k < n // 4)
    assert len(got) == n_inputs * bpl
    for u, per in enumerate(res):
        sigs = [s for _, all_sigs, _ in per for s in all_sigs]
        assert len(got[u]) == len(sigs) == C * len(fis)
        for c in range(C):
            f = got[u][c * len(fis):(c + 1) * len(fis)]
            fr = np.array([s.frequency for s in sigs[c * len(fis):(c + 1) * len(fis)]])
            assert np.all(np.isnan(f[~half])) and np.array_equal(np.isnan(f[half]), np.isnan(d[half]))
            ok = half & ~np.isnan(d)
            assert np.allclose(f[ok] - fr[ok], d[ok] * ch_fs / n, rtol=0, atol=1e-6)    # at the channel rate fs / D
            assert np.all(np.abs(fr - (cf + W.grid_offsets(fs, D)[c] + k * ch_fs / n)) < 1e-6)


@pytest.mark.parametrize("D", [4, 8, 64])
def test_default_taps_are_flat_over_the_neighbours_of_the_central_half(D):
    """A tone passes the channel filter as a tone, so its estimate does not depend on the filter; what the estimator needs is
    that the noise floor it subtracts, and the pulse edges, see no tilt between bins k - 1 and k + 1.  Over k in
    [-n/4 - 1, n/4] the default taps vary by at most 0.078 dB at nperseg 256 (0.071 dB at 1024), and two bins apart by at
    most 0.0184 dB."""
    h = W.default_taps(D)
    for n, ripple, pair in ((256, 0.078, 0.0184), (1024, 0.071, 0.0046)):
        k = np.arange(-n // 4 - 1, n // 4 + 1)
        H = np.abs(np.exp(-2j * np.pi * np.outer(k / (n * D), np.arange(len(h)))) @ h) ** 2   # power gain at the bin centres
        db = 10 * np.log10(H)
        assert db.max() - db.min() <= ripple and np.max(np.abs(db[2:] - db[:-2])) <= pair
