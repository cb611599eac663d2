"""Fine frequency on the B200 (pytest -m gpu): include/rt_engine.h, rt_engine_set_neighbours.

  the neighbour means against the GPU's own cells of this launch and the previous one, and against the float64 oracle, on every
  spectrogram kernel and layout, every sample format, blocks_per_launch 1 and 4, with records carried from the previous launch
  and from the previous unit, and after reset_stream; the estimates against the oracle's and against the true carriers
  records byte-identical with the feature on and off at configs[1] size, also with the survey
  the stream contract: identical bits run to run and alone or in a batch, overflow, a read after an unrefined launch, switching off
  full_band: one estimate per pulse outside the documented DC zones, and the DDC's estimates equal to the filter bank's
"""
import datetime

import numpy as np
import pytest

from oracle import restatement as R
from pyradiotracking_b200 import engine as E
from pyradiotracking_b200 import synth
from pyradiotracking_b200 import wideband as W
from pyradiotracking_b200.analyze import BatchAnalyzer
from pyradiotracking_b200.finefreq import FineFrequency
from tests import finefreq_oracle as FO
from tests import format_oracle as FMT
from tests import parity
from tests.test_fine_frequency import ERR_20DB_MAX

pytestmark = pytest.mark.gpu

T0 = datetime.datetime(2026, 9, 9, 9, 9, 9)
SIGMA = {"cu8": 4 / 127.5, "ci8": 4 / 128, "ci16_le": 0.01, "cf32_le": 0.01}


def _kw(fs, block, nperseg, window, sigma):
    return dict(device="0", calibration_db=0.0, sample_rate=fs, center_freq=150_150_000, fft_nperseg=nperseg, fft_window=window,
                signal_min_duration_ms=8.0, signal_max_duration_ms=40.0,
                signal_threshold_dbw=float(10 * np.log10(2 * sigma ** 2 / fs) + 3.0), snr_threshold_db=5.0, sdr_callback_length=block)


def _capture(fmt, fs, block, nperseg, nb, window, seed, snr_db=20.0):
    """nb blocks of `fmt`: noise and 20 ms tone pulses at fractional-bin carriers, at least four bins apart; one pulse straddles
    every block boundary, so that records carry into the previous block.  -> (raw [nb, 2 block], [(first sample, bin, offset)])"""
    rng = np.random.default_rng(seed)
    win = R.resolve_window(window, nperseg)
    sigma = SIGMA[fmt]
    amp = FO.pulse_amplitude(snr_db, 2 * sigma ** 2, win)
    ln = int(0.02 * fs)
    pulses, truth = [], []
    for b in range(nb):
        lim = nperseg // 2 - 8
        bins = rng.choice(np.r_[-lim:-8:4, 8:lim:4], 4, replace=False)
        for j, k in enumerate(bins):
            s0 = b * block - ln // 2 if (j == 0 and b > 0) else b * block + int(rng.integers(0, block - ln))
            d = rng.uniform(-0.5, 0.5)
            pulses.append((s0, ln, (k + d) / nperseg, amp))
            truth.append((s0, int(k), d))
    x = FO.pulsed_tones(nb * block, pulses, sigma, rng)
    return synth.quantise(x, fmt).reshape(nb, -1), truth


CASES = [  # fmt, nperseg, fs, block, impl, blocks per launch, window
    ("cu8", 256, 300_000, 150_000, E.FFT_GENERIC, 1, "hamming"),       # LINEAR
    ("cu8", 256, 300_000, 150_000, E.FFT_AUTO, 1, "hamming"),          # register kernel, PERM
    ("ci8", 256, 300_000, 150_000, E.FFT_TC256, 1, "hamming"),         # tensor-core kernel, TILE, power scale
    ("ci8", 1024, 2_400_000, 600_000, E.FFT_AUTO, 1, "hann"),          # radix-16
    ("cu8", 4096, 2_400_000, 1_200_000, E.FFT_AUTO, 1, "hann"),        # radix-16
    ("ci16_le", 256, 300_000, 150_000, E.FFT_AUTO, 1, "blackman"),     # generic
    ("cf32_le", 2048, 2_400_000, 1_200_000, E.FFT_AUTO, 1, ("kaiser", 8.0)),
    ("cu8", 256, 300_000, 75_104, E.FFT_AUTO, 4, "hamming"),           # register kernel, ragged blocks
    ("ci8", 256, 300_000, 75_104, E.FFT_AUTO, 4, "hann"),              # register kernel, ragged blocks
    ("ci16_le", 1024, 2_400_000, 600_100, E.FFT_AUTO, 4, "hann"),      # generic, ragged
]


@pytest.mark.parametrize("fmt,nperseg,fs,block,impl,bpl,window", CASES, ids=lambda v: str(v))
def test_neighbours_and_estimates_match_the_cells_and_the_oracle(fmt, nperseg, fs, block, impl, bpl, window):
    launches = 3
    raw, truth = _capture(fmt, fs, block, nperseg, launches * bpl + bpl, window, seed=nperseg + bpl)
    kw = _kw(fs, block, nperseg, window, SIGMA[fmt])
    P = parity.oracle_params(kw)
    ba = BatchAnalyzer(**parity.batch_kwargs(kw, fft_impl=impl, sample_format=fmt, blocks_per_launch=bpl, fine_frequency=True))
    est = FineFrequency(R.resolve_window(window, nperseg))
    T = block // nperseg
    counts = {"carry_launch": 0, "carry_unit": 0, "compared": 0, "truth": 0}
    worst = 0.0
    try:
        eng = ba.engine
        prev32 = prev64 = None                          # the last unit of the previous launch (GPU cells, oracle)
        for k in range(launches + 1):
            if k == launches:                            # one more launch after forgetting the carry
                eng.reset_stream(0)
                prev32 = prev64 = None
            rec = eng.process(raw[k * bpl:(k + 1) * bpl].reshape(1, -1))
            nb = eng.read_neighbours()
            assert len(nb) == len(rec)
            S32 = [eng.read_spectrogram(u).T.astype(np.float64) for u in range(bpl)]
            S64 = [R.spectrogram(FMT.decode_samples(raw[k * bpl + u], fmt), fs, P.fft_window, nperseg)[2] for u in range(bpl)]
            for u in range(bpl):
                sel = rec["stream"] == u
                keys = list(zip(rec["fi"][sel].tolist(), rec["start"][sel].tolist(), rec["end"][sel].tolist()))
                last32 = prev32 if u == 0 else S32[u - 1]
                last64 = prev64 if u == 0 else S64[u - 1]
                carried = rec["start"][sel] < 0
                counts["carry_launch" if u == 0 else "carry_unit"] += int(carried.sum())
                if k == launches and u == 0:
                    assert not carried.any()                # reset_stream: no carry from the previous launch
                got = nb[sel]
                own = FO.neighbours(S32[u], last32, keys)   # float64 sums of the GPU's own fp32 cells
                for f in ("mean_lo", "mean_hi"):
                    assert np.all(np.abs(got[f] - own[f]) <= 1e-12 * own[f]), f
                rm = eng.read_row_means(u)
                lo, hi = (rec["fi"][sel] - 1) % nperseg, (rec["fi"][sel] + 1) % nperseg
                assert np.array_equal(got["row_mean_lo"], rm[lo]) and np.array_equal(got["row_mean_hi"], rm[hi])
                ora = FO.neighbours(S64[u], last64, keys)
                for f in ("mean_lo", "mean_hi", "row_mean_lo", "row_mean_hi"):
                    rel = np.abs(got[f] - ora[f]) / ora[f]
                    assert np.all(rel <= parity.POWER_RTOL), (f, float(rel.max()))
                # estimates: against the oracle's estimator on the same records (neighbours 3 dB above their floor, runs not
                # near a threshold), and against the true carriers
                g = est.offsets(rec["fi"][sel], got["mean_lo"] - got["row_mean_lo"], got["mean_hi"] - got["row_mean_hi"])
                o = est.offsets(rec["fi"][sel], ora["mean_lo"] - ora["row_mean_lo"], ora["mean_hi"] - ora["row_mean_hi"])
                strong = (ora["mean_lo"] > 2 * ora["row_mean_lo"]) & (ora["mean_hi"] > 2 * ora["row_mean_hi"])
                for i, key in enumerate(keys):
                    if strong[i] and not parity.near_threshold(P, S64[u], last64, key) and np.isfinite(o[i]):
                        assert abs(g[i] - o[i]) <= 1e-4, (key, g[i], o[i])
                        counts["compared"] += 1
                b0 = (k * bpl + u) * block
                for s0, kk, d in (truth if nperseg == 256 else []):      # the geometry the CPU bound was pinned at
                    c0, c1 = (s0 - b0) / nperseg, (s0 + int(0.02 * fs) - b0) / nperseg
                    for i, (fi, st, en) in enumerate(keys):
                        if fi == kk % nperseg and st < c1 and en > c0 and st >= c0 - 2 and en <= c1 + 2 and c0 >= -1 and c1 <= T + 1:
                            if np.isfinite(g[i]):
                                worst = max(worst, abs(g[i] - d))
                                counts["truth"] += 1
            prev32, prev64 = S32[-1], S64[-1]
    finally:
        ba.close()
    assert counts["compared"] > 0 and counts["carry_launch"] > 0 and (nperseg != 256 or counts["truth"] >= 4), counts
    if bpl > 1:
        assert counts["carry_unit"] > 0, counts
    assert worst <= ERR_20DB_MAX, worst


def _c2_analyzer(fine, survey=False, **extra):
    w = synth.C2
    return BatchAnalyzer(devices=[str(i) for i in range(w.n_streams)], calibration_db=[0.0] * w.n_streams, sample_rate=w.sample_rate,
                         center_freq=w.center_freq, fft_nperseg=w.nperseg, fft_window="hamming",
                         signal_min_duration_ms=w.signal_min_duration_ms, signal_max_duration_ms=w.signal_max_duration_ms,
                         signal_threshold_dbw=w.signal_threshold_dbw, snr_threshold_db=w.snr_threshold_db,
                         sdr_callback_length=w.block_samples, survey=survey, fine_frequency=fine, **extra)


def test_records_of_configs1_are_unchanged():
    w = synth.C2
    data = synth.make_batch(w, range(w.n_streams), 2)
    recs = {}
    for fine, survey in ((False, False), (True, False), (True, True)):
        ba = _c2_analyzer(fine, survey)
        try:
            eng = ba.engine
            eng.launch(data[0])
            eng.launch(data[1])                    # two launches in flight, as the benchmark runs them
            out = []
            for _ in range(2):
                r = eng.fetch()
                out.append(r.tobytes())
                if fine:
                    assert len(eng.read_neighbours()) == len(r)
            recs[(fine, survey)] = out
        finally:
            ba.close()
    assert recs[(True, False)] == recs[(False, False)] == recs[(True, True)]
    assert all(len(r) > 0 for r in recs[(False, False)])


def _small(n_streams, impl=E.FFT_AUTO, max_records=0):
    kw = _kw(300_000, 150_000, 256, "hamming", SIGMA["cu8"])
    return BatchAnalyzer(**parity.batch_kwargs(kw, devices=[str(i) for i in range(n_streams)], calibration=[0.0] * n_streams,
                                               fft_impl=impl, max_records=max_records))


def _blocks(n_streams, seed):
    return [np.stack([_capture("cu8", 300_000, 150_000, 256, 3, "hamming", seed=seed + s)[0][k] for s in range(n_streams)])
            for k in range(3)]


@pytest.mark.parametrize("impl", [E.FFT_GENERIC, E.FFT_AUTO, E.FFT_TC256])
def test_a_unit_alone_and_in_a_batch_and_run_to_run_gives_the_same_bits(impl):
    def run(rows):
        ba = _small(len(rows[0]), impl)
        try:
            ba.engine.set_neighbours(True)
            out = []
            for blk in rows:
                rec = ba.engine.process(blk)
                out.append((rec, ba.engine.read_neighbours()))
            return out
        finally:
            ba.close()

    blocks = _blocks(4, 40)
    batch, again = run(blocks), run(blocks)
    alone = run([b[2:3] for b in blocks])
    for (ra, na), (rb, nbb), (rc, nc) in zip(batch, again, alone):
        assert ra.tobytes() == rb.tobytes() and na.tobytes() == nbb.tobytes()
        sel = ra["stream"] == 2
        assert nc.tobytes() == na[sel].tobytes() and len(nc) > 0


def test_stream_contract():
    blocks = _blocks(3, 70)
    ba = _small(3)
    try:
        eng = ba.engine
        with pytest.raises(E.EngineError) as ei:   # nothing fetched yet
            eng.read_neighbours()
        assert ei.value.code == E.RT_ERR_INVALID
        eng.launch(blocks[0])                      # launched before the feature was switched on: not refined
        eng.set_neighbours(True)
        eng.launch(blocks[1])
        eng.fetch()
        with pytest.raises(E.EngineError) as ei:
            eng.read_neighbours()
        assert ei.value.code == E.RT_ERR_INVALID
        r1 = eng.fetch()
        n1 = eng.read_neighbours()
        assert len(n1) == len(r1) > 0
        eng.set_neighbours(False)                  # from the next launch on
        eng.launch(blocks[2])
        eng.fetch()
        with pytest.raises(E.EngineError):
            eng.read_neighbours()
    finally:
        ba.close()
    # overflow: entries for the records the fetch returned, equal to the unlimited launch's entries of the same records
    full = _small(3)
    few = _small(3, max_records=5)
    try:
        for a in (full, few):
            a.engine.set_neighbours(True)
            a.engine.process(blocks[0])
        rf, nf = full.engine.process(blocks[1]), full.engine.read_neighbours()
        rs = few.engine.process(blocks[1])
        ns = few.engine.read_neighbours()
        assert few.engine.truncated > 0 and len(rs) == len(ns) == 5
        idx = {r.tobytes(): i for i, r in enumerate(rf)}
        for r, n in zip(rs, ns):
            assert n.tobytes() == nf[idx[r.tobytes()]].tobytes()
    finally:
        full.close()
        few.close()


# ---------------------------------------------------------------------------------------------------------------------------
# full band
# ---------------------------------------------------------------------------------------------------------------------------
FS, D, NPERSEG, CF = 20_000_000, 64, 256, 150_000_000
BW = FS / (D * NPERSEG)                 # channel bin, 1220.7 Hz
HALF = NPERSEG // 2                     # channel spacing in bins


def _wide_keys(block):
    return dict(fft_nperseg=NPERSEG, fft_window="hamming", signal_min_duration_ms=8.0, signal_max_duration_ms=40.0,
                signal_threshold_dbw=float(10 * np.log10(2 * 0.01 ** 2 / (FS / D)) + 3.0), snr_threshold_db=5.0,
                sdr_callback_length=block)


def test_full_band_gives_one_estimate_per_pulse():
    block, nb = 8_000_000, 2
    # carriers in channel bins from the band centre: inside channels, in the overlap of two channels (|k| near 64 of both),
    # and within two bins of a channel centre (the documented DC zone); one 20 ms pulse every 32 ms, so that the shadow filter
    # of each channel keeps the pulse's loudest bin
    inside = [40.3, -1000.27, 2310.41, -3900.18, 5000.33]
    overlap = [64.38, 191.62, -2 * HALF - 63.7, 7 * HALF + 64.12]
    dc = [1.3, 3 * HALF - 1.21, -5 * HALF + 0.4]
    carriers = inside + overlap + dc
    rng = np.random.default_rng(21)
    win = R.resolve_window("hamming", NPERSEG)
    amp = FO.pulse_amplitude(20.0, 2 * 0.01 ** 2, win)   # 20 dB over the channel's floor (the filter has unit gain)
    ln, gap = FS // 50, 640_000
    pulses = [(b * block + 40_000 + j * gap, ln, m * BW / FS, amp) for b in range(nb) for j, m in enumerate(carriers)]
    x = FO.pulsed_tones(nb * block, pulses, 0.01, rng)
    raw = synth.quantise(x, "ci16_le").reshape(nb, -1)
    fb = W.WidebandAnalyzer.full_band(devices=["rx"], calibration_db=[0.0], sample_rate=FS, center_freq=CF, decimation=D,
                                      sample_format="ci16_le", fine_frequency=True, **_wide_keys(block))
    ddc = W.WidebandAnalyzer(devices=["rx"], calibration_db=[0.0], sample_rate=FS, center_freq=CF, offsets_hz=W.grid_offsets(FS, D),
                             decimation=D, taps=fb.ddc.taps, sample_format="ci16_le", fine_frequency=True, **_wide_keys(block))
    dt = datetime.timedelta(seconds=block / FS)
    utc = datetime.timezone.utc
    n_cmp = 0
    try:
        for b in range(nb):
            (chans,) = fb.process_blocks(raw[b][None, :], [T0 + b * dt])
            (fine,) = fb.last_fine_frequencies()
            (fine_all,) = fb.last_fine_frequencies(all_signals=True)
            kept = [s for k, _, _ in chans for s in k]
            assert len(fine) == len(kept) and len(fine_all) == sum(len(a) for _, a, _ in chans)
            (chans_d,) = ddc.process_blocks(raw[b][None, :], [T0 + b * dt])
            (fine_d,) = ddc.last_fine_frequencies(all_signals=True)
            # the DDC on the same grid and taps: the same estimates within 1e-3 bin, Signal for Signal where the keys agree
            oa = od = 0
            for (_, sa, ka), (_, sd, kd) in zip(chans, chans_d):
                fa, fd = fine_all[oa:oa + len(sa)], fine_d[od:od + len(sd)]
                if ka == kd:
                    assert np.array_equal(np.isfinite(fa), np.isfinite(fd))
                    both = np.isfinite(fa)
                    assert np.all(np.abs(fa[both] - fd[both]) <= 1e-3 * BW)
                    n_cmp += int(both.sum())
                oa, od = oa + len(sa), od + len(sd)
            for j, m in enumerate(carriers):
                t0 = (T0 + b * dt + datetime.timedelta(seconds=(40_000 + j * gap) / FS)).astimezone(utc)
                true_f = CF + m * BW
                hits = [f for s, f in zip(kept, fine)
                        if abs(s.frequency - true_f) <= 2.5 * BW and abs((s.ts - t0).total_seconds()) < 0.005 and np.isfinite(f)]
                if m in dc:
                    assert hits == [], (m, hits)
                else:
                    assert len(hits) == 1, (m, hits)
                    assert abs(hits[0] - true_f) <= ERR_20DB_MAX * BW, (m, (hits[0] - true_f) / BW)
    finally:
        fb.close()
        ddc.close()
    assert n_cmp > 0
