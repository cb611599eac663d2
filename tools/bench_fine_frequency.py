"""Cost of the fine frequency (include/rt_engine.h, rt_engine_set_neighbours; finefreq.py) on the GPU: one JSON line per
measurement.

    python tools/bench_fine_frequency.py [--steps 40] [--rounds 3] [--out FILE.jsonl]

  configs1    configs[1]: 64 cu8 streams of 2.4 MS/s in 1-s blocks, nperseg 256 (register kernel, lean scan schedule), from two
              device-resident inputs used in turn (2 x 307 MB, beyond the 126 MB L2), two launches in flight as bench.py runs
              them; neighbour bins off and on alternately (on: the kernel and the copy of the entries, read after every fetch), ms per
              step from CUDA events around `steps` steps that end in a fetch
  full_band   WidebandAnalyzer.full_band on one 20 MS/s ci16_le input in 1-s blocks, D = 64 (127 channels), nperseg 256, from
              device memory, two steps in flight; fine_frequency off and on alternately (on includes the host estimator in
              collect); pulsed tones over the band, so that the launches carry records
Records are compared between the two settings in the same run (`records_equal`), and the records per launch are reported.  The card's name, power limit and max SM
clock are read in the same run and written into every line.
"""
import argparse
import datetime
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_ddc import card  # noqa: E402

KEYS = dict(fft_nperseg=256, fft_window="hamming", signal_min_duration_ms=8.0, signal_max_duration_ms=40.0,
            signal_threshold_dbw=-90.0, snr_threshold_db=5.0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--rounds", type=int, default=3, help="off / on alternations per case")
    args = ap.parse_args()
    import numpy as np
    import torch

    from pyradiotracking_b200 import synth
    from pyradiotracking_b200 import wideband as W
    from pyradiotracking_b200.analyze import BatchAnalyzer

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    info = card()
    lines = []

    def emit(d):
        d.update(info)
        lines.append(d)
        print(json.dumps(d), flush=True)

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    # ---- configs[1]
    w = synth.C2
    host = synth.make_batch(w, range(w.n_streams), 2)
    xs = [torch.from_numpy(host[i]).cuda() for i in range(2)]
    del host

    def c1_run(fine):
        ba = BatchAnalyzer(devices=[str(i) for i in range(w.n_streams)], calibration_db=[0.0] * w.n_streams,
                           sample_rate=w.sample_rate, center_freq=w.center_freq, sdr_callback_length=w.block_samples,
                           fine_frequency=fine, **KEYS)
        eng = ba.engine
        stream = torch.cuda.current_stream()
        eng.set_stream(stream.cuda_stream)
        recs = []
        for i in range(4):                             # warm-up; the records of the two inputs
            eng.launch(xs[i % 2])
            if i >= 1:
                recs.append(eng.fetch().tobytes())
        recs.append(eng.fetch().tobytes())
        torch.cuda.synchronize()
        ev0.record(stream)
        eng.launch(xs[0])
        for i in range(1, args.steps + 1):
            if i < args.steps:
                eng.launch(xs[i % 2])
            eng.fetch()
            if fine:
                eng.read_neighbours()
        eng.join()
        ev1.record(stream)
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / args.steps
        ba.close()
        return ms, recs[-2:]

    ms, recs = {False: [], True: []}, {}
    for _ in range(args.rounds):
        for fine in (False, True):
            m, r = c1_run(fine)
            ms[fine].append(m)
            recs[fine] = r
    off, on = min(ms[False]), min(ms[True])
    cells = w.n_streams * (w.block_samples // 256) * 256
    emit(dict(case="configs1", streams=w.n_streams, fs=w.sample_rate, nperseg=256, input="device", steps=args.steps,
              ms_off=[round(v, 4) for v in ms[False]], ms_on=[round(v, 4) for v in ms[True]], overhead_ms=round(on - off, 4),
              overhead_share=round((on - off) / off, 4), spectrogram_bytes=4 * cells,
              records_per_launch=[len(r) // 40 for r in recs[False]], records_equal=recs[False] == recs[True]))
    del xs

    # ---- full_band, 20 MS/s ci16_le, D = 64
    fs, D = 20_000_000, 64
    rng = np.random.default_rng(1)
    t = np.arange(fs)
    x = 0.01 * (rng.normal(size=fs) + 1j * rng.normal(size=fs))
    for j in range(200):                                                   # 20 ms pulses at 200 carriers over the band
        s0, f = int(rng.integers(0, fs - fs // 50)), rng.uniform(-0.45, 0.45)
        x[s0:s0 + fs // 50] += 0.05 * np.exp(2j * np.pi * f * t[s0:s0 + fs // 50])
    host = synth.quantise(x, "ci16_le")[None, :]
    xs = [torch.from_numpy(host).cuda(), torch.from_numpy(np.roll(host, 2 * 12345, axis=1)).cuda()]
    t0 = datetime.datetime(2026, 1, 1)

    def fb_run(fine):
        wa = W.WidebandAnalyzer.full_band(devices=["0"], calibration_db=[0.0], sample_rate=fs, center_freq=150_000_000, decimation=D,
                                          sample_format="ci16_le", sdr_callback_length=fs, fine_frequency=fine,
                                          **dict(KEYS, signal_threshold_dbw=-75.0))
        keys = []
        for i in range(2):
            wa.submit(xs[i % 2])
            keys.append([k for _, _, k in wa.collect([t0], with_all=True)[0]])
        n_rec = wa.channels.last_record_count
        torch.cuda.synchronize()
        ev0.record()
        pending = 0
        for i in range(args.steps):                    # two steps in flight, like replay()
            wa.submit(xs[i % 2])
            pending += 1
            if pending == 2:
                wa.collect([t0])
                if fine:
                    wa.last_fine_frequencies()
                pending -= 1
        while pending:
            wa.collect([t0])
            pending -= 1
        wa.channels.engine.join()
        ev1.record()
        torch.cuda.synchronize()
        wa.close()
        return ev0.elapsed_time(ev1) / args.steps, keys, n_rec

    ms, keys, n_rec = {False: [], True: []}, {}, 0
    for _ in range(args.rounds):
        for fine in (False, True):
            m, keys[fine], n_rec = fb_run(fine)
            ms[fine].append(m)
    off, on = min(ms[False]), min(ms[True])
    emit(dict(case="full_band", sample_format="ci16_le", fs=fs, decimation=D, channels=2 * D - 1, nperseg=256, input="device",
              steps=args.steps, ms_off=[round(v, 4) for v in ms[False]], ms_on=[round(v, 4) for v in ms[True]],
              overhead_ms=round(on - off, 4), overhead_share=round((on - off) / off, 4), records_per_launch=n_rec,
              records_equal=keys[False] == keys[True]))
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
