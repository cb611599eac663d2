"""Cost of the band survey (include/rt_engine.h, rt_engine_set_survey) on the GPU: one JSON line per measurement.

    python tools/bench_survey.py [--steps 40] [--rounds 3] [--out FILE.jsonl]

  configs1    configs[1]: 64 cu8 streams of 2.4 MS/s in 1-s blocks, nperseg 256 (register kernel, lean scan schedule), from two
              device-resident inputs used in turn (2 x 307 MB, beyond the 126 MB L2), two launches in flight as bench.py runs
              them; survey off and on alternately, ms per step from CUDA events around `steps` steps that end in a fetch
  full_band   WidebandAnalyzer.full_band on one 20 MS/s ci16_le input in 1-s blocks, D = 64 (127 channels), nperseg 256, from
              device memory, two steps in flight; survey off, on, and on with band_survey() after every collect, alternately
Records are compared between the two settings in the same run (`records_equal`).  The card's name, power limit and max SM
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

    def c1_run(survey):
        ba = BatchAnalyzer(devices=[str(i) for i in range(w.n_streams)], calibration_db=[0.0] * w.n_streams,
                           sample_rate=w.sample_rate, center_freq=w.center_freq, sdr_callback_length=w.block_samples,
                           survey=survey, **KEYS)
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
        eng.join()
        ev1.record(stream)
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / args.steps
        ba.close()
        return ms, recs[-2:]

    ms, recs = {False: [], True: []}, {}
    for _ in range(args.rounds):
        for survey in (False, True):
            m, r = c1_run(survey)
            ms[survey].append(m)
            recs[survey] = r
    off, on = min(ms[False]), min(ms[True])
    cells = w.n_streams * (w.block_samples // 256) * 256
    emit(dict(case="configs1", streams=w.n_streams, fs=w.sample_rate, nperseg=256, input="device", steps=args.steps,
              ms_off=[round(v, 4) for v in ms[False]], ms_on=[round(v, 4) for v in ms[True]], overhead_ms=round(on - off, 4),
              overhead_share=round((on - off) / off, 4), spectrogram_bytes=4 * cells,
              records_equal=recs[False] == recs[True]))
    del xs

    # ---- full_band, 20 MS/s ci16_le, D = 64
    fs, D = 20_000_000, 64
    gen = torch.Generator(device="cuda").manual_seed(1)
    xs = [torch.randint(-3000, 3000, (1, 2 * fs), dtype=torch.int16, device="cuda", generator=gen) for _ in range(2)]
    t0 = datetime.datetime(2026, 1, 1)

    def fb_run(survey, stitched):
        wa = W.WidebandAnalyzer.full_band(devices=["0"], calibration_db=[0.0], sample_rate=fs, center_freq=150_000_000, decimation=D,
                                          sample_format="ci16_le", sdr_callback_length=fs, survey=survey, **KEYS)
        for i in range(2):
            wa.submit(xs[i % 2])
            wa.collect([t0])
        torch.cuda.synchronize()
        ev0.record()
        pending = 0
        for i in range(args.steps):                    # two steps in flight, like replay()
            wa.submit(xs[i % 2])
            pending += 1
            if pending == 2:
                wa.collect([t0])
                if stitched:
                    wa.band_survey()
                pending -= 1
        while pending:
            wa.collect([t0])
            pending -= 1
        wa.channels.engine.join()
        ev1.record()
        torch.cuda.synchronize()
        wa.close()
        return ev0.elapsed_time(ev1) / args.steps

    variants = ((False, False), (True, False), (True, True))       # off; on; on and band_survey() after every collect
    ms = {v: [] for v in variants}
    for _ in range(args.rounds):
        for v in variants:
            ms[v].append(fb_run(*v))
    off = min(ms[variants[0]])
    for v in variants[1:]:
        on = min(ms[v])
        emit(dict(case="full_band", sample_format="ci16_le", fs=fs, decimation=D, channels=2 * D - 1, nperseg=256, input="device",
                  steps=args.steps, ms_off=[round(x, 4) for x in ms[variants[0]]], ms_on=[round(x, 4) for x in ms[v]],
                  overhead_ms=round(on - off, 4), overhead_share=round((on - off) / off, 4), band_survey_in_loop=v[1]))
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
