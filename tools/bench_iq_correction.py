"""Cost of the per-block DC and IQ-imbalance correction of the wideband front ends on the GPU: one JSON line per measurement.

    python tools/bench_iq_correction.py [--steps 10] [--out FILE.jsonl]

For one 20 MS/s input in 1-s blocks, device-resident in two buffers used in turn (2 x 80 MB of ci16_le exceed the 126 MB L2;
2 x 40 MB of ci8 do not), in ci16_le and ci8, each with the correction off and on, measured alternately (off, on, off, on) so
that drift between the two shows:
  fbank          FilterBank alone, D = 64, 127 channels, 513 taps: ms per block (CUDA events)
  full_band      WidebandAnalyzer.full_band (filter bank + engine on every channel, nperseg 256), two steps in flight
  ddc            Channelizer alone on the DDC plan of DESIGN §13: 64 channels fs / 64 apart, D = 64, 513 taps
  ddc_analyzer   WidebandAnalyzer on that plan, two steps in flight
The card's name, power limit and max SM clock are read in the same run and written into every line.
"""
import argparse
import datetime
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_ddc import card  # noqa: E402

KEYS = dict(fft_nperseg=256, fft_window="hamming", signal_min_duration_ms=8.0, signal_max_duration_ms=40.0,
            signal_threshold_dbw=-90.0, snr_threshold_db=5.0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=2, help="off / on alternations per case")
    args = ap.parse_args()
    import torch

    from pyradiotracking_b200 import wideband as W

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    info = card()
    lines = []

    def emit(d):
        d.update(info)
        lines.append(d)
        print(json.dumps(d), flush=True)

    gen = torch.Generator(device="cuda").manual_seed(1)

    def device_inputs(fmt, block):
        n = 2 * block
        if fmt == "ci16_le":
            return [torch.randint(-3000, 3000, (1, n), dtype=torch.int16, device="cuda", generator=gen) for _ in range(2)]
        return [torch.randint(-100, 100, (1, n), dtype=torch.int8, device="cuda", generator=gen) for _ in range(2)]

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def time_runs(obj, xs):
        out = obj.run(xs[0])
        for i in range(2):
            obj.run(xs[i % 2], out=out)
        torch.cuda.synchronize()
        ev0.record()
        for i in range(args.steps):
            obj.run(xs[i % 2], out=out)
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / args.steps

    def time_analyzer(wa, xs):
        t0 = datetime.datetime(2026, 1, 1)
        for i in range(2):
            wa.submit(xs[i % 2])
            wa.collect([t0])
        torch.cuda.synchronize()
        tic = time.perf_counter()
        pending = 0
        for i in range(args.steps):                    # two steps in flight, like replay()
            wa.submit(xs[i % 2])
            pending += 1
            if pending == 2:
                wa.collect([t0])
                pending -= 1
        while pending:
            wa.collect([t0])
            pending -= 1
        torch.cuda.synchronize()
        return (time.perf_counter() - tic) * 1e3 / args.steps

    fs, D = 20_000_000, 64
    block = fs
    ddc_offsets = [(c - 64 / 2 + 0.5) * fs / 64 for c in range(64)]
    for fmt in ("ci16_le", "ci8"):
        xs = device_inputs(fmt, block)
        makers = {
            "fbank": (lambda iq: W.FilterBank(fs, block, D, sample_format=fmt, iq_correction=iq), time_runs, 127),
            "full_band": (lambda iq: W.WidebandAnalyzer.full_band(
                devices=["0"], calibration_db=[0.0], sample_rate=fs, center_freq=150_000_000, decimation=D, sample_format=fmt,
                sdr_callback_length=block, iq_correction=iq, **KEYS), time_analyzer, 127),
            "ddc": (lambda iq: W.Channelizer(fs, block, ddc_offsets, D, sample_format=fmt, iq_correction=iq), time_runs, 64),
            "ddc_analyzer": (lambda iq: W.WidebandAnalyzer(
                devices=["0"], calibration_db=[0.0], sample_rate=fs, center_freq=150_000_000, offsets_hz=ddc_offsets, decimation=D,
                sample_format=fmt, sdr_callback_length=block, iq_correction=iq, **KEYS), time_analyzer, 64),
        }
        for case, (make, timer, channels) in makers.items():
            ms = {False: [], True: []}
            for _ in range(args.rounds):
                for iq in (False, True):
                    obj = make(iq)
                    ms[iq].append(timer(obj, xs))
                    obj.close()
            off, on = min(ms[False]), min(ms[True])
            emit(dict(case=case, sample_format=fmt, fs=fs, decimation=D, channels=channels, taps=len(W.default_taps(D)),
                      block_samples=block, input="device", steps=args.steps, ms_off=[round(v, 4) for v in ms[False]],
                      ms_on=[round(v, 4) for v in ms[True]], overhead_ms=round(on - off, 4),
                      overhead_share=round((on - off) / off, 4)))
        del xs
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
