#!/usr/bin/env python
"""Device-resident throughput per input sample format (cu8, ci8, ci16_le, cf32_le) on one GPU.

For configs[1]-shaped batches (64 streams x 2.4 MS/s, nperseg 256) and configs[2] (one 20 MS/s stream, nperseg 1024 / 4096) it
times K launches on HBM-resident input of each format (CUDA events around the launches, like tools/bench_configs.py) and the
spectrogram kernel alone (the engine's per-kernel events), and reports samples/s and input bytes/s: ci16_le and cf32_le move
2x and 4x the bytes of cu8 per sample.  The formats of one configuration are timed in alternating rounds within one process, so
that the cu8 line is measured beside the others.  The card's name and power limit are printed with the numbers.

    python tools/bench_formats.py [--steps 20] [--warmup 5] [--rounds 3] [--out FILE.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

HBM_TBPS = 7.7          # NVIDIA HGX B200 data sheet, per GPU (a bound, not a measured rate)


def card():
    import torch

    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(out[0]), float(out[1])
    except Exception as exc:      # the numbers are still device times; say that the power limit is unknown
        info["power_limit_w"] = f"unavailable ({exc.__class__.__name__})"
    return info


def make_input(w, fmt, n_streams, torch, synth):
    """Two launches' worth of [n_streams, 2 * block_samples] elements of `fmt` on the device (4 distinct streams, repeated)."""
    distinct = [synth.make_stream_format(w, fmt, i, 2) for i in range(min(4, n_streams))]
    host = np.empty((2, n_streams, 2 * w.block_samples), dtype=distinct[0].dtype)
    for s in range(n_streams):
        host[:, s, :] = distinct[s % len(distinct)]
    return torch.from_numpy(host).cuda()


def case(w, fmt, impl, n_streams, torch, BatchAnalyzer):
    ba = BatchAnalyzer(devices=[str(i) for i in range(n_streams)], calibration_db=[0.0] * n_streams, sample_rate=w.sample_rate,
                       center_freq=w.center_freq, fft_nperseg=w.nperseg, fft_window="hamming",
                       signal_min_duration_ms=w.signal_min_duration_ms, signal_max_duration_ms=w.signal_max_duration_ms,
                       signal_threshold_dbw=w.signal_threshold_dbw, snr_threshold_db=w.snr_threshold_db,
                       sdr_callback_length=w.block_samples, cuda_device=0, fft_impl=impl, sample_format=fmt)
    ba.engine.set_stream(torch.cuda.current_stream().cuda_stream)
    return ba


def time_case(ba, dev, steps, warmup, torch):
    eng = ba.engine
    stream = torch.cuda.current_stream()
    for i in range(warmup):
        eng.launch(dev[i % 2])
    for _ in range(min(warmup, 2)):     # the engine keeps the results of the last two launches
        eng.fetch()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(steps):
        eng.launch(dev[i % 2])
    eng.join()
    e1.record(stream)
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / steps
    n_rec = len(eng.fetch())
    # the spectrogram kernel alone: events around it on every launch of a second, shorter run
    eng.enable_timing(1)
    eng.timing(reset=True)
    for i in range(max(4, steps // 4)):
        eng.launch(dev[i % 2])
        eng.fetch()
    tim = eng.timing(reset=True)
    eng.enable_timing(0)
    return step_ms, tim["spectrogram_ms"] / max(1, tim["launches"]), n_rec


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()

    import torch

    from pyradiotracking_b200 import engine as E
    from pyradiotracking_b200 import synth
    from pyradiotracking_b200.analyze import BatchAnalyzer

    if not torch.cuda.is_available():
        raise SystemExit("bench_formats: no CUDA device (nothing here is measured on the CPU)")
    head = card()
    configs = [
        ("configs[1] 64 x 2.4 MS/s n256", synth.C2, 64,
         [("cu8", E.FFT_AUTO), ("cu8", E.FFT_GENERIC), ("ci8", E.FFT_AUTO), ("ci16_le", E.FFT_AUTO), ("cf32_le", E.FFT_AUTO)]),
        ("configs[2] 20 MS/s n1024", synth.C3A, 1, [(f, E.FFT_AUTO) for f in ("cu8", "ci8", "ci16_le", "cf32_le")]),
        ("configs[2] 20 MS/s n4096", synth.C3B, 1, [(f, E.FFT_AUTO) for f in ("cu8", "ci8", "ci16_le", "cf32_le")]),
    ]
    lines = []
    for name, w, n_streams, variants in configs:
        inputs = {fmt: make_input(w, fmt, n_streams, torch, synth) for fmt in {f for f, _ in variants}}
        bas = {v: case(w, v[0], v[1], n_streams, torch, BatchAnalyzer) for v in variants}
        res = {v: [] for v in variants}
        for _ in range(args.rounds):
            for v in variants:
                res[v].append(time_case(bas[v], inputs[v[0]], args.steps, args.warmup, torch))
        for v in variants:
            fmt, impl = v
            steps = sorted(r[0] for r in res[v])
            spec = sorted(r[1] for r in res[v])
            step_ms, spec_ms = steps[len(steps) // 2], spec[len(spec) // 2]
            samples = n_streams * w.block_samples
            nbytes = samples * E.SAMPLE_FORMATS[fmt][2]
            line = dict(config=name, sample_format=fmt, fft_impl=impl, n_streams=n_streams, block_samples=w.block_samples,
                        nperseg=w.nperseg, step_ms_median=round(step_ms, 4), step_ms_all=[round(x, 4) for x in steps],
                        spectrogram_ms_median=round(spec_ms, 4), msps=round(samples / step_ms / 1e3, 1),
                        input_gbps_step=round(nbytes / step_ms / 1e6, 1), input_gbps_spectrogram=round(nbytes / spec_ms / 1e6, 1),
                        input_share_of_hbm_datasheet=round(nbytes / spec_ms / 1e9 / HBM_TBPS, 4),
                        records=res[v][-1][2], **head)
            lines.append(line)
            print(json.dumps(line), flush=True)
        for ba in bas.values():
            ba.close()
        del inputs
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "a") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
