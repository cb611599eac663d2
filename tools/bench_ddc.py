"""Wideband down-converter on the GPU (include/rt_ddc.h): one JSON line per measurement.

    python tools/bench_ddc.py [--steps 5] [--out FILE.jsonl]

  ddc          the DDC alone on the BASELINE configs[2]-scale case (one 20 MS/s input, 1-s blocks, D = 64, 64 channels, the
               default 513 taps), device-resident input, for ci16_le, cf32_le and cu8: ms per block (CUDA events), input
               G samples/s, and real FMA/s (4 L per output) against the 36 T FMA/s lane rate of profiles/r01_ubench_fp32x2.txt
  wideband     WidebandAnalyzer (DDC + engine on the 64 channels, nperseg 256), device-resident input, two steps in flight
  wideband_e2e the same from pinned host buffers, beside the pinned H2D rate of the same bytes measured in the same run
The card's name and power limit are read in the same run and written into every line.
"""
import argparse
import datetime
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

LANE_RATE = 36.0e12        # FFMA / FFMA2 lanes per second, profiles/r01_ubench_fp32x2.txt


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clk = [s.strip() for s in q[0].split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clk)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--steps", type=int, default=5)
    args = ap.parse_args()
    import torch

    from pyradiotracking_b200 import wideband as W

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: nothing to measure")
    info = card()
    fs, D, C = 20_000_000, 64, 64
    block = fs
    offsets = [(c - C / 2 + 0.5) * fs / C for c in range(C)]          # a uniform grid across the band, fs / D apart
    L = len(W.default_taps(D))
    fmas = 4 * L * (block // D) * C
    lines = []

    def emit(d):
        d.update(info)
        lines.append(d)
        print(json.dumps(d), flush=True)

    gen = torch.Generator(device="cuda").manual_seed(1)
    dev_inputs = {
        "ci16_le": torch.randint(-3000, 3000, (1, 2 * block), dtype=torch.int16, device="cuda", generator=gen),
        "cf32_le": torch.randn((1, 2 * block), dtype=torch.float32, device="cuda", generator=gen) * 0.05,
        "cu8": torch.randint(0, 256, (1, 2 * block), dtype=torch.uint8, device="cuda", generator=gen),
    }
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for fmt, x in dev_inputs.items():
        ch = W.Channelizer(fs, block, offsets, D, sample_format=fmt)
        out = ch.run(x)
        for _ in range(2):
            ch.run(x, out=out)
        torch.cuda.synchronize()
        ev0.record()
        for _ in range(args.steps):
            ch.run(x, out=out)
        ev1.record()
        torch.cuda.synchronize()
        ms = ev0.elapsed_time(ev1) / args.steps
        emit(dict(case="ddc", sample_format=fmt, fs=fs, decimation=D, channels=C, taps=L, block_samples=block, steps=args.steps,
                  ms_per_block=round(ms, 4), input_gsps=round(block / ms / 1e6, 3), fma_per_s=float(f"{fmas / ms * 1e3:.4g}"),
                  lane_rate_share=round(fmas / ms * 1e3 / LANE_RATE, 4), bound="fp32 FMA lanes"))
        ch.close()

    keys = dict(fft_nperseg=256, fft_window="hamming", signal_min_duration_ms=8.0, signal_max_duration_ms=40.0,
                signal_threshold_dbw=-90.0, snr_threshold_db=5.0, sdr_callback_length=block)
    t0 = datetime.datetime(2026, 1, 1)
    fmt = "ci16_le"
    x = dev_inputs[fmt]
    pinned = torch.empty((1, 2 * block), dtype=torch.int16, pin_memory=True)
    pinned.copy_(x.cpu())
    for case, src in (("wideband", x), ("wideband_e2e", pinned.numpy())):
        wa = W.WidebandAnalyzer(devices=["0"], calibration_db=[0.0], sample_rate=fs, center_freq=150_000_000, offsets_hz=offsets,
                                decimation=D, sample_format=fmt, **keys)
        for _ in range(2):
            wa.submit(src)
            wa.collect([t0])
        torch.cuda.synchronize()
        tic = time.perf_counter()
        pending = 0
        for _ in range(args.steps):                    # two steps in flight, like replay()
            wa.submit(src)
            pending += 1
            if pending == 2:
                wa.collect([t0])
                pending -= 1
        while pending:
            wa.collect([t0])
            pending -= 1
        torch.cuda.synchronize()
        ms = (time.perf_counter() - tic) * 1e3 / args.steps
        d = dict(case=case, sample_format=fmt, fs=fs, decimation=D, channels=C, taps=L, nperseg=256, steps=args.steps,
                 ms_per_block=round(ms, 3), input_gsps=round(block / ms / 1e6, 3), realtime_factor=round(1e3 / ms, 1))
        if case == "wideband_e2e":
            dst = torch.empty_like(x)
            dst.copy_(pinned, non_blocking=True)
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(args.steps):
                dst.copy_(pinned, non_blocking=True)
            ev1.record()
            torch.cuda.synchronize()
            h2d_ms = ev0.elapsed_time(ev1) / args.steps
            d.update(h2d_ms_per_block=round(h2d_ms, 3), h2d_gbps=round(pinned.numel() * 2 / h2d_ms / 1e6, 2),
                     h2d_gsps=round(block / h2d_ms / 1e6, 3))
        emit(d)
        wa.close()
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
