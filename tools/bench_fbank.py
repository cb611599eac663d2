"""Polyphase FFT filter bank on the GPU (include/rt_fbank.h): one JSON line per measurement.

    python tools/bench_fbank.py [--steps 10] [--out FILE.jsonl]

  fbank            the filter bank alone: one input, 1-s blocks, default 8 D + 1 taps, device-resident input in two buffers
                   used in turn (2 x 80 MB of ci16_le and 2 x 160 MB of cf32_le exceed the 126 MB L2; 2 x 40 MB of cu8 do
                   not), for 20 MS/s at D = 64 (127 channels) in ci16_le, cu8 and cf32_le, and 2.4 MS/s cu8 at D = 8
                   (15 channels): ms per block (CUDA events), input G samples/s, and the share of the HBM bound (input bytes
                   + 8 B per output sample, 2 - 1 / D outputs per input sample, against 7.7 TB/s)
  full_band        WidebandAnalyzer.full_band (filter bank + engine on every channel, nperseg 256), device-resident input,
                   two steps in flight
  full_band_e2e    the same from pinned host memory, beside the pinned H2D rate of the same bytes measured in the same run
  ddc_grid         the down-converter (Channelizer) on the same 127-channel grid, device input, and WidebandAnalyzer on it end
                   to end from pinned host memory (ddc_grid_e2e), for comparison
The card's name and power limit are read in the same run and written into every line.
"""
import argparse
import datetime
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_ddc import card  # noqa: E402

HBM_BYTES_PER_S = 7.7e12     # HGX B200 data sheet, one GPU
KEYS = dict(fft_nperseg=256, fft_window="hamming", signal_min_duration_ms=8.0, signal_max_duration_ms=40.0,
            signal_threshold_dbw=-90.0, snr_threshold_db=5.0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="also write the JSON lines to this file")
    ap.add_argument("--steps", type=int, default=10)
    args = ap.parse_args()
    import torch

    from pyradiotracking_b200 import engine as E
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
        if fmt == "cf32_le":
            return [torch.randn((1, n), dtype=torch.float32, device="cuda", generator=gen) * 0.05 for _ in range(2)]
        return [torch.randint(0, 256, (1, n), dtype=torch.uint8, device="cuda", generator=gen) for _ in range(2)]

    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def time_runs(obj, xs, out):
        for i in range(2):
            obj.run(xs[i % 2], out=out)
        torch.cuda.synchronize()
        ev0.record()
        for i in range(args.steps):
            obj.run(xs[i % 2], out=out)
        ev1.record()
        torch.cuda.synchronize()
        return ev0.elapsed_time(ev1) / args.steps

    def time_analyzer(wa, src):
        t0 = datetime.datetime(2026, 1, 1)
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
        return (time.perf_counter() - tic) * 1e3 / args.steps

    cases = [("ci16_le", 20_000_000, 64), ("cu8", 20_000_000, 64), ("cf32_le", 20_000_000, 64), ("cu8", 2_400_000, 8)]
    for fmt, fs, D in cases:
        block = fs
        C = 2 * D - 1
        L = len(W.default_taps(D))
        xs = device_inputs(fmt, block)
        bytes_in = E.SAMPLE_FORMATS[fmt][2]
        hbm = block * bytes_in + C * (block // D) * 8
        fb = W.FilterBank(fs, block, D, sample_format=fmt)
        ms = time_runs(fb, xs, fb.run(xs[0]))
        fb.close()
        emit(dict(case="fbank", sample_format=fmt, fs=fs, decimation=D, channels=C, taps=L, block_samples=block, steps=args.steps,
                  ms_per_block=round(ms, 4), input_gsps=round(block / ms / 1e6, 3), hbm_bytes_per_block=hbm,
                  hbm_gbps=round(hbm / ms / 1e6, 1), hbm_bound_share=round(hbm / ms * 1e3 / HBM_BYTES_PER_S, 4)))
        pinned = torch.empty(tuple(xs[0].shape), dtype=xs[0].dtype, pin_memory=True)
        pinned.copy_(xs[0].cpu())
        for case, src in (("full_band", xs[0]), ("full_band_e2e", pinned.numpy())):
            wa = W.WidebandAnalyzer.full_band(devices=["0"], calibration_db=[0.0], sample_rate=fs, center_freq=150_000_000,
                                              decimation=D, sample_format=fmt, sdr_callback_length=block, **KEYS)
            ms = time_analyzer(wa, src)
            wa.close()
            d = dict(case=case, sample_format=fmt, fs=fs, decimation=D, channels=C, taps=L, nperseg=256, steps=args.steps,
                     ms_per_block=round(ms, 3), input_gsps=round(block / ms / 1e6, 3), realtime_factor=round(1e3 / ms, 1))
            if case == "full_band_e2e":
                dst = torch.empty_like(xs[0])
                dst.copy_(pinned, non_blocking=True)
                torch.cuda.synchronize()
                ev0.record()
                for _ in range(args.steps):
                    dst.copy_(pinned, non_blocking=True)
                ev1.record()
                torch.cuda.synchronize()
                h2d_ms = ev0.elapsed_time(ev1) / args.steps
                d.update(h2d_ms_per_block=round(h2d_ms, 3), h2d_gbps=round(pinned.numel() * pinned.element_size() / h2d_ms / 1e6, 2),
                         h2d_gsps=round(block / h2d_ms / 1e6, 3))
            emit(d)
        del pinned, xs

    # the DDC on the same 127-channel grid
    fmt, fs, D = "ci16_le", 20_000_000, 64
    block, offsets = fs, W.grid_offsets(fs, D)
    xs = device_inputs(fmt, block)
    ch = W.Channelizer(fs, block, offsets, D, sample_format=fmt)
    ms = time_runs(ch, xs, ch.run(xs[0]))
    ch.close()
    emit(dict(case="ddc_grid", sample_format=fmt, fs=fs, decimation=D, channels=len(offsets), taps=len(W.default_taps(D)),
              block_samples=block, steps=args.steps, ms_per_block=round(ms, 4), input_gsps=round(block / ms / 1e6, 3)))
    pinned = torch.empty(tuple(xs[0].shape), dtype=xs[0].dtype, pin_memory=True)
    pinned.copy_(xs[0].cpu())
    wa = W.WidebandAnalyzer(devices=["0"], calibration_db=[0.0], sample_rate=fs, center_freq=150_000_000, offsets_hz=offsets,
                            decimation=D, sample_format=fmt, sdr_callback_length=block, **KEYS)
    ms = time_analyzer(wa, pinned.numpy())
    wa.close()
    emit(dict(case="ddc_grid_e2e", sample_format=fmt, fs=fs, decimation=D, channels=len(offsets), nperseg=256, steps=args.steps,
              ms_per_block=round(ms, 3), input_gsps=round(block / ms / 1e6, 3), realtime_factor=round(1e3 / ms, 1)))
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
