#!/usr/bin/env python
"""Headline benchmark: IQ Msamples/s from uint8 IQ to Signal records (BASELINE.json `metric`).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c2|c4] [--dump-outputs DIR]

Workloads (one *step* = one engine launch for every stream of the batch; weak scaling: every GPU owns its own 64 streams,
no collective on the data path -- streams are independent analyzers, SURVEY.md section 8e):

  c2 (default)  BASELINE.json configs[1], the configuration the metric is quoted on: 64 concurrent 2.4 MS/s streams per GPU,
                nperseg 256 Hamming, -90 dBW / 5 dB SNR, 8..40 ms; a step = one 1-s callback block of each of the 64
                (distinct, seeded) streams; two alternating blocks (307 MB per step: larger than L2), carry exercised.
  c4            BASELINE.json configs[3]: offline replay of 64 of 512 station channels x 300 kS/s per GPU; a 60-block chunk
                per channel is resident (host: pinned) and replayed with the carry flowing across replays; a step = one
                launch of 10 consecutive callback blocks of every channel (rt_config.blocks_per_launch).

`value`        device-resident: the batch is in HBM before the timed region; K launches timed with CUDA events on the
               launching stream, max over ranks (per-rank times are printed too).
`e2e`          the public API (`BatchAnalyzer.submit` / `collect`) on pinned HOST buffers, two launches in flight: H2D copy,
               kernels, D2H of the records, float64 finalisation, shadow filter, Signal objects; with the per-rank split of the
               host time and the raw concurrent pinned H2D rate of the same bytes (the ceiling of any e2e number).
`roofline`     the spectrogram kernel against the measured HBM copy bandwidth (algorithmic 2 B/sample).
`parity`       the oracle on two streams of the very batch that was timed (BASELINE.md section 4: the gate reported with the number).
`cpu_baseline` the oracle port of the reference's scipy path on ONE host core, one full step of the workload (N = 1 only);
               `--impl reference` runs the same port with one analyzer process per host core.

`--dump-outputs DIR` writes the candidate records (include/rt_engine.h `rt_record`) of the last timed launch, one float64
array per field: stream, fi, start, end, max_lin, row_mean, mean_lin, std_db (with `rank<r>_` in front when N > 1).  The
inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "iq_msamples_per_s"
UNIT = "Msamples/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=["c2", "c4"])
    ap.add_argument("--streams", type=int, default=64, help="streams per GPU")
    ap.add_argument("--profile", action="store_true", help="device-resident region only (for runs under ncu)")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of the timed batch")
    ap.add_argument("--chunk-segs", type=int, default=-1, help="rt_config.chunk_segs (segments per spectrogram CTA); -1 = the workload's default")
    ap.add_argument("--scan-schedule", default="auto", choices=["auto", "serial", "overlap", "lean"], help="rt_config.scan_schedule")
    ap.add_argument("--bpl", type=int, default=0, help="c4: callback blocks per launch (rt_config.blocks_per_launch; 0 = the workload's default, 10)")
    ap.add_argument("--fft-impl", default="auto", choices=["auto", "reg256", "tc256", "generic"],
                    help="spectrogram kernel: auto = reg256 (registers, packed fp32x2); tc256 = tensor-core stage 1 (tcgen05)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the candidate records of the last timed launch to DIR/<field>.npy (float64, one array per rt_record field)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs dumps the records of the GPU path (--impl b200)")
    return args


class Work:
    """What a step is made of."""

    def __init__(self, name, streams):
        from pyradiotracking_b200 import synth

        self.key = name
        self.streams = streams
        self.chunk_segs = 0                                        # rt_config.chunk_segs: 0 = the engine's choice
        if name == "c2":
            self.w, self.bpl, self.n_blk = synth.C2, 1, 2
            self.label = "configs[1]: 64x2.4MS/s nperseg256 hamming -90dBW/5dB 8-40ms"
        else:
            self.w, self.bpl, self.n_blk = synth.C4, 10, 60
            self.label = "configs[3]: replay, 64 of 512 channels x 300kS/s per GPU, 60-block resident chunk, 10 blocks per launch"
            # 640 analyzer units per launch: longer chunks than the engine's latency-minded default for 1171-segment blocks (64)
            # amortise the CTA prologue; measured 0.3258 (64) / 0.3136 (128) / 0.3078 (192) / 0.3057 (256) / 0.3121 (384) ms per launch
            self.chunk_segs = 256
        self.groups = self.n_blk // self.bpl                       # distinct launches before the chunk repeats
        self.samples_per_step = streams * self.bpl * self.w.block_samples
        self.bytes_per_step = 2 * self.samples_per_step

    def config(self, **extra):
        w = self.w
        d = {"workload": self.label, "streams_per_gpu": self.streams, "block_samples": w.block_samples, "blocks_per_launch": self.bpl,
             "distinct_streams": self.streams, "sample_rate": w.sample_rate, "nperseg": w.nperseg}
        d.update(extra)
        return d


def analyzer_kwargs(wk, rank):
    w, n = wk.w, wk.streams
    return dict(
        chunk_segs=wk.chunk_segs, scan_schedule=getattr(wk, "scan_schedule", 0),
        devices=[str(rank * n + i) for i in range(n)], calibration_db=[0.0] * n,
        sample_rate=w.sample_rate, center_freq=w.center_freq, fft_nperseg=w.nperseg, fft_window="hamming",
        signal_min_duration_ms=w.signal_min_duration_ms, signal_max_duration_ms=w.signal_max_duration_ms,
        signal_threshold_dbw=w.signal_threshold_dbw, snr_threshold_db=w.snr_threshold_db,
        sdr_callback_length=w.block_samples, blocks_per_launch=wk.bpl)


def _gen(args):
    from pyradiotracking_b200 import synth

    name, stream, n_blk = args
    return synth.make_stream(synth.WORKLOADS[name], stream, n_blk)


def make_batch(wk, first_stream, procs):
    """uint8 [groups][streams][bpl * block_bytes]: every stream seeded on its own (SURVEY 8d: seed = 1000 * config + stream)."""
    import multiprocessing as mp

    w = wk.w
    out = np.empty((wk.groups, wk.streams, wk.bpl * w.block_bytes), dtype=np.uint8)
    jobs = [(w.name, first_stream + s, wk.n_blk) for s in range(wk.streams)]
    if procs > 1:
        with mp.get_context("fork").Pool(procs) as pool:          # before CUDA is initialised in this process
            it = pool.imap(_gen, jobs, chunksize=1)
            for s, cap in enumerate(it):
                out[:, s, :] = cap.reshape(wk.groups, -1)
    else:
        for s, j in enumerate(jobs):
            out[:, s, :] = _gen(j).reshape(wk.groups, -1)
    return out


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def recorded_traffic():
    """dram bytes per launch of the spectrogram kernel from the committed ncu capture, if any."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get("spectrogram_dram_bytes_per_launch")
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for nm, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path (the reference is pure Python: no oracle/_ref binary; the port is at
# least as fast as the unmodified reference, profiles/r02_cpu_arm_port_vs_reference.txt)
# ----------------------------------------------------------------------------------------------------
def _cpu_analyzers(wk, streams):
    from oracle import restatement as R

    w = wk.w
    P = R.Params.make(sample_rate=w.sample_rate, center_freq=w.center_freq, fft_nperseg=w.nperseg,
                      signal_min_duration_ms=w.signal_min_duration_ms, signal_max_duration_ms=w.signal_max_duration_ms,
                      signal_threshold_dbw=w.signal_threshold_dbw, snr_threshold_db=w.snr_threshold_db)
    return {s: R.OracleAnalyzer(P._replace(device=str(s))) for s in streams}


def _cpu_step(wk, analyzers, caps, step):
    """One step for the streams of `analyzers`: the step's `bpl` consecutive blocks of each, with the carry of earlier steps."""
    import datetime

    t0 = datetime.datetime(2026, 1, 1)
    n_sig = 0
    for s, ora in analyzers.items():
        cap = caps[s]                                              # [blocks, block_bytes]
        for k in range(wk.bpl):
            b = (step * wk.bpl + k) % cap.shape[0]
            n_sig += len(ora.process_block(cap[b], t0)[4])
    return n_sig


def _ref_worker(conn, wk_key, n_streams, streams):
    """One analyzer process (the reference runs one process per SDR, __main__.py:94-140) owning `streams`."""
    from pyradiotracking_b200 import synth

    wk = Work(wk_key, n_streams)
    caps = {s: synth.make_stream(wk.w, s, wk.n_blk) for s in streams}      # outside every timer
    an = _cpu_analyzers(wk, streams)
    conn.send("ready")
    while True:
        msg = conn.recv()
        if msg is None:
            return
        t = time.perf_counter()
        n = _cpu_step(wk, an, caps, msg)
        conn.send((time.perf_counter() - t, n))


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port).  The same config as the GPU arm --
    `streams_per_gpu` streams per step -- dealt over one analyzer process per host core (the reference's own
    process-per-SDR model); a step is timed by the wall clock around all of them."""
    import multiprocessing as mp

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wk = Work(args.workload, args.streams)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    procs = max(1, min(cores, wk.streams))
    # bounded sample: if a full step would not fit the time budget, every process takes fewer streams (stated in `sample`)
    per_stream_s = wk.bpl * wk.w.block_samples / 14e6              # ~14 Msamples/s per core
    budget_s = 150.0
    rounds = max(1, -(-wk.streams // procs))                        # streams per process for the full step
    total_steps = args.warmup + args.steps
    while rounds > 1 and rounds * per_stream_s * total_steps > budget_s:
        rounds -= 1
    step_streams = min(wk.streams, rounds * procs)
    ctx = mp.get_context("fork")
    workers = []
    for p in range(procs):
        mine = list(range(p, step_streams, procs))
        if not mine:
            continue
        a, b = ctx.Pipe()
        pr = ctx.Process(target=_ref_worker, args=(b, wk.key, wk.streams, mine), daemon=True)
        pr.start()
        workers.append((pr, a))
    for _, a in workers:
        assert a.recv() == "ready"
    walls, n_sig = [], 0
    for i in range(total_steps):
        t = time.perf_counter()
        for _, a in workers:
            a.send(i)
        res = [a.recv() for _, a in workers]
        wall = time.perf_counter() - t
        if i >= args.warmup:
            walls.append(wall)
            n_sig += sum(r[1] for r in res)
    for pr, a in workers:
        a.send(None)
        pr.join(timeout=10)
    samples = step_streams * wk.bpl * wk.w.block_samples
    val = samples * len(walls) / sum(walls) / 1e6
    sample = (f"{len(workers)} analyzer processes, {step_streams} of the {wk.streams} streams per step"
              + ("" if step_streams == wk.streams else " (bounded sample)") + f", {wk.bpl} callback block(s) each; oracle port of the scipy path")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(walls) / len(walls), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": wk.config(streams_timed_per_step=step_streams, signals_per_step=n_sig / len(walls)),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": len(workers), "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cpu_port_single(wk):
    """1 core: one full step of the workload (every stream's block(s)) through the oracle port."""
    from pyradiotracking_b200 import synth

    n = wk.streams if wk.key == "c2" else 16                      # ~10-20 s of CPU work either way
    caps = {s: synth.make_stream(wk.w, s, wk.n_blk if wk.key == "c4" else 1) for s in range(n)}
    an = _cpu_analyzers(wk, range(n))
    t = time.perf_counter()
    _cpu_step(wk, an, caps, 0)
    dt = time.perf_counter() - t
    samples = n * wk.bpl * wk.w.block_samples
    return samples / dt / 1e6, f"one step on one core: {n} streams x {wk.bpl} callback block(s) of {wk.w.block_samples} samples, oracle port (numpy pocketfft + run extraction + shadow filter)"


# ----------------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------------
def drain(eng):
    """Fetch (and drop) every launch that has not been fetched yet, so that the next submit / collect pair talks about the same
    launch.  The device-resident loops launch K times and fetch once: up to one result stays in the engine's ring behind them.
    Returns the records of the newest launch fetched here (None if none was left)."""
    from pyradiotracking_b200.engine import RT_ERR_STATE, EngineError

    last = None
    while True:
        try:
            last = eng.fetch()
        except EngineError as e:
            if e.code != RT_ERR_STATE:
                raise
            return last


DUMP_LIMIT_BYTES = 64 << 20


def dump_records(recs, out_dir, prefix=""):
    """One float64 array per rt_record field (integers and float32 values are exact in float64).  Above DUMP_LIMIT_BYTES a
    fixed, seeded sample of the records is written, in record order."""
    per_record = 8 * len(recs.dtype.names)
    if len(recs) * per_record > DUMP_LIMIT_BYTES:
        keep = np.random.default_rng(0).choice(len(recs), DUMP_LIMIT_BYTES // per_record, replace=False)
        recs = recs[np.sort(keep)]
    os.makedirs(out_dir, exist_ok=True)
    for name in recs.dtype.names:
        np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), recs[name].astype(np.float64))


def parity_gate(wk, ba, hnp, streams):
    """The oracle on `streams` of the timed batch: the first two launches from a reset engine (carry from launch 0 to 1)."""
    import datetime

    from oracle import check as C
    from oracle import restatement as R

    w = wk.w
    drain(ba.engine)
    for s in range(wk.streams):
        ba.reset_stream(s)
    P = R.Params.make(sample_rate=w.sample_rate, center_freq=w.center_freq, fft_nperseg=w.nperseg,
                      signal_min_duration_ms=w.signal_min_duration_ms, signal_max_duration_ms=w.signal_max_duration_ms,
                      signal_threshold_dbw=w.signal_threshold_dbw, snr_threshold_db=w.snr_threshold_db)
    t0 = datetime.datetime(2026, 1, 1)
    dt = datetime.timedelta(seconds=w.block_samples / w.sample_rate)
    oras = {s: R.OracleAnalyzer(P._replace(device=ba.devices[s])) for s in streams}
    lasts = {s: None for s in streams}
    tot = C.new_totals()
    n_launch = min(2, wk.groups)
    for g in range(n_launch):
        res = ba.process_blocks(hnp[g], [t0 + g * wk.bpl * dt] * wk.streams)
        for s in streams:
            for k in range(wk.bpl):
                u = s * wk.bpl + k
                blk = hnp[g][s].reshape(wk.bpl, -1)[k]
                _, _, S, found, kept = oras[s].process_block(blk, t0 + (g * wk.bpl + k) * dt)
                filtered, sigs, keys = res[u]
                last_unit = k == wk.bpl - 1 and g == n_launch - 1      # spectrogram cells: one unit per stream is enough
                C.add_block(tot, P, S, lasts[s], found, kept, sigs, keys, filtered,
                            ba.engine.read_spectrogram(u) if last_unit else None, ba.engine.read_row_means(u) if last_unit else None)
                lasts[s] = S
    tot["streams_checked"] = list(streams)
    tot["blocks_per_stream"] = n_launch * wk.bpl
    tot["ok"] = C.verdict(tot)
    return tot


def run_b200(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    wk = Work(args.workload, args.streams)
    if args.chunk_segs >= 0:
        wk.chunk_segs = args.chunk_segs
    if args.bpl > 0 and wk.key == "c4":
        if wk.n_blk % args.bpl:
            raise SystemExit(f"--bpl must divide the {wk.n_blk}-block chunk")
        wk.bpl = args.bpl
        wk.groups = wk.n_blk // wk.bpl
        wk.samples_per_step = wk.streams * wk.bpl * wk.w.block_samples
        wk.bytes_per_step = 2 * wk.samples_per_step
        wk.label = wk.label.replace("10 blocks per launch", f"{wk.bpl} blocks per launch")
    wk.scan_schedule = {"auto": 0, "serial": 1, "overlap": 2, "lean": 3}[args.scan_schedule]
    S = wk.streams

    # every rank keeps to its own share of the host cores: the generator pool, the CUDA driver threads, the finaliser
    affinity = None
    if hasattr(os, "sched_getaffinity"):
        cores = sorted(os.sched_getaffinity(0))
        per = len(cores) // max(1, local_world)
        if local_world > 1 and per >= 2:
            affinity = cores[local * per:(local + 1) * per]
            os.sched_setaffinity(0, affinity)
    n_cores = len(affinity) if affinity else (os.cpu_count() or 1)
    batch = make_batch(wk, rank * S, max(1, min(n_cores, 16)))     # [groups][S][bytes], distinct seeded streams

    import torch
    import torch.distributed as dist

    from pyradiotracking_b200 import engine as _E
    from pyradiotracking_b200.analyze import BatchAnalyzer

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def over_ranks(x):
        """every rank's value, on every rank"""
        if world == 1:
            return [x]
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        out = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    host = torch.empty(batch.shape, dtype=torch.uint8, pin_memory=True)
    hnp = host.numpy()
    hnp[...] = batch
    del batch
    dev = host.cuda()
    impl = {"auto": _E.FFT_AUTO, "reg256": _E.FFT_REG256, "tc256": _E.FFT_TC256, "generic": _E.FFT_GENERIC}[args.fft_impl]
    ba = BatchAnalyzer(**analyzer_kwargs(wk, rank), cuda_device=local, fft_impl=impl)
    eng = ba.engine
    stream = torch.cuda.current_stream()
    eng.set_stream(stream.cuda_stream)
    G = wk.groups

    # ---- device-resident timed region ------------------------------------------------------------
    clocks = ClockSampler(local)      # nvidia-smi needs ~0.2 s before its first line: start it ahead of the warm-up
    clocks.start()
    for i in range(max(args.warmup, 1)):
        eng.launch(dev[i % G])
    n_rec = len(eng.fetch())
    # per-kernel CUDA events (the roofline's kernel time) on every `period`-th launch: an event pair between two spectrogram kernels
    # costs the step a few microseconds of launch gap, so a dozen samples per run are taken rather than one per launch
    eng.enable_timing(max(4, args.steps // 12))
    eng.timing(reset=True)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for i in range(args.steps):
        eng.launch(dev[(args.warmup + i) % G])
    eng.join()          # the scan kernels of the last launch run on the engine's scan stream: wait for them too
    ev1.record(stream)
    barrier()
    ms_ranks = over_ranks(ev0.elapsed_time(ev1))
    ms = max(ms_ranks)
    tim = eng.timing(reset=True)
    eng.enable_timing(0)
    recs = eng.fetch()
    n_rec = len(recs)
    work_items = eng.last_counts()[0]
    newest = drain(eng)          # K launches, one fetch: the newest result is still in the ring
    if args.dump_outputs:
        dump_records(recs if newest is None else newest, args.dump_outputs, f"rank{rank}_" if world > 1 else "")

    # ---- end to end through the public API with host buffers -----------------------------------------
    import datetime

    t0 = datetime.datetime(2026, 1, 1)
    ts = [t0] * S
    e2e = None
    if not args.profile:
        # Two launches in flight (submit i+1 before collect i): the H2D copy and the kernels of the next launch overlap the
        # float64 finalisation of the current one, like a live multi-SDR ingest loop would run.
        e2e_steps = max(3, min(args.steps, 40))      # ~6 ms each (PCIe-bound): the pipeline fill and drain amortise
        for i in range(2):
            ba.process_blocks(hnp[i % G], ts)
        for k in ba.timings:
            ba.timings[k] = 0
        barrier()
        t_e2e = time.perf_counter()
        d2h = n_sig = 0
        t_submit = 0.0
        ba.submit(hnp[0])
        for i in range(e2e_steps):
            if i + 1 < e2e_steps:
                t = time.perf_counter()
                ba.submit(hnp[(i + 1) % G])
                t_submit += time.perf_counter() - t
            res = ba.collect(ts)
            n_sig += sum(len(r[0]) for r in res)
            d2h += 8 + 40 * ba.last_record_count
        torch.cuda.synchronize()
        e2e_own = time.perf_counter() - t_e2e
        barrier()
        e2e_ranks = over_ranks(e2e_own)
        # the ceiling of any e2e number on this box: the same pinned bytes copied to the device by every rank at once
        scratch = torch.empty_like(dev[0])
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n_copy = 10
        c0.record(stream)
        for i in range(n_copy):
            scratch.copy_(host[i % G], non_blocking=True)
        c1.record(stream)
        torch.cuda.synchronize()
        h2d_gbs = over_ranks(n_copy * wk.bytes_per_step / (c0.elapsed_time(c1) * 1e-3) / 1e9)
        barrier()
        del scratch
        tmn = ba.timings
        split = {k: over_ranks(1e3 * v / e2e_steps) for k, v in (("submit_ms", t_submit), ("fetch_wait_ms", tmn["fetch_wait_s"]),
                                                                  ("finalize_ms", tmn["finalize_s"]), ("build_signals_ms", tmn["build_s"]))}
        e2e_s = max(e2e_ranks)
        ceiling = world * min(h2d_gbs) * 1e9 / 2 / 1e6          # Msamples/s if every rank copied at the slowest rank's raw rate
        e2e = {"value": world * wk.samples_per_step * e2e_steps / e2e_s / 1e6, "unit": UNIT,
               "h2d_bytes_per_step": wk.bytes_per_step, "d2h_bytes_per_step": d2h // e2e_steps, "signals_per_step": n_sig / e2e_steps,
               "steps": e2e_steps, "ms_per_step_per_rank": [round(1e3 * x / e2e_steps, 3) for x in e2e_ranks],
               "host_ms_per_step_per_rank": {k: [round(x, 3) for x in v] for k, v in split.items()},
               "raw_pinned_h2d_gbs_per_rank_concurrent": [round(x, 2) for x in h2d_gbs],
               "h2d_ceiling_msamples_per_s": ceiling,
               "frac_of_h2d_ceiling": world * wk.samples_per_step * e2e_steps / e2e_s / 1e6 / ceiling}

    # The timed region of a default run lasts tens of milliseconds -- shorter than nvidia-smi's start-up.  If it yielded fewer
    # than 5 clock samples, keep the GPU under the very same load (untimed launches of the same batch) until it has.
    clock_extra_s = 0.0
    t_ex = time.perf_counter()
    while len(clocks.lines) < 5 and time.perf_counter() - t_ex < 3.0 and clocks.proc is not None:
        for i in range(50):
            eng.launch(dev[i % G])
        eng.join()
        torch.cuda.synchronize()
        clock_extra_s = time.perf_counter() - t_ex
    drain(eng)
    clk = clocks.stop()
    clk["sampled_over"] = "timed region" if clock_extra_s == 0 else f"timed region + {clock_extra_s:.2f} s of identical untimed launches"

    parity = None
    if rank == 0 and not args.profile and not args.no_parity:
        parity = parity_gate(wk, ba, hnp, [0, S // 2 + 5] if S > 6 else list(range(min(S, 2))))
        if not parity["ok"]:
            print("bench.py: PARITY GATE FAILED -- the CUDA path and the oracle disagree on the timed batch: " + json.dumps(parity), file=sys.stderr, flush=True)

    if rank == 0:
        value = world * wk.samples_per_step * args.steps / (ms * 1e-3) / 1e6
        peak, peak_kind = measured_peak()
        k_ms = tim["spectrogram_ms"] / max(1, tim["launches"])
        # consecutive spectrogram kernels run on alternating streams and overlap each other's tails: a kernel's own
        # event-bracketed duration then exceeds the time the GPU spends per launch, which is at most the step time
        k_eff = min(k_ms, ms / args.steps)
        achieved = wk.bytes_per_step / (k_eff * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": wk.config(l2=f"inputs larger than L2 ({wk.bytes_per_step / 1e6:.0f} MB per step, {G} alternating launches)",
                                records_per_step=n_rec, extract_work_items_per_step=work_items, fft_impl=args.fft_impl, chunk_segs=wk.chunk_segs,
                                scan_schedule=args.scan_schedule,
                                host_cores_per_rank=n_cores, cpu_affinity=("all" if affinity is None else f"{affinity[0]}-{affinity[-1]}")),
            "ms_per_step_per_rank": {"min": min(ms_ranks) / args.steps, "median": statistics.median(ms_ranks) / args.steps,
                                     "max": max(ms_ranks) / args.steps, "all": [round(x / args.steps, 5) for x in ms_ranks]},
            "clocks": clk,
            "e2e": e2e,
            "gpu_launches": int(tim["kernels"]),
            "roofline": {"bound": "hbm", "kernel": "spectro_tc256" if args.fft_impl == "tc256" else "spectro_reg256_v8", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": recorded_traffic() if wk.key == "c2" else None, "peak_source": peak_kind,
                         "algorithmic_bytes_per_launch": wk.bytes_per_step, "kernel_ms": k_eff,
                         "kernel_ms_event_bracketed": k_ms,
                         "kernel_share_of_step": k_eff / (ms / args.steps),
                         "other_kernels_ms": {k: tim[k] / max(1, tim["launches"]) for k in ("rowmean_ms", "probe_ms", "extract_ms")}},
            "parity": parity,
        }
        if world == 1 and not args.profile:
            v, sample = cpu_port_single(wk)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "sample": sample}
        print(json.dumps(line), flush=True)
    ba.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
