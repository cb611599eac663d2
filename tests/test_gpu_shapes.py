"""Every shape the engine accepts, against the float64 oracle or against itself, on the B200 (pytest -m gpu).

  A  every nperseg that no other test reaches (8 ... 2048): the generic Stockham kernel with and without its final radix-2
     pass, probe CTAs of 8 ... 256 threads, probe strides up to 300 columns, ragged tails, carries across block boundaries
  B  tiny blocks (T = 2 ... 65 columns, ragged): hand-built column-aligned bursts put a run at each edge of the scan
  C  the same records whatever the batch: probe kernels with 8 / 16 / 32 columns per thread on every layout, the widened and
     the plain extraction, the register kernel's chunk lengths
  D  blocks_per_launch > 1 on every layout, at aligned and ragged block lengths
  E  engines of different nperseg alive in one process
"""
import datetime
import functools

import numpy as np
import pytest

from oracle import restatement as R
from pyradiotracking_b200 import engine as E
from pyradiotracking_b200 import synth
from pyradiotracking_b200.analyze import BatchAnalyzer
from tests import parity

pytestmark = pytest.mark.gpu

T0 = datetime.datetime(2026, 5, 5, 5, 5, 5)
FS = 300_000


def _kw(fs, block, nperseg, window="hamming", min_ms=8.0, max_ms=40.0, thr_dbw=-90.0, snr_db=5.0):
    return dict(device="0", calibration_db=0.0, sample_rate=fs, center_freq=150_150_000, fft_nperseg=nperseg, fft_window=window,
                signal_min_duration_ms=min_ms, signal_max_duration_ms=max_ms, signal_threshold_dbw=thr_dbw, snr_threshold_db=snr_db,
                sdr_callback_length=block)


def _workload(fs, block, nperseg, **over):
    return synth.Workload(90, f"shape-{nperseg}-{fs}-{block}", fs, block, nperseg=nperseg, **over)


def _impls(nperseg, window="hamming"):
    """Every kernel that serves this nperseg: the generic one always, AUTO where it picks another, TC256 where it applies."""
    if nperseg in (1024, 4096):
        return [E.FFT_GENERIC, E.FFT_AUTO]           # AUTO = radix-16 Stockham kernel
    if nperseg != 256:
        return [E.FFT_GENERIC]
    impls = [E.FFT_GENERIC, E.FFT_AUTO]               # AUTO = register kernel
    if window in ("hamming", "hann", "boxcar"):
        impls.append(E.FFT_TC256)
    return impls


def _ts(kw, b):
    return parity.block_ts(T0, b, kw["sdr_callback_length"], kw["sample_rate"])


def _oracle(kw, cap, reset_at=None):
    """[(S, last, found)] for the blocks of one stream; `reset_at`: forget the previous block before that one."""
    P = parity.oracle_params(kw)
    ora = R.OracleAnalyzer(P)
    out = []
    for b in range(len(cap)):
        if b == reset_at:
            ora.last = None
        last = ora.last
        _, _, S, found, _ = ora.process_block(cap[b], _ts(kw, b))
        out.append((S, last, found))
    return P, out


def _strip(rec, unit):
    r = rec[rec["stream"] == unit].copy()
    r["stream"] = 0
    return r


def _run_vs_oracle(kw, cap, impl, tag, spectrogram=True, **extra):
    """One stream, block by block, through BatchAnalyzer: records against the oracle (tests/parity.py); returns the totals,
    the number of carried records and the keys of every block."""
    P, want = _oracle(kw, cap)
    ba = BatchAnalyzer(**parity.batch_kwargs(kw, fft_impl=impl, **extra))
    tot = dict(oracle=0, gpu=0, near_threshold_mismatch=0)
    carried = 0
    try:
        for b, (S, last, found) in enumerate(want):
            _, sigs, keys = ba.process_blocks(cap[b][None, :], [_ts(kw, b)])[0]
            st = parity.compare_block(P, S, last, found, sigs, keys)
            if spectrogram:
                spec, rm = ba.engine.read_spectrogram(0), ba.engine.read_row_means(0)
                if kw["fft_window"] == "boxcar":
                    # the DC bin of a detrended, boxcar-windowed segment is zero: both sides hold rounding residue there, so its
                    # relative error means nothing; it must stay far below anything that could decide a run
                    assert spec[:, 0].max() < 1e-2 * P.signal_threshold
                    S, spec, rm = S[1:], spec[:, 1:], rm[1:]
                parity.compare_spectrogram(P, S, spec, rm, tag=f"{tag}/b{b}")
            for k in tot:
                tot[k] += st[k]
            carried += sum(1 for k in keys if k[1] < 0)
    finally:
        ba.close()
    return tot, carried


# ---------------------------------------------------------------------------------------------------------------------------
# A: every nperseg against the oracle
# ---------------------------------------------------------------------------------------------------------------------------
A_CASES = [  # nperseg, fs, block_samples, blocks, window
    (8, 300_000, 300_000, 3, "hamming"),          # T = 37 500, probe stride 300, widened extraction; probe CTAs of 8 threads
    (8, 2_400_000, 2_400_000, 2, "hamming"),      # T = 300 000: plain LINEAR extraction, carry walks of thousands of columns
    (16, 300_000, 250_123, 3, "hamming"),         # ragged tail
    (32, 300_000, 300_000, 3, "hann"),            # odd log2: final radix-2 pass
    (128, 300_000, 300_000, 3, "boxcar"),         # odd log2
    (64, 1_024_000, 1_024_000, 3, "boxcar"),      # even log2
    (2048, 2_400_000, 2_400_000, 3, "hamming"),   # odd log2, 8 bin blocks per probe CTA; T = 1171 and a remainder
]


@pytest.mark.parametrize("nperseg,fs,block,nb,window", A_CASES, ids=lambda v: str(v) if not isinstance(v, str) else v)
def test_every_nperseg_matches_the_oracle(nperseg, fs, block, nb, window):
    w = _workload(fs, block, nperseg, amp_lsb=(10.0, 30.0))
    cap = synth.make_stream(w, 1, nb)                          # one burst straddles every block boundary (stream 0's burst at
                                                               # 2.4 MS/s lies so close to DC that nperseg 8's detrend removes it)
    kw = _kw(fs, block, nperseg, window)
    for impl in _impls(nperseg, window):
        tot, carried = _run_vs_oracle(kw, cap, impl, tag=f"shapes/n{nperseg}/fs{fs}/impl{impl}")
        assert tot["gpu"] >= 5 and tot["near_threshold_mismatch"] == 0, (impl, tot)
        assert carried >= 1, impl                              # a straddling burst was re-found from the next block


# ---------------------------------------------------------------------------------------------------------------------------
# B: tiny blocks with hand-built runs at the edges of the scan
# ---------------------------------------------------------------------------------------------------------------------------
B_BLOCKS, B_RESET = 8, 5
B_TONE_DBW, B_SIGMA = -62.0, 1.0       # tone cells 13 dB over the threshold below at every nperseg; noise of 1 LSB: cells 32 dB under
                                        # the tones, so that a not-above neighbour inside a window stays out of the float32 deep tail


def _tone_capture(n, T, r, masks, seed):
    """uint8 [B_BLOCKS, 2 (T n + r)]: dithering noise plus, for every (bin k, mask [B_BLOCKS, T]), a bin-centred complex tone of
    B_TONE_DBW per cell on exactly the segments the mask sets.  Under a boxcar window such a tone lights its own bin only, and
    only in those columns; the r samples after the last whole segment of every block are never analysed."""
    N = T * n + r
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((B_BLOCKS, N, 2)) * B_SIGMA
    t = np.arange(n)
    amp = 127.5 * np.sqrt(10 ** (B_TONE_DBW / 10) * FS / n)     # boxcar, bin-centred: cell power (amp / 127.5)^2 n / fs
    for k, m in masks.items():
        tone = amp * np.exp(2j * np.pi * k * t / n)
        for b, c in zip(*np.nonzero(m)):
            x[b, c * n:(c + 1) * n, 0] += tone.real
            x[b, c * n:(c + 1) * n, 1] += tone.imag
    return np.clip(np.rint(x + 127.5), 0, 255).astype(np.uint8).reshape(B_BLOCKS, 2 * N)


def _edge_masks(n, T):
    """Column masks of five bins (the runs each one makes are listed in test_tiny_blocks_match_the_oracle)."""
    A, B, C, D, Ebin = (k * n // 8 for k in (1, 2, 3, 5, 6))
    m = {k: np.zeros((B_BLOCKS, T), dtype=bool) for k in (A, B, C, D, Ebin)}
    for b in range(B_BLOCKS):
        if b % 2:
            m[A][b, max(0, T - 4):T - 1] = True            # last above cell T - 2: kept
            m[B][b, max(0, T - 3):T] = True                # last above cell T - 1: touches the block end, dropped
            m[C][b, :] = True                              # whole block ...
            if T >= 5:
                m[D][b, :] = True
        elif b >= 2:
            m[C][b, 0] = True                              # ... and one column more: start == -(T - 1), end == 1
            if T >= 5:
                m[D][b, :3] = True                         # ... and three columns more: longer than the maximum duration
    short = max(1, min(2, T - 1))
    m[Ebin][0, :short] = True                              # from column 0 of the first block: start == 0
    m[Ebin][B_RESET - 1, T - 1] = True                     # would be carried into the next block, ...
    m[Ebin][B_RESET, :short] = True                        # ... which follows reset_stream: start == 0 again
    return (A, B, C, D, Ebin), m


B_KERNELS = [(256, E.FFT_AUTO), (256, E.FFT_GENERIC), (256, E.FFT_TC256), (1024, E.FFT_AUTO), (1024, E.FFT_GENERIC), (8, E.FFT_GENERIC)]
B_KERNEL_IDS = ["n256-reg", "n256-generic", "n256-tc", "n1024-r16", "n1024-generic", "n8-generic"]


@pytest.mark.parametrize("T", [2, 3, 5, 8, 9, 31, 33, 65])
@pytest.mark.parametrize("nperseg,impl", B_KERNELS, ids=B_KERNEL_IDS)
def test_tiny_blocks_match_the_oracle(nperseg, impl, T):
    """T whole segments plus a ragged remainder per block, probe stride 1 (minimum duration 0), maximum duration T + 1.5 columns,
    8 consecutive blocks with reset_stream before block 5.  Per bin:
      A  odd blocks: a run whose last above cell is T - 2 (record, end == T - 1)
      B  odd blocks: a run whose last above cell is T - 1 (touches the block end: no record)
      C  odd blocks whole, next block column 0: the carry walk runs into start_min (record (C, -(T - 1), 1))
      D  like C with three columns in the next block: T + 3 columns, over the maximum (no record; T >= 5)
      E  columns 0 ... of the first block and of the block after reset_stream (record with start == 0)"""
    fs = FS
    r = nperseg // 2 + 3 if nperseg > 8 else 3
    block = T * nperseg + r
    dt_ms = 1000.0 * nperseg / fs
    kw = _kw(fs, block, nperseg, "boxcar", min_ms=0.0, max_ms=(T + 1.5) * dt_ms, thr_dbw=-75.0, snr_db=-30.0)
    (A, B, C, D, Ebin), masks = _edge_masks(nperseg, T)
    cap = _tone_capture(nperseg, T, r, masks, seed=T)
    P, want = _oracle(kw, cap, reset_at=B_RESET)
    ba = BatchAnalyzer(**parity.batch_kwargs(kw, fft_impl=impl))
    try:
        assert ba.engine.T == T and ba.plan.stride == 1
        for b, (S, last, found) in enumerate(want):
            if b == B_RESET:
                ba.reset_stream(0)
            _, sigs, keys = ba.process_blocks(cap[b][None, :], [_ts(kw, b)])[0]
            st = parity.compare_block(P, S, last, found, sigs, keys)
            assert st["near_threshold_mismatch"] == 0, (b, st)
            if b % 2:
                assert any(k[0] == A and k[2] == T - 1 for k in keys), (b, keys)
                assert not any(k[0] == B for k in keys), (b, keys)
            elif b >= 2:
                assert (C, -(T - 1), 1) in keys, (b, keys)
                assert not any(k[0] == D for k in keys), (b, keys)
            if b in (0, B_RESET):
                assert any(k[0] == Ebin and k[1] == 0 for k in keys), (b, keys)
            else:
                assert not any(k[0] == Ebin and k[1] >= 0 for k in keys), (b, keys)
    finally:
        ba.close()


# ---------------------------------------------------------------------------------------------------------------------------
# C: the same records whatever the batch
# ---------------------------------------------------------------------------------------------------------------------------
def _alone_and_batched(kw, caps, batch_sizes, loose_row_mean=False, **extra):
    """Records of every capture run alone, and of batches of `batch_sizes` streams (stream s = caps[s % len(caps)]); every
    stream of a batch must equal its capture alone, byte for byte (`loose_row_mean`: except row_mean, within 1e-6 relative)."""
    nb = len(caps[0])
    alone = []
    for c in caps:
        ba = BatchAnalyzer(**parity.batch_kwargs(kw, **extra))
        try:
            alone.append([ba.engine.process(c[b][None, :]) for b in range(nb)])
        finally:
            ba.close()
    assert sum(len(r) for r in alone[0]) > 0
    for n in batch_sizes:
        ba = BatchAnalyzer(**parity.batch_kwargs(kw, devices=[str(i) for i in range(n)], calibration=[0.0] * n, **extra))
        try:
            for b in range(nb):
                rec = ba.engine.process(np.stack([caps[s % len(caps)][b] for s in range(n)]))
                for s in range(n):
                    got, want = _strip(rec, s), alone[s % len(caps)][b]
                    if loose_row_mean and len(got) == len(want):
                        np.testing.assert_allclose(got["row_mean"], want["row_mean"], rtol=1e-6, atol=0)
                        got["row_mean"] = want["row_mean"]
                    if got.tobytes() != want.tobytes():
                        diff = {x.tobytes() for x in got} ^ {x.tobytes() for x in want}
                        fields = [f for f in E.RECORD_DTYPE.names if len(got) == len(want) and (got[f] != want[f]).any()]
                        pytest.fail(f"batch of {n}, stream {s}, block {b}: {len(got)} vs {len(want)} records alone, "
                                    f"{len(diff)} differ, fields {fields}")
        finally:
            ba.close()
    return alone


C_LAYOUTS = [(E.FFT_AUTO, dict(scan_schedule=E.SCAN_OVERLAP)), (E.FFT_GENERIC, {}), (E.FFT_TC256, {})]


@pytest.mark.parametrize("impl,extra", C_LAYOUTS, ids=["perm", "linear", "tile"])
def test_batch_composition_does_not_change_the_records(impl, extra):
    """nperseg 256 at 300 kS/s: T = 1171, probe stride 9, 131 probe columns.  The probe kernel takes the fewest probe columns per
    thread whose grid fits one wave of 148 CTAs: alone ceil(131 / 8) * 1 = 17 <= 148 (8 columns), a batch of 12
    ceil(131 / 16) * 12 = 108 <= 148 (16 columns; 17 * 12 = 204 does not fit), a batch of 24 ceil(131 / 32) * 24 = 120 <= 148
    (32 columns; 9 * 24 = 216 does not fit).

    The tensor-core kernel sums each stream's rows over warp-group runs whose split depends on the batch size (tc_first_run /
    tc_last_run), so its row means may differ in the last bits between a stream alone and in a batch; every other field must
    still be identical."""
    w = synth.C1
    kw = _kw(w.sample_rate, w.block_samples, 256)
    caps = [synth.make_stream(w, 40 + i, 3) for i in range(4)]
    _alone_and_batched(kw, caps, [12, 24], loose_row_mean=impl == E.FFT_TC256, fft_impl=impl, **extra)
    for c in caps:                                            # every distinct capture against the oracle
        tot, _ = _run_vs_oracle(kw, c, impl, tag=f"shapes/batch/impl{impl}", spectrogram=False, **extra)
        assert tot["near_threshold_mismatch"] == 0 and tot["gpu"] > 0


def test_nperseg_8_alone_equals_a_batch_of_8():
    """nperseg 8 at 300 kS/s: probe stride 300, so a run's backward walk stays open for up to 10 rounds.  Alone (T = 37 500) the
    extraction widens its forward walk (streams x T < 300 000), in a batch of 8 (300 000) it does not: the float64 sums of a
    record must not depend on that."""
    w = _workload(FS, FS, 8, amp_lsb=(10.0, 30.0), pulses_per_block=(8, 8), pulse_ms=(12.0, 36.0))
    kw = _kw(FS, FS, 8)
    caps = [synth.make_stream(w, i, 3) for i in range(2)]
    _alone_and_batched(kw, caps, [8], fft_impl=E.FFT_GENERIC)
    tot, carried = _run_vs_oracle(kw, caps[0], E.FFT_GENERIC, tag="shapes/n8-batch", spectrogram=False)
    assert tot["near_threshold_mismatch"] == 0 and tot["gpu"] >= 5


@pytest.mark.parametrize("chunk_segs", [8, 24, 256, 2048])
def test_register_kernel_chunk_lengths_match_the_oracle(chunk_segs):
    """rt_config.chunk_segs groups the row sums differently (2048 > T: one chunk per stream): within tolerance, not bitwise."""
    w = synth.C1
    kw = _kw(w.sample_rate, w.block_samples, 256)
    cap = synth.make_stream(w, 7, 3)
    tot, carried = _run_vs_oracle(kw, cap, E.FFT_REG256, tag=f"shapes/chunk{chunk_segs}", chunk_segs=chunk_segs)
    assert tot["gpu"] >= 5 and tot["near_threshold_mismatch"] == 0 and carried >= 1


# ---------------------------------------------------------------------------------------------------------------------------
# D: blocks_per_launch on every layout
# ---------------------------------------------------------------------------------------------------------------------------
D_STREAMS, D_BLOCKS = 3, 7


@functools.lru_cache(maxsize=None)
def _d_capture(nperseg, block):
    w = _workload(FS, block, nperseg, amp_lsb=(10.0, 30.0))
    return np.stack([synth.make_stream(w, s, D_BLOCKS) for s in range(D_STREAMS)], axis=1)      # [blocks, streams, 2 block]


@functools.lru_cache(maxsize=None)
def _d_one_block_per_launch(nperseg, impl, block):
    kw = _kw(FS, block, nperseg)
    cap = _d_capture(nperseg, block)
    ba = BatchAnalyzer(**parity.batch_kwargs(kw, devices=[str(s) for s in range(D_STREAMS)], calibration=[0.0] * D_STREAMS, fft_impl=impl))
    try:
        return [ba.engine.process(cap[b]) for b in range(D_BLOCKS)]
    finally:
        ba.close()


D_KERNELS = [(256, E.FFT_AUTO), (256, E.FFT_GENERIC), (1024, E.FFT_AUTO), (512, E.FFT_GENERIC), (8, E.FFT_GENERIC)]


@pytest.mark.parametrize("block", [300_000, 250_123], ids=["aligned", "ragged"])
@pytest.mark.parametrize("bpl", [2, 3])
@pytest.mark.parametrize("nperseg,impl", D_KERNELS, ids=["n256-auto", "n256-generic", "n1024-auto", "n512-generic", "n8-generic"])
def test_blocks_per_launch_equal_one_block_per_launch(nperseg, impl, bpl, block):
    """3 streams x 7 blocks (the last launch padded).  Where the same spectrogram kernel runs, every analyzer unit equals the
    one-block-per-launch run byte for byte (the carry of unit s is unit s - 1 of the same launch).  At a ragged length the
    register and the radix-16 kernel cannot read the blocks of a launch with 16-byte copies and the generic kernel runs: those
    units are checked against the oracle."""
    kw = _kw(FS, block, nperseg)
    cap = _d_capture(nperseg, block)
    same_kernel = not (impl == E.FFT_AUTO and nperseg in (256, 1024) and block % 8)
    one = _d_one_block_per_launch(nperseg, impl, block)
    oracle = None if same_kernel else [_oracle(dict(kw, device=str(s)), cap[:, s]) for s in range(D_STREAMS)]
    ba = BatchAnalyzer(**parity.batch_kwargs(kw, devices=[str(s) for s in range(D_STREAMS)], calibration=[0.0] * D_STREAMS,
                                             fft_impl=impl, blocks_per_launch=bpl))
    n_rec = 0
    try:
        for b0 in range(0, D_BLOCKS, bpl):
            blk = np.zeros((D_STREAMS, bpl, cap.shape[2]), dtype=np.uint8)
            nblk = min(bpl, D_BLOCKS - b0)
            blk[:, :nblk] = cap[b0:b0 + nblk].transpose(1, 0, 2)
            rec = ba.engine.process(blk)
            per_unit = None if same_kernel else ba.finalize(rec, [_ts(kw, b0)] * D_STREAMS)
            for s in range(D_STREAMS):
                for j in range(nblk):
                    u, b = s * bpl + j, b0 + j
                    if same_kernel:
                        assert _strip(rec, u).tobytes() == _strip(one[b], s).tobytes(), (s, b)
                        n_rec += len(_strip(one[b], s))
                    else:
                        P, want = oracle[s]
                        S, last, found = want[b]
                        sigs, keys = per_unit[u]
                        st = parity.compare_block(P, S, last, found, sigs, keys)
                        assert st["near_threshold_mismatch"] == 0, (s, b, st)
                        n_rec += len(keys)
    finally:
        ba.close()
    assert n_rec >= 20


# ---------------------------------------------------------------------------------------------------------------------------
# E: engines of different nperseg in one process
# ---------------------------------------------------------------------------------------------------------------------------
def test_engines_of_different_nperseg_share_the_process():
    """The generic kernel's shared-memory limit is a property of the kernel: an engine created later with a smaller nperseg must
    not take away what a larger one needs (81 936 bytes at 4096)."""
    setups = [(4096, 2_400_000, 2_400_000), (256, FS, FS), (512, FS, FS)]        # created in this order
    runs = []
    try:
        for n, fs, block in setups:
            kw = _kw(fs, block, n)
            cap = synth.make_stream(_workload(fs, block, n, amp_lsb=(10.0, 30.0)), 1, 2)
            ba = BatchAnalyzer(**parity.batch_kwargs(kw, fft_impl=E.FFT_GENERIC))
            ba.engine                                                                  # create it now
            runs.append((kw, cap, ba) + _oracle(kw, cap))
        for b in range(2):                                                             # interleaved launches
            for kw, cap, ba, P, want in runs:
                S, last, found = want[b]
                _, sigs, keys = ba.process_blocks(cap[b][None, :], [_ts(kw, b)])[0]
                st = parity.compare_block(P, S, last, found, sigs, keys)
                assert st["near_threshold_mismatch"] == 0 and st["gpu"] > 0, (kw["fft_nperseg"], st)
                parity.compare_spectrogram(P, S, ba.engine.read_spectrogram(0), ba.engine.read_row_means(0),
                                           tag=f"shapes/shared/n{kw['fft_nperseg']}/b{b}")
    finally:
        for r in runs:
            r[2].close()


def test_radix16_fallback_after_a_smaller_engine_exists():
    """nperseg 4096 AUTO fed device input that is not 16-byte aligned: the radix-16 kernel cannot take it and the launch runs
    the generic kernel, after an engine with a smaller nperseg was created."""
    torch = pytest.importorskip("torch")
    n, fs, block = 4096, 2_400_000, 2_400_000
    kw = _kw(fs, block, n)
    cap = synth.make_stream(_workload(fs, block, n, amp_lsb=(10.0, 30.0)), 2, 2)
    P, want = _oracle(kw, cap)
    big = BatchAnalyzer(**parity.batch_kwargs(kw, fft_impl=E.FFT_AUTO))
    small = BatchAnalyzer(**parity.batch_kwargs(_kw(FS, FS, 256), fft_impl=E.FFT_GENERIC))
    try:
        big.engine
        small.engine
        small_cap = synth.make_stream(synth.C1, 3, 2)
        for b in range(2):
            buf = torch.empty(cap.shape[1] + 16, dtype=torch.uint8, device="cuda")
            view = buf[2:2 + cap.shape[1]]                                             # 2-byte aligned, not 16-byte aligned
            view.copy_(torch.from_numpy(cap[b]))
            assert view.data_ptr() % 16 != 0
            S, last, found = want[b]
            _, sigs, keys = big.process_blocks(view, [_ts(kw, b)])[0]
            st = parity.compare_block(P, S, last, found, sigs, keys)
            assert st["near_threshold_mismatch"] == 0 and st["gpu"] > 0, st
            parity.compare_spectrogram(P, S, big.engine.read_spectrogram(0), big.engine.read_row_means(0), tag=f"shapes/r16-fallback/b{b}")
            assert len(small.engine.process(small_cap[b][None, :])) > 0
    finally:
        big.close()
        small.close()
