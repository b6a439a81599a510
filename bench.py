#!/usr/bin/env python
"""bench.py — the benchmark of the B200 signal path: one JSON result line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload at N=1 = BASELINE.json configs[1] ("c2"): 256 streams x 1080p, CHROM_GREEN ROI sampling,
[DETREND_LINEAR, FILTER_FIR], Welch HR, W=300, T=64 frames per stream resident in HBM per step (102 GB of the
180 GB, far larger than the 126 MB L2, so nothing is cached between steps; `--frames-per-step 32` = the round-1 depth:
the launch ramp / tail and ~80 MB of dirty window scratch left in L2 cost F1 0.64 of the HBM peak there against 0.74 at 64,
profiles/r2q_discard_depth_ab.txt).  One step = the whole hot path over
one batch: ROI-sample S*T frames, push, and evaluate the sliding window after EVERY frame, as the
reference's process() does (S*T window jobs -> R bpm + P ptt each).  metric = ROI-sampled frames/s.
N>1: every rank owns S streams (weak scaling, no data-path collective); the 24-byte per-job records are
all-gathered over NCCL inside the timed region, one step behind the compute (bpv.dist.RecordGather).

`--impl reference` times the UNMODIFIED reference (`baseline/_ref`, a git-ignored copy of the reference's own
modules that `__graft_entry__.build()` makes where the upstream project is checked out at `__graft_entry__.REFERENCE`):
`SignalProcessor.process` per frame, one process per host core, one stream each.  The oracle port
(`oracle/bpv_oracle.py`) is the fallback when that copy is missing, and is reported beside it.

`--dump-outputs DIR` writes what the last timed step returned (`dump_outputs`), for comparing two builds output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, 'bp-from-video_b200')
REF_DIR = os.path.join(ROOT, 'baseline', '_ref')
REF_MODULES = ('signal_processor.py', 'signal_data.py', 'roi.py', 'model.py', 'profiler.py', 'exceptions.py')
sys.path.insert(0, PKG)
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: S, H, W, T, window, channel, methods, transform, fps, kwargs
    'c2': dict(S=256, H=1080, W=1920, T=64, window=300, channel='CHROM_GREEN', methods=['DETREND_LINEAR', 'FILTER_FIR'],
               transform='PGRAM_WELCH', fps=30.0, kw={},
               desc='BASELINE configs[1]: 256 streams 1080p 30 fps, chrom-green ROI + detrend + FIR + Welch HR'),
    'c2small': dict(S=32, H=1080, W=1920, T=8, window=300, channel='CHROM_GREEN', methods=['DETREND_LINEAR', 'FILTER_FIR'],
                    transform='PGRAM_WELCH', fps=30.0, kw={}, desc='reduced c2 for quick checks (not a bench line)'),
}
# The other shapes BASELINE.json names, reported beside the headline (`other_shapes`): one new frame per stream per step.
# irregular = cumsum(1/fps (1 + U(-0.3, 0.3))) timestamps; p_nan = missed detections (NaN samples).
OTHER_SHAPES = {
    'c1_batched': dict(S=4096, H=480, W=640, T=1, window=300, channel='GREEN', methods=['FILTER_BUTTER'], transform='PGRAM_LS',
                       fps=30.0, kw=dict(min_freq=0.7), irregular=False, p_nan=0.01,
                       desc='configs[0] shape batched: 4096 streams 640x480, green-mean + Butterworth 0.7-4 Hz + Lomb-Scargle (F = n), 10 s window'),
    'c3': dict(S=4096, H=0, W=0, T=1, window=300, channel='GREEN', methods=[], transform='PGRAM_LS', fps=30.0,
               kw=dict(ls_num_freqs=2048), irregular=True, p_nan=0.05,
               desc='configs[2]: 4096 streams, irregular timestamps, Lomb-Scargle on a 2048-frequency grid, no interpolation (signals only)'),
    'c4': dict(S=1024, H=720, W=1280, T=1, window=1200, channel='GREEN', methods=['INTERP_CUBIC', 'FILTER_BUTTER'],
               transform='PGRAM_LS', fps=120.0, kw={}, irregular=True, p_nan=0.01,
               desc='configs[3]: 1024 streams 720p 120 fps, cubic-spline resample + Butterworth + Lomb-Scargle HR + PTT over 2399 lags'),
    'c5': dict(S=65536, H=480, W=640, T=1, window=300, channel='GREEN', methods=['FILTER_BUTTER'], transform='PGRAM_LS',
               fps=30.0, kw=dict(min_freq=0.7), irregular=False, p_nan=0.01,
               desc='configs[4]: 65536 streams x 10 s windows over all GPUs, ROI -> Butterworth -> Lomb-Scargle -> HR -> PTT + NCCL record gather'),
}
METRIC, UNIT = 'roi_sampled_frames_per_s', 'frames/s'
# --dump-outputs: the StepResult fields a caller of BatchedSignalProcessor.step receives
DUMP_FIELDS = ('samples', 'peak_freq', 'peak_idx', 'peak_mag', 'lag_sec', 'lag_idx', 'lag_corr', 'status')
DUMP_MAX_BYTES = 64 << 20
# dram__bytes_read.sum + dram__bytes_write.sum of one c2 F1 launch of 16 384 frames (ncu --set full; profiles/r2y_c2_summary.md:
# 664.3 + 4.0 and 664.4 + 5.9 MB for the two captured launches, same boxes); 337.2 MB for the 8192-frame launch of round 1
ROI_NCU_TRAFFIC_BYTES = 669.3e6
FRAME_PERIOD_MS = 1000.0 / 30.0


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return json.load(open(p))['hbm_gbs'], 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def shape_config(name, wl, world=1, windows='every_frame'):
    """The `config` object of the JSON line: identical in both arms for the same workload."""
    S, T = wl['S'], wl['T']
    jobs = S * (T if windows == 'every_frame' else 1)
    return {'workload': name, 'desc': wl['desc'], 'streams_per_gpu': S, 'frames_per_stream_per_step': T,
            'frame': f"{wl['W']}x{wl['H']}x3 u8 BGR", 'window': wl['window'], 'rois': 2, 'windows': windows,
            'window_jobs_per_step': jobs * world,
            'l2_policy': f"inputs ({S * T * wl['H'] * wl['W'] * 3 / 1e9:.0f} GB of frames per GPU) larger than the 126 MB L2",
            'parallelism': f'streams sharded x{world}, NCCL all-gather of per-stream records' if world > 1 else 'single GPU'}


# ------------------------------------------------------------------------------------------------
# CPU arms: the unmodified reference (baseline/_ref) or the oracle port, one stream per host core
# ------------------------------------------------------------------------------------------------
_W = {}          # per-worker state (processor, synthetic feed)


def reference_available():
    return all(os.path.exists(os.path.join(REF_DIR, m)) for m in REF_MODULES)


def _cpu_init(wl, kind, seed_base):
    """Pool initializer: build ONE stream's processor in this worker and bring its window to steady state."""
    import warnings
    warnings.simplefilter('ignore')
    os.environ['OMP_NUM_THREADS'] = os.environ['OPENBLAS_NUM_THREADS'] = '1'
    from bpv import synth
    seed = seed_base + os.getpid() % 100000
    rng = np.random.default_rng(seed)
    H, W, win = max(wl['H'], 8), max(wl['W'], 8), wl['window']
    n_feed = 4096
    ts = synth.timestamps(rng, win + n_feed, wl['fps'], irregular=wl.get('irregular', False),
                          drop=0.05 if wl.get('irregular', False) else 0.0, origin=1.0)
    raw0 = synth.raw_signals(rng, ts[:win], p_nan=wl.get('p_nan', 0.0))
    pool = rng.integers(0, 256, (4, H, W, 3), dtype=np.uint8)       # 4 distinct frames, cycled
    _W.update(kind=kind, wl=wl, ts=ts, pool=pool, i=0, win=win)
    if kind == 'reference':
        for name in ('roi', 'signal_data', 'signal_processor', 'model', 'profiler', 'exceptions'):
            sys.modules.pop(name, None)
        if PKG in sys.path:
            sys.path.remove(PKG)              # our drop-in modules of the same names must not shadow the reference's
        sys.path.insert(0, REF_DIR)
        import signal_processor as sp
        import profiler
        assert os.path.dirname(os.path.abspath(sp.__file__)) == REF_DIR, sp.__file__
        profiler.profiler.enabled = False     # as pbp.py:11 (cProfile off)
        sys.path.insert(1, PKG)
        proc = sp.SignalProcessor(None, 1, win, 50, color_channel=sp.SignalColorChannel[wl['channel']],
                                  processing_methods=[sp.SignalProcessingMethod[m] for m in wl['methods']],
                                  spectrum_transform=sp.SignalSpectrumTransform[wl['transform']], **wl['kw'])
        for k in range(win):                  # steady state through the reference's own ring API (signal_data.py:94-98)
            proc.store.sg_raw.add_samples(float(ts[k]), [float(raw0[0, k]), float(raw0[1, k])])
        _W.update(proc=proc, det=synth.detections(rng, n_feed, H, W))
    else:
        from oracle import bpv_oracle as orc
        st = orc.OracleStream(2, 1, win, 50, getattr(orc, wl['channel']), [getattr(orc, m) for m in wl['methods']],
                              getattr(orc, wl['transform']), **wl['kw'])
        st.t[:] = ts[:win]
        st.raw[:] = raw0
        _W.update(proc=st, boxes=synth.roi_boxes(rng, n_feed, H, W), NO_BOX=synth.NO_BOX)


def _cpu_run(frames):
    """Time `frames` calls of the per-frame step in this worker; returns (seconds, frames)."""
    from bpv import synth
    w = _W
    t0 = time.perf_counter()
    for _ in range(frames):
        i = w['i']
        w['i'] += 1
        ts = float(w['ts'][w['win'] + i])
        frame = w['pool'][i % 4]
        if w['kind'] == 'reference':
            w['proc'].process(synth.FrameData(frame, ts), synth.ModelResults(w['det'], i % len(w['det']['present'])))
        else:
            b = w['boxes'][i % len(w['boxes'])]
            rois = [(np.nan,) * 6 if b[r, 0] == w['NO_BOX'] else (0, 0, *[int(v) for v in b[r]]) for r in range(2)]
            w['proc'].process(frame, ts, rois)
    return time.perf_counter() - t0, frames


class CpuArm:
    """`procs` worker processes, one stream each (streams are independent); rates exclude process start + prefill."""

    def __init__(self, wl, kind, procs):
        import multiprocessing as mp
        self.kind, self.procs = kind, procs
        self.pool = mp.get_context('spawn').Pool(procs, initializer=_cpu_init, initargs=(wl, kind, 1000))

    def step(self, frames_per_core):
        res = self.pool.map(_cpu_run, [frames_per_core] * self.procs, chunksize=1)
        return sum(f / t for t, f in res), max(t for t, _ in res)        # aggregate frames/s, slowest worker seconds

    def close(self):
        self.pool.terminate()
        self.pool.join()


def cpu_rate(wl, kind, procs, frames_per_core, reps=1, warm=1):
    arm = CpuArm(wl, kind, procs)
    try:
        for _ in range(warm):
            arm.step(max(1, frames_per_core // 4))
        out = [arm.step(frames_per_core) for _ in range(reps)]
    finally:
        arm.close()
    return out


def run_reference(args, wl):
    """--impl reference: the reference's own CPU implementation of the path on all host cores.  Each "step" is a bounded
    sample of the workload (a few frames of one stream per core); rank 0 only."""
    if int(os.environ.get('RANK', 0)) != 0:
        return
    cores = os.cpu_count() or 1
    kind = 'reference' if reference_available() and not args.port else 'port'
    per_frame = 0.025 if kind == 'reference' else 0.006           # s per frame per core (c2), to size a step
    total = max(1, args.warmup + args.steps)
    per = int(max(4, min(args.ref_frames, args.ref_budget_s / (total * per_frame))))
    arm = CpuArm(wl, kind, cores)
    try:
        for _ in range(args.warmup):
            arm.step(per)
        res = [arm.step(per) for _ in range(args.steps)]
    finally:
        arm.close()
    v = float(np.median([r for r, _ in res]))
    what = ('the UNMODIFIED reference (baseline/_ref copy of signal_processor.py / signal_data.py / roi.py): '
            'SignalProcessor.process per frame incl. calc_rois, deques and copy.deepcopy' if kind == 'reference'
            else 'oracle port of SignalProcessor.process per frame (numpy/scipy, same calls as the reference)')
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': 1e3 * float(np.median([t for _, t in res])), 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': shape_config(args.workload, wl, 1, args.windows),
        'cpu_baseline': {'value': v, 'unit': UNIT, 'cores': cores, 'kind': kind,
                         'sample': f'each step = {cores} streams x {per} steady-state frames (window prefilled), {what}, '
                                   f'one process per core, cProfile off'},
        'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '20',
                                          '-i', str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        reasons = set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            for k, nm in enumerate(names):
                if len(r) > 4 + k and r[4 + k].lower().startswith('active'):
                    reasons.add(nm)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def make_frames_device(torch, S, T, H, W, seed, dev):
    """Synthetic frames in HBM: skin-tone base + per-(stream, frame) pulse on G + uniform noise +-8 (SURVEY 8d)."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    frames = torch.empty((S, T, H, W, 3), dtype=torch.uint8, device=dev)
    base = torch.tensor([110, 140, 190], dtype=torch.int16, device=dev)
    f_pulse = torch.rand(S, generator=g, device=dev) * 2.2 + 0.8
    tt = (torch.arange(T, device=dev) + 1) / 30.0
    pulse = (2.0 * torch.sin(2 * math.pi * f_pulse[:, None] * tt[None, :])).round().to(torch.int16)   # [S, T]
    chunk = max(1, min(S, int(2.5e8 // (T * H * W * 3))))
    for s in range(0, S, chunk):
        e = min(S, s + chunk)
        noise = torch.randint(-8, 9, (e - s, T, H, W, 3), generator=g, device=dev, dtype=torch.int16)
        noise += base
        noise[..., 1] += pulse[s:e][:, :, None, None]
        frames[s:e] = noise.clamp_(0, 255).to(torch.uint8)
        del noise
    return frames


def device_signals(torch, S, n, fps, irregular, p_nan, seed, dev):
    """Signals-only synthetic input generated on the device: timestamps f64 [S, n] (regular (i+1)/fps, or the cumulative
    sum of jittered periods with a per-stream origin) and ROI-mean-like samples f64 [S, n, 2] (DC 120, pulse 0.5, drift,
    noise 0.15; ROI 1 delayed by 30 ms; p_nan of the samples missing)."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    f64 = torch.float64
    if irregular:
        dt = (1.0 / fps) * (1.0 + (torch.rand((S, n), generator=g, device=dev, dtype=f64) * 0.6 - 0.3))
        ts = torch.cumsum(dt, dim=1) + torch.rand((S, 1), generator=g, device=dev, dtype=f64) * 1000.0
    else:
        ts = ((torch.arange(n, device=dev, dtype=f64) + 1) / fps)[None, :].expand(S, n).contiguous()
    f = torch.rand((S, 1, 1), generator=g, device=dev, dtype=f64) * 2.2 + 0.8
    r = torch.arange(2, device=dev, dtype=f64)[None, None, :]
    tt = (ts - ts[:, :1])[:, :, None] - 0.03 * r
    y = (120.0 + 3.0 * r + 0.5 * torch.sin(2 * math.pi * f * tt) + 0.1 * torch.sin(4 * math.pi * f * tt + 0.7)
         + 0.3 * torch.sin(2 * math.pi * 0.11 * tt + r) + 0.15 * torch.randn((S, n, 2), generator=g, device=dev, dtype=f64))
    if p_nan > 0:
        y = torch.where(torch.rand((S, n, 2), generator=g, device=dev) < p_nan, torch.full_like(y, float('nan')), y)
    return ts.contiguous(), y.contiguous()


def roi_bytes(boxes_np, H, W):
    x0, y0, x1, y1 = [boxes_np[..., i].astype(np.int64) for i in range(4)]
    valid = boxes_np[..., 0] != np.iinfo(np.int32).min

    def sl(a, b, L):
        a = np.where(a < 0, np.maximum(a + L, 0), np.minimum(a, L))
        b = np.where(b < 0, np.maximum(b + L, 0), np.minimum(b, L))
        return np.maximum(b - a, 0)
    return int((3 * sl(x0, x1, W) * sl(y0, y1, H) * valid).sum())


def granule_bytes(boxes_np, H, W, row_stride, frame_stride, gran):
    """Bytes of the distinct `gran`-byte aligned granules the ROI rows of a launch touch (frame f at f*frame_stride):
    the DRAM traffic an ideal kernel generates when the L2 fills in `gran`-byte units."""
    b = boxes_np.reshape(-1, boxes_np.shape[-2], 4).astype(np.int64)
    total = 0
    for r in range(b.shape[1]):
        x0, y0, x1, y1 = b[:, r, 0], b[:, r, 1], b[:, r, 2], b[:, r, 3]
        valid = x0 != np.iinfo(np.int32).min
        cl = lambda a, L: np.where(a < 0, np.maximum(a + L, 0), np.minimum(a, L))
        xs, xe, ys, ye = cl(x0, W), cl(x1, W), cl(y0, H), cl(y1, H)
        ok = valid & (xe > xs) & (ye > ys)
        f = np.arange(b.shape[0])[ok]
        xs, xe, ys, ye = xs[ok], xe[ok], ys[ok], ye[ok]
        for i in range(f.size):
            rows = np.arange(ys[i], ye[i])
            a = f[i] * frame_stride + rows * row_stride + 3 * xs[i]
            e = f[i] * frame_stride + rows * row_stride + 3 * xe[i] - 1
            total += int(((e // gran) - (a // gran) + 1).sum()) * gran
    return total


def measure_fma_peaks(torch, dev):
    """FP64 and FP32 FMA throughput of this GPU, measured live (bpv_probe_fma: 8 independent FMA chains per thread,
    148 x 8 CTAs of 256 threads), best of 3; TFLOP/s with 2 flop per FMA."""
    from bpv import ops
    sink = torch.zeros(2, dtype=torch.float64, device=dev)
    out = {}
    for name, iters in (('f64', 1 << 13), ('f32', 1 << 15)):
        best = 0.0
        for _ in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            n = ops.probe_fma(name, iters, 148 * 8, sink)
            e1.record()
            torch.cuda.synchronize(dev)
            best = max(best, 2.0 * n / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        out[name] = best
    return out


def measure_pcie(torch, dev):
    """Host -> device copy bandwidth from pinned memory (GB/s), 256 MiB, best of 3."""
    h = torch.empty(256 << 20, dtype=torch.uint8, pin_memory=True)
    d = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    best = 0.0
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        d.copy_(h, non_blocking=True)
        e1.record()
        torch.cuda.synchronize(dev)
        best = max(best, h.numel() / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    return best


def measure_pcie_concurrent(torch, dev, tdist, world):
    """N > 1: every rank copies 256 MiB of pinned memory to its GPU AT THE SAME TIME, 8 times back to back; returns
    (sum over ranks, slowest rank) in GB/s — the host-side ceiling the N-GPU e2e number lives under (the GPUs' PCIe links share
    host bridges / memory channels), measured with nothing of this repo's kernels involved."""
    h = torch.empty(256 << 20, dtype=torch.uint8, pin_memory=True)
    d = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    d.copy_(h, non_blocking=True)
    torch.cuda.synchronize(dev)
    tdist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(8):
        d.copy_(h, non_blocking=True)
    e1.record()
    torch.cuda.synchronize(dev)
    mine = 8 * h.numel() / (e0.elapsed_time(e1) * 1e-3) / 1e9
    t = torch.tensor([mine, -mine], dtype=torch.float64, device=dev)
    tot = t.clone()
    tdist.all_reduce(tot, op=tdist.ReduceOp.SUM)
    tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
    return float(tot[0].item()), float(-t[1].item())


def time_family_wrappers(torch, ops, fam, only=None):
    """Wrap the ops launchers (all, or those named in `only`) so every call is bracketed by CUDA events on the stream it
    launches on."""
    names = dict(roi_sample='roi', ring_push='push', window_preprocess='preprocess', window_design='design',
                 window_filter='preprocess', window_spectrum='spectrum', window_xcorr='xcorr', window_welch_xcorr='spectrum_xcorr')
    if only is not None:
        names = {k: v for k, v in names.items() if k in only}
    orig = {k: getattr(ops, k) for k in names}

    def timed(fn, key):
        def wrap(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn(*a, **k)
            e1.record()
            fam.setdefault(key, []).append((e0, e1))
            return out
        return wrap
    for k, fn in orig.items():
        setattr(ops, k, timed(fn, names[k]))
    return orig


def _time_launches(torch, fn, iters=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(iters + 1)]
    ev[0].record()
    for i in range(iters):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    return float(np.median([ev[i].elapsed_time(ev[i + 1]) for i in range(iters)]))


def run_ingest_resized(torch, frames, boxes_np, channel, peak):
    """SURVEY 8f row 2 beside the headline: F1 with the VideoReader resize fused in front (1080p frames in HBM sampled as if
    cv2.resize had produced 720p; boxes scaled to the 720p frame).  Same frames / launch size as the timed region."""
    from bpv import ops, synth
    S, T, H, W = frames.shape[:4]
    dh, dw = H * 2 // 3, W * 2 // 3
    b = boxes_np.reshape(S * T, 2, 4).copy()
    ok = b[..., 0] != synth.NO_BOX
    b[ok] = np.rint(b[ok] * (dw / W)).astype(np.int32)
    bd = torch.from_numpy(b).to(frames.device)
    fr = frames.view(S * T, H, W, 3)
    ms = _time_launches(torch, lambda: ops.roi_sample_resized(fr, dh, dw, bd, channel))
    src_bytes = roi_bytes(boxes_np, H, W)                     # the source footprint of the scaled boxes ~ the original boxes
    return {'resized_720p': {'us_per_launch': ms * 1e3, 'frames_per_s': S * T / ms * 1e3, 'alg_bytes': int(src_bytes),
                             'gbs': src_bytes / ms / 1e6, 'frac_hbm': src_bytes / ms / 1e6 / peak,
                             'desc': f'{S * T} frames {W}x{H} BGR in HBM, boxes in the {dw}x{dh} frame cv2.resize would produce; 3 B per source pixel'}}


def run_ingest_nv12(torch, dev, boxes_np, S, T, H, W, channel, peak):
    """F1 straight from NV12 decoder surfaces (1.5 B/px) in HBM, same boxes and launch size as the timed region."""
    from bpv import ops
    nv = torch.empty((S * T, H * 3 // 2, W), dtype=torch.uint8, device=dev)
    for i in range(0, S * T, 256):
        nv[i:i + 256].random_(0, 256)
    bd = torch.from_numpy(boxes_np.reshape(S * T, 2, 4).copy()).to(dev)
    ms = _time_launches(torch, lambda: ops.roi_sample_nv12(nv, H, W, bd, channel))
    alg = roi_bytes(boxes_np, H, W) / 2                       # 1.5 B/px instead of 3
    del nv
    torch.cuda.empty_cache()
    return {'nv12': {'us_per_launch': ms * 1e3, 'frames_per_s': S * T / ms * 1e3, 'alg_bytes': int(alg), 'gbs': alg / ms / 1e6,
                     'frac_hbm': alg / ms / 1e6 / peak,
                     'desc': f'{S * T} NV12 surfaces {W}x{H} (Y plane + interleaved UV plane) in HBM; 1.5 B per ROI pixel'}}


def run_other_shape(torch, name, wl, dev, world, steps=6, with_frames=True):
    """One of the other BASELINE shapes on this rank's GPU: prefill the rings, then `steps` timed steps of one new frame per
    stream (F1 when the shape has frames, push, F2, F3, F4; window evaluated once per step per stream); N > 1: + gather."""
    from bpv import _cabi, dist as bdist, synth
    from bpv.engine import BatchedSignalProcessor
    import torch.distributed as tdist
    S = wl['S'] // world if name == 'c5' else wl['S']
    H, W, win, T = wl['H'], wl['W'], wl['window'], wl['T']
    frames_bytes = S * T * H * W * 3
    use_frames = with_frames and H > 0 and frames_bytes <= 24e9
    Tpre = 50
    eng = BatchedSignalProcessor(S, 2, signal_max_samples=win, max_frames_per_step=Tpre,
                                 color_channel=getattr(_cabi, wl['channel']), processing_methods=[getattr(_cabi, m) for m in wl['methods']],
                                 spectrum_transform=getattr(_cabi, wl['transform']), windows='last', device=dev,
                                 roi_pixels_hint=int(0.05 * W * 0.06 * H), **wl['kw'])
    n_total = win + steps + 4
    ts, y = device_signals(torch, S, n_total, wl['fps'], wl['irregular'], wl['p_nan'], 4321 + int(os.environ.get('RANK', 0)), dev)
    for a in range(0, win, Tpre):
        b = min(win, a + Tpre)
        eng.step_signals(y[:, a:b].contiguous(), ts[:, a:b].contiguous())
    frames = boxes = None
    if use_frames:
        rng = np.random.default_rng(99)
        frames = make_frames_device(torch, S, T, H, W, 5, dev)
        one = synth.roi_boxes(rng, 64, H, W)
        boxes = torch.from_numpy(one[np.arange(S) % 64][:, None]).to(dev).contiguous()      # [S, 1, R, 4]
    rg = bdist.RecordGather()

    def one_step(k):
        tk = ts[:, win + k:win + k + 1].contiguous()
        if use_frames:
            res = eng.step(frames, boxes, tk)
        else:
            res = eng.step_signals(y[:, win + k:win + k + 1].contiguous(), tk)
        if world > 1:
            rg.launch(res.packed32())
            rg.collect()
        return res
    for k in range(3):
        one_step(k)
    if world > 1:
        tdist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(3, 3 + steps):
        res = one_step(k)
    if world > 1:
        rg.flush()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    if world > 1:
        tt = torch.tensor([ms], dtype=torch.float64, device=dev)
        tdist.all_reduce(tt, op=tdist.ReduceOp.MAX)
        ms = float(tt.item())
    finite = float(torch.isfinite(res.peak_freq).double().mean().item())
    out = {'desc': wl['desc'], 'streams': S * world, 'streams_per_gpu': S, 'window': win, 'ms_per_step': ms,
           'windows_per_s': S * world / (ms * 1e-3), 'frames_in_hbm': bool(use_frames), 'finite_hr_frac': finite}
    if name == 'c5':
        out['frame_period_ms'] = FRAME_PERIOD_MS
        out['under_one_frame_period'] = bool(ms < FRAME_PERIOD_MS)
    del eng, frames, ts, y
    torch.cuda.empty_cache()
    return out


def run_latency_c1(torch, dev, frames_n=60):
    """BASELINE configs[0] as the reference runs it: ONE 640x480 stream through the drop-in SignalProcessor.process()
    (host frame in, SignalStore of numpy objects out), per-frame latency in steady state."""
    import signal_processor as sp
    from bpv import synth
    assert os.path.dirname(os.path.abspath(sp.__file__)) == PKG, sp.__file__
    rng = np.random.default_rng(3)
    H, W, win = 480, 640, 300
    proc = sp.SignalProcessor(None, 1, win, 50, color_channel=sp.SignalColorChannel.GREEN,
                              processing_methods=[sp.SignalProcessingMethod.FILTER_BUTTER],
                              spectrum_transform=sp.SignalSpectrumTransform.PGRAM_LS, min_freq=0.7)
    n = win + frames_n + 8
    ts = synth.timestamps(rng, n, 30.0)
    det = synth.detections(rng, n, H, W)
    pool = synth.frames(rng, ts[:8], H, W)
    for i in range(win + 8):
        proc.process(synth.FrameData(pool[i % 8], float(ts[i])), synth.ModelResults(det, i))
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for i in range(win + 8, n):
        store = proc.process(synth.FrameData(pool[i % 8], float(ts[i])), synth.ModelResults(det, i))
    dt = (time.perf_counter() - t0) / frames_n
    bpm = [float(v) for v in np.asarray(store.sg_bpm.signals[0].y)[-1:]]
    return {'ms_per_frame': dt * 1e3, 'frames_per_s': 1.0 / dt, 'last_bpm': bpm,
            'how': 'drop-in SignalProcessor.process (S=1 engine, store_arrays=True): host BGR frame in, deep-copied SignalStore out'}


def dump_outputs(res, out_dir):
    """Write the StepResult `res` as out_dir/<field>.npy, float64 (the int32 bins and status convert exactly).  The inputs
    of a run are fixed by its arguments, so two builds of the project run with the same arguments compare file for file.
    Every file holds finite values: the path reports "none" as NaN (a missed detection or a box outside the frame gives a
    NaN ROI sample, a window without a peak NaN bpm), so each floating-point field is written with its non-finite entries
    as 0 beside <field>_nonfinite.npy, which holds 1 where the value was NaN, 2 for +inf, 3 for -inf and 0 elsewhere.
    All of it is written: at c2 it is 2.8 MB, and the frames in HBM bound any shape far below DUMP_MAX_BYTES."""
    arrays = {}
    for k in DUMP_FIELDS:
        t = getattr(res, k)
        a = t.double().cpu().numpy()
        if t.is_floating_point():
            bad = ~np.isfinite(a)
            arrays[f'{k}_nonfinite'] = np.select([np.isnan(a), a > 0], [1.0, 2.0], 3.0) * bad
            a = np.where(bad, 0.0, a)
        arrays[k] = a
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise ValueError(f'--dump-outputs: {total} bytes of outputs, more than {DUMP_MAX_BYTES}')
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f'{k}.npy'), a)


def run_gpu(args, wl):
    import torch
    from bpv import _cabi, dist as bdist, synth
    from bpv.engine import BatchedSignalProcessor
    import torch.distributed as tdist
    rank, local, world = bdist.init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    numa = bdist.bind_to_gpu_numa_node(local) if args.numa else None
    S, T, H, W, win = wl['S'], wl['T'], wl['H'], wl['W'], wl['window']
    methods = [getattr(_cabi, m) for m in wl['methods']]
    eng = BatchedSignalProcessor(S, 2, signal_max_samples=win, max_frames_per_step=T, color_channel=getattr(_cabi, wl['channel']),
                                 processing_methods=methods, spectrum_transform=getattr(_cabi, wl['transform']),
                                 windows=args.windows, device=dev, roi_pixels_hint=int(0.05 * W * 0.06 * H), **wl['kw'])
    rng = np.random.default_rng(1234 + rank)
    frames = make_frames_device(torch, S, T, H, W, 77 + rank, dev)
    boxes_np = np.stack([synth.roi_boxes(rng, T, H, W) for _ in range(S)])
    boxes = torch.from_numpy(boxes_np).to(dev)
    alg_roi_bytes = roi_bytes(boxes_np, H, W)
    fps = wl['fps']
    # prefill the rings with `win` synthetic samples so every timed window is full (steady state)
    ts0 = np.stack([synth.timestamps(rng, win, fps) for _ in range(S)])
    raw0 = np.stack([synth.raw_signals(rng, ts0[s]).T for s in range(S)])            # [S, win, R]
    eng.windows, keep = 'last', eng.windows
    for a in range(0, win, T):
        eng.step_signals(torch.from_numpy(raw0[:, a:a + T].copy()).to(dev), torch.from_numpy(ts0[:, a:a + T].copy()).to(dev))
    eng.windows = keep
    t_next = [float(ts0[0, -1])]
    W_UP = max(3, args.warmup)
    # timestamps of every step are synthetic inputs too: resident in HBM before the timed region ([steps, S, T] float64)
    PROF_STEPS = min(args.steps, 20)                          # family profile pass after the timed region
    n_steps = W_UP + args.steps + PROF_STEPS
    ts_all = (t_next[0] + (torch.arange(n_steps * T, device=dev, dtype=torch.float64) + 1) / fps).view(n_steps, 1, T).expand(n_steps, S, T).contiguous()
    t_next[0] += n_steps * T / fps
    step_no = [0]
    gather = bdist.RecordGather()
    recbuf = [None, None]

    def one_step():
        ts = ts_all[step_no[0]]
        k = step_no[0] & 1
        step_no[0] += 1
        res = eng.step(frames, boxes, ts)
        recbuf[k] = res.packed32(out=recbuf[k])           # the 24-byte record per window job (bpm, ptt, bins)
        gather.launch(recbuf[k])                          # N > 1: NCCL all-gather, collected one step later
        gather.collect()
        return res

    def barrier():
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize(dev)

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
        time.sleep(0.1)
    for _ in range(W_UP):
        one_step()
    barrier()
    # ---- timed region: exactly K steps between two CUDA events; inside it only F1 (the roofline kernel) is bracketed by
    # its own events — every extra event pair costs launch-queue time that is not part of the path
    from bpv import ops
    fam = {}
    orig = time_family_wrappers(torch, ops, fam, only=('roi_sample',))
    barrier()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(args.steps):
        res = one_step()
    gather.flush()
    stop.record()
    barrier()
    for k, fn in orig.items():
        setattr(ops, k, fn)
    if args.dump_outputs and rank == 0:
        dump_outputs(res, args.dump_outputs)              # before the profile pass below reuses the result buffers
    ms = start.elapsed_time(stop)
    launches_per_step = eng.launches_per_step + 1            # of the timed steps: the engine's own count + pack_records32
    clk = clocks.stop() if rank == 0 else None
    if world > 1:
        tt = torch.tensor([ms], dtype=torch.float64, device=dev)
        tdist.all_reduce(tt, op=tdist.ReduceOp.MAX)
        ms = float(tt.item())
    roi_ms = float(np.mean([a.elapsed_time(b) for a, b in fam['roi']]))
    # ---- the other kernel families (informational `kernels` block, `roofline_by_time`): the same steps again, right after
    # the timed region, with every launcher bracketed by events on its launch stream
    fam = {}
    prof_steps = PROF_STEPS
    orig = time_family_wrappers(torch, ops, fam)
    for _ in range(prof_steps):
        one_step()
    gather.flush()
    barrier()
    for k, fn in orig.items():
        setattr(ops, k, fn)
    fam_ms = {k: float(np.mean([a.elapsed_time(b) for a, b in v])) for k, v in fam.items() if v}
    # ring_push may be called twice per step (timestamps ahead of the samples): per-step time = sum of its calls
    calls_per_step = {k: len(v) / prof_steps for k, v in fam.items() if v}
    fam_ms = {k: fam_ms[k] * calls_per_step[k] for k in fam_ms}
    fam_ms['roi'] = roi_ms                                   # F1: the in-region measurement
    rec_cols = int(recbuf[0].shape[1])

    # ---- e2e: the same step through the public API with HOST inputs (pinned), results read back to host.
    # Frames stay in pinned host memory and F1 reads the ROI rows straight over PCIe (zero-copy): only the
    # bytes the path needs cross the bus; boxes + timestamps are copied H2D; bpm/ptt records copied D2H.
    Te = min(T, args.e2e_frames)
    host_frames = torch.empty((S, Te, H, W, 3), dtype=torch.uint8, pin_memory=True)
    host_frames.copy_(frames[:, :Te])
    host_boxes = torch.from_numpy(boxes_np[:, :Te].copy()).pin_memory()
    host_ts = torch.empty((S, Te), dtype=torch.float64, pin_memory=True)
    jobs_e = S * (Te if args.windows == 'every_frame' else 1)
    host_out = torch.empty((jobs_e, 2 * 2 + 2 * 1), dtype=torch.float64, pin_memory=True)
    e2e_roi_bytes = roi_bytes(boxes_np[:, :Te], H, W)

    # Two-stage software pipeline over two CUDA streams: F1 of batch k+1 (PCIe bound: ROI rows read straight from
    # pinned host memory) runs on a side stream while the window pipeline of batch k runs on the main stream and its
    # records are copied back.  Every batch's inputs start in host memory and its results end in host memory inside
    # the timed region; K batches are timed from the first F1 launch to the last result landing on the host.
    side = torch.cuda.Stream(device=dev)
    main = torch.cuda.current_stream()
    sbuf = [torch.empty((S, Te, 2), dtype=torch.float64, device=dev) for _ in range(2)]
    bbuf = [torch.empty((S, Te, 2, 4), dtype=torch.int32, device=dev) for _ in range(2)]
    evs = [torch.cuda.Event() for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]
    dev_out = torch.empty((jobs_e, 6), dtype=torch.float64, device=dev)

    def launch_f1(k):
        side.wait_event(done[k % 2])                        # buffer k%2 is free once batch k-2 has consumed it
        with torch.cuda.stream(side):
            bbuf[k % 2].copy_(host_boxes, non_blocking=True)
            eng.roi_samples(host_frames, bbuf[k % 2], out=sbuf[k % 2])
            evs[k % 2].record(side)

    def finish(k):
        host_ts.copy_(torch.from_numpy((t_next[0] + (np.arange(Te) + 1) / fps)[None, :].repeat(S, 0)))
        t_next[0] += Te / fps
        main.wait_event(evs[k % 2])
        r = eng.step_signals(sbuf[k % 2], host_ts.to(dev, non_blocking=True))
        done[k % 2].record(main)
        host_out.copy_(r.packed(out=dev_out), non_blocking=True)
        main.synchronize()

    def run_e2e(K):
        launch_f1(0)
        for k in range(K):
            if k + 1 < K:
                launch_f1(k + 1)
            finish(k)

    run_e2e(4)
    barrier()
    ke = max(4, min(args.steps, 40))
    t0 = time.perf_counter()
    run_e2e(ke)
    barrier()
    e2e_s = (time.perf_counter() - t0) / ke
    if world > 1:
        tt = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        tdist.all_reduce(tt, op=tdist.ReduceOp.MAX)
        e2e_s = float(tt.item())
    del host_frames
    fma = measure_fma_peaks(torch, dev) if rank == 0 else None
    pcie_conc = measure_pcie_concurrent(torch, dev, tdist, world) if world > 1 else None
    pcie = measure_pcie(torch, dev) if rank == 0 else None
    sched = {'overlap_mask': eng.overlap, 'design_cache': eng._dcache is not None}
    # ---- ingest variants of F1 (SURVEY 8f row 2), informational: same launch size, frames / surfaces resident in HBM
    ingest = {}
    if rank == 0 and world == 1 and not args.no_other:
        try:
            ingest.update(run_ingest_resized(torch, frames, boxes_np, getattr(_cabi, wl['channel']), peaks()[0]))
        except Exception as e:
            ingest['resized_720p'] = {'error': f'{type(e).__name__}: {e}'[:300]}
    del frames, eng
    torch.cuda.empty_cache()
    if rank == 0 and world == 1 and not args.no_other:
        try:
            ingest.update(run_ingest_nv12(torch, dev, boxes_np, S, T, H, W, getattr(_cabi, wl['channel']), peaks()[0]))
        except Exception as e:
            ingest['nv12'] = {'error': f'{type(e).__name__}: {e}'[:300]}

    # ---- the other named shapes (every rank takes part when N > 1: c5 is sharded over the ranks)
    other = {}
    if not args.no_other:
        names = ['c5'] if world > 1 else ['c1_batched', 'c3', 'c4', 'c5']
        for nm in names:
            try:
                other[nm] = run_other_shape(torch, nm, OTHER_SHAPES[nm], dev, world)
            except Exception as e:                           # a failed side measurement must not lose the headline
                other[nm] = {'error': f'{type(e).__name__}: {e}'[:300]}
    lat = None
    if rank == 0 and world == 1 and not args.no_other:
        try:
            lat = run_latency_c1(torch, dev)
        except Exception as e:
            lat = {'error': f'{type(e).__name__}: {e}'[:300]}
    if rank != 0:
        return
    peak, peak_src = peaks()
    jobs = S * (T if args.windows == 'every_frame' else 1)
    nsig = jobs * 2
    taps = 127
    # algorithmic bytes / flops per launch (DESIGN.md §Kernels)
    alg = {
        'roi': alg_roi_bytes + S * T * 2 * (16 + 8),
        'push': S * T * 3 * 8 * 2,
        'design': jobs * (win * 8 + 520 * 8),
        'preprocess': nsig * win * (8 + 8 + 8 + 8),          # ring t,y in + proc x,y out (float64)
        'spectrum': nsig * win * 16 + nsig * 24,
        'xcorr': jobs * (3 * win * 8 + 24),
    }
    alg['spectrum_xcorr'] = alg['spectrum'] + alg['xcorr']       # overlap bit 4: both in one grid
    if 'design' not in fam_ms and 'preprocess' in fam_ms:
        alg['preprocess'] += alg['design']
    total_fam = sum(fam_ms.values())
    kernels = {k: {'ms': fam_ms[k], 'share': fam_ms[k] / total_fam, 'alg_bytes': alg[k],
                   'gbs': alg[k] / fam_ms[k] / 1e6, 'frac_hbm': alg[k] / fam_ms[k] / 1e6 / peak} for k in fam_ms}
    dom = max(fam_ms, key=fam_ms.get)
    total_frames = world * S * T * args.steps
    value = total_frames / (ms / 1e3)
    # FP64 work of the F2 filter kernel as executed (DESIGN.md §4): merged FIR n x (2 taps - 1) FMAs per signal + detrend.
    # The filter DESIGN is not in this figure: with the design cache a regular-fps workload designs (almost) nothing.
    f2_flop = nsig * (2.0 * win * (2 * taps - 1) + 16.0 * win)
    # the same work by SURVEY.md 8(d)'s per-unit figure for the reference's two-pass filtfilt over the padded signal
    f2_flop_survey = nsig * (2.0 * (win + 2 * min(win - 1, 3 * taps)) * taps * 2 + 8.0 * win)
    f2_ms = fam_ms.get('preprocess', 0.0)
    g64 = granule_bytes(boxes_np, H, W, 3 * W, H * W * 3, 64)
    g32 = granule_bytes(boxes_np, H, W, 3 * W, H * W * 3, 32)
    cpu = None
    if world == 1 and not args.no_cpu:
        kind = 'reference' if reference_available() and not args.port else 'port'
        per = args.cpu_frames if kind == 'reference' else args.cpu_frames * 4
        rate, secs = cpu_rate(wl, kind, os.cpu_count() or 1, per, reps=1, warm=1)[0]
        cpu = {'value': rate, 'unit': UNIT, 'cores': os.cpu_count() or 1, 'kind': kind,
               'sample': f'{os.cpu_count()} streams x {per} steady-state frames (window prefilled), '
                         + ('UNMODIFIED reference SignalProcessor.process per frame (baseline/_ref)' if kind == 'reference'
                            else 'oracle port of SignalProcessor.process per frame')
                         + f', one process per core; {secs:.1f} s of CPU work per core'}
        if kind == 'reference':
            prate, _ = cpu_rate(wl, 'port', os.cpu_count() or 1, per * 2, reps=1, warm=1)[0]
            cpu['oracle_port_value'] = prate
        if not args.no_other:
            # CPU numbers beside the other shapes: the reference where it can run the shape (c3's fixed 2048-frequency grid
            # is an extension kwarg, so the oracle port stands in), a few frames per core
            for nm in other:
                o = OTHER_SHAPES[nm]
                k2 = 'port' if (nm == 'c3' or kind == 'port') else 'reference'
                try:
                    r2, s2 = cpu_rate(o, k2, os.cpu_count() or 1, 3 if nm in ('c3', 'c4') else 8, reps=1, warm=1)[0]
                    other[nm]['cpu'] = {'windows_per_s': r2, 'cores': os.cpu_count() or 1, 'kind': k2,
                                        'ms_per_frame_per_core': 1e3 * (os.cpu_count() or 1) / r2}
                    other[nm]['speedup_vs_cpu'] = other[nm]['windows_per_s'] / r2 if 'windows_per_s' in other[nm] else None
                except Exception as e:
                    other[nm]['cpu'] = {'error': f'{type(e).__name__}: {e}'[:200]}
        if lat is not None and 'ms_per_frame' in lat:
            try:
                c1 = dict(OTHER_SHAPES['c1_batched'])
                r1, _ = cpu_rate(c1, kind, 1, 24, reps=1, warm=1)[0]
                lat['reference_ms_per_frame'] = 1e3 / r1
                lat['reference_kind'] = kind
            except Exception as e:
                lat['reference_error'] = f'{type(e).__name__}: {e}'[:200]
    e2e_value = world * S * Te / e2e_s
    e2e_h2d = int(e2e_roi_bytes + host_boxes.numel() * 4 + host_ts.numel() * 8)
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': W_UP,
        'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic',
        'config': shape_config(args.workload, wl, world, args.windows),
        'windows_per_s': world * jobs * args.steps / (ms / 1e3),
        # F1 is the HBM-bound kernel the metric is quoted on ("ROI-sampled frames/s (%HBM peak)") and moves most of the
        # step's DRAM traffic; the dominant family BY TIME is FP64-bound filter work (roofline_by_time, FP64 peak).
        'roofline': {'kernel': 'roi (roi_staged_kernel)', 'bound': 'hbm', 'achieved': kernels['roi']['gbs'], 'peak': peak,
                     'unit': 'GB/s', 'frac': kernels['roi']['frac_hbm'], 'traffic': (ROI_NCU_TRAFFIC_BYTES * T / 64.0) if args.workload == 'c2' else None,
                     'peak_source': peak_src, 'alg_bytes': alg['roi'],
                     'granule64_bytes': g64, 'granule32_bytes': g32,
                     'note': 'achieved = algorithmic bytes (sum of 3*w*h over the ROIs of a launch + boxes + outputs) / mean '
                             'CUDA-event time of the F1 launches inside the timed region; traffic = dram__bytes_read+write of '
                             'one launch from ncu --set full (same boxes); granule64_bytes = bytes of the distinct 64-byte '
                             'granules the ROI rows touch = the least DRAM traffic at the smallest L2 fill granule PTX exposes '
                             '(L2::64B), granule32_bytes the same at sector size'},
        'roofline_by_time': {'kernel': 'F2 window_preprocess_kernel (detrend + filtfilt as one merged 253-tap FIR, float64)',
                             'bound': 'fp64', 'achieved': f2_flop / (f2_ms * 1e-3) / 1e12 if f2_ms else None,
                             'peak': fma['f64'] if fma else None, 'unit': 'TFLOP/s',
                             'frac': (f2_flop / (f2_ms * 1e-3) / 1e12) / fma['f64'] if fma and f2_ms else None,
                             'flop_per_launch': f2_flop, 'flop_per_launch_survey_figure': f2_flop_survey, 'ms': f2_ms,
                             'peak_source': 'bpv_probe_fma float64, measured live in this run',
                             'note': 'dominant family of the step by CUDA-event time: ' + dom},
        'fma_peaks_tflops': fma,
        'kernels': kernels,
        'kernels_note': 'roi: CUDA events around every F1 launch INSIDE the timed region; the other families: the same steps replayed '
                        'right after it with every launcher bracketed by events (families on different streams overlap)',
        # libbpv kernels launched inside the timed region: the engine's step (roi, ring push, firls design, preprocess,
        # spectrum, xcorr) + pack_records32 for the result record
        'gpu_launches': launches_per_step * args.steps,
        'schedule': dict(sched, note='bpv/engine.py: overlap bit 1 = filter design beside F1, bit 2 = xcorr beside the spectrum (their '
                                     'family times then overlap), bit 4 = Welch + xcorr as ONE grid of interleaved CTAs (family '
                                     'spectrum_xcorr); design_cache = filter designs looked up by the bits of fs'),
        'record_bytes_per_job': 4 * rec_cols,
        'numa': numa,
        'clocks': clk,
        'e2e': {'value': e2e_value, 'unit': UNIT,
                'h2d_bytes_per_step': e2e_h2d, 'd2h_bytes_per_step': int(host_out.numel() * 8),
                'frames_per_stream_per_step': Te, 'pcie_gbs_measured': pcie,
                'pcie_frac': (e2e_h2d / e2e_s / 1e9) / pcie if pcie else None,
                'pcie_gbs_concurrent_sum': pcie_conc[0] if pcie_conc else None,
                'pcie_gbs_concurrent_slowest_rank': pcie_conc[1] if pcie_conc else None,
                'pcie_frac_concurrent': (world * e2e_h2d / e2e_s / 1e9) / pcie_conc[0] if pcie_conc else None,
                'how': 'BatchedSignalProcessor.roi_samples + step_signals on pinned HOST frames/boxes/timestamps; F1 reads the '
                       'ROI rows zero-copy over PCIe (the other 99.5 % of each frame never crosses the bus, so h2d_bytes_per_step '
                       'counts the ROI bytes + boxes + timestamps) on a side stream, overlapped with the previous batch\'s window '
                       f'pipeline; records copied back to host every batch; wall clock.  {Te} frames per stream per batch instead of '
                       f'the {T} of the device-timed region: the whole batch must sit in PINNED host memory '
                       f'({S * Te * H * W * 3 / 1e9:.1f} GB pinned at {Te}, {S * T * H * W * 3 / 1e9:.0f} GB at {T}); the rate is PCIe bound '
                       '(pcie_frac = ROI bytes/s over the measured pinned-copy bandwidth)'},
    }
    if cpu is not None:
        line['cpu_baseline'] = cpu
    if ingest:
        line['ingest'] = ingest
    if other:
        line['other_shapes'] = other
    if lat is not None:
        line['latency_c1'] = lat
    print(json.dumps(line), flush=True)


def _shutdown():
    try:
        import torch.distributed as tdist
        if tdist.is_available() and tdist.is_initialized():
            tdist.destroy_process_group()
    except Exception:
        pass


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200, help='timed steps (>= 1)')
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='bpv', choices=['bpv', 'reference'])
    ap.add_argument('--workload', default='c2', choices=list(WORKLOADS))
    ap.add_argument('--windows', default='every_frame', choices=['every_frame', 'last'])
    ap.add_argument('--frames-per-step', type=int, default=0, help='frames per stream per step (batch depth T); 0 = the workload default')
    ap.add_argument('--ref-frames', type=int, default=64, help='reference arm: at most this many frames per core per step')
    ap.add_argument('--ref-budget-s', type=float, default=90.0, help='reference arm: CPU seconds per core for all steps')
    ap.add_argument('--cpu-frames', type=int, default=400, help='cpu_baseline of the GPU arm: frames per core')
    ap.add_argument('--e2e-frames', type=int, default=8, help='frames per stream per e2e step (pinned host memory)')
    ap.add_argument('--port', action='store_true', help='CPU arms: time the oracle port even if baseline/_ref exists')
    ap.add_argument('--bind-numa', dest='numa', action='store_true', help='N > 1: bind each rank to the CPUs of its GPU\'s NUMA node')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-other', action='store_true', help='skip the other_shapes / latency blocks')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the results of the last timed step as DIR/<name>.npy '
                                                          '(rank 0\'s streams when N > 1)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'bpv':
        ap.error('--dump-outputs writes the results of the GPU path (--impl bpv)')
    wl = dict(WORKLOADS[args.workload])
    if args.frames_per_step > 0:
        wl['T'] = args.frames_per_step
    if args.impl == 'reference':
        run_reference(args, wl)
    else:
        try:
            run_gpu(args, wl)
        finally:
            _shutdown()


if __name__ == '__main__':
    main()
