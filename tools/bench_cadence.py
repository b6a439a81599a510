"""Cost of window cadences (BatchedSignalProcessor window_stride / window_phase) on signals-only input.

Two shapes:
  c2    256 streams x 64 frames per step, window 300, DETREND_LINEAR + FIR, Welch.  Variants: k = 1 (every frame, the
        default path), k = 4, 16, 64 with phase 0 (the lockstep kernels with head_step = k), and per-stream k drawn from
        {15, 30, 60} with random phases (the strided job map).  Each round times `iters` back-to-back steps per variant.
  live  4096 streams x 1 frame per step, window 300, Butterworth + Lomb-Scargle: a live system that steps once per frame.
        Variants: every frame; k = 30 with phase 0 (one step in 30 carries every stream's job, the others none); k = 30
        with phase s mod 30 (the same work spread over the steps, on the job map).  Each round times one 30-step cycle per
        variant, step by step: the mean step and the worst step of the cycle.
Variants alternate round after round; round 0 warms every shape up and is dropped.  Steps are timed with CUDA events.  A
separate pass under torch.profiler (CUDA activities) sums the device time of each kernel family per step.  Prints the
card's name, power limit and max SM clock, then one JSON line per shape.  Needs a CUDA device; there is no CPU fallback.

    python tools/bench_cadence.py [--rounds 5] [--iters 10] [--shapes c2,live] [--no-profile]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
ap.add_argument('--rounds', type=int, default=5)
ap.add_argument('--iters', type=int, default=10)
ap.add_argument('--shapes', default='c2,live')
ap.add_argument('--no-profile', action='store_true')
ARGS = ap.parse_args()
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'bp-from-video_b200'))
from bench import OTHER_SHAPES, WORKLOADS, device_signals  # noqa: E402
from bpv import _cabi  # noqa: E402
from bpv.engine import BatchedSignalProcessor  # noqa: E402

FAMILIES = (('jobmap', ('stream_jobs',)), ('push', ('ring_push',)), ('design', ('job_butter', 'job_firls', 'design_probe', 'miss_')),
            ('f2', ('window_preprocess',)), ('f3', ('welch', 'ls_', 'dft', 'spectrum')), ('f4', ('xcorr',)),
            ('means', ('running_mean',)))
CYCLE = 30


def card():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else torch.cuda.get_device_name()


def family(name):
    for fam, keys in FAMILIES:
        if any(k in name for k in keys):
            return fam
    return 'other'


def variants(shape, S):
    """name -> (window_stride, window_phase)."""
    if shape == 'c2':
        rng = np.random.default_rng(7)
        k = rng.choice([15, 30, 60], S)
        return {'k1': (1, 0), 'k4': (4, 0), 'k16': (16, 0), 'k64': (64, 0), 'k15_30_60': (k, rng.integers(0, 2 ** 20, S) % k)}
    return {'every_frame': (1, 0), 'k30_aligned': (CYCLE, 0), 'k30_staggered': (CYCLE, np.arange(S) % CYCLE)}


def run_shape(name, wl, rounds, iters):
    S, T, W = wl['S'], wl['T'], wl['window']
    kw = dict(processing_methods=[getattr(_cabi, m) for m in wl['methods']], spectrum_transform=getattr(_cabi, wl['transform']),
              **wl['kw'])
    per_round = iters if name == 'c2' else CYCLE
    fill = (W + T - 1) // T * T
    nsteps = (rounds + 2) * per_round + 2
    n = fill + T * (nsteps + 1)
    ts, y = device_signals(torch, S, n, wl['fps'], wl.get('irregular', False), wl.get('p_nan', 0.0), 4321, 'cuda')
    vs = variants(name, S)
    engines, head, jobs = {}, {}, {v: [] for v in vs}
    for v, (k, ph) in vs.items():
        eng = BatchedSignalProcessor(S, 2, signal_max_samples=W, max_frames_per_step=T, **kw)
        for a in range(0, fill, T):                                    # fill the windows at every frame (level steps)
            eng.step_signals(y[:, a:a + T].contiguous(), ts[:, a:a + T].contiguous())
        eng.window_stride, eng.window_phase = k, ph
        engines[v], head[v] = eng, fill
    # live: the 30-step cycle of every variant starts at the same count, so every cycle holds each stream's one job
    torch.cuda.synchronize()

    def step(v):
        g = head[v]
        res = engines[v].step_signals(y[:, g:g + T], ts[:, g:g + T])
        jobs[v].append(res.peak_freq.shape[0])
        head[v] = g + T

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(per_round + 1)]
    times = {v: [] for v in vs}
    for rnd in range(rounds + 1):
        for v in vs:
            torch.cuda.synchronize()
            ev[0].record()
            for i in range(per_round):
                step(v)
                ev[i + 1].record()
            torch.cuda.synchronize()
            if rnd:
                times[v].append([ev[i].elapsed_time(ev[i + 1]) for i in range(per_round)])
    out = dict(shape=name, S=S, T=T, window=W, rounds=rounds, steps_per_round=per_round, unit='ms')
    for v in vs:
        whole = [sum(r) / per_round for r in times[v]]                 # mean step of each round
        out[v] = dict(step=dict(median=statistics.median(whole), min=min(whole), max=max(whole)),
                      mean_jobs=float(np.mean(jobs[v])), launches_per_step=engines[v].launches_per_step)
        if name == 'live':
            worst = [max(r) for r in times[v]]
            out[v]['worst_step'] = dict(median=statistics.median(worst), max=max(worst))
            out[v]['max_jobs'] = int(max(jobs[v]))
    if not ARGS.no_profile:
        from torch.profiler import ProfilerActivity, profile
        for v in vs:
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(per_round):
                    step(v)
                torch.cuda.synchronize()
            fam = {}
            for e in prof.key_averages():
                if e.device_type.name == 'CUDA' and not e.key.startswith(('Memcpy', 'Memset')):
                    f = family(e.key)
                    fam[f] = fam.get(f, 0.0) + e.self_device_time_total / per_round
            out[v]['kernel_us_per_step'] = {k: round(x, 1) for k, x in sorted(fam.items())}
    return out


def main():
    if not torch.cuda.is_available():
        raise SystemExit('bench_cadence: needs a CUDA device (no CPU fallback)')
    print(f'card: {card()}', flush=True)
    shapes = {'c2': WORKLOADS['c2'], 'live': OTHER_SHAPES['c1_batched']}
    for name in ARGS.shapes.split(','):
        print(json.dumps(run_shape(name, shapes[name], ARGS.rounds, ARGS.iters)), flush=True)


if __name__ == '__main__':
    main()
