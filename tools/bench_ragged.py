"""Cost of ragged steps (BatchedSignalProcessor frame_counts) on signals-only input.

Two shapes: c2 (256 streams x 64 frames per step, window 300, DETREND_LINEAR + FIR, Welch) and c5 (65 536 streams x 1 frame,
window 300, Butterworth + Lomb-Scargle).  Three variants per shape, timed in alternation round after round:
  lockstep  frame_counts = None: the lockstep kernels (run this with --pkg <checkout of the parent>/bp-from-video_b200 to
            time the parent's engine on the same input; only this variant exists there)
  forced    level counts through the job-map path (BPV_FORCE_JOBMAP): the price of the map
  random    counts drawn uniformly from 0..T per stream and step: J falls, and so should F2 / F3 / F4.  Each stream takes
            the next n_s frames of its own timeline (no gaps), so its sampling rate, and the design cache, behave as for a
            camera that delivers fewer frames per step rather than one that drops frames
Whole steps are timed with CUDA events around `iters` back-to-back steps.  A separate pass under torch.profiler (CUDA
activities) sums the device time of each kernel family per step.  Prints the card's name, power limit and max SM clock,
then one JSON line per shape.  Needs a CUDA device; there is no CPU fallback.

    python tools/bench_ragged.py [--rounds 5] [--iters 10] [--shapes c2,c5] [--variants lockstep,forced,random] [--pkg DIR]
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
ap.add_argument('--shapes', default='c2,c5')
ap.add_argument('--variants', default='lockstep,forced,random')
ap.add_argument('--pkg', default=os.path.join(ROOT, 'bp-from-video_b200'), help='bp-from-video_b200 directory to time')
ap.add_argument('--no-profile', action='store_true')
ARGS = ap.parse_args()
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.abspath(ARGS.pkg))
from bench import OTHER_SHAPES, WORKLOADS, device_signals  # noqa: E402
from bpv import _cabi  # noqa: E402
from bpv.engine import BatchedSignalProcessor  # noqa: E402

FAMILIES = (('jobmap', ('stream_jobs',)), ('push', ('ring_push',)), ('design', ('job_butter', 'job_firls', 'design_probe', 'miss_')),
            ('f2', ('window_preprocess',)), ('f3', ('welch', 'ls_', 'dft', 'spectrum')), ('f4', ('xcorr',)),
            ('means', ('running_mean',)))


def card():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else torch.cuda.get_device_name()


def family(name):
    for fam, keys in FAMILIES:
        if any(k in name for k in keys):
            return fam
    return 'other'


def run_shape(name, wl, variants, rounds, iters):
    S, T, W = wl['S'], wl['T'], wl['window']
    kw = dict(processing_methods=[getattr(_cabi, m) for m in wl['methods']], spectrum_transform=getattr(_cabi, wl['transform']),
              **wl['kw'])
    nsteps = (rounds + 1) * iters + iters + 2
    n = W + T * (nsteps + 1)
    ts, y = device_signals(torch, S, n, wl['fps'], wl.get('irregular', False), wl.get('p_nan', 0.0), 4321, 'cuda')
    rng = np.random.default_rng(5)
    engines, head, counts = {}, {}, {}
    for v in variants:
        eng = BatchedSignalProcessor(S, 2, signal_max_samples=W, max_frames_per_step=T, **kw)
        for a in range(0, W, T):                                      # fill the windows (level steps)
            eng.step_signals(y[:, a:min(W, a + T)].contiguous(), ts[:, a:min(W, a + T)].contiguous())
        if v == 'forced':
            eng.force_jobmap = True
        engines[v], head[v] = eng, (W + T - 1) // T * T
        counts[v] = [None] * nsteps if v != 'random' else [rng.integers(0, T + 1, S) for _ in range(nsteps)]
    # random: the inputs of every step gathered up front from each stream's own position (outside the timed region)
    inputs = []
    if 'random' in variants:
        pos = np.full(S, head['random'], dtype=np.int64)
        rows = torch.arange(S, device='cuda')[:, None]
        for fc in counts['random']:
            idx = torch.from_numpy(np.minimum(pos[:, None] + np.arange(T), n - 1)).cuda()
            inputs.append((y[rows, idx].contiguous(), ts[rows, idx].contiguous()))
            pos += fc
    jobs = {v: [] for v in variants}

    def step(v):
        g = head[v]
        k = (g - W) // T
        fc = counts[v][k]
        if fc is None:
            engines[v].step_signals(y[:, g:g + T].contiguous(), ts[:, g:g + T].contiguous())
            jobs[v].append(S * T)
        else:
            engines[v].step_signals(*inputs[k], frame_counts=fc)
            jobs[v].append(int(fc.sum()))
        head[v] = g + T

    def timed(v):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(iters):
            step(v)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    times = {v: [] for v in variants}
    for rnd in range(rounds + 1):                                     # round 0 warms every shape up and is dropped
        for v in variants:
            t = timed(v)
            if rnd:
                times[v].append(t)
    out = dict(shape=name, S=S, T=T, window=W, rounds=rounds, iters=iters, unit='ms')
    for v in variants:
        out[v] = dict(step=dict(median=statistics.median(times[v]), min=min(times[v]), max=max(times[v])),
                      mean_jobs=float(np.mean(jobs[v])), launches_per_step=engines[v].launches_per_step)
    if not ARGS.no_profile:
        from torch.profiler import ProfilerActivity, profile
        for v in variants:
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(iters):
                    step(v)
                torch.cuda.synchronize()
            fam = {}
            for e in prof.key_averages():
                if e.device_type.name == 'CUDA' and not e.key.startswith(('Memcpy', 'Memset')):
                    f = family(e.key)
                    fam[f] = fam.get(f, 0.0) + e.self_device_time_total / iters
            out[v]['kernel_us_per_step'] = {k: round(x, 1) for k, x in sorted(fam.items())}
    return out


def main():
    if not torch.cuda.is_available():
        raise SystemExit('bench_ragged: needs a CUDA device (no CPU fallback)')
    print(f'card: {card()}', flush=True)
    print(f'package: {os.path.relpath(os.path.abspath(ARGS.pkg), ROOT)}', flush=True)
    shapes = {'c2': WORKLOADS['c2'], 'c5': OTHER_SHAPES['c5']}
    for name in ARGS.shapes.split(','):
        print(json.dumps(run_shape(name, shapes[name], ARGS.variants.split(','), ARGS.rounds, ARGS.iters)), flush=True)


if __name__ == '__main__':
    main()
