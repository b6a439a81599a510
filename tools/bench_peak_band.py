"""Cost of the band-limited peak search (BatchedSignalProcessor freq_band / lag_band) on signals-only input.

Two shapes of bench.py: c2 (256 streams x 64 frames per step, window 300, DETREND_LINEAR + FIR, Welch, 16 384 window jobs per
step) and c4 (1024 streams x 1 frame, window 1200, INTERP_CUBIC + BUTTER, Lomb-Scargle, 2399 lags per pair).  Three variants
are timed in alternation, round after round: no band, the unbounded band (-inf, inf), and the reference's configured ranges
(0.8, 4.0) Hz / (-0.5, 0.5) s.  Per variant, CUDA events around
  - the F3 launch (ops.window_spectrum) and the F4 launch (ops.window_xcorr) on the processed windows of a step,
  - a whole engine step (step_signals, default overlap).
Prints the card's name and power limit, then one JSON line per shape.  Needs a CUDA device; there is no CPU fallback.

    python tools/bench_peak_band.py [--rounds 5] [--iters 20]
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'bp-from-video_b200'))
from bench import OTHER_SHAPES, WORKLOADS, device_signals  # noqa: E402
from bpv import _cabi, ops  # noqa: E402
from bpv.engine import BatchedSignalProcessor  # noqa: E402

VARIANTS = {'none': (None, None), 'unbounded': ((-math.inf, math.inf), (-math.inf, math.inf)),
            'configured': ((0.8, 4.0), (-0.5, 0.5))}


def card():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else torch.cuda.get_device_name()


def timed(fn, iters):
    """Mean milliseconds of fn() over `iters` back-to-back calls, by CUDA events on the current stream."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def run_shape(name, wl, rounds, iters):
    S, T, W = wl['S'], wl['T'], wl['window']
    kw = dict(processing_methods=[getattr(_cabi, m) for m in wl['methods']], spectrum_transform=getattr(_cabi, wl['transform']),
              **wl['kw'])
    n = W + T * ((rounds + 1) * iters + 2)                            # every timed step gets new samples
    ts, y = device_signals(torch, S, n, wl['fps'], wl.get('irregular', False), wl.get('p_nan', 0.0), 4321, 'cuda')
    engines = {}
    for v, (fb, lb) in VARIANTS.items():
        eng = BatchedSignalProcessor(S, 2, signal_max_samples=W, max_frames_per_step=max(T, 50), freq_band=fb, lag_band=lb, **kw)
        for a in range(0, W, 50):                                     # fill the windows
            eng.step_signals(y[:, a:min(W, a + 50)].contiguous(), ts[:, a:min(W, a + 50)].contiguous())
        engines[v] = eng
    # processed windows of one steady-state step (stored by a separate engine), for the F3 / F4 launches on their own
    cap = BatchedSignalProcessor(S, 2, signal_max_samples=W, max_frames_per_step=max(T, 50), store_arrays=True, **kw)
    for a in range(0, W, 50):
        cap.step_signals(y[:, a:min(W, a + 50)].contiguous(), ts[:, a:min(W, a + 50)].contiguous())
    res = cap.step_signals(y[:, W:W + T].contiguous(), ts[:, W:W + T].contiguous())
    px, py = res.arrays['proc_x'], res.arrays['proc_y']
    p = cap._params(cap.count - T, 1, T)
    ws = torch.zeros(max(_cabi.lib().bpv_spectrum_workspace_bytes(p, ops.max_bins(p)), 16), dtype=torch.uint8, device='cuda')
    times = {v: dict(f3=[], f4=[], step=[]) for v in VARIANTS}
    head = {v: W for v in VARIANTS}
    for rnd in range(rounds + 1):                                     # round 0 warms every shape up and is dropped
        for v, (fb, lb) in VARIANTS.items():
            f3 = timed(lambda: ops.window_spectrum(px, py, p, store=False, workspace=ws, band=fb), iters)
            f4 = timed(lambda: ops.window_xcorr(px, py, p, store=False, band=lb), iters)
            eng = engines[v]

            def step():
                g = head[v]
                eng.step_signals(y[:, g:g + T].contiguous(), ts[:, g:g + T].contiguous())
                head[v] = g + T
            st = timed(step, iters)
            if rnd:
                times[v]['f3'].append(f3)
                times[v]['f4'].append(f4)
                times[v]['step'].append(st)
    out = dict(shape=name, S=S, T=T, window=W, jobs_per_step=S * T, lags=2 * W - 1, rounds=rounds, iters=iters, unit='ms')
    for v in VARIANTS:
        out[v] = {k: dict(median=statistics.median(x), min=min(x), max=max(x)) for k, x in times[v].items()}
    for k in ('f3', 'f4', 'step'):
        out[f'configured_over_none_{k}'] = out['configured'][k]['median'] / out['none'][k]['median']
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--shapes', default='c2,c4')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_peak_band: needs a CUDA device (no CPU fallback)')
    print(f'card: {card()}', flush=True)
    shapes = {'c2': WORKLOADS['c2'], 'c4': OTHER_SHAPES['c4']}
    for name in a.shapes.split(','):
        print(json.dumps(run_shape(name, shapes[name], a.rounds, a.iters)), flush=True)


if __name__ == '__main__':
    main()
