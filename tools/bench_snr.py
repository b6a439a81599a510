"""Cost of the per-window spectral SNR (BatchedSignalProcessor snr / min_snr_db, include/bpv.h bpv_window_snr) on
signals-only input.

Two shapes:
  c2    256 streams x 64 frames per step, window 300, DETREND_LINEAR + FIR, Welch (129 bins): 16 384 window jobs a step.
  c4ls  1024 streams x 1 frame per step, window 1200 at 120 fps, INTERP_CUBIC + Butterworth, Lomb-Scargle (F = n).
Variants: 'off' (snr=False), 'on' (snr=True), 'gated' (snr=True, min_snr_db=3).  Every engine keeps running means
(peak_max_samples=30), so the variants differ only by the SNR.  Variants alternate round after round; round 0 warms every
shape up and is dropped.  Steps are timed with CUDA events over `iters` back-to-back steps.  Then, on the processed windows
and spectra of the last step, CUDA events time over `reps` calls each: bpv_window_snr alone, and F3 (bpv_window_spectrum)
with the spectrum stored (what snr=True makes F3 do) and without it.  Prints the card's name, power limit and max SM clock,
then one JSON line per shape.  Needs a CUDA device; there is no CPU fallback.

    python tools/bench_snr.py [--rounds 5] [--iters 10] [--reps 50] [--shapes c2,c4ls]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
ap.add_argument('--rounds', type=int, default=5)
ap.add_argument('--iters', type=int, default=10)
ap.add_argument('--reps', type=int, default=50)
ap.add_argument('--shapes', default='c2,c4ls')
ARGS = ap.parse_args()
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'bp-from-video_b200'))
from bench import OTHER_SHAPES, WORKLOADS, device_signals  # noqa: E402
from bpv import _cabi, ops  # noqa: E402
from bpv.engine import BatchedSignalProcessor  # noqa: E402

VARIANTS = {'off': dict(), 'on': dict(snr=True), 'gated': dict(snr=True, min_snr_db=3.0)}


def card():
    r = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else torch.cuda.get_device_name()


def timed(fn, reps):
    """Mean device time of one call in microseconds: CUDA events around `reps` back-to-back calls."""
    fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) * 1000.0 / reps


def run_shape(name, wl, rounds, iters, reps):
    S, T, W = wl['S'], wl['T'], wl['window']
    kw = dict(processing_methods=[getattr(_cabi, m) for m in wl['methods']], spectrum_transform=getattr(_cabi, wl['transform']),
              **wl['kw'])
    fill = (W + T - 1) // T * T
    n = fill + T * ((rounds + 1) * iters + 2)
    ts, y = device_signals(torch, S, n, wl['fps'], wl.get('irregular', False), wl.get('p_nan', 0.0), 4321, 'cuda')
    engines, head, res = {}, {}, {}
    for v, extra in VARIANTS.items():
        eng = BatchedSignalProcessor(S, 2, signal_max_samples=W, max_frames_per_step=T, peak_max_samples=30, **kw, **extra)
        for a in range(0, fill, T):
            eng.step_signals(y[:, a:a + T].contiguous(), ts[:, a:a + T].contiguous())
        engines[v], head[v] = eng, fill
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    times = {v: [] for v in VARIANTS}
    for rnd in range(rounds + 1):
        for v in VARIANTS:
            torch.cuda.synchronize()
            ev[0].record()
            for _ in range(iters):
                g = head[v]
                res[v] = engines[v].step_signals(y[:, g:g + T], ts[:, g:g + T])
                head[v] = g + T
            ev[1].record()
            torch.cuda.synchronize()
            if rnd:
                times[v].append(ev[0].elapsed_time(ev[1]) / iters)
    out = dict(shape=name, S=S, T=T, window=W, jobs=int(res['off'].peak_freq.shape[0]), rounds=rounds, steps_per_round=iters,
               unit='ms')
    for v in VARIANTS:
        out[v] = dict(step=dict(median=statistics.median(times[v]), min=min(times[v]), max=max(times[v])),
                      launches_per_step=engines[v].launches_per_step)
    # kernels on the last step's processed windows / stored spectra of the 'gated' engine (nothing else runs meanwhile)
    eng, r = engines['gated'], res['gated']
    J = r.peak_freq.shape[0]
    sp = eng._out[(eng._turn - 1) % eng._nbuf][0]
    f, m, nb = sp['freqs'][:J], sp['mags'][:J], sp['num_bins'][:J]
    band = (eng.kw['min_freq'], eng.kw['max_freq'])
    out['snr_kernel_us'] = round(timed(lambda: ops.window_snr(f, m, nb, r.peak_idx, eng.transform, band), reps), 2)
    out['snr_gated_kernel_us'] = round(timed(lambda: ops.window_snr(f, m, nb, r.peak_idx, eng.transform, band, min_snr_db=3.0,
                                                                    peak_freq=r.peak_freq, lag_sec=r.lag_sec), reps), 2)
    out['spectrum_bytes_read_by_snr'] = int(2 * 4 * f.numel())
    proc = eng._proc[0]
    px, py = proc[0, :J], proc[1, :J]
    p = ops.jobs_params(eng._params(0, 1, 1), J)
    stored = ops._spectrum_out(p, True, None, eng.device)
    scratch = ops._spectrum_out(p, False, None, eng.device)
    out['f3_stored_us'] = round(timed(lambda: ops.window_spectrum(px, py, p, store=True, out=stored, workspace=eng._ws_spec), reps), 2)
    out['f3_not_stored_us'] = round(timed(lambda: ops.window_spectrum(px, py, p, store=False, out=scratch, workspace=eng._ws_spec),
                                          reps), 2)
    return out


def main():
    if not torch.cuda.is_available():
        raise SystemExit('bench_snr: needs a CUDA device (no CPU fallback)')
    print(f'card: {card()}', flush=True)
    shapes = {'c2': WORKLOADS['c2'], 'c4ls': dict(OTHER_SHAPES['c4'], T=1)}
    for name in ARGS.shapes.split(','):
        print(json.dumps(run_shape(name, shapes[name], ARGS.rounds, ARGS.iters, ARGS.reps)), flush=True)


if __name__ == '__main__':
    main()
