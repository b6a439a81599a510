"""Launchers: torch tensors (device memory + stream plumbing only) -> libbpv C-ABI calls.

Every function enqueues on torch's current CUDA stream and returns device tensors; nothing here
computes on the host.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _cabi
from ._cabi import WindowParams, check, lib, ptr, stream_handle


def _run(dev: torch.device, name: str, *args) -> None:
    """Call libbpv entry point `name` with `args` + the current stream of `dev`, with `dev` as the CUDA device of the
    calling thread: kernels are enqueued on the GPU that owns the tensors, whatever the caller's current device is."""
    fn = getattr(lib(), name)
    if dev.type != 'cuda':
        raise _cabi.BpvError(f'{name}: tensors must live on a CUDA device (no CPU fallback)')
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    if idx != torch.cuda.current_device():
        with torch.cuda.device(idx):
            check(fn(*args, stream_handle(idx)), name)
    else:
        check(fn(*args, stream_handle(idx)), name)


def _require(cond: bool, msg: str) -> None:
    """Argument check that survives `python -O` (unlike assert)."""
    if not cond:
        raise ValueError(msg)


def _dev_accessible(t: torch.Tensor) -> bool:
    return t.is_cuda or t.is_pinned()


def roi_sample(frames: torch.Tensor, boxes: torch.Tensor, mode: int, *, want_sums: bool = False,
               roi_pixels_hint: int = 0, out_value: torch.Tensor | None = None):
    """F1.  frames uint8 [N,H,W,3] (CUDA, or pinned host memory for the zero-copy path; rows may be
    strided), boxes int32 [N,R,4] (CUDA).  Returns (value f64 [N,R], sums u64-as-int64 [N,R,4] | None).
    Reference: signal_processor.py:176-193."""
    _require(frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[-1] == 3, 'bad argument: ' + 'frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[-1] == 3')
    _require(_dev_accessible(frames), 'frames must live in CUDA or pinned host memory')
    _require(frames.stride(3) == 1 and frames.stride(2) == 3, 'pixels must be packed BGR')
    N, H, W, _ = frames.shape
    _require(boxes.is_cuda and boxes.dtype == torch.int32 and boxes.is_contiguous() and boxes.shape[0] == N and boxes.shape[2] == 4, 'bad argument: ' + 'boxes.is_cuda and boxes.dtype == torch.int32 and boxes.is_contiguous() and boxes.shape[0] == N and boxes.shape[2] == 4')
    R = boxes.shape[1]
    dev = boxes.device
    if out_value is None:
        out_value = torch.empty((N, R), dtype=torch.float64, device=dev)
    sums = torch.empty((N, R, 4), dtype=torch.int64, device=dev) if want_sums else None
    fstride = frames.stride(0) if N > 1 else H * frames.stride(1)
    _run(boxes.device, 'bpv_roi_sample_u8', ptr(frames), None, fstride, frames.stride(1), H, W, N, ptr(boxes), R, int(mode),
                                  ptr(sums), ptr(out_value), int(roi_pixels_hint))
    return out_value, sums


def roi_sample_ptrs(frame_ptrs: torch.Tensor, H: int, W: int, row_stride: int, boxes: torch.Tensor, mode: int, *,
                    want_sums: bool = False, roi_pixels_hint: int = 0):
    """F1 over frames living in separate allocations: frame_ptrs int64 [N] (CUDA) of device-accessible
    addresses."""
    N = frame_ptrs.numel()
    R = boxes.shape[1]
    out_value = torch.empty((N, R), dtype=torch.float64, device=boxes.device)
    sums = torch.empty((N, R, 4), dtype=torch.int64, device=boxes.device) if want_sums else None
    _run(boxes.device, 'bpv_roi_sample_u8', None, ptr(frame_ptrs), 0, row_stride, H, W, N, ptr(boxes), R, int(mode),
                                  ptr(sums), ptr(out_value), int(roi_pixels_hint))
    return out_value, sums


def calc_rois(present, bbox, points, num_points, rel_bbox, hist, g0: int, want_locations: bool = False):
    """Batched calc_rois + ROI smoothing (signal_processor.py:133-155, 304-305).  present u8 [S,T,R], bbox i32 [S,T,R,4],
    points i32 [S,T,R,K,2], num_points i32 [R], rel_bbox f64 [R,4], hist f64 [S,R,H,6] (state, NaN-initialised).
    Returns boxes i32 [S,T,R,4] (+ locations, smoothed f64 [S,T,R,6] when want_locations)."""
    S, T, R = present.shape
    K, H = points.shape[3], hist.shape[2]
    dev = present.device
    boxes = torch.empty((S, T, R, 4), dtype=torch.int32, device=dev)
    loc = torch.empty((S, T, R, 6), dtype=torch.float64, device=dev) if want_locations else None
    smo = torch.empty((S, T, R, 6), dtype=torch.float64, device=dev) if want_locations else None
    _run(present.device, 'bpv_calc_rois', ptr(present), ptr(bbox), ptr(points), ptr(num_points), ptr(rel_bbox), S, T, R, K, H, int(g0),
                              ptr(hist), ptr(loc), ptr(smo), ptr(boxes))
    return (boxes, loc, smo) if want_locations else boxes


def running_mean(ring, g0: int, values, scale: float):
    """Push values [S,T,C] * scale into ring [S,C,H] and return (mean, mean_int) f64 [S,T,C] after each push
    (sg_bpm / sg_ptt + get_means, signal_processor.py:310, 312; signal_data.py:60-63)."""
    S, C_, H = ring.shape
    T = values.shape[1]
    _require(values.shape == (S, T, C_) and values.is_contiguous(), 'bad argument: ' + 'values.shape == (S, T, C_) and values.is_contiguous()')
    mean = torch.empty((S, T, C_), dtype=torch.float64, device=ring.device)
    mean_int = torch.empty((S, T, C_), dtype=torch.float64, device=ring.device)
    _run(ring.device, 'bpv_running_mean', ptr(ring), S, C_, H, int(g0), T, ptr(values), float(scale), ptr(mean), ptr(mean_int))
    return mean, mean_int


def ring_push(ring_t: torch.Tensor, ring_y: torch.Tensor, g0: int, ts: torch.Tensor | None, values: torch.Tensor | None):
    """Append T samples per stream (signal_data.py:31-35, 94-98).  ring_t f64 [S,cap], ring_y f64 [S,R,cap],
    ts f64 [S,T], values f64 [S,T,R]; either of ts / values may be None (timestamps pushed ahead of the samples)."""
    S, R, cap = ring_y.shape
    if ts is None and values is None:
        raise ValueError('ring_push: nothing to push')
    T = ts.shape[1] if ts is not None else values.shape[1]
    if ts is not None and not (ts.shape == (S, T) and ts.is_contiguous()):
        raise ValueError('ring_push: ts must be a contiguous [S, T] tensor')
    if values is not None and not (values.shape == (S, T, R) and values.is_contiguous()):
        raise ValueError('ring_push: values must be a contiguous [S, T, R] tensor')
    _run(ring_y.device, 'bpv_ring_push', ptr(ring_t), ptr(ring_y), S, R, cap, int(g0), T, ptr(ts), ptr(values))


def ring_push_ragged(ring_t, ring_y, g0: torch.Tensor, n: torch.Tensor, ts: torch.Tensor | None, values: torch.Tensor | None):
    """Ragged push (include/bpv.h bpv_ring_push_ragged): stream s appends its first n[s] rows of ts f64 [S,T] / values
    f64 [S,T,R] at global indices g0[s] ...  g0 int64 [S], n int32 [S] on the device; g0 is not advanced."""
    S, R, cap = ring_y.shape
    if ts is None and values is None:
        raise ValueError('ring_push_ragged: nothing to push')
    T = ts.shape[1] if ts is not None else values.shape[1]
    _require(ts is None or (tuple(ts.shape) == (S, T) and ts.is_contiguous()), 'ring_push_ragged: ts must be a contiguous [S, T] tensor')
    _require(values is None or (tuple(values.shape) == (S, T, R) and values.is_contiguous()),
             'ring_push_ragged: values must be a contiguous [S, T, R] tensor')
    _require(g0.dtype == torch.int64 and n.dtype == torch.int32 and g0.numel() == n.numel() == S, 'ring_push_ragged: g0 int64 [S], n int32 [S]')
    _run(ring_y.device, 'bpv_ring_push_ragged', ptr(ring_t), ptr(ring_y), S, R, cap, ptr(g0), ptr(n), T, ptr(ts), ptr(values))


def stream_jobs(g0: torch.Tensor, n: torch.Tensor, last_only: bool, num_jobs: int, job_stream: torch.Tensor,
                job_head: torch.Tensor, stream_job0: torch.Tensor, g0_next: torch.Tensor) -> None:
    """Job map of a ragged step on the device (include/bpv.h bpv_stream_jobs): job_stream i32 / job_head i64 [>= num_jobs],
    stream_job0 i32 [S+1], g0_next i64 [S] = g0 + n.  num_jobs must be the sum of the job counts."""
    S = g0.numel()
    _require(n.numel() == S and stream_job0.numel() == S + 1 and g0_next.numel() == S, 'stream_jobs: sizes do not match')
    _require(job_stream.numel() >= num_jobs and job_head.numel() >= num_jobs, 'stream_jobs: job map buffers too small')
    _run(g0.device, 'bpv_stream_jobs', S, ptr(g0), ptr(n), int(bool(last_only)), int(num_jobs), ptr(job_stream), ptr(job_head),
         ptr(stream_job0), ptr(g0_next))


def running_mean_jobs(ring, g0: torch.Tensor, stream_job0: torch.Tensor, values, scale: float):
    """running_mean over the job map of a ragged step (include/bpv.h bpv_running_mean_jobs): values [J,C]; returns (mean,
    mean_int) f64 [J,C].  g0 int64 [S] = the streams' history counts (not advanced)."""
    S, C_, H = ring.shape
    J = values.shape[0]
    _require(values.dim() == 2 and values.shape[1] == C_ and values.is_contiguous(), 'running_mean_jobs: values must be [J, C]')
    mean = torch.empty((J, C_), dtype=torch.float64, device=ring.device)
    mean_int = torch.empty((J, C_), dtype=torch.float64, device=ring.device)
    _run(ring.device, 'bpv_running_mean_jobs', ptr(ring), S, C_, H, ptr(g0), ptr(stream_job0), ptr(values), float(scale),
         ptr(mean), ptr(mean_int))
    return mean, mean_int


def make_params(S, R, cap, window, head0, head_step, jobs_per_stream, methods, transform, *, butter_order=16,
                butter_min_bw=0.1, fir_taps=127, fir_df=0.3, min_freq=0.8, max_freq=4.0, ls_num_freqs=0) -> WindowParams:
    p = WindowParams()
    p.S, p.R, p.cap, p.window = S, R, cap, window
    p.head0, p.head_step, p.jobs_per_stream = head0, head_step, jobs_per_stream
    if len(methods) > _cabi.MAX_METHODS:
        raise ValueError('too many processing methods')
    p.num_methods = len(methods)
    for i, m in enumerate(methods):
        p.methods[i] = int(m)
    p.transform = int(transform)
    p.butter_order, p.fir_taps, p.ls_num_freqs = butter_order, fir_taps, int(ls_num_freqs or 0)
    p.butter_min_bw, p.fir_df, p.min_freq, p.max_freq = butter_min_bw, fir_df, min_freq, max_freq
    return p


def _pre_buffers(ring_y, p, proc_x, proc_y, status, workspace):
    J = p.S * p.jobs_per_stream
    dev = ring_y.device
    proc_x = torch.empty((J, p.R, p.window), dtype=torch.float64, device=dev) if proc_x is None else proc_x
    proc_y = torch.empty((J, p.R, p.window), dtype=torch.float64, device=dev) if proc_y is None else proc_y
    status = torch.empty((J, p.R), dtype=torch.int32, device=dev) if status is None else status
    need = lib().bpv_window_workspace_bytes(C.byref(p))
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    return proc_x, proc_y, status, workspace


def window_preprocess(ring_t, ring_y, p: WindowParams, proc_x=None, proc_y=None, status=None, workspace=None):
    """F2 (signal_processor.py:196-245).  Returns proc_x, proc_y f64 [J,R,window], status i32 [J,R]."""
    proc_x, proc_y, status, workspace = _pre_buffers(ring_y, p, proc_x, proc_y, status, workspace)
    _run(ring_y.device, 'bpv_window_preprocess', ptr(ring_t), ptr(ring_y), C.byref(p), ptr(workspace), workspace.numel(),
                                      ptr(proc_x), ptr(proc_y), ptr(status))
    return proc_x, proc_y, status


def new_design_cache(device) -> torch.Tensor:
    """A zero-initialised design cache (include/bpv.h bpv_window_design): keep it across steps, zero it when the filter
    parameters change."""
    return torch.zeros(lib().bpv_design_cache_bytes(), dtype=torch.uint8, device=device)


def window_design(ring_t, p: WindowParams, workspace, cache=None):
    """make_filter of every window job into `workspace` (signal_processor.py:158-173): needs only the timestamps, so
    it can run on another stream beside the ROI sampling of the same frames.  cache = new_design_cache(...) tensor:
    sampling rates that were designed before are looked up instead."""
    _run(ring_t.device, 'bpv_window_design', ptr(ring_t), C.byref(p), ptr(workspace), workspace.numel(),
         ptr(cache), 0 if cache is None else cache.numel())


def window_filter(ring_t, ring_y, p: WindowParams, workspace, proc_x=None, proc_y=None, status=None, cache=None):
    """F2 given the designs `window_design` left in `workspace` (and `cache`, when one was used)."""
    proc_x, proc_y, status, workspace = _pre_buffers(ring_y, p, proc_x, proc_y, status, workspace)
    _run(ring_y.device, 'bpv_window_filter', ptr(ring_t), ptr(ring_y), C.byref(p), ptr(workspace), workspace.numel(),
         ptr(cache), 0 if cache is None else cache.numel(), ptr(proc_x), ptr(proc_y), ptr(status))
    return proc_x, proc_y, status


def jobs_params(p: WindowParams, num_jobs: int) -> WindowParams:
    """The params F3 / F4 (and the per-job output shapes) see for the num_jobs jobs of a job map: S = num_jobs,
    jobs_per_stream = 1 (include/bpv.h: F3 and F4 only use S * jobs_per_stream)."""
    q = WindowParams.from_buffer_copy(p)
    q.S, q.jobs_per_stream, q.head0, q.head_step = int(num_jobs), 1, 0, 0
    return q


def window_design_jobs(ring_t, p: WindowParams, workspace, job_stream, job_head, num_jobs: int, cache=None):
    """window_design over a job map (include/bpv.h bpv_window_design_jobs): p describes the rings."""
    _run(ring_t.device, 'bpv_window_design_jobs', ptr(ring_t), C.byref(p), ptr(workspace), workspace.numel(),
         ptr(cache), 0 if cache is None else cache.numel(), ptr(job_stream), ptr(job_head), int(num_jobs))


def window_filter_jobs(ring_t, ring_y, p: WindowParams, workspace, job_stream, job_head, num_jobs: int, proc_x=None, proc_y=None,
                       status=None, cache=None):
    """window_filter over a job map (include/bpv.h bpv_window_filter_jobs).  Returns proc_x, proc_y f64 [J,R,window],
    status i32 [J,R] for the J = num_jobs jobs."""
    proc_x, proc_y, status, workspace = _pre_buffers(ring_y, jobs_params(p, num_jobs), proc_x, proc_y, status, workspace)
    _run(ring_y.device, 'bpv_window_filter_jobs', ptr(ring_t), ptr(ring_y), C.byref(p), ptr(workspace), workspace.numel(),
         ptr(cache), 0 if cache is None else cache.numel(), ptr(proc_x), ptr(proc_y), ptr(status), ptr(job_stream), ptr(job_head),
         int(num_jobs))
    return proc_x, proc_y, status


def probe_fma(dtype: str, iters: int, blocks: int, sink: torch.Tensor) -> int:
    """Enqueue the FMA throughput probe (bench.py); returns the number of FMAs it executes."""
    with torch.cuda.device(sink.device):
        n = lib().bpv_probe_fma(1 if dtype == 'f64' else 0, int(iters), int(blocks), ptr(sink), stream_handle(sink.device.index))
    if n < 0:
        check(int(-n), 'bpv_probe_fma')
    return int(n)


def max_bins(p: WindowParams) -> int:
    if p.transform == _cabi.PGRAM_LS:
        return p.ls_num_freqs if p.ls_num_freqs > 0 else p.window
    if p.transform == _cabi.DFT_RFFT:
        return p.window // 2 + 1
    return min(256, p.window) // 2 + 1


def _spectrum_out(p: WindowParams, store: bool, out, dev) -> dict:
    """Result tensors of F3 (missing ones are allocated): freqs, mags f32 [J,R,max_bins] | None, num_bins i32, peak_idx i32,
    peak_freq f64, peak_mag f64 [J,R]."""
    J, mb = p.S * p.jobs_per_stream, max_bins(p)
    o = out or {}
    if store:
        if 'freqs' not in o:
            o['freqs'] = torch.full((J, p.R, mb), float('nan'), dtype=torch.float32, device=dev)
        if 'mags' not in o:
            o['mags'] = torch.full((J, p.R, mb), float('nan'), dtype=torch.float32, device=dev)
    else:
        o['freqs'] = o['mags'] = None
    if 'num_bins' not in o:
        o['num_bins'] = torch.empty((J, p.R), dtype=torch.int32, device=dev)
    if 'peak_idx' not in o:
        o['peak_idx'] = torch.empty((J, p.R), dtype=torch.int32, device=dev)
    if 'peak_freq' not in o:
        o['peak_freq'] = torch.empty((J, p.R), dtype=torch.float64, device=dev)
    if 'peak_mag' not in o:
        o['peak_mag'] = torch.empty((J, p.R), dtype=torch.float64, device=dev)
    return o


def _xcorr_out(p: WindowParams, store: bool, out, dev) -> dict:
    """Result tensors of F4 (missing ones are allocated): lags, corr f32 [J,P,2W-1] | None, num_lags, lag_idx i32,
    lag_sec, lag_corr f64 [J,P]."""
    J, P, L = p.S * p.jobs_per_stream, p.R * (p.R - 1) // 2, 2 * p.window - 1
    o = out or {}
    if store:
        if 'lags' not in o:
            o['lags'] = torch.full((J, P, L), float('nan'), dtype=torch.float32, device=dev)
        if 'corr' not in o:
            o['corr'] = torch.full((J, P, L), float('nan'), dtype=torch.float32, device=dev)
    else:
        o['lags'] = o['corr'] = None
    if 'num_lags' not in o:
        o['num_lags'] = torch.empty((J, P), dtype=torch.int32, device=dev)
    if 'lag_idx' not in o:
        o['lag_idx'] = torch.empty((J, P), dtype=torch.int32, device=dev)
    if 'lag_sec' not in o:
        o['lag_sec'] = torch.empty((J, P), dtype=torch.float64, device=dev)
    if 'lag_corr' not in o:
        o['lag_corr'] = torch.empty((J, P), dtype=torch.float64, device=dev)
    return o


def window_welch_xcorr(proc_x, proc_y, p: WindowParams, store: bool = True, out_spectrum=None, out_xcorr=None):
    """F3 (PGRAM_WELCH) + F4 of the same window jobs in ONE grid of interleaved Welch / xcorr CTAs (include/bpv.h
    bpv_window_welch_xcorr).  Returns the dicts of window_spectrum and window_xcorr; same values bit for bit."""
    if p.transform != _cabi.PGRAM_WELCH or p.R < 2:
        raise ValueError('window_welch_xcorr: PGRAM_WELCH and at least two ROIs')
    dev = proc_y.device
    sp, xc = _spectrum_out(p, store, out_spectrum, dev), _xcorr_out(p, store, out_xcorr, dev)
    _run(dev, 'bpv_window_welch_xcorr', ptr(proc_x), ptr(proc_y), C.byref(p), max_bins(p), ptr(sp['freqs']), ptr(sp['mags']),
         ptr(sp['num_bins']), ptr(sp['peak_idx']), ptr(sp['peak_freq']), ptr(sp['peak_mag']), ptr(xc['lags']), ptr(xc['corr']),
         ptr(xc['num_lags']), ptr(xc['lag_idx']), ptr(xc['lag_sec']), ptr(xc['lag_corr']))
    return sp, xc


def peak_band(band, name: str = 'band'):
    """None, or (lo, hi) as two floats: the search range of a band-limited peak (Signal.get_peak(lo, hi), signal_data.py:65-70).
    Infinite bounds are allowed and lo > hi gives no peak, as get_peak does; NaN bounds are rejected."""
    if band is None:
        return None
    try:
        lo, hi = (float(v) for v in band)
    except (TypeError, ValueError):
        raise ValueError(f'{name} must be None or a (lo, hi) pair of numbers, not {band!r}') from None
    if lo != lo or hi != hi:
        raise ValueError(f'{name} has a NaN bound: {band!r}')
    return lo, hi


def window_spectrum(proc_x, proc_y, p: WindowParams, store: bool = True, out=None, workspace=None, band=None):
    """F3 + HR peak (signal_processor.py:248-277, 310).  Returns dict(freqs, mags f32 [J,R,max_bins] | None,
    num_bins i32, peak_idx i32, peak_freq f64, peak_mag f64 [J,R]).
    band = (min_freq, max_freq): the peak is the first maximum over the bins whose frequency lies in the band, as a single
    transform_signal(s).get_peak() finds it (include/bpv.h bpv_window_spectrum_band); the spectrum itself does not change.
    None searches every bin, as process() does."""
    band = peak_band(band)
    dev = proc_y.device
    mb = max_bins(p)
    o = _spectrum_out(p, store, out, dev)
    # scratch for the coarse spectrum when it is not stored; for DFT_RFFT also the persistent twiddle operand images of the
    # tensor-core kernel (zero-initialised: a header tells the kernel whether they are built) — pass the same workspace
    # every call to build them once
    need = lib().bpv_spectrum_workspace_bytes(C.byref(p), mb) if (not store or p.transform == _cabi.DFT_RFFT) else 0
    if need and (workspace is None or workspace.numel() < need):
        workspace = torch.zeros(need, dtype=torch.uint8, device=dev)
    args = (ptr(proc_x), ptr(proc_y), C.byref(p), mb, ptr(workspace) if need else None, need, ptr(o['freqs']), ptr(o['mags']),
            ptr(o['num_bins']), ptr(o['peak_idx']), ptr(o['peak_freq']), ptr(o['peak_mag']))
    if band is None:
        _run(proc_y.device, 'bpv_window_spectrum', *args)
    else:
        _run(proc_y.device, 'bpv_window_spectrum_band', *args, *band)
    return o


def window_xcorr(proc_x, proc_y, p: WindowParams, store: bool = True, out=None, band=None):
    """F4 pairwise xcorr + lag peak (signal_processor.py:280-299, 312).
    band = (min_lag, max_lag) in seconds: the peak is the first maximum over the lags inside the band, as a single
    correlate_signal_pair(a, b).get_peak() finds it (include/bpv.h bpv_window_xcorr_band); the correlation does not change.
    None searches every lag, as process() does."""
    band = peak_band(band)
    P = p.R * (p.R - 1) // 2
    o = _xcorr_out(p, store, out, proc_y.device)
    if P > 0:
        args = (ptr(proc_x), ptr(proc_y), C.byref(p), ptr(o['lags']), ptr(o['corr']), ptr(o['num_lags']), ptr(o['lag_idx']),
                ptr(o['lag_sec']), ptr(o['lag_corr']))
        if band is None:
            _run(proc_y.device, 'bpv_window_xcorr', *args)
        else:
            _run(proc_y.device, 'bpv_window_xcorr_band', *args, *band)
    return o


def butter_sos_design(fs: torch.Tensor, p: WindowParams):
    out = torch.empty((fs.numel(), p.butter_order, 6), dtype=torch.float64, device=fs.device)
    _run(fs.device, 'bpv_butter_sos_design', ptr(fs), fs.numel(), C.byref(p), ptr(out))
    return out


def firls_design(fs: torch.Tensor, p: WindowParams):
    out = torch.empty((fs.numel(), p.fir_taps), dtype=torch.float64, device=fs.device)
    _run(fs.device, 'bpv_firls_design', ptr(fs), fs.numel(), C.byref(p), ptr(out))
    return out


def view_boxes(boxes: torch.Tensor, view_w: int, view_h: int, left: int = 0, flip_horizontally: bool = False, out=None):
    """Map boxes int32 [..., 4] expressed in the VideoReader view (portrait crop frame[:, left:left+view_w], optional
    horizontal flip; video_reader.py:97-103) onto the decoded frame (SURVEY.md 8f row 2).  No pixel is copied."""
    _require(boxes.is_cuda and boxes.dtype == torch.int32 and boxes.is_contiguous() and boxes.shape[-1] == 4, 'bad argument: ' + 'boxes.is_cuda and boxes.dtype == torch.int32 and boxes.is_contiguous() and boxes.shape[-1] == 4')
    out = torch.empty_like(boxes) if out is None else out
    _run(boxes.device, 'bpv_view_boxes', ptr(boxes), boxes.numel() // 4, int(view_w), int(view_h), int(left), int(bool(flip_horizontally)),
                               ptr(out))
    return out


def pack_records(peak_freq, lag_sec, peak_idx, lag_idx, out=None):
    """[J, 2R + 2P] float64 record (bpm, ptt_ms, peak_idx, lag_idx) (signal_processor.py:310, 312)."""
    J, R = peak_freq.shape
    P = lag_sec.shape[1]
    if out is None:
        out = torch.empty((J, 2 * R + 2 * P), dtype=torch.float64, device=peak_freq.device)
    _run(peak_freq.device, 'bpv_pack_records', ptr(peak_freq), ptr(lag_sec) if P else None, ptr(peak_idx), ptr(lag_idx) if P else None,
                                 J, R, P, ptr(out))
    return out


def pack_records32(peak_freq, lag_sec, peak_idx, lag_idx, out=None):
    """[J, 2R + 2P] int32 words: (bpm f32, ptt_ms f32, peak_idx i32, lag_idx i32) — the 24-byte record of SURVEY.md 8(e).
    `unpack_records32` splits it again."""
    J, R = peak_freq.shape
    P = lag_sec.shape[1]
    if out is None:
        out = torch.empty((J, 2 * R + 2 * P), dtype=torch.int32, device=peak_freq.device)
    _run(peak_freq.device, 'bpv_pack_records32', ptr(peak_freq), ptr(lag_sec) if P else None, ptr(peak_idx), ptr(lag_idx) if P else None,
         J, R, P, ptr(out))
    return out


def scratch_discard(*tensors) -> None:
    """Drop the L2 lines of dead scratch tensors without writing them back to DRAM (include/bpv.h bpv_scratch_discard).
    Their contents are undefined afterwards."""
    for t in tensors:
        _require(t.is_cuda and t.is_contiguous(), 'scratch_discard: contiguous CUDA tensors only')
        _run(t.device, 'bpv_scratch_discard', ptr(t), t.numel() * t.element_size())


def unpack_records32(rec: torch.Tensor, R: int, P: int):
    """(bpm f32 [J,R], ptt_ms f32 [J,P], peak_idx i32 [J,R], lag_idx i32 [J,P]) views of a packed int32 record tensor."""
    f = rec.view(torch.float32)
    return f[:, :R], f[:, R:R + P], rec[:, R + P:2 * R + P], rec[:, 2 * R + P:]


def dft256_tc(z: torch.Tensor) -> torch.Tensor:
    """256-point DFT of real segments z f32 [rows, 256] on the tensor cores (tcgen05, 3xTF32): returns f32 [rows, 256] with
    [:, :129] = Re X[0..128] and [:, 129:] = -Im X[1..127]."""
    _require(z.is_cuda and z.dtype == torch.float32 and z.is_contiguous() and z.dim() == 2 and z.shape[1] == 256, 'bad argument: ' + 'z.is_cuda and z.dtype == torch.float32 and z.is_contiguous() and z.dim() == 2 and z.shape[1] == 256')
    d = torch.empty_like(z)
    _run(z.device, 'bpv_dft256_tc', ptr(z), z.shape[0], ptr(d))
    return d


def roi_sample_nv12(frames: torch.Tensor, H: int, W: int, boxes: torch.Tensor, mode: int, *, want_sums: bool = False):
    """F1 on NV12 frames: frames uint8 [N, 3H/2, pitch] (Y plane rows then interleaved UV rows; CUDA or pinned host
    memory), boxes int32 [N, R, 4] in pixel coordinates of the H x W image.  Returns (value f64 [N,R], sums | None): the
    sums of the BGR frame cv2.cvtColor(nv12, COLOR_YUV2BGR_NV12) would give (SURVEY.md 8f row 2)."""
    _require(frames.dtype == torch.uint8 and frames.dim() == 3 and frames.shape[1] == H * 3 // 2 and frames.stride(2) == 1, 'bad argument: ' + 'frames.dtype == torch.uint8 and frames.dim() == 3 and frames.shape[1] == H * 3 // 2 and frames.stride(2) == 1')
    _require(_dev_accessible(frames) and boxes.is_cuda and boxes.dtype == torch.int32 and boxes.is_contiguous(), 'bad argument: ' + '_dev_accessible(frames) and boxes.is_cuda and boxes.dtype == torch.int32 and boxes.is_contiguous()')
    N, R = boxes.shape[0], boxes.shape[1]
    _require(frames.shape[0] == N, 'bad argument: ' + 'frames.shape[0] == N')
    out_value = torch.empty((N, R), dtype=torch.float64, device=boxes.device)
    sums = torch.empty((N, R, 4), dtype=torch.int64, device=boxes.device) if want_sums else None
    fstride = frames.stride(0) if N > 1 else frames.shape[1] * frames.stride(1)
    _run(boxes.device, 'bpv_roi_sample_nv12', ptr(frames), fstride, frames.stride(1), H, W, N, ptr(boxes), R, int(mode), ptr(sums),
                                    ptr(out_value))
    return out_value, sums


def roi_sample_resized(frames: torch.Tensor, dst_h: int, dst_w: int, boxes: torch.Tensor, mode: int, *, want_sums: bool = False):
    """F1 on frames the reference would first have resized with cv2.resize(frame, (dst_w, dst_h)) (video_reader.py:95-96):
    frames uint8 [N, H, W, 3] source frames, boxes int32 [N, R, 4] in the RESIZED frame.  Bit-exact with sampling
    cv2.resize's output; the resized frame is never materialised (SURVEY.md 8f row 2)."""
    _require(frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[-1] == 3 and _dev_accessible(frames), 'bad argument: ' + 'frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[-1] == 3 and _dev_accessible(frames)')
    _require(frames.stride(3) == 1 and frames.stride(2) == 3, 'pixels must be packed BGR')
    N, H, W, _ = frames.shape
    _require(boxes.is_cuda and boxes.dtype == torch.int32 and boxes.is_contiguous() and boxes.shape[0] == N and boxes.shape[2] == 4, 'bad argument: ' + 'boxes.is_cuda and boxes.dtype == torch.int32 and boxes.is_contiguous() and boxes.shape[0] == N and boxes.shape[2] == 4')
    R = boxes.shape[1]
    out_value = torch.empty((N, R), dtype=torch.float64, device=boxes.device)
    sums = torch.empty((N, R, 4), dtype=torch.int64, device=boxes.device) if want_sums else None
    fstride = frames.stride(0) if N > 1 else H * frames.stride(1)
    _run(boxes.device, 'bpv_roi_sample_resized_u8', ptr(frames), fstride, frames.stride(1), H, W, int(dst_h), int(dst_w), N, ptr(boxes), R,
                                          int(mode), ptr(sums), ptr(out_value))
    return out_value, sums


def roi_sample_masked(frames: torch.Tensor, masks: torch.Tensor, categories, boxes: torch.Tensor, mode: int, *,
                      want_sums: bool = False):
    """F1 through a segmentation mask (SURVEY.md 8f row 4): frames uint8 [N, H, W, 3], masks uint8 [N, H, W] per-pixel
    categories (the person segmenter's category_mask, inference_runner.py:154-166), categories = one int for all ROIs or
    an int32 [R] tensor / sequence; boxes int32 [N, R, 4].  Only pixels whose category matches contribute; returns
    (value f64 [N, R], sums (sumB, sumG, sumR, N_selected) | None)."""
    if not (frames.dtype == torch.uint8 and frames.dim() == 4 and frames.shape[-1] == 3 and _dev_accessible(frames)):
        raise ValueError('roi_sample_masked: frames must be uint8 [N, H, W, 3] in CUDA or pinned host memory')
    if not (frames.stride(3) == 1 and frames.stride(2) == 3):
        raise ValueError('roi_sample_masked: pixels must be packed BGR')
    N, H, W, _ = frames.shape
    if not (masks.dtype == torch.uint8 and tuple(masks.shape) == (N, H, W) and masks.stride(2) == 1 and _dev_accessible(masks)):
        raise ValueError('roi_sample_masked: masks must be uint8 [N, H, W] with contiguous rows')
    if not (boxes.is_cuda and boxes.dtype == torch.int32 and boxes.is_contiguous() and boxes.shape[0] == N and boxes.shape[2] == 4):
        raise ValueError('roi_sample_masked: boxes must be a contiguous CUDA int32 [N, R, 4] tensor')
    R = boxes.shape[1]
    dev = boxes.device
    if isinstance(categories, int):
        categories = [categories] * R
    if not torch.is_tensor(categories):
        categories = torch.tensor(list(categories), dtype=torch.int32, device=dev)
    if not (categories.dtype == torch.int32 and categories.numel() == R and categories.device == dev):
        raise ValueError(f'roi_sample_masked: categories must be {R} int32 values on {dev}')
    out_value = torch.empty((N, R), dtype=torch.float64, device=dev)
    sums = torch.empty((N, R, 4), dtype=torch.int64, device=dev) if want_sums else None
    fstride = frames.stride(0) if N > 1 else H * frames.stride(1)
    mstride = masks.stride(0) if N > 1 else H * masks.stride(1)
    _run(dev, 'bpv_roi_sample_masked_u8', ptr(frames), fstride, frames.stride(1), ptr(masks), mstride, masks.stride(1), H, W, N,
         ptr(boxes), R, ptr(categories.contiguous()), int(mode), ptr(sums), ptr(out_value))
    return out_value, sums
