"""BatchedSignalProcessor — the reference's SignalProcessor.process() (signal_processor.py:302-313)
vectorised over S independent video streams on one GPU.

Per step (T frames per stream):
  1. F1  ROI sampling of S*T frames                       (sample_signals, :306)
  2.     push samples + timestamps into the device rings   (sg_raw.add_samples, :307)
  3. F2  preprocessing of every window job                 (process_signals, :308)
  4. F3  spectrum + heart-rate peak                        (transform_signals + get_peaks, :309-310)
  5. F4  pairwise xcorr + PTT lag peak                     (correlate_signals + get_peaks, :311-312)
A window job is one evaluation of a stream's sliding window.  `windows='every_frame'` evaluates the
window after every pushed frame, exactly as the reference does; `windows='last'` only after the last
frame of the step.  All state lives in HBM: ring_t f64 [S, cap], ring_y f64 [S, R, cap].

ROI boxes are inputs (calc_rois / detection are upstream of the path, SURVEY.md §8).  torch is used for
device allocations and the stream handle only; every computation is a libbpv kernel.

Lifetime of results: the tensors of a StepResult are views of `result_buffers` rotating buffer sets owned by the
engine (no allocation per step).  With the default of 2 a result stays valid while the NEXT step runs and is
overwritten by the one after; hold results longer by cloning them or by raising `result_buffers`.

Overlap (`overlap`, bit mask; default from the environment variable BPV_OVERLAP, else OVERLAP_DEFAULT):
  1  the filter design of the step (it needs only the timestamps) runs on a side stream beside F1
  2  F4 (cross-correlation) runs on a side stream beside F3 (spectrum): both only read the processed windows
  4  F3 + F4 as ONE grid of interleaved Welch / xcorr CTAs (PGRAM_WELCH, windows up to 320 samples, >= 2 ROIs; takes precedence
     over 2 where it applies).  Measured SLOWER than bit 2 (profiles/r4g: 272.9 against 227.5 us for the pair, step 0.7255 against
     0.6840 ms) although the two kernels are bound by different things: not in the default mask, kept as a measurement switch.
     It has no band-limited peak search: with `freq_band` or `lag_band` set, the step runs the two kernels of bit 2 instead.

Peak search ranges (`freq_band`, `lag_band`; default None).  process() searches the heart-rate peak over EVERY spectrum bin
and the PTT lag over EVERY correlation lag: SignalGroup resets the ranges that transform_signal / correlate_signal_pair set
(signal_processor.py:272, 294; signal_data.py:82-86), and None keeps that behaviour bit for bit.  A (lo, hi) pair limits the
search as Signal.get_peak(lo, hi) does (signal_data.py:65-70): the peak is the first maximum over the bins (lags) whose
reported frequency in Hz (lag in seconds) lies in [lo, hi]; fewer than two such entries give no peak (NaN, index -1).  The
ranges the reference configures are freq_band=(min_freq, max_freq) and lag_band=(-0.5, 0.5).  Spectra, correlations and
the stored arrays do not depend on the bands; peak_idx / lag_idx still index the full arrays, and the running means and
packed records take the band-limited peaks.  Both are plain attributes: assign a new pair (or None) between steps.

Ragged steps (`frame_counts` of step / step_signals): real streams do not advance in lockstep — cameras join and leave, run
at different frame rates, drop frames.  frame_counts = n_s in 0..T per stream (host sequence, numpy array or CPU tensor):
stream s takes rows [:n_s] of its T input rows and behaves exactly like its own BatchedSignalProcessor(1, R, ...) fed only
those frames (one reference SignalProcessor per camera).  It contributes n_s window jobs ('every_frame') or one job when
n_s > 0 ('last'); jobs are laid out stream-major and in frame order (StepResult.job_offsets / job_stream), which with every
n_s = T is the lockstep layout.  Sample counts, running-mean history lengths and ROI smoothing rows are per stream
(`counts`; `count` is their common value), and reset(streams=[...]) empties chosen streams only.  A step with every
n_s = T from level counts runs the lockstep kernels unchanged; any other step builds a job map on the device
(bpv_stream_jobs) and runs the job-map instantiations of the push, design and filter kernels, F3 / F4 over the J jobs
(every overlap schedule, the fused grid of bit 4 included, works unchanged: F3 / F4 only see J processed windows).  A step
in which no stream takes a frame enqueues nothing.  step_detections stays lockstep.  BPV_FORCE_JOBMAP=1 (attribute
`force_jobmap`) sends level steps through the job-map path too: a measurement switch (tools/bench_ragged.py).

Cadence (`window_stride` k_s, `window_phase` phi_s; one int, or one per stream; default 1 / 0): a display that updates the
heart rate and PTT at 1-2 Hz needs no window job for each of 30 frames a second.  Stream s evaluates its window after its
m-th sample (m = 1, 2, ...) exactly when (m + phi_s) % k_s == 0, with 0 <= phi_s < k_s.  The count is the stream's own, so
the cadence carries across steps, frame_counts, reassignment of the attributes and state_dict(); reset(streams=...) starts
it over.  Each job equals, bit for bit, the 'every_frame' row with the same head; the running means push one value per
evaluated job.  Staggered phases (phi_s = s % k) spread the jobs of equal cadences evenly over the steps: a lower worst step
for a higher mean, since a step of few jobs runs its launches at their latency floor (profiles/r6b: 4096 streams, k = 30,
mean 0.156 -> 0.387 ms, worst 0.783 -> 0.478 ms on a B200 at 1000 W).  A step of S x T frames from level counts with one k
and one phi runs the lockstep kernels with head_step = k; any other strided step builds its job map on the device
(bpv_stream_jobs_strided).  A step can push frames and have no job (k > T, or between cadence points): it samples and pushes
its frames and returns a zero-row result.  k = 1 and phi = 0 everywhere is the 'every_frame' step, unchanged; a stride needs
windows='every_frame' ('last' has its own cadence).  Bad settings raise ValueError at the step, before anything is enqueued.
`cadence_jobs` is the host planning of both paths.

Signal quality (`snr`, `snr_half_width`, `min_snr_db`; default off).  Every window job returns a heart rate, whether its ROI
held a pulsing forehead, a face that turned away or a dark frame, and peak_mag is no quality measure (its unit depends on
the transform, and for DFT / Welch it scales with the signal).  snr=True adds StepResult.snr_db f64 [J, R], the spectral SNR of
de Haan & Jeanne (IEEE TBME 2013), dimensionless and scale-free, computed by one kernel (include/bpv.h bpv_window_snr) from the
spectrum F3 stores: on the stored float32 values widened to float64, the bin power P_k is m_k^2 for DFT_RFFT (amplitude
spectrum) and m_k for PGRAM_WELCH / PGRAM_LS; B = the bins k < num_bins with a finite m_k and lo <= f_k <= hi; a bin is in the
template when |f_k - f0| <= snr_half_width or |f_k - 2 f0| <= snr_half_width (f0 = f_{peak_idx}, in Hz; default 0.125 Hz =
7.5 bpm: the peak bin and its two neighbours on the 0.1 Hz DFT grid of 10 s at 30 fps, where 0.1 Hz would put a neighbour in
or out on float32 rounding, and on the 0.117 Hz Welch grid); snr_db = 10 log10(S_sig / S_noise) with IEEE semantics (0/x ->
-inf, x/0 -> +inf, 0/0 -> NaN), NaN when there is no peak or |B| < 2.  The band is freq_band when set, else (min_freq,
max_freq); an unbanded DC peak (0 bpm) therefore gets -inf.  B is decided on the stored float32 frequencies, so it can differ
from the band-limited peak search (float64) in a bin within float32 rounding of lo or hi.  min_snr_db (dB, -inf allowed; a plain
attribute, reassignable between steps; needs snr=True) gates what the running means push: a heart rate is accepted when snr_db
>= min_snr_db (NaN is rejected), a pair's PTT when both of its ROIs are, and a rejected value enters the history as NaN (which
np.nanmean skips).  peak_freq, lag_sec, the indices and the packed records stay ungated; the gate adds no state.  The kernel runs
on the main stream after F3 (and after the xcorr event) on every path: one more launch per step.  Memory: F3 then stores its
spectrum into the result buffers even with store_arrays=False (res.arrays stays empty): 2 x 4 B x Jmax x R x max_bins per
result buffer, 34 MB for c2 (16 384 jobs, R = 2, 129 Welch bins), 134 MB for 4096 jobs of a 2048-bin Lomb-Scargle grid.
snr=False takes exactly the path and launches of an engine without the feature.
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _cabi, ops

EVERY_FRAME, LAST = 'every_frame', 'last'
OVERLAP_DESIGN, OVERLAP_XCORR, OVERLAP_FUSED = 1, 2, 4
OVERLAP_DEFAULT = OVERLAP_DESIGN | OVERLAP_XCORR    # measured on c2 (profiles/r2k_overlap_ab.txt): 0.474 ms serial, 0.467 xcorr only, 0.461 both
STATE_VERSION = 2          # 2: per-stream sample / running-mean counts (version 1 states hold one level count)


def cadence_jobs(counts, n, stride, phase):
    """Window jobs of a strided step (module docstring, cadence) from host int64 arrays (or ints) of the streams' sample
    counts c, frames taken n, strides k and phases phi: (jobs per stream, J, first heads).  Stream s takes
    q = (c + n + phi) // k - b jobs with b = (c + phi) // k; job i has its newest sample at (b + 1 + i) * k - phi - 1."""
    b = (counts + phase) // stride
    jobs = (counts + n + phase) // stride - b
    return jobs, int(np.sum(jobs)), (b + 1) * stride - phase - 1


@dataclass
class StepResult:
    """Device tensors for the J window jobs of one step.  A lockstep step has J = S * jobs_per_stream (job =
    s*jobs_per_stream + j; 0 jobs per stream for a strided step between cadence points); a ragged or per-stream strided
    step (module docstring) has jobs_per_stream = None and the jobs of stream s in rows job_offsets[s]:job_offsets[s+1],
    in frame order."""
    jobs_per_stream: int | None
    samples: torch.Tensor | None          # f64 [S, T, R]   raw ROI samples of this step
    peak_freq: torch.Tensor               # f64 [J, R]      Hz (NaN = none)
    peak_idx: torch.Tensor                # i32 [J, R]
    peak_mag: torch.Tensor                # f64 [J, R]
    lag_sec: torch.Tensor                 # f64 [J, P]
    lag_idx: torch.Tensor                 # i32 [J, P]
    lag_corr: torch.Tensor                # f64 [J, P]
    status: torch.Tensor                  # i32 [J, R]
    arrays: dict = field(default_factory=dict)   # proc_x/proc_y/freqs/mags/lags/corr/num_bins/num_lags when stored
    means: dict = field(default_factory=dict)    # mean_bpm, mean_bpm_int [J, R], mean_ptt, mean_ptt_int [J, P] when tracked
    _job_offsets: np.ndarray | None = field(default=None, repr=False)   # host int64 [S+1] of a ragged step
    _job_stream: torch.Tensor | None = field(default=None, repr=False)  # device int32 [J] of a ragged step
    snr_db: torch.Tensor | None = None    # f64 [J, R]      spectral SNR of the heart-rate peak (engine snr=True)

    @property
    def job_offsets(self) -> np.ndarray:
        """Host int64 [S+1]: the jobs of stream s are rows job_offsets[s]:job_offsets[s+1]."""
        if self._job_offsets is None:
            S = self.peak_freq.shape[0] // self.jobs_per_stream
            self._job_offsets = np.arange(S + 1, dtype=np.int64) * self.jobs_per_stream
        return self._job_offsets

    @property
    def job_stream(self) -> torch.Tensor:
        """Device int32 [J]: the stream of each job (built on first use for a lockstep step)."""
        if self._job_stream is None:
            off = self.job_offsets
            rows = np.repeat(np.arange(len(off) - 1, dtype=np.int32), np.diff(off))
            self._job_stream = torch.from_numpy(rows).to(self.peak_freq.device)
        return self._job_stream

    @property
    def bpm(self):                        # signal_processor.py:310  f * 60
        return self.peak_freq * 60

    @property
    def ptt_ms(self):                     # signal_processor.py:312  t * 1000
        return self.lag_sec * 1000

    def packed(self, out: torch.Tensor | None = None) -> torch.Tensor:
        """[J, 2R + 2P] float64 record (bpm, ptt_ms, peak_idx, lag_idx): full-precision host read-back."""
        return ops.pack_records(self.peak_freq, self.lag_sec, self.peak_idx, self.lag_idx, out=out)

    def packed32(self, out: torch.Tensor | None = None) -> torch.Tensor:
        """[J, 2R + 2P] int32 words (bpm f32, ptt_ms f32, peak_idx i32, lag_idx i32): the 24-byte record of SURVEY.md
        8(e) that the multi-GPU gather moves (`ops.unpack_records32` splits it)."""
        return ops.pack_records32(self.peak_freq, self.lag_sec, self.peak_idx, self.lag_idx, out=out)


class BatchedSignalProcessor:
    def __init__(self, num_streams: int, num_rois: int = 2, *, signal_max_samples: int = 250,
                 max_frames_per_step: int = 1, color_channel: int = _cabi.GREEN, processing_methods=(_cabi.FILTER_BUTTER,),
                 spectrum_transform: int = _cabi.PGRAM_LS, butter_order: int = 16, butter_min_bw: float = 0.1,
                 fir_taps: int = 127, fir_df: float = 0.3, min_freq: float = 0.8, max_freq: float = 4.0,
                 ls_num_freqs: int | None = None, windows: str = EVERY_FRAME, store_arrays: bool = False,
                 device: str | torch.device = 'cuda', roi_pixels_hint: int = 0, peak_max_samples: int = 0,
                 result_buffers: int = 2, overlap: int | None = None, design_cache: bool | None = None,
                 freq_band: tuple[float, float] | None = None, lag_band: tuple[float, float] | None = None,
                 window_stride=1, window_phase=0, snr: bool = False, snr_half_width: float = ops.SNR_HALF_WIDTH,
                 min_snr_db: float | None = None):
        _cabi.lib()  # fail loudly if the CUDA library is missing: there is no CPU fallback
        if not torch.cuda.is_available():
            raise _cabi.BpvError('BatchedSignalProcessor needs a CUDA device (no CPU fallback)')
        if windows not in (EVERY_FRAME, LAST):
            raise ValueError(f"windows must be '{EVERY_FRAME}' or '{LAST}', not {windows!r}")
        if int(num_streams) < 1 or int(num_rois) < 1 or int(signal_max_samples) < 1 or int(max_frames_per_step) < 1:
            raise ValueError('num_streams, num_rois, signal_max_samples and max_frames_per_step must be positive')
        if int(result_buffers) < 1:
            raise ValueError('result_buffers must be >= 1')
        self.S, self.R, self.P = int(num_streams), int(num_rois), math.comb(int(num_rois), 2)
        self.W = int(signal_max_samples)
        self.Tmax = int(max_frames_per_step)
        self.cap = self.W + self.Tmax
        self.color_channel = int(color_channel)
        self.methods = [int(m) for m in processing_methods]
        self.transform = int(spectrum_transform)
        self.kw = dict(butter_order=butter_order, butter_min_bw=butter_min_bw, fir_taps=fir_taps, fir_df=fir_df,
                       min_freq=min_freq, max_freq=max_freq, ls_num_freqs=int(ls_num_freqs or 0))
        self.windows, self.store_arrays = windows, bool(store_arrays)
        # peak search ranges (module docstring): None = every bin / lag, as process()
        self.freq_band = ops.peak_band(freq_band, 'freq_band')
        self.lag_band = ops.peak_band(lag_band, 'lag_band')
        # signal quality (module docstring): fixed at construction, since F3 then stores its spectrum into the result buffers
        self.snr = bool(snr)
        self.snr_half_width = ops.snr_half_width(snr_half_width)
        self._min_snr_db = None
        self.min_snr_db = min_snr_db
        self.roi_pixels_hint = int(roi_pixels_hint)
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise _cabi.BpvError('BatchedSignalProcessor needs a CUDA device (no CPU fallback)')
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        if overlap is None:
            env = os.environ.get('BPV_OVERLAP')
            overlap = int(env) if env not in (None, '') else OVERLAP_DEFAULT
        self.overlap = int(overlap)
        dev, f64 = self.device, torch.float64
        self.ring_t = torch.full((self.S, self.cap), float('nan'), dtype=f64, device=dev)
        self.ring_y = torch.full((self.S, self.R, self.cap), float('nan'), dtype=f64, device=dev)
        # samples pushed per stream so far (global index of the next sample) and bpm / ptt history lengths: an int while every
        # stream holds the same count (the lockstep path), else a host int64 [S] array (the `counts` property)
        self._cnt = self._mcnt = 0
        # device copies for the job-map path: the sample counts (ping-pong: bpv_stream_jobs writes the advanced ones), valid
        # while _g0_ok; the history counts are uploaded for every ragged step that tracks running means
        self._g0 = [torch.zeros(self.S, dtype=torch.int64, device=dev) for _ in range(2)]
        self._g0_ok = True
        self._mg0 = torch.zeros(self.S, dtype=torch.int64, device=dev) if int(peak_max_samples) else None
        self._ndev = torch.zeros(self.S, dtype=torch.int32, device=dev)
        self._jobmap = [None] * int(result_buffers)          # per result buffer: job_stream i32 [Jmax], job_head i64, stream_job0 i32
        # per result buffer: pinned staging of the host counts a job-map step uploads, and an event after those copies (the
        # host waits on it before refilling the buffer: a fresh pinned allocation per step would call cudaHostAlloc)
        self._staging = [None] * int(result_buffers)
        # measurement switch: level counts take the job-map path too (tools/bench_ragged.py)
        self.force_jobmap = os.environ.get('BPV_FORCE_JOBMAP', '0') == '1'
        Jmax = self.S * (self.Tmax if windows == EVERY_FRAME else 1)
        self._Jmax = Jmax
        self._nbuf = int(result_buffers)
        self._turn = 0
        self._samples = [torch.empty((self.S, self.Tmax, self.R), dtype=f64, device=dev) for _ in range(self._nbuf)]
        # the processed windows are results only when the arrays are stored; otherwise scratch between F2 and F3 / F4
        nproc = self._nbuf if self.store_arrays else 1
        self._proc = [torch.empty((2, Jmax, self.R, self.W), dtype=f64, device=dev) for _ in range(nproc)]   # [x | y]
        self._status = [torch.empty((Jmax, self.R), dtype=torch.int32, device=dev) for _ in range(self._nbuf)]
        self._out = [None] * self._nbuf          # per result buffer: F3 / F4 outputs of Jmax jobs, sliced to each step's J
        p = self._params(0, 1, self.Tmax if windows == EVERY_FRAME else 1)
        self._mb = ops.max_bins(p)
        need = max(_cabi.lib().bpv_window_workspace_bytes(p), 16)
        self._ws = torch.empty(need, dtype=torch.uint8, device=dev)                 # per-job filter designs
        need = max(_cabi.lib().bpv_spectrum_workspace_bytes(p, self._mb), 16)
        self._ws_spec = torch.zeros(need, dtype=torch.uint8, device=dev)    # zeroed: holds the DFT twiddle images' header
        self.launches_per_step = self._extra_launches = 0
        self._has_filter = any(m in (_cabi.FILTER_BUTTER, _cabi.FILTER_FIR) for m in self.methods)
        # design cache (include/bpv.h bpv_window_design): make_filter is a pure function of fs, so sampling rates that were
        # designed before — constant-fps streams: every window of every stream on that clock — are looked up, not redesigned
        if design_cache is None:
            design_cache = os.environ.get('BPV_DESIGN_CACHE', '1') != '0'
        self._dcache = ops.new_design_cache(dev) if design_cache else None
        self._dcache_sig = None
        # measured (profiles/r2q_discard_depth_ab.txt): at 8192 jobs per step the discard saves 2.2 us of F1 and costs 4 us itself; at
        # 16 384 jobs the scratch (157 MB) no longer fits L2 and has been written back before F1 starts -> off by default
        self.discard_scratch = os.environ.get('BPV_DISCARD', '0') == '1'
        self._side = None
        self._side_hi = None
        self._ev = None
        # SURVEY.md §8(f) row 3: sg_bpm / sg_ptt histories and their running means on the device (0 = off)
        self.peak_max_samples = int(peak_max_samples)
        self._bpm_ring = self._ptt_ring = None
        if self.peak_max_samples:
            self._bpm_ring = torch.full((self.S, self.R, self.peak_max_samples), float('nan'), dtype=f64, device=dev)
            self._ptt_ring = torch.full((self.S, max(self.P, 1), self.peak_max_samples), float('nan'), dtype=f64, device=dev)
        self._roi_hist = None
        self._roi_count = 0
        # window cadence (module docstring): plain attributes, checked at every step; the device copies of a strided job-map
        # step are uploaded when they change
        self.window_stride, self.window_phase = window_stride, window_phase
        self._cad_dev = self._cad_host = None
        self._cadence()

    # ------------------------------------------------------------------------------------------
    def _params(self, head0: int, head_step: int, jobs: int) -> _cabi.WindowParams:
        return ops.make_params(self.S, self.R, self.cap, self.W, head0, head_step, jobs, self.methods, self.transform, **self.kw)

    def _streams(self):
        """Side stream + events of the overlapped schedule (created on first use, on the engine's device)."""
        if self._side is None:
            with torch.cuda.device(self.device):
                self._side = torch.cuda.Stream(device=self.device)
                # BPV_DESIGN_PRIO=1 puts the design probe (512 CTAs, F2 waits for it) on a high-priority stream: its CTAs are then
                # placed as soon as F1's retire instead of behind the 32 768 F1 CTAs already queued.  Measured (profiles/r4b): the
                # probe finishes 90 us earlier, the step gains 2 us (0.7011 -> 0.6990 ms) and F1 loses 2.4 us to the probe's CTAs
                # (0.722 -> 0.708 of the HBM peak by the events around it) -> off by default
                prio = -1 if os.environ.get('BPV_DESIGN_PRIO', '0') == '1' else 0
                self._side_hi = torch.cuda.Stream(device=self.device, priority=prio)
                self._ev = {k: torch.cuda.Event() for k in ('ts', 'design', 'pre', 'xc')}
        return self._side, self._ev

    @property
    def min_snr_db(self) -> float | None:
        """SNR gate of the running means in dB (module docstring, signal quality); None = no gate.  Reassignable between
        steps; needs snr=True."""
        return self._min_snr_db

    @min_snr_db.setter
    def min_snr_db(self, value) -> None:
        value = ops.snr_threshold(value)
        if value is not None and not self.snr:
            raise ValueError('min_snr_db needs an engine built with snr=True')
        self._min_snr_db = value

    # per-stream counts (module docstring: ragged steps)
    @property
    def counts(self) -> np.ndarray:
        """Host int64 [S]: samples pushed so far per stream."""
        return np.full(self.S, self._cnt, dtype=np.int64) if isinstance(self._cnt, int) else self._cnt.copy()

    @property
    def count(self) -> int:
        """The samples pushed per stream while every stream holds the same count; raises ValueError otherwise (see
        `counts`).  Assigning it sets every stream's count."""
        if not isinstance(self._cnt, int):
            raise ValueError('count: the streams hold different sample counts; read `counts`')
        return self._cnt

    @count.setter
    def count(self, value: int) -> None:
        self._cnt = int(value)
        self._g0_ok = False

    def _level(self, a: np.ndarray):
        """a as one int when every stream holds the same value (the lockstep path's form), else as the array."""
        return int(a[0]) if (a == a[0]).all() else a

    def _host_ints(self, value, name: str, scalar: bool = False) -> np.ndarray:
        """value (host sequence / numpy array / CPU int tensor of S integers; one integer for every stream when `scalar`)
        as int64 [S]."""
        if torch.is_tensor(value):
            if value.device.type != 'cpu':
                raise ValueError(f'{name} must live on the host (a sequence, numpy array or CPU tensor): the engine '
                                 'needs the job count without synchronising with the device')
            value = value.numpy()
        a = np.asarray(value)
        if scalar and a.shape == ():
            a = np.full(self.S, a)
        if a.shape != (self.S,):
            raise ValueError(f'{name} must hold {self.S} values, got shape {a.shape}')
        if a.dtype.kind not in 'iu' and not (a.dtype.kind == 'f' and np.array_equal(a, np.floor(a))):
            raise ValueError(f'{name} must be integers, got {a.dtype}')
        return a.astype(np.int64)

    def _frame_counts(self, frame_counts, T: int):
        """frame_counts (host sequence / numpy array / CPU int tensor of S values in 0..T) as int64 [S], or None."""
        if frame_counts is None:
            return None
        a = self._host_ints(frame_counts, 'frame_counts')
        if a.size and (a.min() < 0 or a.max() > T):
            raise ValueError(f'frame_counts must lie in [0, {T}]')
        return a

    def _cadence(self):
        """window_stride / window_phase checked for the coming step: None for the default (a job after every frame), else
        dict(k=, phase= host int64 [S], uniform= one k and one phase for every stream)."""
        k, ph = self.window_stride, self.window_phase
        if type(k) is int and type(ph) is int and k == 1 and ph == 0:
            return None
        k, ph = self._host_ints(k, 'window_stride', True), self._host_ints(ph, 'window_phase', True)
        if k.min() < 1 or k.max() > np.iinfo(np.int32).max:
            raise ValueError('window_stride must lie in [1, 2^31)')
        if ph.min() < 0 or (ph >= k).any():
            raise ValueError('window_phase must lie in [0, window_stride)')
        if k.max() == 1:
            return None
        if self.windows == LAST:
            raise ValueError("window_stride != 1 needs windows='every_frame' ('last' has its own cadence)")
        return dict(k=k, phase=ph, uniform=bool((k == k[0]).all() and (ph == ph[0]).all()))

    def _lockstep(self, n, T: int, cad) -> bool:
        """The lockstep path serves a step in which every stream takes T frames from the same counts with the same cadence."""
        return ((n is None or bool((n == T).all())) and isinstance(self._cnt, int) and isinstance(self._mcnt, int)
                and (cad is None or cad['uniform']) and not self.force_jobmap)

    def _plan(self, n, T: int, cad) -> dict | None:
        """Host side of a step: None for a lockstep step at the default cadence; for a strided lockstep step its head0,
        head_step, jobs per stream and J; for a job-map step the per-stream frame counts, job counts, offsets and J."""
        if self._lockstep(n, T, cad):
            if cad is None:
                return None
            k, ph = int(cad['k'][0]), int(cad['phase'][0])
            jobs, _, head0 = cadence_jobs(self._cnt, T, k, ph)
            return dict(lock=True, head0=head0, head_step=k, jobs=jobs, J=self.S * jobs)
        n = np.full(self.S, T, dtype=np.int64) if n is None else n
        if cad is not None:
            jobs = cadence_jobs(self.counts, n, cad['k'], cad['phase'])[0]
        else:
            jobs = n if self.windows == EVERY_FRAME else (n > 0).astype(np.int64)
        off = np.zeros(self.S + 1, dtype=np.int64)
        np.cumsum(jobs, out=off[1:])
        return dict(lock=False, n=n, jobs=jobs, off=off, J=int(off[-1]), T=T, mapped=False, cad=cad)

    def _lock_jobs(self, T: int, plan):
        """(head0, head_step, jobs per stream) of a lockstep step from the current count."""
        if plan is not None:
            return plan['head0'], plan['head_step'], plan['jobs']
        if self.windows == EVERY_FRAME:
            return self._cnt, 1, T
        return self._cnt + T - 1, 1, 1

    def _map_jobs(self, plan: dict, turn: int) -> None:
        """Upload the step's frame counts (and the sample counts when the device copy is stale) and build the job map of
        the plan on the device (bpv_stream_jobs), into the buffers of result turn `turn`."""
        dev = self.device
        if self._jobmap[turn] is None:
            self._jobmap[turn] = (torch.empty(self._Jmax, dtype=torch.int32, device=dev),
                                  torch.empty(self._Jmax, dtype=torch.int64, device=dev),
                                  torch.empty(self.S + 1, dtype=torch.int32, device=dev))
        pin = self._pinned(turn)
        pin['n'].numpy()[:] = plan['n']
        self._ndev.copy_(pin['n'], non_blocking=True)
        if not self._g0_ok:
            pin['g0'].numpy()[:] = self.counts
            self._g0[0].copy_(pin['g0'], non_blocking=True)
            self._g0_ok = True
        js, jh, sj0 = self._jobmap[turn]
        if plan['cad'] is None:
            ops.stream_jobs(self._g0[0], self._ndev, self.windows == LAST, plan['J'], js, jh, sj0, self._g0[1])
        else:
            kd, pd = self._cadence_dev(plan['cad'], pin)
            ops.stream_jobs_strided(self._g0[0], self._ndev, kd, pd, plan['J'], js, jh, sj0, self._g0[1])
        plan['mapped'] = True

    def _cadence_dev(self, cad: dict, pin: dict):
        """Device int32 [S] copies of the strides and phases, uploaded through the pinned staging `pin` when they changed."""
        if self._cad_dev is None:
            self._cad_dev = tuple(torch.empty(self.S, dtype=torch.int32, device=self.device) for _ in range(2))
        host = self._cad_host
        if host is None or not (np.array_equal(host[0], cad['k']) and np.array_equal(host[1], cad['phase'])):
            pin['k'].numpy()[:] = cad['k']
            pin['ph'].numpy()[:] = cad['phase']
            self._cad_dev[0].copy_(pin['k'], non_blocking=True)
            self._cad_dev[1].copy_(pin['ph'], non_blocking=True)
            self._cad_host = (cad['k'].copy(), cad['phase'].copy())
        return self._cad_dev

    def _pinned(self, turn: int) -> dict:
        """Pinned staging buffers of result turn `turn`, once the device has consumed their previous contents."""
        if self._staging[turn] is None:
            mk = lambda dt: torch.empty(self.S, dtype=dt).pin_memory()
            self._staging[turn] = dict(n=mk(torch.int32), g0=mk(torch.int64), m0=mk(torch.int64), k=mk(torch.int32),
                                       ph=mk(torch.int32), ev=torch.cuda.Event(), used=False)
        pin = self._staging[turn]
        if pin['used']:
            pin['ev'].synchronize()
            pin['used'] = False
        return pin

    def _check_step(self, S, T, boxes=None):
        if S != self.S or not 1 <= T <= self.Tmax:
            raise ValueError(f'step: expected {self.S} streams and 1..{self.Tmax} frames per stream, got {S} x {T}')
        if boxes is not None and tuple(boxes.shape) != (S, T, self.R, 4):
            raise ValueError(f'step: boxes must be int32 [{S}, {T}, {self.R}, 4], got {tuple(boxes.shape)}')

    def step(self, frames: torch.Tensor, boxes: torch.Tensor, timestamps: torch.Tensor, view=None, nv12_size=None,
             resize_to=None, masks: torch.Tensor | None = None, mask_category=0, frame_counts=None) -> StepResult:
        """frames uint8 [S, T, H, W, 3] (HBM, or pinned host memory: the ROI kernel then reads the ROI rows
        straight over PCIe), boxes int32 [S, T, R, 4] (device), timestamps float64 [S, T] (device).
        view = (view_w, view_h, left, flip_horizontally): the boxes are expressed in the reference VideoReader's
        cropped / mirrored view of the decoded frames (video_reader.py:97-103) and are mapped back onto `frames`
        on the device; nothing is copied.
        nv12_size = (H, W): frames are NV12 decoder buffers uint8 [S, T, 3H/2, pitch]; the ROI is sampled from the planes
        with OpenCV's integer BT.601 conversion, i.e. as from the BGR frame cv2.VideoCapture would have produced.
        masks uint8 [S, T, H, W] + mask_category (one int, or one per ROI): only ROI pixels whose segmentation category
        matches contribute (SURVEY.md §8(f) row 4; category masks as InferenceResults.person_segmenter, inference_runner.py:154-166).
        frame_counts: S values n_s in 0..T on the host (module docstring, ragged steps): stream s takes rows [:n_s] of its T
        frames.  F1 still samples all S x T rows; the rows a stream does not take cost next to nothing when their boxes
        are BPV_NO_BOX (x0 = NO_BOX).  A step in which no stream takes a frame enqueues nothing (samples = None)."""
        S, T = frames.shape[:2]
        self._check_step(S, T, boxes)
        cad = self._cadence()
        if self.snr:
            self.snr_half_width = ops.snr_half_width(self.snr_half_width)
        n = self._frame_counts(frame_counts, T)
        if n is not None and not n.any():
            return self._empty_step(None)
        self._extra_launches = 0
        with torch.cuda.device(self.device):
            if view is not None:
                boxes = ops.view_boxes(boxes.contiguous(), *view)
                self._extra_launches = 1
            if resize_to is not None:
                # boxes live in the frame cv2.resize(frame, (dst_w, dst_h)) would produce (video_reader.py:95-96); pixels
                # are generated on the fly with OpenCV's integer bilinear arithmetic, the resized frame is never materialised
                dst_h, dst_w = resize_to
                val, _ = ops.roi_sample_resized(frames.view(S * T, *frames.shape[2:]), dst_h, dst_w,
                                                boxes.reshape(S * T, self.R, 4).contiguous(), self.color_channel)
                return self.step_signals(val.view(S, T, self.R), timestamps, _count_roi=True, frame_counts=n)
            if nv12_size is not None:
                H, W = nv12_size
                val, _ = ops.roi_sample_nv12(frames.view(S * T, *frames.shape[2:]), H, W,
                                             boxes.reshape(S * T, self.R, 4).contiguous(), self.color_channel)
                return self.step_signals(val.view(S, T, self.R), timestamps, _count_roi=True, frame_counts=n)
            if masks is not None:
                val, _ = ops.roi_sample_masked(frames.view(S * T, *frames.shape[2:]), masks.view(S * T, *masks.shape[2:]),
                                               mask_category, boxes.reshape(S * T, self.R, 4).contiguous(),
                                               self.color_channel)
                return self.step_signals(val.view(S, T, self.R), timestamps, _count_roi=True, frame_counts=n)
            samples = self._samples[self._turn][:, :T]
            if T != self.Tmax:
                samples = torch.empty((S, T, self.R), dtype=torch.float64, device=self.device)
            plan = self._plan(n, T, cad)
            design_ahead = (bool(self.overlap & OVERLAP_DESIGN)
                            and any(m in (_cabi.FILTER_BUTTER, _cabi.FILTER_FIR) for m in self.methods)
                            and (plan is None or plan['J'] > 0))      # a step without jobs has nothing to design
            if design_ahead and (plan is None or plan['lock']):
                self._design_ahead(timestamps, T, plan)
            elif design_ahead:
                self._design_ahead_jobs(timestamps, plan)
            ops.roi_sample(frames.view(S * T, *frames.shape[2:]), boxes.view(S * T, self.R, 4), self.color_channel,
                           roi_pixels_hint=self.roi_pixels_hint, out_value=samples.view(S * T, self.R))
            return self.step_signals(samples, timestamps, _count_roi=True, _designed=design_ahead, frame_counts=n, _plan=plan)

    def _design_ahead(self, timestamps: torch.Tensor, T: int, plan) -> None:
        """Push the step's timestamps and start the filter design of its window jobs on the side stream: make_filter
        depends on nothing else (signal_processor.py:158-173), so it runs beside F1 instead of between F1 and F2."""
        _, ev = self._streams()
        side = self._side_hi
        main = torch.cuda.current_stream(self.device)
        ops.ring_push(self.ring_t, self.ring_y, self._cnt, timestamps.contiguous(), None)
        ev['ts'].record(main)
        head0, head_step, jobs = self._lock_jobs(T, plan)
        p = self._params(head0, head_step, jobs)
        side.wait_event(ev['ts'])
        with torch.cuda.stream(side):
            ops.window_design(self.ring_t, p, self._ws, self._cache())
            ev['design'].record(side)

    def _design_ahead_jobs(self, timestamps: torch.Tensor, plan: dict) -> None:
        """_design_ahead for a job-map step: ragged timestamp push, job map, then the design of the mapped jobs on the
        side stream."""
        _, ev = self._streams()
        side = self._side_hi
        main = torch.cuda.current_stream(self.device)
        self._map_jobs(plan, self._turn)
        ops.ring_push_ragged(self.ring_t, self.ring_y, self._g0[0], self._ndev, timestamps.contiguous(), None)
        ev['ts'].record(main)
        js, jh, _ = self._jobmap[self._turn]
        side.wait_event(ev['ts'])
        with torch.cuda.stream(side):
            ops.window_design_jobs(self.ring_t, self._params(0, 1, 1), self._ws, js, jh, plan['J'], self._cache())
            ev['design'].record(side)

    def _cache(self):
        """The design cache, emptied whenever the filter parameters it was filled under have changed (the drop-in
        SignalProcessor lets callers edit them between frames)."""
        if self._dcache is None:
            return None
        sig = tuple(sorted(self.kw.items()))
        if sig != self._dcache_sig:
            if self._dcache_sig is not None:
                self._dcache.zero_()
            self._dcache_sig = sig
        return self._dcache

    # ------------------------------------------------------------------------------------------
    # SURVEY.md §8(f) row 1: calc_rois + ROI smoothing on the device for batched landmark tensors
    def set_roi_configs(self, relative_bboxes, num_points, roi_max_samples: int = 1):
        """relative_bboxes [R][4] (left, top, right, bottom) and the number of anchor landmarks per ROI, as in
        roi.ROIConfig (roi.py:8-13); roi_max_samples = length of the smoothing history (signal_processor.py:47)."""
        if len(relative_bboxes) != self.R or len(num_points) != self.R:
            raise ValueError(f'set_roi_configs: expected {self.R} ROI configs')
        self._rel = torch.tensor(relative_bboxes, dtype=torch.float64, device=self.device).contiguous()
        self._npts = torch.tensor(num_points, dtype=torch.int32, device=self.device)
        self._roi_hist = torch.full((self.S, self.R, int(roi_max_samples), 6), float('nan'), dtype=torch.float64, device=self.device)
        self._roi_count = 0

    def step_detections(self, frames, present, bbox, points, timestamps, want_locations: bool = False):
        """One step from detector outputs instead of boxes: present u8 [S,T,R], bbox i32 [S,T,R,4] (largest detection
        of the ROI's model), points i32 [S,T,R,K,2] (the landmarks the ROI config selects).  Returns (StepResult, boxes
        [, locations, smoothed])."""
        if self._roi_hist is None:
            raise ValueError('step_detections: call set_roi_configs first')
        out = ops.calc_rois(present, bbox, points, self._npts, self._rel, self._roi_hist, self._roi_count, want_locations)
        self._roi_count += present.shape[1]
        boxes = out[0] if want_locations else out
        res = self.step(frames, boxes, timestamps)
        return (res, *out) if want_locations else (res, boxes)

    def roi_samples(self, frames: torch.Tensor, boxes: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """F1 only, on the current stream: float64 [S, T, R] samples of frames uint8 [S, T, H, W, 3].  Lets a caller
        overlap the ROI sampling of the next batch (e.g. zero-copy from pinned host memory, PCIe bound) with the
        window pipeline of the current one: run this on a side stream, then `step_signals` on the main stream."""
        S, T = frames.shape[:2]
        if S != self.S or tuple(boxes.shape) != (S, T, self.R, 4):
            raise ValueError('roi_samples: frames [S, T, H, W, 3] / boxes [S, T, R, 4] do not match the engine')
        if out is None:
            out = torch.empty((S, T, self.R), dtype=torch.float64, device=self.device)
        ops.roi_sample(frames.view(S * T, *frames.shape[2:]), boxes.view(S * T, self.R, 4), self.color_channel,
                       roi_pixels_hint=self.roi_pixels_hint, out_value=out.view(S * T, self.R))
        return out

    def step_signals(self, samples: torch.Tensor, timestamps: torch.Tensor, _count_roi: bool = False,
                     _designed: bool = False, frame_counts=None, _plan: dict | None = None) -> StepResult:
        """Signals-only entry: samples float64 [S, T, R] (already ROI-sampled), timestamps float64 [S, T].
        frame_counts: as in `step`; stream s takes rows [:n_s] of its samples and timestamps, the others are not read."""
        S, T, R = samples.shape
        self._check_step(S, T)
        if R != self.R or tuple(timestamps.shape) != (S, T):
            raise ValueError(f'step_signals: samples must be [S, T, {self.R}] and timestamps [S, T]')
        cad = self._cadence()
        if self.snr:
            self.snr_half_width = ops.snr_half_width(self.snr_half_width)
        n = self._frame_counts(frame_counts, T)
        if n is not None and not n.any():
            return self._empty_step(samples)
        if _plan is None:
            _plan = self._plan(n, T, cad)
        with torch.cuda.device(self.device):
            return self._step_signals(samples, timestamps, S, T, _count_roi, _designed, _plan)

    def _empty_step(self, samples, jobs_per_stream=None, launches: int = 0) -> StepResult:
        """A result of zero jobs.  A step in which no stream takes a frame enqueues nothing and changes no state; a strided
        step without jobs has pushed its frames (`launches`)."""
        dev, f64, f32, i32 = self.device, torch.float64, torch.float32, torch.int32
        R, P, W = self.R, self.P, self.W
        e = lambda *shape, dt=f64: torch.empty(shape, dtype=dt, device=dev)
        arrays, means = {}, {}
        if self.store_arrays:
            arrays = dict(proc_x=e(0, R, W), proc_y=e(0, R, W), freqs=e(0, R, self._mb, dt=f32), mags=e(0, R, self._mb, dt=f32),
                          num_bins=e(0, R, dt=i32), lags=e(0, P, 2 * W - 1, dt=f32), corr=e(0, P, 2 * W - 1, dt=f32),
                          num_lags=e(0, P, dt=i32))
        if self.peak_max_samples:
            means = dict(mean_bpm=e(0, R), mean_bpm_int=e(0, R))
            if P:
                means.update(mean_ptt=e(0, P), mean_ptt_int=e(0, P))
        self.launches_per_step = launches
        return StepResult(jobs_per_stream, samples, e(0, R), e(0, R, dt=i32), e(0, R), e(0, P), e(0, P, dt=i32), e(0, P),
                          e(0, R, dt=i32), arrays, means, _job_offsets=np.zeros(self.S + 1, dtype=np.int64),
                          _job_stream=e(0, dt=i32), snr_db=e(0, R) if self.snr else None)

    def _outputs(self, turn: int, J: int):
        """F3 / F4 (and SNR, with snr=True) output dicts of a step: views of the first J rows of result turn `turn`'s
        Jmax-row buffers.  With snr=True F3 stores its spectrum even when the arrays are not stored."""
        if self._out[turn] is None:
            pm = ops.jobs_params(self._params(0, 1, 1), self._Jmax)
            e = lambda C_: torch.empty((self._Jmax, C_), dtype=torch.float64, device=self.device)
            q = {}
            if self.snr:
                q['snr_db'] = e(self.R)
                if self.peak_max_samples:       # the gate only acts on the running means
                    q.update(gated_freq=e(self.R), gated_lag=e(self.P))
            self._out[turn] = (ops._spectrum_out(pm, self.store_arrays or self.snr, None, self.device),
                               ops._xcorr_out(pm, self.store_arrays, None, self.device), q)
        return [{k: None if v is None else v[:J] for k, v in d.items()} for d in self._out[turn]]

    def _step_signals(self, samples, timestamps, S, T, _count_roi, _designed, plan=None) -> StepResult:
        main = torch.cuda.current_stream(self.device)
        turn = self._turn
        self._turn = (turn + 1) % self._nbuf
        has_filter = any(m in (_cabi.FILTER_BUTTER, _cabi.FILTER_FIR) for m in self.methods)
        lock = plan is None or plan['lock']
        roi_launches = 1 + self._extra_launches if _count_roi else 0
        if lock:
            head0, head_step, jobs = self._lock_jobs(T, plan)
            ops.ring_push(self.ring_t, self.ring_y, self._cnt, None if _designed else timestamps.contiguous(), samples.contiguous())
            self._cnt += T
            self._g0_ok = False
            if jobs == 0:                       # a strided step between cadence points: F1 + push
                return self._empty_step(samples, 0, roi_launches + 1)
            p = self._params(head0, head_step, jobs)
            pj, J = p, S * jobs
        else:
            # job-map path: stream s pushes n_s frames and owns jobs job_offsets[s]:job_offsets[s+1]; F3 / F4 see the J jobs
            # as J streams of one job (include/bpv.h)
            if not plan['mapped']:
                self._map_jobs(plan, turn)
            ops.ring_push_ragged(self.ring_t, self.ring_y, self._g0[0], self._ndev, None if _designed else timestamps.contiguous(),
                                 samples.contiguous())
            jobs, J = None, plan['J']
            if J == 0:                          # a strided step between cadence points: F1 + map + push
                self._advance(plan, turn, main)
                return self._empty_step(samples, None, roi_launches + 2)
            p = self._params(0, 1, 1)
            pj = ops.jobs_params(p, J)
            js, jh, sj0 = self._jobmap[turn]
        proc = self._proc[turn % len(self._proc)]
        px, py, st = proc[0, :J], proc[1, :J], self._status[turn][:J]
        if _designed:
            main.wait_event(self._ev['design'])
        elif has_filter and lock:
            ops.window_design(self.ring_t, p, self._ws, self._cache())
        elif has_filter:
            ops.window_design_jobs(self.ring_t, p, self._ws, js, jh, J, self._cache())
        if lock:
            ops.window_filter(self.ring_t, self.ring_y, p, self._ws, px, py, st, cache=self._dcache if has_filter else None)
        else:
            ops.window_filter_jobs(self.ring_t, self.ring_y, p, self._ws, js, jh, J, px, py, st,
                                   cache=self._dcache if has_filter else None)
        spo, xco, qo = self._outputs(turn, J)
        p = pj
        # (windows over 320 samples: the entry point itself runs the two stand-alone launches, on this stream)
        fb, lb = ops.peak_band(self.freq_band, 'freq_band'), ops.peak_band(self.lag_band, 'lag_band')
        fused = (bool(self.overlap & OVERLAP_FUSED) and self.P > 0 and self.transform == _cabi.PGRAM_WELCH
                 and fb is None and lb is None)       # the fused grid has no band: two kernels instead
        store_spec = self.store_arrays or self.snr
        if fused:
            sp, xc = ops.window_welch_xcorr(px, py, p, store=store_spec, out_spectrum=spo, out_xcorr=xco,
                                            store_xcorr=self.store_arrays)
        elif (self.overlap & OVERLAP_XCORR) and self.P:
            # launch order matters for co-residency: the spectrum kernels' CTAs are small (Welch: 24 KB of shared memory),
            # the xcorr CTAs large (51 KB); with xcorr first its 4 CTAs fill an SM's shared memory and the spectrum only
            # gets in as they retire (168 us for the pair against 103 + 75 serial); spectrum first leaves room for two xcorr
            # CTAs beside five Welch CTAs.  BPV_XC_FIRST=1 restores the other order (measurement switch).
            side, ev = self._streams()
            ev['pre'].record(main)
            side.wait_event(ev['pre'])
            xc_first = os.environ.get('BPV_XC_FIRST', '') == '1'
            if not xc_first:
                sp = ops.window_spectrum(px, py, p, store=store_spec, workspace=self._ws_spec, out=spo, band=fb)
            with torch.cuda.stream(side):
                xc = ops.window_xcorr(px, py, p, store=self.store_arrays, out=xco, band=lb)
                ev['xc'].record(side)
            if xc_first:
                sp = ops.window_spectrum(px, py, p, store=store_spec, workspace=self._ws_spec, out=spo, band=fb)
            main.wait_event(ev['xc'])
        else:
            sp = ops.window_spectrum(px, py, p, store=store_spec, workspace=self._ws_spec, out=spo, band=fb)
            xc = ops.window_xcorr(px, py, p, store=self.store_arrays, out=xco, band=lb)
        gate = self.snr and self._min_snr_db is not None and self.peak_max_samples > 0
        if self.snr:
            # after F3 and, on the two-stream schedule, after the xcorr event: the gate reads lag_sec
            band = fb if fb is not None else (self.kw['min_freq'], self.kw['max_freq'])
            qo = ops.window_snr(sp['freqs'], sp['mags'], sp['num_bins'], sp['peak_idx'], self.transform, band, self.snr_half_width,
                                min_snr_db=self._min_snr_db if gate else None, peak_freq=sp['peak_freq'] if gate else None,
                                lag_sec=xc['lag_sec'] if gate else None, out=qo)
        if not self.store_arrays and self.discard_scratch:
            # the processed windows are dead now: drop their dirty L2 lines instead of letting the next step's ROI sampling
            # push them out to DRAM (F1 64.5 -> 69.7 us with 80 MB of dirty scratch in L2, profiles/r2p_f1_dirty.txt)
            if J == self._Jmax:
                ops.scratch_discard(proc)
            else:
                ops.scratch_discard(px, py)
        n_design = sum(1 for m in set(self.methods) if m in (_cabi.FILTER_BUTTER, _cabi.FILTER_FIR))
        n_pre = 1 + n_design + (1 if n_design and self._dcache is not None else 0)     # filter + designs (+ cache probe)
        n_spec = 2 if self.transform == _cabi.PGRAM_LS else 1
        if self.transform == _cabi.DFT_RFFT and 16 <= self.W <= 2048:
            env = os.environ.get('BPV_DFT_TC')
            interp = any(m in (_cabi.INTERP_LINEAR, _cabi.INTERP_CUBIC) for m in self.methods)
            if (env[:1] == '1') if env is not None else interp:
                n_spec = 6              # dft_image + seal + dft_split + dft_tc_tma2 + dft_peak kernels + spectrum_dense_kernel for the flagged windows
        n_push = (2 if _designed else 1) + (0 if lock else 1)          # (+ the job map)
        self.launches_per_step = roi_launches + n_push + n_pre + n_spec + (1 if self.P and not (fused and self.W <= 320) else 0)
        if not self.store_arrays and self.discard_scratch:
            self.launches_per_step += 1 if J == self._Jmax else 2
        self.launches_per_step += 1 if self.snr else 0
        arrays = {}
        if self.store_arrays:
            arrays = dict(proc_x=px, proc_y=py, freqs=sp['freqs'], mags=sp['mags'], num_bins=sp['num_bins'],
                          lags=xc['lags'], corr=xc['corr'], num_lags=xc['num_lags'])
        # the running means push the gated values: a rejected heart rate / PTT enters the history as NaN
        bpm_in = qo['gated_freq'] if gate else sp['peak_freq']
        ptt_in = qo['gated_lag'] if gate else xc['lag_sec']
        snr_db = qo['snr_db'] if self.snr else None
        means = {}
        if self.peak_max_samples and lock:
            mb, mbi = ops.running_mean(self._bpm_ring, self._mcnt, bpm_in.view(S, jobs, self.R), 60.0)
            means = dict(mean_bpm=mb.view(J, self.R), mean_bpm_int=mbi.view(J, self.R))
            if self.P:
                mp, mpi = ops.running_mean(self._ptt_ring, self._mcnt, ptt_in.view(S, jobs, self.P), 1000.0)
                means.update(mean_ptt=mp.view(J, self.P), mean_ptt_int=mpi.view(J, self.P))
            self._mcnt += jobs
            self.launches_per_step += 2 if self.P else 1
        elif self.peak_max_samples:
            mcnt = np.full(self.S, self._mcnt, dtype=np.int64) if isinstance(self._mcnt, int) else self._mcnt
            pin = self._pinned(turn)
            pin['m0'].numpy()[:] = mcnt
            self._mg0.copy_(pin['m0'], non_blocking=True)
            mb, mbi = ops.running_mean_jobs(self._bpm_ring, self._mg0, sj0, bpm_in, 60.0)
            means = dict(mean_bpm=mb, mean_bpm_int=mbi)
            if self.P:
                mp, mpi = ops.running_mean_jobs(self._ptt_ring, self._mg0, sj0, ptt_in, 1000.0)
                means.update(mean_ptt=mp, mean_ptt_int=mpi)
            self._mcnt = self._level(mcnt + plan['jobs'])
            self.launches_per_step += 2 if self.P else 1
        if lock:
            return StepResult(jobs, samples, sp['peak_freq'], sp['peak_idx'], sp['peak_mag'], xc['lag_sec'], xc['lag_idx'],
                              xc['lag_corr'], st, arrays, means, snr_db=snr_db)
        self._advance(plan, turn, main)
        return StepResult(None, samples, sp['peak_freq'], sp['peak_idx'], sp['peak_mag'], xc['lag_sec'], xc['lag_idx'],
                          xc['lag_corr'], st, arrays, means, _job_offsets=plan['off'], _job_stream=js[:J], snr_db=snr_db)

    def _advance(self, plan: dict, turn: int, main) -> None:
        """End of a job-map step on the host: the staging of `turn` is in flight until the device passes this point, and
        the counts advance by the frames taken."""
        self._staging[turn]['ev'].record(main)
        self._staging[turn]['used'] = True
        self._cnt = self._level(self.counts + plan['n'])
        self._g0.reverse()                      # bpv_stream_jobs left the advanced counts in the other buffer

    # ------------------------------------------------------------------------------------------
    # SURVEY.md §8(f) row 3: snapshot / resume of the per-stream state (the reference's deepcopy(store), :313, is the
    # only "checkpoint" it has; long-running batched streams need the device rings and histories)
    def _signature(self) -> dict:
        return dict(S=self.S, R=self.R, W=self.W, cap=self.cap, peak_max_samples=self.peak_max_samples,
                    roi_max_samples=0 if self._roi_hist is None else int(self._roi_hist.shape[2]))

    def state_dict(self) -> dict:
        """Everything a run needs to continue bit-for-bit: raw-sample rings and their per-stream counts, the bpm / ptt
        histories of the running means and their per-stream lengths, the ROI smoothing history.  Tensors and counts are
        copied to the host."""
        torch.cuda.synchronize(self.device)
        cpu = lambda t: None if t is None else t.detach().to('cpu', copy=True)
        mcnt = np.full(self.S, self._mcnt, dtype=np.int64) if isinstance(self._mcnt, int) else self._mcnt.copy()
        return dict(version=STATE_VERSION, signature=self._signature(), counts=self.counts,
                    ring_t=cpu(self.ring_t), ring_y=cpu(self.ring_y),
                    mean_counts=mcnt, bpm_ring=cpu(self._bpm_ring), ptt_ring=cpu(self._ptt_ring),
                    roi_count=int(self._roi_count), roi_hist=cpu(self._roi_hist))

    def load_state_dict(self, state: dict) -> None:
        """Load a state_dict() of an engine of the same geometry; version 1 states (one count for every stream) load too."""
        version = state.get('version')
        if version not in (1, STATE_VERSION):
            raise ValueError(f"load_state_dict: unsupported state version {version!r}")
        if version == 1:
            counts, mcnt = np.full(self.S, int(state['count']), np.int64), np.full(self.S, int(state['mean_count']), np.int64)
        else:
            counts, mcnt = np.asarray(state['counts'], dtype=np.int64), np.asarray(state['mean_counts'], dtype=np.int64)
            if counts.shape != (self.S,) or mcnt.shape != (self.S,):
                raise ValueError(f'load_state_dict: counts of {counts.shape} / {mcnt.shape} streams, expected ({self.S},)')
        if state['signature'] != self._signature():
            raise ValueError(f"load_state_dict: state of a different engine geometry {state['signature']} != {self._signature()}")

        def put(dst, src, name):
            if (dst is None) != (src is None):
                raise ValueError(f'load_state_dict: {name} present on one side only')
            if dst is not None:
                if tuple(dst.shape) != tuple(src.shape) or dst.dtype != src.dtype:
                    raise ValueError(f'load_state_dict: {name} has shape {tuple(src.shape)}, expected {tuple(dst.shape)}')
                dst.copy_(src)
        put(self.ring_t, state['ring_t'], 'ring_t')
        put(self.ring_y, state['ring_y'], 'ring_y')
        put(self._bpm_ring, state['bpm_ring'], 'bpm_ring')
        put(self._ptt_ring, state['ptt_ring'], 'ptt_ring')
        put(self._roi_hist, state['roi_hist'], 'roi_hist')
        self._cnt, self._mcnt, self._roi_count = self._level(counts), self._level(mcnt), int(state['roi_count'])
        self._g0_ok = False

    def reset(self, streams=None):
        """Back to the state of a freshly constructed engine: empty rings AND empty bpm / ptt / ROI histories.
        streams = indices of some streams (e.g. cameras that disconnected): only their ring rows, bpm / ptt history rows and
        ROI smoothing rows are emptied and their counts zeroed; every other stream keeps its state bit for bit."""
        nan = float('nan')
        if streams is None:
            self.ring_t.fill_(nan)
            self.ring_y.fill_(nan)
            self.count = 0
            for t in (self._bpm_ring, self._ptt_ring, self._roi_hist):
                if t is not None:
                    t.fill_(nan)
            self._mcnt = self._roi_count = 0
            return
        idx = np.unique(np.asarray(streams, dtype=np.int64).reshape(-1))
        if idx.size and (idx[0] < 0 or idx[-1] >= self.S):
            raise ValueError(f'reset: stream indices must lie in [0, {self.S})')
        if not idx.size:
            return
        rows = torch.from_numpy(idx).to(self.device)
        for t in (self.ring_t, self.ring_y, self._bpm_ring, self._ptt_ring, self._roi_hist):
            if t is not None:
                t.index_fill_(0, rows, nan)
        counts = self.counts
        counts[idx] = 0
        self._cnt = self._level(counts)
        mcnt = np.full(self.S, self._mcnt, dtype=np.int64) if isinstance(self._mcnt, int) else self._mcnt.copy()
        mcnt[idx] = 0
        self._mcnt = self._level(mcnt)
        self._g0_ok = False
