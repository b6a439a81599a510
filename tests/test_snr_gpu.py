"""GPU: per-window spectral SNR of the heart-rate peak and the SNR-gated running means (include/bpv.h bpv_window_snr,
BatchedSignalProcessor(snr=True, snr_half_width=..., min_snr_db=...)).

The kernel is held to tests/snr_oracle.py on the spectra the engine itself stored (the definition reads only those arrays,
so membership of every bin is decided identically and only the summation order and log10 differ), and to scipy's
float64 spectra of the same processed windows.  An engine with snr=True must leave every other output bit for bit as an
engine without it, and the gated running means must equal np.nanmean over a host-gated history.
"""
import math
import warnings

import numpy as np
import pytest
import torch

from oracle import bpv_oracle as orc
from tests import helpers as h
from tests import snr_oracle as so

pytestmark = pytest.mark.gpu

FIELDS = ('peak_freq', 'peak_idx', 'peak_mag', 'lag_sec', 'lag_idx', 'lag_corr', 'status')
C2 = dict(processing_methods=[orc.DETREND_LINEAR, orc.FILTER_FIR], spectrum_transform=orc.PGRAM_WELCH)
C4 = dict(processing_methods=[orc.INTERP_CUBIC, orc.FILTER_BUTTER], spectrum_transform=orc.PGRAM_LS)


def workload(S, R, n, seed, fps=30.0, ac=None, p_nan=0.02):
    """Timestamps [S, n] and samples [S, R, n] of S synthetic streams (bpv.synth)."""
    from bpv import synth
    rng = np.random.default_rng(seed)
    ts = np.stack([synth.timestamps(rng, n, fps, irregular=True, drop=0.03, origin=rng.uniform(0, 100)) for _ in range(S)])
    ys = np.stack([synth.raw_signals(rng, ts[s], R=R, p_nan=p_nan, **({} if ac is None else dict(ac=ac[s])))
                   for s in range(S)])
    return ts, ys


def feed(eng, ts, ys, g0, T, frame_counts=None):
    """One step_signals of frames g0 .. g0+T-1 of every stream."""
    y = torch.from_numpy(np.ascontiguousarray(ys[:, :, g0:g0 + T].transpose(0, 2, 1))).cuda()
    return eng.step_signals(y, torch.from_numpy(np.ascontiguousarray(ts[:, g0:g0 + T])).cuda(), frame_counts=frame_counts)


def host(res):
    """Copies of a result's fields, arrays, means and snr_db (results are views of rotating buffers)."""
    cp = lambda t: None if t is None else t.cpu().numpy().copy()
    return dict({k: cp(getattr(res, k)) for k in FIELDS}, arrays={k: cp(v) for k, v in res.arrays.items()},
                means={k: cp(v) for k, v in res.means.items()}, snr_db=cp(res.snr_db), off=res.job_offsets.copy())


def same_nan(a, b):
    """Equal with NaN == NaN and the same signs of infinity."""
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return a.shape == b.shape and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


def check_snr(got, want, tol=1e-9):
    """snr_db within tol dB, with NaN and +-inf in the same places."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape
    fin = np.isfinite(want)
    assert np.array_equal(np.isnan(got), np.isnan(want)), np.argwhere(np.isnan(got) != np.isnan(want))[:5]
    assert np.array_equal(got[np.isinf(want)], want[np.isinf(want)]) and np.array_equal(np.isinf(got), np.isinf(want))
    if fin.any():
        err = np.abs(got[fin] - want[fin])
        assert err.max() <= tol, (err.max(), np.argmax(err))
    return int(fin.sum())


# ------------------------------------------------------------------------------------------------
# 1. the kernel against the oracle, on the engine's own stored spectra
# ------------------------------------------------------------------------------------------------
PATHS = [   # (engine kwargs, W, fps, BPV_DFT_TC)
    (C2, 64, 30.0, None),                                                                           # Welch warm-up (n < 256)
    (C2, 300, 30.0, None),                                                                          # c2: Welch, n < 256 and 256
    (dict(processing_methods=[orc.DIFF_1], spectrum_transform=orc.DFT_RFFT), 300, 30.0, '0'),       # float64 DFT
    (dict(processing_methods=[orc.INTERP_CUBIC, orc.FILTER_BUTTER], spectrum_transform=orc.DFT_RFFT), 250, 30.0, None),  # TC DFT
    (dict(processing_methods=[orc.FILTER_BUTTER], spectrum_transform=orc.PGRAM_LS, min_freq=0.7), 250, 30.0, None),      # LS F = n
    (dict(processing_methods=[orc.DETREND_CONST], spectrum_transform=orc.PGRAM_LS, ls_num_freqs=2048), 300, 30.0, None),  # fixed grid
    (C4, 1200, 120.0, None),                                                                        # c4 chain
]


@pytest.mark.parametrize('R', [1, 2, 4])
@pytest.mark.parametrize('kw,W,fps,tc', PATHS, ids=lambda v: str(v).replace(' ', ''))
def test_kernel_matches_oracle_on_stored_spectra(kw, W, fps, tc, R, monkeypatch):
    from bpv import ops
    if tc is not None:
        monkeypatch.setenv('BPV_DFT_TC', tc)
    if R == 4 and W >= 1200:
        pytest.skip('R = 4 is covered at the shorter windows')
    S, T = (2, 100) if W >= 1200 else (3, max(4, W // 6))
    steps = W // T + 2
    ts, ys = workload(S, R, T * steps, W + R, fps=fps)
    band_cfg = (kw.get('min_freq', 0.8), kw.get('max_freq', 4.0))
    from bpv.engine import BatchedSignalProcessor
    eng = BatchedSignalProcessor(S, R, signal_max_samples=W, max_frames_per_step=T, store_arrays=True, snr=True, **kw)
    transform = eng.transform
    checked = 0
    for i in range(steps):
        res = feed(eng, ts, ys, i * T, T)
        if i not in (0, steps // 2, steps - 1):
            continue
        a = res.arrays
        f, m, nb, pk = (a['freqs'].cpu().numpy(), a['mags'].cpu().numpy(), a['num_bins'].cpu().numpy(), res.peak_idx.cpu().numpy())
        # the engine's own result: the configured band, the default half width
        checked += check_snr(res.snr_db.cpu().numpy(), so.snr_all(f, m, nb, pk, transform, *band_cfg, 0.125))
        # the entry point over other bands and half widths, on the same stored arrays
        for band in [(-math.inf, math.inf), (0.7, 3.0), (1.0, 1.05), (4.0, 0.8)]:
            for hw in (0.0, 0.05, 0.125, 0.4):
                o = ops.window_snr(a['freqs'], a['mags'], a['num_bins'], res.peak_idx, transform, band, hw)
                checked += check_snr(o['snr_db'].cpu().numpy(), so.snr_all(f, m, nb, pk, transform, *band, hw))
    assert checked > 0


def test_gated_outputs_are_exact():
    from bpv import ops
    from bpv.engine import BatchedSignalProcessor
    S, R, T, W = 6, 3, 50, 300
    ts, ys = workload(S, R, 400, 11, ac=[0.5, 0.0, 0.05, 0.5, 0.0, 0.2])
    eng = BatchedSignalProcessor(S, R, signal_max_samples=W, max_frames_per_step=T, store_arrays=True, snr=True, **C2)
    for i in range(8):
        res = feed(eng, ts, ys, i * T, T)
    a = res.arrays
    snr = res.snr_db.cpu().numpy()
    for thr in (-math.inf, 0.0, 3.0, float(np.nanmedian(snr[np.isfinite(snr)])), math.inf):
        o = ops.window_snr(a['freqs'], a['mags'], a['num_bins'], res.peak_idx, eng.transform, (0.8, 4.0), 0.125, min_snr_db=thr,
                           peak_freq=res.peak_freq, lag_sec=res.lag_sec)
        assert same_nan(o['snr_db'].cpu().numpy(), snr)
        gf, gl = so.gate(snr, res.peak_freq.cpu().numpy(), res.lag_sec.cpu().numpy(), thr)
        assert same_nan(o['gated_freq'].cpu().numpy(), gf) and same_nan(o['gated_lag'].cpu().numpy(), gl), thr


def test_many_rois_loop_over_the_warps():
    """R = 11 (more ROIs than warps of a CTA; 55 pairs): the kernel against the oracle and the gate."""
    from bpv import ops
    J, R, mb = 37, 11, 129
    rng = np.random.default_rng(3)
    f = np.tile((np.arange(mb) * 0.1171875).astype(np.float32), (J, R, 1))
    m = rng.exponential(1.0, (J, R, mb)).astype(np.float32)
    m[rng.uniform(size=m.shape) < 0.02] = np.nan
    nb = rng.integers(0, mb + 1, (J, R)).astype(np.int32)
    pk = np.where(nb > 0, rng.integers(0, mb, (J, R)) % np.maximum(nb, 1), -1).astype(np.int32)
    pk[0, :3] = -1
    pf = rng.uniform(0.5, 3.0, (J, R))
    ls = rng.uniform(-0.5, 0.5, (J, R * (R - 1) // 2))
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).cuda()
    o = ops.window_snr(d(f), d(m), d(nb), d(pk), so.PGRAM_WELCH, (0.8, 4.0), 0.125, min_snr_db=-1.0, peak_freq=d(pf), lag_sec=d(ls))
    want = so.snr_all(f, m, nb, pk, so.PGRAM_WELCH, 0.8, 4.0, 0.125)
    check_snr(o['snr_db'].cpu().numpy(), want)
    gf, gl = so.gate(want, pf, ls, -1.0)
    assert same_nan(o['gated_freq'].cpu().numpy(), gf) and same_nan(o['gated_lag'].cpu().numpy(), gl)


# ------------------------------------------------------------------------------------------------
# 2. against scipy's float64 spectra of the same processed windows
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('chain', ['c2', 'c4'])
def test_snr_matches_scipy_spectra(chain):
    from bpv.engine import BatchedSignalProcessor
    kw, W, fps, T = (C2, 300, 30.0, 50) if chain == 'c2' else (C4, 1200, 120.0, 100)
    S, R = 3, 2
    steps = W // T + 1
    ts, ys = workload(S, R, T * steps, 21, fps=fps)
    eng = BatchedSignalProcessor(S, R, signal_max_samples=W, max_frames_per_step=T, store_arrays=True, snr=True, **kw)
    for i in range(steps):
        res = feed(eng, ts, ys, i * T, T)
    a = {k: v.cpu().numpy() for k, v in res.arrays.items()}
    snr, pk = res.snr_db.cpu().numpy(), res.peak_idx.cpu().numpy()
    rows = np.arange(0, snr.shape[0], 7 if chain == 'c2' else 19)
    n = 0
    for j in rows:
        for r in range(R):
            ef, em = orc.spectrum(a['proc_x'][j, r], a['proc_y'][j, r], eng.transform)
            nb = int(a['num_bins'][j, r])
            assert len(em) == nb
            # membership from the engine's stored frequencies, powers from scipy's float64 spectrum
            f32 = a['freqs'][j, r, :nb]
            want = so.snr_db(f32, em, nb, pk[j, r], eng.transform, 0.8, 4.0, 0.125, exact_mags=True)
            if np.isfinite(want):
                assert abs(snr[j, r] - want) <= 1e-3, (j, r, snr[j, r], want)
                n += 1
            else:
                assert same_nan(snr[j, r], want)
    assert n >= len(rows)


# ------------------------------------------------------------------------------------------------
# 3. nothing else moves
# ------------------------------------------------------------------------------------------------
def _pair(kw, S, R, T, W, steps, seed, counts=None, **engkw):
    """Run an snr=False and an snr=True engine on the same inputs; every other output must be equal bit for bit."""
    from bpv.engine import BatchedSignalProcessor
    ts, ys = workload(S, R, T * steps, seed)
    engs = [BatchedSignalProcessor(S, R, signal_max_samples=W, max_frames_per_step=T, snr=q, peak_max_samples=9, **kw, **engkw)
            for q in (False, True)]
    g = np.zeros(S, dtype=np.int64)
    cnt = 0
    for i in range(steps):
        n = None if counts is None else counts[i]
        outs = []
        for e in engs:
            if n is None:
                outs.append((host(feed(e, ts, ys, i * T, T)), e.launches_per_step))
            else:       # stream s takes its next n[s] frames
                idx = g[:, None] + np.arange(T)[None, :]
                tt = np.take_along_axis(ts, np.minimum(idx, ts.shape[1] - 1), axis=1)
                yy = np.take_along_axis(ys, np.minimum(idx, ts.shape[1] - 1)[:, None, :].repeat(R, 1), axis=2)
                outs.append((host(feed(e, tt, yy, 0, T, frame_counts=n)), e.launches_per_step))
        if n is not None:
            g += n
        (a, la), (b, lb) = outs
        assert a['snr_db'] is None and b['snr_db'] is not None and b['snr_db'].shape == a['peak_freq'].shape
        for k in FIELDS:
            assert same_nan(a[k], b[k]), (i, k)
        assert np.array_equal(a['off'], b['off'])
        assert a['arrays'].keys() == b['arrays'].keys()
        for k in a['arrays']:
            assert same_nan(a['arrays'][k], b['arrays'][k]), (i, k)
        for k in a['means']:
            assert same_nan(a['means'][k], b['means'][k]), (i, k)
        assert lb == la + (1 if a['peak_freq'].shape[0] else 0), (i, la, lb)
        cnt += a['peak_freq'].shape[0]
    assert cnt > 0
    return engs


@pytest.mark.parametrize('overlap', [0, 3, 5])
@pytest.mark.parametrize('store', [False, True])
def test_snr_moves_nothing_else_lockstep(overlap, store):
    _pair(C2, 4, 2, 16, 64, 8, 5, overlap=overlap, store_arrays=store)


@pytest.mark.parametrize('overlap', [0, 3, 5])
def test_snr_moves_nothing_else_ragged(overlap):
    rng = np.random.default_rng(8)
    counts = [rng.integers(0, 17, 5) for _ in range(10)]
    counts[3][:] = 0
    _pair(C2, 5, 2, 16, 64, 10, 6, counts=counts, overlap=overlap)


@pytest.mark.parametrize('kw', [C4, dict(processing_methods=[orc.INTERP_CUBIC, orc.FILTER_BUTTER], spectrum_transform=orc.DFT_RFFT)],
                         ids=['c4', 'dft_tc'])
def test_snr_moves_nothing_else_other_transforms(kw):
    _pair(kw, 3, 2, 16, 96, 8, 7)
    _pair(kw, 3, 2, 16, 96, 8, 7, design_cache=False)


def test_snr_moves_nothing_else_strided():
    _pair(C2, 4, 2, 8, 64, 12, 9, window_stride=[3, 5, 1, 9], window_phase=[0, 2, 0, 4])
    _pair(C2, 4, 2, 8, 64, 12, 9, window_stride=12, window_phase=5)          # uniform: lockstep with head_step, zero-job steps


# ------------------------------------------------------------------------------------------------
# 4. it separates pulse from noise
# ------------------------------------------------------------------------------------------------
def test_pulse_streams_above_noise_streams():
    """16 streams with a pulse (ac 0.5) against 16 of drift and noise only (ac 0), c2 chain, every full window: the lowest
    pulse SNR lies above the highest noise SNR.  Found with this seed: pulse min 2.04 dB, noise max 1.29 dB, a margin of
    0.76 dB (the 0.125 Hz template keeps the peak bin and its neighbours; the rest of the Hann main lobe counts as noise)."""
    from bpv.engine import BatchedSignalProcessor
    S, R, W, T = 32, 2, 300, 60
    ac = [0.5] * 16 + [0.0] * 16
    ts, ys = workload(S, R, 600, 123, ac=ac, p_nan=0.0)
    eng = BatchedSignalProcessor(S, R, signal_max_samples=W, max_frames_per_step=T, snr=True, freq_band=(0.8, 4.0), **C2)
    snr = []
    for i in range(10):
        res = feed(eng, ts, ys, i * T, T)
        if (i + 1) * T >= W:                      # full windows only
            snr.append(res.snr_db.cpu().numpy().reshape(S, T, R))
    snr = np.concatenate(snr, axis=1)             # [S, jobs, R]
    pulse, noise = snr[:16], snr[16:]
    assert np.isfinite(pulse).all()
    lo_pulse, hi_noise = pulse.min(), np.nanmax(np.where(np.isnan(noise), -np.inf, noise))
    print(f'\nfull-window SNR: pulse streams min {lo_pulse:.2f} dB, noise streams max {hi_noise:.2f} dB, '
          f'margin {lo_pulse - hi_noise:.2f} dB')
    assert lo_pulse > hi_noise


# ------------------------------------------------------------------------------------------------
# 5. gating of the running means
# ------------------------------------------------------------------------------------------------
def _nanmean_last(hist, H):
    with np.errstate(all='ignore'), warnings.catch_warnings():
        warnings.simplefilter('ignore')
        return np.nanmean(np.asarray(hist[-H:]), axis=0)


def _gated_run(eng, ts, ys, T, steps, thresholds, counts=None, hist=None, start=0, g=None):
    """Steps start .. steps-1 with threshold thresholds[i]; checks every job's running means against a host history of
    gated values.  Returns the histories and per-stream offsets for a continuation."""
    S, R = ys.shape[:2]
    H = eng.peak_max_samples
    hist = hist if hist is not None else ([[] for _ in range(S)], [[] for _ in range(S)])
    g = np.zeros(S, dtype=np.int64) if g is None else g
    for i in range(start, steps):
        eng.min_snr_db = thresholds[i]
        if counts is None:
            res = feed(eng, ts, ys, i * T, T)
            n = np.full(S, T)
        else:
            n = counts[i]
            idx = np.minimum(g[:, None] + np.arange(T)[None, :], ts.shape[1] - 1)
            tt = np.take_along_axis(ts, idx, axis=1)
            yy = np.take_along_axis(ys, idx[:, None, :].repeat(R, 1), axis=2)
            res = feed(eng, tt, yy, 0, T, frame_counts=n)
        g += n
        r = host(res)
        if not r['peak_freq'].shape[0]:
            continue
        thr = -math.inf if thresholds[i] is None else thresholds[i]
        gf, gl = so.gate(r['snr_db'], r['peak_freq'], r['lag_sec'], thr) if thresholds[i] is not None else (r['peak_freq'], r['lag_sec'])
        off = r['off']
        for s in range(S):
            for j in range(off[s], off[s + 1]):
                hist[0][s].append(gf[j] * 60)
                hist[1][s].append(gl[j] * 1000)
                assert h.close(r['means']['mean_bpm'][j], _nanmean_last(hist[0][s], H), rtol=1e-12, atol_frac=0), (i, s, j)
                assert h.close(r['means']['mean_ptt'][j], _nanmean_last(hist[1][s], H), rtol=1e-12, atol_frac=0), (i, s, j)
    return hist, g


def _gate_engine(S, R, W, T, **kw):
    from bpv.engine import BatchedSignalProcessor
    return BatchedSignalProcessor(S, R, signal_max_samples=W, max_frames_per_step=T, snr=True, peak_max_samples=10,
                                  freq_band=(0.8, 4.0), **C2, **kw)


def _thresholds(steps):
    return [[3.0, 3.0, 0.0, None, 6.0, -math.inf, 3.0, 10.0, 3.0, 1.0, 3.0, 3.0][i % 12] for i in range(steps)]


def test_gated_running_means_lockstep():
    S, R, W, T, steps = 6, 3, 64, 12, 12
    ts, ys = workload(S, R, T * steps, 31, ac=[0.5, 0.0, 0.1, 0.5, 0.02, 0.3])
    _gated_run(_gate_engine(S, R, W, T), ts, ys, T, steps, _thresholds(steps))


def test_gated_running_means_ragged_and_strided():
    S, R, W, T, steps = 5, 2, 64, 12, 14
    ts, ys = workload(S, R, T * steps, 32, ac=[0.5, 0.0, 0.1, 0.5, 0.02])
    rng = np.random.default_rng(4)
    counts = [rng.integers(0, T + 1, S) for _ in range(steps)]
    _gated_run(_gate_engine(S, R, W, T), ts, ys, T, steps, _thresholds(steps), counts=counts)
    _gated_run(_gate_engine(S, R, W, T, window_stride=[1, 2, 3, 5, 7], window_phase=[0, 1, 2, 0, 6]), ts, ys, T, steps,
               _thresholds(steps))
    _gated_run(_gate_engine(S, R, W, T, window_stride=[2, 2, 3, 5, 13], window_phase=[0, 1, 2, 0, 6]), ts, ys, T, steps,
               _thresholds(steps), counts=counts)


def test_no_threshold_is_the_engine_without_snr():
    from bpv.engine import BatchedSignalProcessor
    S, R, W, T, steps = 4, 2, 64, 12, 8
    ts, ys = workload(S, R, T * steps, 33)
    engs = [BatchedSignalProcessor(S, R, signal_max_samples=W, max_frames_per_step=T, peak_max_samples=10, **C2, **q)
            for q in (dict(), dict(snr=True, min_snr_db=None))]
    for i in range(steps):
        a, b = (host(feed(e, ts, ys, i * T, T)) for e in engs)
        for k in a['means']:
            assert same_nan(a['means'][k], b['means'][k])


def test_gated_resume_equals_the_uninterrupted_run():
    import pickle
    S, R, W, T, steps = 4, 2, 64, 12, 12
    ts, ys = workload(S, R, T * steps, 34, ac=[0.5, 0.0, 0.1, 0.5])
    thr = _thresholds(steps)
    full = _gate_engine(S, R, W, T)
    first = _gate_engine(S, R, W, T)
    hist, g = _gated_run(first, ts, ys, T, 6, thr)
    state = pickle.loads(pickle.dumps(first.state_dict()))
    resumed = _gate_engine(S, R, W, T, min_snr_db=3.0)
    resumed.load_state_dict(state)
    _gated_run(resumed, ts, ys, T, steps, thr, hist=hist, start=6, g=g)       # continues the host history
    # bit for bit: every step of a second resumed engine equals the uninterrupted run's
    again = _gate_engine(S, R, W, T)
    again.load_state_dict(state)
    for i in range(steps):
        full.min_snr_db = thr[i]
        a = host(feed(full, ts, ys, i * T, T))
        if i >= 6:
            again.min_snr_db = thr[i]
            b = host(feed(again, ts, ys, i * T, T))
            for k in a['means']:
                assert same_nan(a['means'][k], b['means'][k]), (i, k)
            assert same_nan(a['snr_db'], b['snr_db']) and same_nan(a['peak_freq'], b['peak_freq'])


# ------------------------------------------------------------------------------------------------
# 6. zero-job steps, launch counts, arguments
# ------------------------------------------------------------------------------------------------
def test_zero_job_steps_and_launch_counts():
    from bpv.engine import BatchedSignalProcessor
    S, R, W, T = 4, 2, 64, 8
    ts, ys = workload(S, R, 64, 35)
    mk = lambda **kw: [BatchedSignalProcessor(S, R, signal_max_samples=W, max_frames_per_step=T, snr=q, **C2, **kw)
                       for q in (False, True)]
    # lockstep, job map (ragged), fused overlap: one more launch
    for kw, n in [(dict(), None), (dict(), [8, 3, 0, 5]), (dict(overlap=5), None), (dict(overlap=0, peak_max_samples=4), None)]:
        a, b = mk(**kw)
        ra, rb = feed(a, ts, ys, 0, T, frame_counts=n), feed(b, ts, ys, 0, T, frame_counts=n)
        assert rb.snr_db.shape == (ra.peak_freq.shape[0], R) and ra.snr_db is None
        assert b.launches_per_step == a.launches_per_step + 1, kw
    # a step in which no stream takes a frame, and a strided step between cadence points: zero rows, no SNR launch
    for kw, n in [(dict(), [0, 0, 0, 0]), (dict(window_stride=20), None), (dict(window_stride=[20, 20, 30, 40]), None)]:
        a, b = mk(**kw)
        ra, rb = feed(a, ts, ys, 0, T, frame_counts=n), feed(b, ts, ys, 0, T, frame_counts=n)
        assert rb.snr_db.shape == (0, R) and rb.snr_db.dtype == torch.float64 and ra.snr_db is None
        assert b.launches_per_step == a.launches_per_step, kw


def test_engine_arguments():
    from bpv.engine import BatchedSignalProcessor
    mk = lambda **kw: BatchedSignalProcessor(2, 2, signal_max_samples=16, **kw)
    for bad in [dict(min_snr_db=3.0), dict(snr=True, min_snr_db=math.nan), dict(snr=True, snr_half_width=-0.1),
                dict(snr=True, snr_half_width=math.inf), dict(snr=True, min_snr_db='x')]:
        with pytest.raises(ValueError):
            mk(**bad)
    eng = mk()
    with pytest.raises(ValueError):
        eng.min_snr_db = 3.0                       # snr=False
    eng.min_snr_db = None
    eng = mk(snr=True, min_snr_db=-math.inf)
    eng.min_snr_db = 3
    assert eng.min_snr_db == 3.0
    with pytest.raises(ValueError):
        eng.min_snr_db = math.nan
    eng.snr_half_width = -1.0
    ts, ys = workload(2, 2, 4, 1)
    with pytest.raises(ValueError):
        feed(eng, ts, ys, 0, 1)
    assert eng.count == 0                          # rejected before anything was enqueued
    eng.snr_half_width = 0.2
    assert feed(eng, ts, ys, 0, 1).snr_db.shape == (2, 2)
