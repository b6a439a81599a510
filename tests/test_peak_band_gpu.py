"""GPU: band-limited heart-rate and PTT peak search (include/bpv.h bpv_window_spectrum_band / bpv_window_xcorr_band,
BatchedSignalProcessor(freq_band=..., lag_band=...)).

Each kernel that writes a peak is fed the oracle's processed windows and held to bo.peak_in_band applied to the oracle's
spectrum / correlation of the same window, with the x values the kernel reports (the contract: a bin or lag is eligible
iff lo <= x_k <= hi for the float64 x_k the kernel computes).  Peak / lag indices are bit-exact from MIN_N valid samples
on; values are held to the bars of tests/test_window_gpu.py.
"""
import itertools
import math
import warnings

import numpy as np
import pytest
import torch

from oracle import bpv_oracle as orc
from tests import band_oracle as bo
from tests import helpers as h
from tests.test_window_gpu import make_windows, oracle_proc, params

pytestmark = pytest.mark.gpu
MIN_N = 4
WIDE = (-1e300, 1e300)          # finite, so the band kernels run, yet every bin / lag is inside


def kernel_x(px, py, transform, kw):
    """The float64 frequency the spectrum kernels report for every bin of one processed window (k * fval from
    fs = (m - 1) / (x_last - x_first) over the finite x; np.linspace's value for Lomb-Scargle)."""
    p = orc._params(kw)
    n = int(np.isfinite(py).sum())
    xf = px[np.isfinite(px)]
    if n < 2 or xf.size < 2:
        return np.zeros(0)
    fs = 1.0 / ((xf[-1] - xf[0]) / float(xf.size - 1))
    if not np.isfinite(fs):
        return np.zeros(0)
    if transform == orc.PGRAM_LS:
        F = int(p['ls_num_freqs'] or n)
        if F == 1:
            return np.array([p['min_freq']])
        step = (p['max_freq'] - p['min_freq']) / float(F - 1)
        x = np.arange(F, dtype=float) * step + p['min_freq']
        x[-1] = p['max_freq']
        return x
    N = n if transform == orc.DFT_RFFT else min(n, 256)
    return np.arange(N // 2 + 1, dtype=float) * (1.0 / (N * (1.0 / fs)))


def oracle_spectra(px, py, transform, kw):
    """{(s, r): (kernel x, oracle magnitudes)} of every window."""
    out = {}
    for s, r in np.ndindex(*px.shape[:2]):
        ef, em = orc.spectrum(px[s, r], py[s, r], transform, **kw)
        xk = kernel_x(px[s, r], py[s, r], transform, kw)
        assert len(xk) == len(ef)
        out[s, r] = xk, em
    return out


def check_spectrum(o, px, py, spectra, band):
    pi, pf, pm = (o[k].cpu().numpy() for k in ('peak_idx', 'peak_freq', 'peak_mag'))
    S, R = pi.shape
    for s in range(S):
        for r in range(R):
            xk, em = spectra[s, r]
            if int(np.isfinite(py[s, r]).sum()) < MIN_N:
                continue
            ex, ey, ei = bo.peak_in_band(xk, em, *band)
            assert pi[s, r] == ei, (s, r, band, pi[s, r], ei)
            if ei >= 0:
                assert pf[s, r] == xk[ei] and band[0] <= pf[s, r] <= band[1]
                np.testing.assert_allclose(pm[s, r], ey, rtol=1e-7, atol=1e-9 * max(1.0, abs(ey)))
            else:
                assert np.isnan(pf[s, r]) and np.isnan(pm[s, r])


def spectrum_bands(px, py, transform, kw):
    """The reference's configured range, others, and bands cut from signal (0, 0)'s own bins: edges exactly on k * fval,
    exactly one bin (-> no peak), an empty and an inverted band."""
    x0 = kernel_x(px[0, 0], py[0, 0], transform, kw)
    assert len(x0) >= 9
    return [(0.8, 4.0), (0.3, 2.0), (x0[2], x0[len(x0) // 2]), (x0[3], x0[3]), (x0[3] + 1e-9, x0[4] - 1e-9), (4.0, 0.8), (-math.inf, 1.5)]


SPEC_PATHS = [   # (transform, methods, kw, W, fps, BPV_DFT_TC): every kernel that writes peak_idx
    (orc.PGRAM_WELCH, [orc.DETREND_LINEAR, orc.FILTER_FIR], {}, 64, 30.0, None),       # welch_warp: direct-DFT warm-up branch
    (orc.PGRAM_WELCH, [orc.DETREND_LINEAR, orc.FILTER_FIR], {}, 300, 30.0, None),      # welch_warp: FFT + direct branches
    (orc.PGRAM_WELCH, [], {}, 600, 120.0, None),                                        # spectrum_dense_kernel (W > 512)
    (orc.DFT_RFFT, [orc.DIFF_1], {}, 300, 30.0, '0'),                                   # float64 DFT
    (orc.DFT_RFFT, [orc.INTERP_CUBIC, orc.FILTER_BUTTER], {}, 300, 30.0, None),         # dft_tc + dft_peak_kernel (+ flagged)
    (orc.DFT_RFFT, [], {}, 64, 30.0, '1'),                                              # forced TC, holed windows flagged
    (orc.PGRAM_LS, [orc.FILTER_BUTTER], dict(min_freq=0.7), 64, 30.0, None),            # ls_peak_warp_kernel
    (orc.PGRAM_LS, [orc.INTERP_CUBIC, orc.FILTER_BUTTER], {}, 300, 30.0, None),
    (orc.PGRAM_LS, [orc.DETREND_CONST], dict(ls_num_freqs=512), 300, 30.0, None),       # fixed grid
    (orc.PGRAM_LS, [], {}, 3300, 120.0, None),                                          # ls_peak_kernel (CTA per signal)
]


@pytest.mark.parametrize('transform,methods,kw,W,fps,tc', SPEC_PATHS, ids=lambda v: str(v).replace(' ', ''))
def test_band_spectrum_matches_oracle(transform, methods, kw, W, fps, tc, monkeypatch):
    from bpv import ops
    if tc is not None:
        monkeypatch.setenv('BPV_DFT_TC', tc)
    S, R = (3, 2) if W > 1000 else (12, 2)
    fill = [min(f, W) for f in [W, W, W, W - 1, W // 2, 257, 130, 40, 9, 5, 4, 2]][:S]
    t, y = make_windows(W * 7 + transform + len(methods), S, W, R, fps=fps, fill=fill, p_nan=0.0 if tc == '1' else 0.03)
    if tc == '1':
        y[1, 0, W // 3] = np.nan                         # a hole in a full window: taken by the float64 kernel
    px, py = oracle_proc(t, y, methods)
    p = params(S, R, W, methods, transform, **kw)
    dx, dy = torch.from_numpy(px).cuda(), torch.from_numpy(py).cuda()
    base = ops.window_spectrum(dx, dy, p, store=True)
    spectra = oracle_spectra(px, py, transform, kw)
    for band in spectrum_bands(px, py, transform, kw):
        for store in (True, False):
            o = ops.window_spectrum(dx, dy, p, store=store, band=band)
            torch.cuda.synchronize()
            check_spectrum(o, px, py, spectra, band)
            if store:   # the spectrum does not depend on the band
                for k in ('freqs', 'mags', 'num_bins'):
                    assert torch.equal(o[k].nan_to_num(-7.0), base[k].nan_to_num(-7.0)), (band, k)
    one = ops.window_spectrum(dx, dy, p, band=spectrum_bands(px, py, transform, kw)[3])
    assert int(one['peak_idx'][0, 0]) == -1              # exactly one eligible bin: no peak


IDENTITY = [(orc.PGRAM_WELCH, [orc.DETREND_LINEAR, orc.FILTER_FIR], 300, None), (orc.PGRAM_WELCH, [], 600, None),
            (orc.DFT_RFFT, [orc.DIFF_1], 300, '0'), (orc.DFT_RFFT, [orc.INTERP_CUBIC, orc.FILTER_BUTTER], 300, None),
            (orc.PGRAM_LS, [orc.FILTER_BUTTER], 250, None), (orc.PGRAM_LS, [], 3300, None)]


@pytest.mark.parametrize('transform,methods,W,tc', IDENTITY, ids=lambda v: str(v).replace(' ', ''))
def test_unbounded_band_is_the_default_search(transform, methods, W, tc, monkeypatch):
    """(-inf, inf) gives the bits of the existing entry point; a finite band that holds every bin runs the band kernels
    and must give them too (their coarse maximum, candidate set and write-back then equal the unbanded ones)."""
    from bpv import ops
    if tc is not None:
        monkeypatch.setenv('BPV_DFT_TC', tc)
    S, R = (3, 2) if W > 1000 else (10, 2)
    fill = [min(f, W) for f in [W, W, W - 1, W // 2, 130, 40, 5, 3, 2, 0]][:S]
    t, y = make_windows(W * 3 + transform, S, W, R, fill=fill)
    px, py = oracle_proc(t, y, methods)
    p = params(S, R, W, methods, transform)
    dx, dy = torch.from_numpy(px).cuda(), torch.from_numpy(py).cuda()
    for store in (True, False):
        ref = ops.window_spectrum(dx, dy, p, store=store)
        for band in [(-math.inf, math.inf), WIDE]:
            o = ops.window_spectrum(dx, dy, p, store=store, band=band)
            for k, v in ref.items():
                assert (v is None) == (o[k] is None)
                if v is not None:
                    assert torch.equal(o[k].nan_to_num(-7.0), v.nan_to_num(-7.0)), (band, k)


def lag_x(px, py, a, b):
    """Lag in seconds of every lag index, as the xcorr kernels report it (= orc.xcorr's lags)."""
    return orc.xcorr(px[a], py[a], py[b])[0]


def check_xcorr(o, px, py, band):
    li, ls, lc = (o[k].cpu().numpy() for k in ('lag_idx', 'lag_sec', 'lag_corr'))
    S, R = px.shape[:2]
    for s in range(S):
        for k, (a, b) in enumerate(itertools.combinations(range(R), 2)):
            el, ec = orc.xcorr(px[s, a], py[s, a], py[s, b])
            if int((np.isfinite(py[s, a]) & np.isfinite(py[s, b])).sum()) < MIN_N:
                continue
            ex, ey, ei = bo.peak_in_band(el, ec, *band)
            assert li[s, k] == ei, (s, k, band, li[s, k], ei)
            if ei >= 0:
                assert ls[s, k] == ex and band[0] <= ls[s, k] <= band[1]
                np.testing.assert_allclose(lc[s, k], ey, rtol=1e-9)
            else:
                assert np.isnan(ls[s, k]) and np.isnan(lc[s, k])


def xcorr_bands(px, py):
    """As spectrum_bands, cut from the lags of pair (0, 1) of the job px, py [R, W]."""
    x0 = lag_x(px, py, 0, 1)
    s = np.unique(x0)
    assert s.size >= 9
    return [(-0.5, 0.5), (0.0, 0.3), (s[1], s[len(s) // 2]), (s[2], s[2]), (s[3] + 1e-12, s[4] - 1e-12), (0.5, -0.5), (-math.inf, 0.0)]


@pytest.mark.parametrize('W,fps', [(64, 30.0), (250, 30.0), (300, 30.0), (1200, 120.0)])
def test_band_xcorr_matches_oracle(W, fps):
    """W = 64 / 250 / 300: coarse values in registers (ONE; generic, LD 53 and LD 63 instantiations); 1200: cv[] path;
    R = 3 (three pairs).  (xcorr_kernel, the CTA-per-pair fallback, needs more shared memory than the warp kernel at every
    window length, so no shape reaches it.)"""
    from bpv import ops
    S, R = 10, 3
    fill = [min(f, W) for f in [W, W - 1, W // 2, 130, 40, 9, 5, 3, 2, 0]][:S]
    t, y = make_windows(W * 11 + 5, S, W, R, fps=fps, fill=fill)
    methods = [orc.DETREND_LINEAR]
    px, py = oracle_proc(t, y, methods)
    p = params(S, R, W, methods)
    dx, dy = torch.from_numpy(px).cuda(), torch.from_numpy(py).cuda()
    base = ops.window_xcorr(dx, dy, p, store=True)
    for band in xcorr_bands(px[0], py[0]):
        for store in (True, False):
            o = ops.window_xcorr(dx, dy, p, store=store, band=band)
            torch.cuda.synchronize()
            check_xcorr(o, px, py, band)
            if store:
                for k in ('lags', 'corr', 'num_lags'):
                    assert torch.equal(o[k].nan_to_num(-7.0), base[k].nan_to_num(-7.0)), (band, k)
    for band in [(-math.inf, math.inf), WIDE]:
        o = ops.window_xcorr(dx, dy, p, store=True, band=band)
        for k, v in base.items():
            assert torch.equal(o[k].nan_to_num(-7.0), v.nan_to_num(-7.0)), (band, k)


def test_band_xcorr_non_monotone_timestamps():
    """Timestamps out of order (accepted outside INTERP_CUBIC): the lag of index k is not monotone in k, so eligibility is
    decided lag by lag."""
    from bpv import ops
    S, R, W = 6, 2, 300
    t, y = make_windows(77, S, W, R, fill=[W, W, 200, 64, 40, 9])
    rng = np.random.default_rng(5)
    for s in range(S):
        idx = np.flatnonzero(np.isfinite(t[s]))
        for _ in range(len(idx) // 6):
            i, j = rng.choice(idx, 2, replace=False)
            t[s, [i, j]] = t[s, [j, i]]
    px, py = oracle_proc(t, y, [orc.DETREND_CONST])
    lags = lag_x(px[0], py[0], 0, 1)
    assert (np.diff(lags) < 0).any()
    p = params(S, R, W, [orc.DETREND_CONST])
    dx, dy = torch.from_numpy(px).cuda(), torch.from_numpy(py).cuda()
    for band in [(-0.5, 0.5), (0.2, 1.0), (-3.0, -0.1)]:
        check_xcorr(ops.window_xcorr(dx, dy, p, band=band), px, py, band)


@pytest.mark.parametrize('transform,W,tc', [(orc.DFT_RFFT, 300, '0'), (orc.DFT_RFFT, 300, '1'), (orc.PGRAM_WELCH, 600, None),
                                            (orc.PGRAM_WELCH, 300, None)])
def test_band_dc_dominated_and_ties(transform, W, tc, monkeypatch):
    """A large DC level wins the all-bins search (0 bpm); the band finds the pulse.  An all-zero window ties every bin:
    the first in-band bin wins."""
    from bpv import ops
    if tc is not None:
        monkeypatch.setenv('BPV_DFT_TC', tc)
    S, R = 4, 2
    t = np.tile(np.arange(W, dtype=float) / 30.0 + 3.0, (S, 1))
    y = np.empty((S, R, W))
    y[:, 0] = 5.0 + 0.3 * np.sin(2 * np.pi * 1.3 * t)          # DFT: the DC bin dominates
    if transform == orc.PGRAM_WELCH:                            # Welch removes each segment's mean: a steep trend dominates
        y[:, 0] += np.linspace(0, 30.0, W)
    y[:, 1] = 0.0                                               # ties everywhere
    y[2, 0, 17] = np.nan                                                          # a hole
    px, py = oracle_proc(t, y, [])
    p = params(S, R, W, [], transform)
    dx, dy = torch.from_numpy(px).cuda(), torch.from_numpy(py).cuda()
    allb = ops.window_spectrum(dx, dy, p)
    band = ops.window_spectrum(dx, dy, p, band=(0.8, 4.0))
    check_spectrum(band, px, py, oracle_spectra(px, py, transform, {}), (0.8, 4.0))
    a, b = allb['peak_idx'].cpu().numpy(), band['peak_idx'].cpu().numpy()
    assert (a[:, 0] <= 2).all() and (b[:, 0] > 2).all()
    assert np.allclose(band['peak_freq'].cpu().numpy()[:, 0], 1.3, atol=0.2)
    x1 = kernel_x(px[0, 1], py[0, 1], transform, {})
    assert (b[:, 1] == int(np.flatnonzero(x1 >= 0.8)[0])).all()


# ------------------------------------------------------------------------------------------------
# the engine
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', ['c2_detrend_fir_welch', 'c4_cubic_butter_ls', 'diff1_dft', 'long_window_c2'])
def test_golden_replay_with_configured_ranges(name):
    """The reference-generated spectra / correlations of a golden case, searched over the configured ranges
    (Signal.get_peak(min_freq, max_freq) / (-0.5, 0.5)), against the engine run with those bands."""
    from bpv.engine import BatchedSignalProcessor
    channel, methods, transform, window, n, fps, irregular, p_none, roi_ms, kw = h.CASES[name]
    g = h.load_case(name)
    pr = orc._params(kw)
    fb, lb = (pr['min_freq'], pr['max_freq']), (-0.5, 0.5)
    eng = BatchedSignalProcessor(1, 2, signal_max_samples=window, processing_methods=[h.METHOD[m] for m in methods],
                                 spectrum_transform=h.TRANSFORM[transform], store_arrays=True, freq_band=fb, lag_band=lb, **kw)
    full_at = set(int(i) for i in g['full_at'])
    checked = 0
    for i in range(n):
        res = eng.step_signals(torch.tensor(g['raw'][i][None, None], dtype=torch.float64, device='cuda'),
                               torch.tensor([[g['ts'][i]]], dtype=torch.float64, device='cuda'))
        if i not in full_at:
            continue
        pi, pf = res.peak_idx.cpu().numpy()[0], res.peak_freq.cpu().numpy()[0]
        li, ls = res.lag_idx.cpu().numpy()[0], res.lag_sec.cpu().numpy()[0]
        nvalid = np.isfinite(g['raw'][:i + 1][-window:]).sum(axis=0)
        py_dev = res.arrays['proc_y'].cpu().numpy()[0]
        rawmax = np.nanmax(np.abs(g['raw'][:i + 1][-window:]), axis=0, initial=1.0)
        resid = [not np.isfinite(py_dev[r]).any() or np.nanmax(np.abs(py_dev[r])) < 1e-9 * rawmax[r] for r in range(2)]
        for r in range(2):
            if nvalid[r] < MIN_N or resid[r]:
                continue
            ex, ey, ei = bo.peak_in_band(g[f'f{i}_spec_x{r}'], g[f'f{i}_spec_y{r}'], *fb)
            assert pi[r] == ei, (name, i, r, pi[r], ei)
            assert h.close(pf[r], ex, rtol=1e-12, atol_frac=0), (name, i, r)
            checked += 1
        joint = int(np.isfinite(g['raw'][:i + 1][-window:]).all(axis=1).sum())
        if joint >= MIN_N and not any(resid):
            ex, ey, ei = bo.peak_in_band(g[f'f{i}_corr_x0'], g[f'f{i}_corr_y0'], *lb)
            assert li[0] == ei, (name, i, li[0], ei)
            assert h.close(ls[0], ex, rtol=1e-12, atol_frac=0)
            checked += 1
    assert checked >= 6


def _engine_run(S, T, steps, seed, **kw):
    from bpv import synth
    from bpv.engine import BatchedSignalProcessor
    rng = np.random.default_rng(seed)
    W = kw.pop('W', 40)
    n = T * steps
    ts = np.stack([synth.timestamps(rng, n, 30.0, irregular=True, drop=0.05, origin=rng.uniform(0, 100)) for _ in range(S)])
    ys = np.stack([synth.raw_signals(rng, ts[s], R=kw.get('num_rois', 2), p_nan=0.03) for s in range(S)])   # [S, R, n]
    eng = BatchedSignalProcessor(S, signal_max_samples=W, max_frames_per_step=T, **kw)
    out = []
    for g0 in range(0, n, T):
        res = eng.step_signals(torch.from_numpy(np.ascontiguousarray(ys[:, :, g0:g0 + T].transpose(0, 2, 1))).cuda(),
                               torch.from_numpy(ts[:, g0:g0 + T].copy()).cuda())
        # results are views of rotating buffers: keep copies
        snap = {k: getattr(res, k).clone() for k in ('peak_freq', 'peak_idx', 'peak_mag', 'lag_sec', 'lag_idx', 'lag_corr')}
        out.append((snap, {k: v.clone() for k, v in res.arrays.items()}, {k: v.clone() for k, v in res.means.items()},
                    res.packed().clone(), eng.launches_per_step))
    return eng, out


def test_engine_band_means_records_and_arrays():
    """Running means over the band peaks equal the oracle's nanmean of the band peaks; the packed record carries the band
    peaks; the stored arrays are those of a run without a band; bands can be changed between steps."""
    S, T, steps, R = 3, 4, 14, 3            # R = 3: P = 3 pairs
    common = dict(num_rois=R, processing_methods=[orc.DETREND_LINEAR, orc.FILTER_FIR], spectrum_transform=orc.PGRAM_WELCH,
                  store_arrays=True, peak_max_samples=8)
    _, plain = _engine_run(S, T, steps, 9, **common)
    eng, band = _engine_run(S, T, steps, 9, freq_band=(0.8, 4.0), lag_band=(-0.5, 0.5), **common)
    assert eng.freq_band == (0.8, 4.0) and eng.lag_band == (-0.5, 0.5)
    hist_b, hist_p = [], []
    differs = False
    for (rb, ab, mb, pb, nb), (rp, ap, mp, pp, np_) in zip(band, plain):
        assert nb == np_
        for k in ab:
            assert torch.equal(ab[k].nan_to_num(-7.0), ap[k].nan_to_num(-7.0)), k
        pf, ls = rb['peak_freq'].cpu().numpy(), rb['lag_sec'].cpu().numpy()
        assert (~np.isfinite(pf) | ((pf >= 0.8) & (pf <= 4.0))).all()
        assert (~np.isfinite(ls) | ((ls >= -0.5) & (ls <= 0.5))).all()
        differs |= not torch.equal(rb['peak_idx'], rp['peak_idx']) or not torch.equal(rb['lag_idx'], rp['lag_idx'])
        rec = pb.cpu().numpy()
        assert h.same(rec[:, :R], pf * 60) and h.same(rec[:, R:2 * R], ls * 1000)
        hist_b.append(pf.reshape(S, T, R))
        hist_p.append(ls.reshape(S, T, R))  # [S, T, P]
        # running means: nanmean over the last peak_max_samples band peaks of each stream
        allf = np.concatenate(hist_b, axis=1) * 60
        allp = np.concatenate(hist_p, axis=1) * 1000
        mbpm, mptt = mb['mean_bpm'].cpu().numpy().reshape(S, T, R), mb['mean_ptt'].cpu().numpy().reshape(S, T, R)
        for s in range(S):
            for t in range(T):
                end = allf.shape[1] - T + t + 1
                with np.errstate(all='ignore'), warnings.catch_warnings():
                    warnings.simplefilter('ignore')
                    ef = np.nanmean(allf[s, max(0, end - 8):end], axis=0)
                    ep = np.nanmean(allp[s, max(0, end - 8):end], axis=0)
                assert h.close(mbpm[s, t], ef, rtol=1e-12, atol_frac=0) and h.close(mptt[s, t], ep, rtol=1e-12, atol_frac=0)
    assert differs                      # the bands changed some peaks of this run
    # editable between steps: back to None gives the unbanded peaks on the same windows
    eng.freq_band = eng.lag_band = None
    assert eng.freq_band is None


@pytest.mark.parametrize('W', [64, 300])
def test_engine_band_fused_overlap_falls_back(W):
    """Overlap bit 4 (the fused Welch + xcorr grid, which has no band) with a band set runs the two-kernel schedule: same
    bits as the default schedule with the same band, and the launch count of that schedule."""
    common = dict(num_rois=2, processing_methods=[orc.DETREND_LINEAR, orc.FILTER_FIR], spectrum_transform=orc.PGRAM_WELCH,
                  store_arrays=True, freq_band=(0.8, 4.0), lag_band=(-0.5, 0.5), W=W)
    _, dflt = _engine_run(3, 4, 6 if W > 100 else 20, 13, **common)
    _, fused = _engine_run(3, 4, 6 if W > 100 else 20, 13, overlap=4 | 1, **common)
    _, serial = _engine_run(3, 4, 6 if W > 100 else 20, 13, overlap=1, **common)
    for (rd, ad, _, pd, nd), (rf, af, _, pf, nf), (_, _, _, _, ns) in zip(dflt, fused, serial):
        assert torch.equal(pd.nan_to_num(-7.0), pf.nan_to_num(-7.0))
        for k in rd:
            assert torch.equal(rd[k].nan_to_num(-7.0), rf[k].nan_to_num(-7.0)), k
        assert nf == ns == nd


def test_engine_rejects_bad_bands():
    from bpv.engine import BatchedSignalProcessor
    for bad in [dict(freq_band=(math.nan, 4.0)), dict(lag_band=(0.0,)), dict(lag_band='x')]:
        with pytest.raises(ValueError):
            BatchedSignalProcessor(1, 2, signal_max_samples=16, **bad)
