"""Shared helpers for the parity tests (golden replay, comparisons)."""
import os

import numpy as np

from __graft_entry__ import REFERENCE   # the upstream checkout build() stages from; live-reference tests skip without it
from oracle import bpv_oracle as orc

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
NO_REFERENCE = f'no checkout of the reference at {REFERENCE}'
METHOD = dict(DIFF_1=orc.DIFF_1, DIFF_2=orc.DIFF_2, INTERP_LINEAR=orc.INTERP_LINEAR, INTERP_CUBIC=orc.INTERP_CUBIC,
              DETREND_CONST=orc.DETREND_CONST, DETREND_LINEAR=orc.DETREND_LINEAR, FILTER_BUTTER=orc.FILTER_BUTTER,
              FILTER_FIR=orc.FILTER_FIR)
TRANSFORM = dict(DFT_RFFT=orc.DFT_RFFT, PGRAM_WELCH=orc.PGRAM_WELCH, PGRAM_LS=orc.PGRAM_LS)
CHANNEL = dict(GREEN=orc.GREEN, CHROM_GREEN=orc.CHROM_GREEN)

# golden case table (also imported by tests/golden/make_golden.py):
# name: (channel, methods, transform, window, n_frames, fps, irregular, p_none, roi_max_samples, kwargs)
CASES = {
    'c1_butter_ls':      ('GREEN', ['FILTER_BUTTER'], 'PGRAM_LS', 48, 70, 30, False, 0.03, 1, dict(min_freq=0.7)),
    'c2_detrend_fir_welch': ('CHROM_GREEN', ['DETREND_LINEAR', 'FILTER_FIR'], 'PGRAM_WELCH', 48, 70, 30, False, 0.03, 1, {}),
    'c4_cubic_butter_ls': ('GREEN', ['INTERP_CUBIC', 'FILTER_BUTTER'], 'PGRAM_LS', 56, 72, 120, True, 0.05, 1, {}),
    'diff1_dft':         ('GREEN', ['DIFF_1'], 'DFT_RFFT', 40, 60, 30, False, 0.02, 1, {}),
    'diff2_welch':       ('CHROM_GREEN', ['DIFF_2'], 'PGRAM_WELCH', 40, 60, 30, True, 0.02, 2, {}),
    'lin_const_fir_dft': ('GREEN', ['INTERP_LINEAR', 'DETREND_CONST', 'FILTER_FIR'], 'DFT_RFFT', 40, 60, 25, True, 0.05, 3, {}),
    'none_ls':           ('CHROM_GREEN', [], 'PGRAM_LS', 40, 60, 30, True, 0.05, 1, {}),
    'lowfs_butter_ls':   ('GREEN', ['DETREND_LINEAR', 'FILTER_BUTTER'], 'PGRAM_LS', 40, 56, 7.5, False, 0.0, 1, {}),
    'long_window_c2':    ('CHROM_GREEN', ['DETREND_LINEAR', 'FILTER_FIR'], 'PGRAM_WELCH', 300, 306, 30, False, 0.01, 1, {}),
    'long_window_c1':    ('GREEN', ['FILTER_BUTTER'], 'PGRAM_LS', 300, 306, 30, False, 0.01, 1, dict(min_freq=0.7)),
}
# added after the first ten (generated with their own seeds, SEEDS below): other method chains, filter orders, tap counts,
# frame rates and ROI smoothing lengths
CASES.update({
    'diff1_butter4_welch':  ('GREEN', ['DIFF_1', 'FILTER_BUTTER'], 'PGRAM_WELCH', 44, 64, 30, True, 0.04, 2, dict(butter_order=4)),
    'cubic_lin_fir31_ls':   ('CHROM_GREEN', ['INTERP_CUBIC', 'DETREND_LINEAR', 'FILTER_FIR'], 'PGRAM_LS', 52, 70, 60, True, 0.04, 1,
                             dict(fir_taps=31, min_freq=0.7)),
    'const_dft_smooth3':    ('CHROM_GREEN', ['DETREND_CONST'], 'DFT_RFFT', 36, 50, 24, False, 0.10, 3, {}),
    'lin_diff2_butter8_ls': ('GREEN', ['INTERP_LINEAR', 'DIFF_2', 'FILTER_BUTTER'], 'PGRAM_LS', 40, 58, 15, True, 0.02, 1,
                             dict(butter_order=8, max_freq=3.0)),
})
SEEDS = {name: 100 + k for k, name in enumerate(list(CASES)[:10])}
SEEDS.update(diff1_butter4_welch=500, cubic_lin_fir31_ls=501, const_dft_smooth3=502, lin_diff2_butter8_ls=503)
# cases that are NOT committed as fixtures: tests/test_oracle_golden.py::test_live_differential_vs_reference runs the
# reference on them in a subprocess (where REFERENCE exists) and demands exact equality with the oracle, so the pin does
# not rest on the frozen files alone
LIVE_CASES = {
    'live_diff2_butter2_dft':       ('GREEN', ['DIFF_2', 'FILTER_BUTTER'], 'DFT_RFFT', 38, 54, 30, True, 0.03, 1, dict(butter_order=2)),
    'live_cubic_const_fir63_welch': ('CHROM_GREEN', ['INTERP_CUBIC', 'DETREND_CONST', 'FILTER_FIR'], 'PGRAM_WELCH', 48, 66, 50, True, 0.03, 2,
                                     dict(fir_taps=63)),
    'live_lin_detrend_ls_lowfs':    ('GREEN', ['INTERP_LINEAR', 'DETREND_LINEAR'], 'PGRAM_LS', 32, 48, 10, True, 0.05, 1, {}),
}
IMG_H, IMG_W = 60, 80
REL = [(-0.00, -0.10, 0.20, 0.05), (-0.10, -0.10, 0.10, 0.10)]  # roi.py:26,28
LMK = [[151], [0, 9]]                                            # roi.py:19,21-22


def load_case(name):
    g = np.load(os.path.join(GOLDEN, f'{name}.npz'))
    return {k: g[k] for k in g.files}


def case_frames(g):
    from bpv import synth
    return synth.frames(np.random.default_rng(int(g['seed']) + 1000), g['ts'], IMG_H, IMG_W, f_pulse=1.3)


def case_rois(g, i):
    """The reference's calc_rois (via the oracle restatement) on the stored detections."""
    rois = []
    for r in range(2):
        if not g['present'][i, r]:
            rois.append((np.nan,) * 6)
            continue
        if r == 0:
            pts = np.zeros((478, 2), np.int64)
            pts[151] = g['face_pt'][i]
            det = [(tuple(int(v) for v in g['face_bbox'][i]), pts)]
        else:
            pts = np.zeros((21, 2), np.int64)
            pts[0], pts[9] = g['hand_pts'][i, 0], g['hand_pts'][i, 1]
            det = [(tuple(int(v) for v in g['hand_bbox'][i]), pts)]
        rois.append(orc.calc_roi(det, LMK[r], REL[r]))
    return rois


def same(a, b):
    """Exact equality with NaN == NaN."""
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return a.shape == b.shape and bool(np.all((a == b) | (np.isnan(a) & np.isnan(b))))


def close(a, b, rtol=1e-4, atol_frac=1e-5, atol=0.0):
    """|a-b| <= rtol*|b| + atol_frac*max|b| + atol  with NaN == NaN (north_star: rtol 1e-4).
    `atol` covers outputs that are pure rounding residue of a much larger input (e.g. a detrended
    2-sample window): pass eps-level * input scale."""
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    if a.shape != b.shape:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    if not np.array_equal(na, nb):
        return False
    if b.size == 0 or nb.all():
        return True
    scale = np.nanmax(np.abs(b))
    return bool(np.all(np.abs(a - b)[~nb] <= rtol * np.abs(b)[~nb] + atol_frac * scale + atol))
