"""CPU: the restatement of the per-window spectral SNR (tests/snr_oracle.py) on hand-built spectra, and the argument checks
of bpv_window_snr, which return before anything is enqueued on a device."""
import ctypes as C
import math

import numpy as np
import pytest

from tests import snr_oracle as so

F = np.arange(11, dtype=np.float32) * np.float32(0.5)          # 0, 0.5, ..., 5 Hz


def snr(m, pk, lo=0.7, hi=4.0, hw=0.125, transform=so.PGRAM_WELCH, f=F, nb=None):
    m = np.asarray(m, dtype=np.float32)
    return so.snr_db(f, m, len(m) if nb is None else nb, pk, transform, lo, hi, hw)


def test_signal_over_noise_in_db():
    m = np.full(11, 1.0)
    m[2] = 50.0                     # f0 = 1 Hz; harmonic 2 Hz = bin 4; band 0.7..4 = bins 2..8
    m[4] = 10.0
    assert snr(m, 2) == pytest.approx(10 * math.log10(60.0 / 5.0), abs=1e-12)


def test_no_peak_and_too_few_bins():
    m = np.arange(11, dtype=float) + 1
    assert math.isnan(snr(m, -1))
    assert math.isnan(snr(m, 3, lo=1.5, hi=1.5))               # |B| = 1
    assert math.isnan(snr(m, 3, lo=2.0, hi=1.0))               # inverted band: B empty
    assert math.isnan(snr(m, 9, nb=8))                         # the peak lies beyond num_bins
    m2 = m.copy()
    m2[[3, 4, 5, 6, 7, 8]] = np.nan
    assert math.isnan(snr(m2, 2, lo=0.7, hi=4.0))              # one finite bin left in the band


def test_ieee_division():
    m = np.zeros(11)
    m[2] = 3.0
    assert snr(m, 2) == math.inf                               # S_noise = 0
    m = np.zeros(11)
    m[6] = 3.0
    assert snr(m, 2) == -math.inf                              # S_sig = 0
    assert math.isnan(snr(np.zeros(11), 2))                    # 0 / 0


def test_dc_peak_is_minus_infinity():
    m = np.linspace(1.0, 2.0, 11)
    m[0] = 100.0
    assert snr(m, 0) == -math.inf                              # template {0 Hz, 0 Hz} lies below the band


def test_harmonic_outside_the_band():
    m = np.ones(11)
    m[6] = 9.0                                                 # f0 = 3 Hz, harmonic 6 Hz outside the band and the grid
    m[8] = 99.0                                                # 4 Hz: in the band, not in the template
    s_sig, s_noise = 9.0, 1.0 * 5 + 99.0
    assert snr(m, 6) == pytest.approx(10 * math.log10(s_sig / s_noise), abs=1e-12)


def test_template_edges_are_inclusive_and_zero_width():
    m = np.ones(11)
    m[2] = 8.0
    # hw = 0.5 exactly: bins 1, 3 (f0 -/+ 0.5) and 3, 5 (2 f0 -/+ 0.5) inside; band 0..5 holds all 11 bins
    got = snr(m, 2, lo=0.0, hi=5.0, hw=0.5)
    assert got == pytest.approx(10 * math.log10((1 + 8.0 + 1 + 1 + 1) / 6.0), abs=1e-12)   # bins 1..5 vs 0, 6..10
    got0 = snr(m, 2, lo=0.0, hi=5.0, hw=0.0)                   # delta = 0: the peak and the harmonic bin only
    assert got0 == pytest.approx(10 * math.log10((8.0 + 1.0) / 9.0), abs=1e-12)
    assert snr(m, 2, lo=0.0, hi=5.0, hw=0.4999) == pytest.approx(got0, abs=1e-12)


def test_lomb_scargle_grid_not_starting_at_zero():
    f = np.linspace(0.8, 4.0, 33).astype(np.float32)           # the LS grid of (min_freq, max_freq)
    m = np.full(33, 0.01, dtype=np.float32)
    m[5] = np.float32(0.9)                                     # f0 = 1.3 Hz, harmonic 2.6 Hz = bin 18
    m[18] = np.float32(0.2)
    f64, m64 = f.astype(np.float64), m.astype(np.float64)
    tm = (np.abs(f64 - f64[5]) <= 0.125) | (np.abs(f64 - 2 * f64[5]) <= 0.125)
    assert tm.sum() == 6                                       # 0.1 Hz grid: peak and harmonic bins with both neighbours
    want = 10 * math.log10(m64[tm].sum() / m64[~tm].sum())
    assert so.snr_db(f, m, 33, 5, so.PGRAM_LS, 0.8, 4.0, 0.125) == pytest.approx(want, abs=1e-12)


def test_dft_power_is_the_square():
    m = np.ones(11)
    m[2] = 3.0
    m[4] = 2.0
    dft = snr(m, 2, transform=so.DFT_RFFT)
    assert dft == pytest.approx(10 * math.log10((9.0 + 4.0) / 5.0), abs=1e-12)
    assert snr(m, 2, transform=so.PGRAM_LS) == pytest.approx(10 * math.log10(5.0 / 5.0), abs=1e-12)


def test_gate():
    s = np.array([[3.0, 2.9, math.nan], [math.inf, -math.inf, 3.0]])
    pf = np.arange(6, dtype=float).reshape(2, 3) + 1
    ls = np.arange(6, dtype=float).reshape(2, 3) * 0.1
    gf, gl = so.gate(s, pf, ls, 3.0)
    assert np.array_equal(np.isnan(gf), [[False, True, True], [False, True, False]])
    # pairs (0, 1), (0, 2), (1, 2): job 0 accepts ROI 0 only; job 1 accepts ROIs 0 and 2
    assert np.array_equal(np.isnan(gl), [[True, True, True], [True, False, True]])
    assert gl[1, 1] == ls[1, 1]
    gf, gl = so.gate(s, pf, ls, -math.inf)                      # -inf accepts every value but NaN
    assert np.isnan(gf).sum() == 1 and np.isnan(gl).sum() == 2


def test_window_snr_rejects_bad_arguments_before_touching_the_gpu():
    """-1 = BPV_E_INVALID for every bad argument, before the first CUDA call; J = 0 with valid arguments enqueues nothing."""
    from bpv import _cabi
    lib = _cabi.lib()
    buf = (C.c_uint8 * 4096)()
    a = C.cast(buf, C.c_void_p)        # a non-NULL address that is never dereferenced
    inf, nan = math.inf, math.nan
    good = dict(spec_f=a, spec_mag=a, num_bins=a, peak_idx=a, J=4, R=2, max_bins=9, transform=_cabi.PGRAM_WELCH, lo=0.8,
                hi=4.0, hw=0.125, peak_freq=a, lag_sec=a, P=1, thr=3.0, snr=a, gf=a, gl=a)

    def call(**kw):
        v = {**good, **kw}
        return lib.bpv_window_snr(v['spec_f'], v['spec_mag'], v['num_bins'], v['peak_idx'], v['J'], v['R'], v['max_bins'],
                                  v['transform'], v['lo'], v['hi'], v['hw'], v['peak_freq'], v['lag_sec'], v['P'], v['thr'],
                                  v['snr'], v['gf'], v['gl'], None)
    bad = [dict(lo=nan), dict(hi=nan), dict(hw=-0.1), dict(hw=inf), dict(hw=nan), dict(thr=nan), dict(J=-1), dict(R=0),
           dict(max_bins=0), dict(P=0), dict(R=3, P=1), dict(transform=0), dict(transform=4),
           dict(spec_f=None), dict(spec_mag=None), dict(num_bins=None), dict(peak_idx=None), dict(snr=None),
           dict(peak_freq=None), dict(lag_sec=None)]
    for kw in bad:
        assert call(**kw) == -1, kw
        assert b'bpv_window_snr' in lib.bpv_last_error(), kw
    # valid with J = 0: nothing to do.  -inf thresholds, infinite and inverted bands, zero width and no gated outputs are fine
    ok = [dict(), dict(thr=-inf), dict(lo=-inf, hi=inf), dict(lo=4.0, hi=0.8), dict(hw=0.0), dict(gf=None, peak_freq=None),
          dict(gl=None, lag_sec=None), dict(R=1, P=0, gl=None, lag_sec=None), dict(transform=_cabi.DFT_RFFT),
          dict(transform=_cabi.PGRAM_LS)]
    for kw in ok:
        assert call(J=0, **kw) == 0, kw


def test_python_arguments():
    from bpv import ops
    assert ops.snr_half_width(0) == 0.0 and ops.snr_half_width(0.125) == 0.125
    for bad in (-1e-9, math.inf, math.nan, 'x', None):
        with pytest.raises(ValueError):
            ops.snr_half_width(bad)
    assert ops.snr_threshold(None) is None and ops.snr_threshold(3) == 3.0 and ops.snr_threshold(-math.inf) == -math.inf
    for bad in (math.nan, 'x', (1, 2)):
        with pytest.raises(ValueError):
            ops.snr_threshold(bad)
