"""numpy restatement of the per-window spectral SNR and its gate (include/bpv.h bpv_window_snr) for the SNR tests.

It sits beside the tests, as band_oracle.py does: oracle/ stays the frozen restatement of what process() computes, and
process() has no SNR.
"""
import itertools

import numpy as np

DFT_RFFT, PGRAM_WELCH, PGRAM_LS = 1, 2, 3


def snr_db(f, m, num_bins, peak_idx, transform, lo, hi, half_width, exact_mags=False):
    """The SNR of one stored spectrum: f, m [>= num_bins] as F3 stored them (float32), widened to float64.
    P_k = m_k^2 (DFT_RFFT) or m_k; B = {k < num_bins : m_k finite, lo <= f_k <= hi}; template = |f_k - f0| <= hw or
    |f_k - 2 f0| <= hw with f0 = f[peak_idx]; 10 log10(S_sig / S_noise) with IEEE division; NaN without a peak or |B| < 2.
    exact_mags: take m as float64 values (e.g. scipy's spectrum) instead of rounding them to float32 first."""
    nb = int(num_bins)
    if peak_idx < 0 or peak_idx >= nb:
        return np.nan
    f = np.asarray(f[:nb], dtype=np.float32).astype(np.float64)
    m = np.asarray(m[:nb], dtype=np.float64 if exact_mags else np.float32).astype(np.float64)
    with np.errstate(invalid='ignore'):
        inb = np.isfinite(m) & (lo <= f) & (f <= hi)
    if inb.sum() < 2:
        return np.nan
    pw = m * m if transform == DFT_RFFT else m
    f0 = f[peak_idx]
    tmpl = (np.abs(f - f0) <= half_width) | (np.abs(f - 2.0 * f0) <= half_width)
    s_sig, s_noise = pw[inb & tmpl].sum(), pw[inb & ~tmpl].sum()
    with np.errstate(divide='ignore', invalid='ignore'):
        return float(10.0 * np.log10(np.float64(s_sig) / np.float64(s_noise)))


def snr_all(freqs, mags, num_bins, peak_idx, transform, lo, hi, half_width):
    """snr_db over [J, R] stored spectra (host arrays)."""
    J, R = num_bins.shape
    out = np.empty((J, R))
    for j, r in np.ndindex(J, R):
        out[j, r] = snr_db(freqs[j, r], mags[j, r], num_bins[j, r], peak_idx[j, r], transform, lo, hi, half_width)
    return out


def gate(snr, peak_freq, lag_sec, min_snr_db):
    """(gated_freq [J, R], gated_lag [J, P]): the values where accepted, NaN elsewhere.  A heart rate is accepted when
    snr >= min_snr_db (NaN rejected); the PTT of pair (a, b), itertools.combinations order, when both a and b are."""
    with np.errstate(invalid='ignore'):
        ok = np.asarray(snr) >= min_snr_db
    gf = np.where(ok, peak_freq, np.nan)
    R = ok.shape[1]
    pairs = list(itertools.combinations(range(R), 2))
    gl = np.full(np.shape(lag_sec), np.nan)
    for q, (a, b) in enumerate(pairs):
        both = ok[:, a] & ok[:, b]
        gl[both, q] = np.asarray(lag_sec)[both, q]
    return gf, gl
