"""Restatement of the band-limited peak search for the parity tests of the band-limited peak entry points.

It sits beside the tests rather than in oracle/, which stays the frozen restatement of what process() computes (`peak`
there is the search after SignalGroup's range reset); this is the search a single Signal.get_peak(min_x, max_x) runs.
"""
import numpy as np


def peak_in_band(x, y, lo, hi):
    """signal_data.py:65-70 with explicit bounds, Signal.get_peak(lo, hi): the first maximum of y over the entries with
    lo <= x <= hi and a finite y; fewer than two such entries -> no peak.  What a single transform_signal(s).get_peak()
    (range (min_freq, max_freq), signal_processor.py:272) or correlate_signal_pair(a, b).get_peak() (range (min_lag,
    max_lag), :294) returns before SignalGroup resets the range.  Returns the triple of `peak`."""
    x, y = np.asarray(x, dtype=float), np.asarray(y, dtype=float)
    with np.errstate(invalid='ignore'):
        u = (lo <= x) & (x <= hi) & np.isfinite(y)
    if u.sum() < 2:
        return np.nan, np.nan, -1
    i = int(np.argmax(y[u]))
    return x[u][i], y[u][i], int(np.flatnonzero(u)[i])
