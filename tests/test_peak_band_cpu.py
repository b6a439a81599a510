"""CPU: the band-limited peak search.  Its restatement of Signal.get_peak(min_x, max_x) (tests/band_oracle.py) against the
drop-in and the reference's signal_data on every stored golden spectrum / correlation, and the argument checks of the C ABI
entry points that run before anything is enqueued on a device."""
import ctypes
import glob
import importlib.util
import math
import os
import re
import warnings

import numpy as np
import pytest

from oracle import bpv_oracle as orc
from tests import band_oracle as bo
from tests import helpers as h


def _arrays():
    """Every stored spectrum and correlation of the committed fixtures: (name, x, y)."""
    out = []
    for path in sorted(glob.glob(os.path.join(h.GOLDEN, '*.npz'))):
        g = np.load(path)
        for k in g.files:
            m = re.fullmatch(r'(f\d+)_(spec|corr)_x(\d+)', k)
            if m:
                out.append((f'{os.path.basename(path)}:{k}', g[k], g[k.replace('_x', '_y', 1)], m.group(2)))
    assert len(out) > 100
    return out


def _bands(x, kind):
    """Bands that matter: the reference's configured ranges, edges exactly on an entry, exactly one eligible entry, two,
    an empty band, an inverted band and the unbounded one."""
    bands = [(-math.inf, math.inf), (1.0, 0.5), (1e9, 2e9)]
    bands += [(0.8, 4.0), (0.7, 3.0)] if kind == 'spec' else [(-0.5, 0.5), (0.0, 0.5), (-0.5, 0.0)]
    xf = x[np.isfinite(x)]
    if xf.size:
        s = np.unique(xf)
        bands += [(s[0], s[-1]), (s[len(s) // 2], s[len(s) // 2])]            # full span on the edges; a single entry
        if s.size >= 2:
            bands += [(s[1], s[-2]), (s[0], s[1]), (s[-2], s[-1])]              # edges exactly on entries; two entries
    return bands


def _ref_peak(sd, x, y, lo, hi):
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        return sd.Signal(list(x), list(y)).get_peak(lo, hi)


def _check_against(sd):
    n = 0
    for name, x, y, kind in _arrays():
        for lo, hi in _bands(x, kind):
            ex, ey = _ref_peak(sd, x, y, lo, hi)
            gx, gy, gi = bo.peak_in_band(x, y, lo, hi)
            assert h.same([gx, gy], [ex, ey]), (name, lo, hi, (gx, gy), (ex, ey))
            if gi >= 0:
                assert x[gi] == gx and y[gi] == gy and lo <= gx <= hi
                assert not (np.isfinite(y) & (x >= lo) & (x <= hi) & (y > gy)).any()
            n += 1
    return n


def test_peak_in_band_matches_dropin_get_peak():
    import signal_data as sd
    assert _check_against(sd) > 1000


@pytest.mark.skipif(not os.path.isdir(h.REFERENCE), reason=h.NO_REFERENCE)
def test_peak_in_band_matches_reference_get_peak():
    spec = importlib.util.spec_from_file_location('ref_signal_data', os.path.join(h.REFERENCE, 'signal_data.py'))
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    assert _check_against(ref) > 1000


def test_peak_in_band_edge_cases():
    x = np.array([0.0, 0.5, 1.0, 1.5, 2.0])
    y = np.array([9.0, 1.0, 3.0, 3.0, np.nan])
    assert bo.peak_in_band(x, y, 0.5, 2.0)[2] == 2          # tie: the first maximum; NaN magnitude never eligible
    assert bo.peak_in_band(x, y, 1.0, 1.0)[2] == -1         # exactly one eligible entry: no peak
    assert bo.peak_in_band(x, y, 1.2, 1.3)[2] == -1         # empty
    assert bo.peak_in_band(x, y, 2.0, 0.0)[2] == -1         # inverted
    assert bo.peak_in_band(x, y, -np.inf, np.inf)[:3] == orc.peak(x, y)[:3]
    assert bo.peak_in_band(x, y, 0.0, 0.5)[2] == 0


def test_band_entry_points_reject_nan_bounds():
    """A NaN bound is an argument error (BPV_E_INVALID) returned before any CUDA call, so it holds without a device."""
    from bpv import _cabi, ops
    lib = _cabi.lib()
    p = ops.make_params(1, 2, 16, 16, 15, 1, 1, [], _cabi.PGRAM_WELCH)
    buf = (ctypes.c_double * 64)()
    fake = ctypes.cast(buf, ctypes.c_void_p)
    for lo, hi in [(math.nan, 1.0), (0.0, math.nan), (math.nan, math.nan)]:
        rc = lib.bpv_window_spectrum_band(fake, fake, ctypes.byref(p), 9, None, 0, None, None, fake, fake, fake, fake, lo, hi, None)
        assert rc == -1 and b'NaN' in lib.bpv_last_error(), rc
        rc = lib.bpv_window_xcorr_band(fake, fake, ctypes.byref(p), None, None, fake, fake, fake, fake, lo, hi, None)
        assert rc == -1 and b'NaN' in lib.bpv_last_error(), rc


def test_band_arguments_are_validated_in_python():
    from bpv import ops
    assert ops.peak_band(None) is None
    assert ops.peak_band((0.8, 4)) == (0.8, 4.0)
    assert ops.peak_band([-math.inf, math.inf]) == (-math.inf, math.inf)
    assert ops.peak_band((2.0, 1.0)) == (2.0, 1.0)                       # inverted: allowed, gives no peak
    for bad in [(math.nan, 1.0), (0.0, float('nan')), (1.0,), (1.0, 2.0, 3.0), 'ab', 3.0]:
        with pytest.raises(ValueError):
            ops.peak_band(bad)
