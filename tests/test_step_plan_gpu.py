"""GPU: settings of the batched engine that can be reassigned between steps take effect at the next step as a whole.  A bad
peak band raises before the step enqueues anything; a switch of transform or ls_num_freqs resizes F3's output buffers,
the zero-row result and the spectrum workspace to the new bin count."""
import math

import numpy as np
import pytest
import torch

from oracle import bpv_oracle as orc

pytestmark = pytest.mark.gpu

S, R, T = 5, 2, 6


def _data(seed, n, W):
    from bpv import synth
    rng = np.random.default_rng(seed)
    ts = np.stack([synth.timestamps(rng, n, 30.0, irregular=True, drop=0.03, origin=rng.uniform(0, 50)) for _ in range(S)])
    ys = np.stack([synth.raw_signals(rng, ts[s], R=R, f_pulse=1.1 + 0.1 * s, p_nan=0.02) for s in range(S)]).transpose(0, 2, 1)
    return ts, np.ascontiguousarray(ys)


def _step_inputs(ts, ys, i):
    sl = slice(i * T, (i + 1) * T)
    return torch.from_numpy(ys[:, sl].copy()).cuda(), torch.from_numpy(ts[:, sl].copy()).cuda()


@pytest.mark.parametrize('path', ['lockstep', 'jobmap'])
def test_bad_band_raises_before_anything_is_enqueued(path):
    """A NaN, one-element or string band assigned between steps raises at the next step before its first launch: the
    counts, the result turn and the rings stay as the previous step left them, and a good band then steps normally."""
    from bpv.engine import BatchedSignalProcessor
    ts, ys = _data(1, 3 * T, 48)
    eng = BatchedSignalProcessor(S, R, signal_max_samples=48, max_frames_per_step=T, processing_methods=[orc.FILTER_BUTTER],
                                 spectrum_transform=orc.PGRAM_WELCH, peak_max_samples=8, store_arrays=True)
    eng.force_jobmap = path == 'jobmap'
    eng.step_signals(*_step_inputs(ts, ys, 0))
    torch.cuda.synchronize()
    state = (eng.counts, eng.mean_counts, eng._turn, eng.ring_t.clone(), eng.ring_y.clone(), eng._bpm_ring.clone())
    smp, tst = _step_inputs(ts, ys, 1)
    for name in ('freq_band', 'lag_band'):
        for bad in ((math.nan, 4.0), (0.5,), 'band'):
            setattr(eng, name, bad)
            with pytest.raises(ValueError):
                eng.step_signals(smp, tst)
            with pytest.raises(ValueError):
                eng.step_signals(smp, tst, frame_counts=[T, 1, 0, 2, T])
            torch.cuda.synchronize()
            assert np.array_equal(eng.counts, state[0]) and np.array_equal(eng.mean_counts, state[1]) and eng._turn == state[2]
            for a, b in zip((eng.ring_t, eng.ring_y, eng._bpm_ring), state[3:]):
                assert torch.equal(a.isnan(), b.isnan()) and torch.equal(a.nan_to_num(), b.nan_to_num())
        setattr(eng, name, None)
    eng.freq_band = (0.8, 4.0)
    res = eng.step_signals(smp, tst)
    assert res.peak_freq.shape[0] == S * T and np.array_equal(eng.counts, state[0] + T)


def _host(res):
    out = {k: getattr(res, k).cpu().numpy() for k in ('peak_freq', 'peak_idx', 'peak_mag', 'lag_sec', 'lag_idx', 'lag_corr',
                                                      'status', 'snr_db')}
    out.update({k: v.cpu().numpy() for k, v in res.arrays.items()})
    return out


def _same(a, b, tag):
    assert a.keys() == b.keys(), tag
    for k in a:
        assert a[k].shape == b[k].shape and a[k].dtype == b[k].dtype, (tag, k, a[k].shape, b[k].shape)
        assert np.array_equal(a[k].view(np.uint8), b[k].view(np.uint8)), (tag, k)


def test_transform_and_bin_count_switches_resize_the_spectrum_buffers():
    """An engine with store_arrays and snr runs Welch steps (126 bins at a 250-sample window), then switches to Lomb-Scargle
    (250 bins), then raises ls_num_freqs to 400.  At J = Jmax, every output of every step after a switch is bit-identical
    to that of an engine built with the new setting and fed the same steps, and a zero-row result has the new bin count."""
    from bpv.engine import BatchedSignalProcessor
    W, steps = 250, 9
    ts, ys = _data(2, steps * T, W)
    kw = dict(signal_max_samples=W, max_frames_per_step=T, processing_methods=[orc.DETREND_LINEAR, orc.FILTER_BUTTER],
              store_arrays=True, snr=True)
    eng = BatchedSignalProcessor(S, R, spectrum_transform=orc.PGRAM_WELCH, **kw)
    refs = {3: BatchedSignalProcessor(S, R, spectrum_transform=orc.PGRAM_LS, **kw),
            6: BatchedSignalProcessor(S, R, spectrum_transform=orc.PGRAM_LS, ls_num_freqs=400, **kw)}
    for i in range(steps):
        if i == 3:
            eng.transform = orc.PGRAM_LS
        if i == 6:
            eng.kw['ls_num_freqs'] = 400
        smp, tst = _step_inputs(ts, ys, i)
        got = _host(eng.step_signals(smp, tst))
        outs = {k: _host(r.step_signals(smp, tst)) for k, r in refs.items()}
        assert got['freqs'].shape == (S * T, R, 126 if i < 3 else 250 if i < 6 else 400), i
        if i >= 3:
            _same(got, outs[3 if i < 6 else 6], i)
        empty = eng.step_signals(smp, tst, frame_counts=np.zeros(S, dtype=np.int64))
        assert empty.arrays['freqs'].shape == (0, R, got['freqs'].shape[2]), i
