"""GPU tests of the round-2 rows: mask-weighted ROI sampling (SURVEY 8f-4), engine state_dict / resume (8f-3), result
lifetime (rotating buffers), the overlapped schedules, device placement, the split design / filter entry points, the
24-byte record, and the merged forward.backward FIR against the two-pass filtfilt of the oracle."""
import numpy as np
import pytest
import torch

from oracle import bpv_oracle as orc
from tests import helpers as h

pytestmark = pytest.mark.gpu


def _boxes(rng, N, R, H, W):
    from bpv import synth
    b = np.zeros((N, R, 4), dtype=np.int32)
    for i in range(N):
        for r in range(R):
            kind = rng.integers(0, 10)
            x0, y0 = int(rng.integers(-W // 2, W)), int(rng.integers(-H // 2, H))
            x1, y1 = x0 + int(rng.integers(0, W // 2 + 3)), y0 + int(rng.integers(0, H // 2 + 3))
            b[i, r] = (x0, y0, x1, y1)
            if kind == 0:
                b[i, r, 0] = synth.NO_BOX
            elif kind == 1:
                b[i, r] = (W - 3, H - 2, W + 50, H + 50)          # clamped at the far corner
            elif kind == 2:
                b[i, r] = (-7, -5, -1, -1)                        # negative wrap
    return b


@pytest.mark.parametrize('shape', [(37, 53), (48, 64), (61, 100)])      # W % 4 != 0 -> byte path, W % 4 == 0 -> word path
@pytest.mark.parametrize('channel', [orc.GREEN, orc.CHROM_GREEN])
def test_masked_roi_sampling_bit_exact(shape, channel):
    from bpv import ops, synth
    H, W = shape
    rng = np.random.default_rng(H * 1000 + W + channel)
    N, R = 24, 3
    frames = rng.integers(0, 256, (N, H, W, 3), dtype=np.uint8)
    masks = rng.integers(0, 6, (N, H, W), dtype=np.uint8)
    masks[3] = 3                                                   # everything selected for category 3
    masks[4] = 0                                                   # nothing selected for categories 2 / 3 -> NaN
    boxes = _boxes(rng, N, R, H, W)
    cats = [3, 2, 3]
    val, sums = ops.roi_sample_masked(torch.from_numpy(frames).cuda(), torch.from_numpy(masks).cuda(), cats,
                                      torch.from_numpy(boxes).cuda(), channel, want_sums=True)
    val, sums = val.cpu().numpy(), sums.cpu().numpy()
    for i in range(N):
        for r in range(R):
            b = boxes[i, r]
            sroi = (np.nan,) * 6 if b[0] == synth.NO_BOX else (0, 0, int(b[0]), int(b[1]), int(b[2]), int(b[3]))
            ref, rs = orc.roi_sample_masked(frames[i], masks[i], cats[r], sroi, channel)
            assert h.same(val[i, r], ref), (i, r, val[i, r], ref)
            if b[0] != synth.NO_BOX:
                assert tuple(int(v) for v in sums[i, r]) == rs, (i, r)
    # an all-pass mask reproduces the unmasked kernel bit for bit
    ones = torch.full((N, H, W), 5, dtype=torch.uint8, device='cuda')
    v_all, _ = ops.roi_sample_masked(torch.from_numpy(frames).cuda(), ones, 5, torch.from_numpy(boxes).cuda(), channel)
    v_ref, _ = ops.roi_sample(torch.from_numpy(frames).cuda(), torch.from_numpy(boxes).cuda(), channel)
    assert h.same(v_all.cpu().numpy(), v_ref.cpu().numpy())


def test_masked_roi_strided_views():
    """Cropped views (row stride > 3W, odd offsets) take the byte path and still match."""
    from bpv import ops
    rng = np.random.default_rng(7)
    big = rng.integers(0, 256, (6, 40, 70, 3), dtype=np.uint8)
    bigm = rng.integers(0, 4, (6, 40, 70), dtype=np.uint8)
    fr, mk = torch.from_numpy(big).cuda()[:, :, 5:58], torch.from_numpy(bigm).cuda()[:, :, 5:58]
    boxes = _boxes(rng, 6, 2, 40, 53)
    val, _ = ops.roi_sample_masked(fr, mk, 1, torch.from_numpy(boxes).cuda(), orc.GREEN)
    from bpv import synth
    for i in range(6):
        for r in range(2):
            b = boxes[i, r]
            sroi = (np.nan,) * 6 if b[0] == synth.NO_BOX else (0, 0, int(b[0]), int(b[1]), int(b[2]), int(b[3]))
            ref, _ = orc.roi_sample_masked(big[i][:, 5:58], bigm[i][:, 5:58], 1, sroi, orc.GREEN)
            assert h.same(val[i, r].item(), ref)


def _engine(S=6, W=48, T=4, **kw):
    from bpv.engine import BatchedSignalProcessor
    base = dict(signal_max_samples=W, max_frames_per_step=T, color_channel=orc.CHROM_GREEN,
                processing_methods=[orc.DETREND_LINEAR, orc.FILTER_FIR], spectrum_transform=orc.PGRAM_WELCH, peak_max_samples=5)
    base.update(kw)
    return BatchedSignalProcessor(S, 2, **base)


def _signal_steps(seed, S, T, steps, fps=30.0):
    from bpv import synth
    rng = np.random.default_rng(seed)
    ts = np.stack([synth.timestamps(rng, T * steps, fps, irregular=True, drop=0.03, origin=rng.uniform(0, 9)) for _ in range(S)])
    raw = np.stack([synth.raw_signals(rng, ts[s], R=2, p_nan=0.03).T for s in range(S)])          # [S, N, R]
    return [(torch.from_numpy(raw[:, k * T:(k + 1) * T].copy()).cuda(), torch.from_numpy(ts[:, k * T:(k + 1) * T].copy()).cuda())
            for k in range(steps)]


def _snap(res):
    return {k: getattr(res, k).clone() for k in ('peak_freq', 'peak_idx', 'peak_mag', 'lag_sec', 'lag_idx', 'lag_corr', 'status')} | \
           {k: v.clone() for k, v in res.means.items()}


def _same(a, b):
    return all(torch.equal(a[k].view(torch.int64) if a[k].dtype == torch.float64 else a[k],
                           b[k].view(torch.int64) if b[k].dtype == torch.float64 else b[k]) for k in a)


def test_state_dict_resume_is_bit_exact():
    """A run interrupted after step k and resumed in a NEW engine from state_dict() equals the uninterrupted run bit for
    bit: rings, sample count, bpm / ptt histories of the running means (SURVEY 8f-3)."""
    S, T, steps, cut = 6, 4, 30, 17
    feed = _signal_steps(11, S, T, steps)
    a = _engine(S, 48, T)
    full = [_snap(a.step_signals(*f)) for f in feed]
    b = _engine(S, 48, T)
    for f in feed[:cut]:
        b.step_signals(*f)
    state = b.state_dict()
    assert all(not v.is_cuda for v in state.values() if torch.is_tensor(v))
    import pickle
    state = pickle.loads(pickle.dumps(state))                    # survives a checkpoint file
    c = _engine(S, 48, T)
    c.load_state_dict(state)
    for k, f in enumerate(feed[cut:]):
        assert _same(_snap(c.step_signals(*f)), full[cut + k]), k
    # reset() forgets the histories too: a reset engine replays the run from the start
    c.reset()
    for k, f in enumerate(feed[:8]):
        assert _same(_snap(c.step_signals(*f)), full[k]), k
    with pytest.raises(ValueError):
        _engine(S + 1, 48, T).load_state_dict(state)


def test_state_dict_covers_roi_history():
    from bpv.engine import BatchedSignalProcessor
    rng = np.random.default_rng(5)
    S, T, R, K, H, W = 3, 2, 2, 2, 60, 80
    mk = lambda: BatchedSignalProcessor(S, R, signal_max_samples=16, max_frames_per_step=T, processing_methods=[], spectrum_transform=orc.DFT_RFFT)
    a, b = mk(), mk()
    for e in (a, b):
        e.set_roi_configs(h.REL, [1, 2], roi_max_samples=3)
    def det(k):
        g = np.random.default_rng(100 + k)
        present = torch.from_numpy((g.random((S, T, R)) > 0.2).astype(np.uint8)).cuda()
        bbox = torch.from_numpy(g.integers(5, 50, (S, T, R, 4)).astype(np.int32)).cuda()
        bbox[..., 2:] += bbox[..., :2]
        pts = torch.from_numpy(g.integers(5, 55, (S, T, R, K, 2)).astype(np.int32)).cuda()
        fr = torch.from_numpy(g.integers(0, 256, (S, T, H, W, 3), dtype=np.uint8)).cuda()
        ts = torch.from_numpy(np.tile((np.arange(T) + 1 + k * T) / 30.0, (S, 1))).cuda()
        return fr, present, bbox, pts, ts
    for k in range(3):
        a.step_detections(*det(k))
        b.step_detections(*det(k))
    c = mk()
    c.set_roi_configs(h.REL, [1, 2], roi_max_samples=3)
    c.load_state_dict(b.state_dict())
    for k in range(3, 6):
        ra, ba = a.step_detections(*det(k))
        rc, bc = c.step_detections(*det(k))
        assert torch.equal(ba, bc) and _same(_snap(ra), _snap(rc))


def test_results_survive_the_next_step():
    """StepResult tensors are views of rotating buffers: with result_buffers=2 (default) the result of step k is intact
    after step k+1 and overwritten by step k+2; result_buffers=1 aliases immediately (documented in bpv/engine.py)."""
    S, T = 5, 3
    feed = _signal_steps(3, S, T, 6)
    eng = _engine(S, 48, T, store_arrays=True)
    r0 = eng.step_signals(*feed[0])
    keep = _snap(r0)
    keep_proc = r0.arrays['proc_y'].clone()
    eng.step_signals(*feed[1])
    torch.cuda.synchronize()
    assert _same(_snap(r0), keep) and torch.equal(r0.arrays['proc_y'].view(torch.int64), keep_proc.view(torch.int64))
    r2 = eng.step_signals(*feed[2])
    assert r2.peak_freq.data_ptr() == r0.peak_freq.data_ptr()          # the slot has been reused
    one = _engine(S, 48, T, result_buffers=1)
    q0 = one.step_signals(*feed[0])
    q1 = one.step_signals(*feed[1])
    assert q0.peak_freq.data_ptr() == q1.peak_freq.data_ptr()


@pytest.mark.parametrize('methods,transform', [([orc.DETREND_LINEAR, orc.FILTER_FIR], orc.PGRAM_WELCH),
                                               ([orc.FILTER_BUTTER], orc.PGRAM_LS)])
def test_overlapped_schedules_equal_the_serial_one(methods, transform):
    """overlap = 0 / 1 / 2 / 3 (filter design beside F1, xcorr beside the spectrum) produce identical bits."""
    from bpv import synth
    S, T, H, W = 4, 3, 48, 64
    rng = np.random.default_rng(21)
    frames = torch.from_numpy(rng.integers(0, 256, (S, T, H, W, 3), dtype=np.uint8)).cuda()
    boxes = torch.from_numpy(np.stack([synth.roi_boxes(rng, T, H, W) for _ in range(S)])).cuda()
    outs = []
    for ov in (0, 1, 2, 3):
        eng = _engine(S, 40, T, processing_methods=methods, spectrum_transform=transform, overlap=ov)
        run = []
        for k in range(16):
            ts = torch.from_numpy(np.tile((np.arange(T) + 1 + k * T) / 30.0, (S, 1))).cuda()
            run.append(_snap(eng.step(frames.roll(k, dims=1), boxes, ts)))
        torch.cuda.synchronize()
        outs.append(run)
    for ov in (1, 2, 3):
        assert all(_same(x, y) for x, y in zip(outs[0], outs[ov])), ov


def test_split_design_and_filter_equal_preprocess():
    from tests.test_window_gpu import make_windows, to_ring, params
    from bpv import ops, _cabi
    S, R, W = 40, 2, 300
    t, y = make_windows(9, S, W, R, fill=[W, W - 1, 200, 127, 126, 60, 3, 2, 1, 0])
    rt, ry = to_ring(t, y)
    p = params(S, R, W, [orc.DETREND_LINEAR, orc.FILTER_FIR, orc.FILTER_BUTTER])
    px, py, st = ops.window_preprocess(rt, ry, p)
    ws = torch.empty(_cabi.lib().bpv_window_workspace_bytes(p), dtype=torch.uint8, device='cuda')
    ops.window_design(rt, p, ws)
    qx, qy, qs = ops.window_filter(rt, ry, p, ws)
    assert torch.equal(st, qs) and torch.equal(py.view(torch.int64), qy.view(torch.int64)) and torch.equal(px.view(torch.int64), qx.view(torch.int64))


@pytest.mark.parametrize('W,taps', [(300, 127), (250, 127), (1200, 127), (128, 127), (127, 127), (126, 127), (64, 31), (300, 31), (31, 31)])
def test_fir_merged_path_matches_two_pass_filtfilt(W, taps):
    """Windows of n >= taps samples run filtfilt as ONE symmetric 2*taps-1 tap filter (autocorrelation of the taps, from the
    design kernel); shorter ones the two-pass form.  Both against scipy.signal.filtfilt through the oracle."""
    from tests.test_window_gpu import make_windows, to_ring, params, TIGHT
    from bpv import ops
    S, R = 24, 2
    fill = [W, W - 1, max(W - 5, 0), taps + 1, taps, taps - 1, taps // 2, 5]
    t, y = make_windows(1000 + W + taps, S, W, R, fps=30.0, fill=[min(f, W) for f in fill], p_nan=0.0)
    rt, ry = to_ring(t, y)
    p = params(S, R, W, [orc.FILTER_FIR], fir_taps=taps)
    px, py, st = ops.window_preprocess(rt, ry, p)
    py, st = py.cpu().numpy(), st.cpu().numpy()
    checked = 0
    for s in range(S):
        for r in range(R):
            if st[s, r] != 0:
                continue
            _, ref = orc.preprocess(t[s], y[s, r], [orc.FILTER_FIR], fir_taps=taps)
            scale = np.nanmax(np.abs(ref))
            np.testing.assert_allclose(py[s, r], ref, rtol=0, atol=TIGHT * scale, equal_nan=True, err_msg=f'{s} {r}')
            checked += 1
    assert checked >= S


def test_packed32_record_roundtrip():
    from bpv import ops
    S, T = 5, 3
    eng = _engine(S, 48, T)
    for f in _signal_steps(8, S, T, 20):
        res = eng.step_signals(*f)
    rec = res.packed32()
    assert rec.dtype == torch.int32 and rec.shape == (S * T, 6) and rec.element_size() * rec.shape[1] == 24
    bpm, ptt, pi, li = ops.unpack_records32(rec, 2, 1)
    assert torch.equal(pi, res.peak_idx) and torch.equal(li, res.lag_idx)
    assert h.same(bpm.cpu().numpy(), res.bpm.to(torch.float32).cpu().numpy())
    assert h.same(ptt.cpu().numpy(), res.ptt_ms.to(torch.float32).cpu().numpy())


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason='needs 2 GPUs')
def test_engine_on_second_gpu_while_current_device_is_first():
    """ADVICE r1: kernels must be enqueued on the GPU that owns the tensors, whatever the caller's current device."""
    S, T = 4, 3
    feed = _signal_steps(14, S, T, 18)
    torch.cuda.set_device(0)
    a = _engine(S, 40, T, device='cuda:0')
    b = _engine(S, 40, T, device='cuda:1')
    for f in feed:
        ra = a.step_signals(*f)
        rb = b.step_signals(f[0].to('cuda:1'), f[1].to('cuda:1'))
    assert torch.cuda.current_device() == 0
    assert rb.peak_freq.device == torch.device('cuda:1')
    sa, sb = _snap(ra), {k: v.to('cuda:0') for k, v in _snap(rb).items()}
    assert _same(sa, sb)


@pytest.mark.parametrize('methods', [[orc.FILTER_BUTTER], [orc.INTERP_CUBIC, orc.FILTER_BUTTER], [orc.DETREND_LINEAR, orc.FILTER_BUTTER, orc.DIFF_1],
                                     [orc.FILTER_FIR, orc.FILTER_BUTTER]])
@pytest.mark.parametrize('R', [1, 2, 3])
def test_two_signal_butterworth_cascade_is_bit_identical(methods, R, monkeypatch):
    """FILTER_BUTTER runs two signals per warp (lanes 0-15 / 16-31 each own a 16-section cascade); the arithmetic per lane
    is that of the one-signal-per-warp kernel (BPV_SOS_SINGLE=1), so every output bit must agree — for odd signal counts,
    pairs that straddle window jobs (R = 1, 3), windows of different lengths in one warp, guard failures and bad bands."""
    from tests.test_window_gpu import make_windows, to_ring, params
    from bpv import ops
    S, W = 45, 120
    fill = [W, W - 1, 100, 64, 33, 17, 5, 3, 2, 1, 0]
    t, y = make_windows(77 + R, S, W, R, fps=30.0, fill=fill)
    t[7] = np.where(np.isfinite(t[7]), t[7][np.isfinite(t[7])][0] + np.arange(W) * 3.0, np.nan)      # 0.33 fps: no valid pass band left
    rt, ry = to_ring(t, y)
    p = params(S, R, W, methods, fir_taps=31)
    monkeypatch.delenv('BPV_SOS_SINGLE', raising=False)
    px2, py2, st2 = ops.window_preprocess(rt, ry, p)
    monkeypatch.setenv('BPV_SOS_SINGLE', '1')
    px1, py1, st1 = ops.window_preprocess(rt, ry, p)
    assert torch.equal(st1, st2)
    assert torch.equal(py1.view(torch.int64), py2.view(torch.int64))
    assert torch.equal(px1.view(torch.int64), px2.view(torch.int64))
    assert int((st1 == 0).sum()) > S // 2 and int((st1 == 3).sum()) >= 1


@pytest.mark.parametrize('methods,transform', [([orc.DETREND_LINEAR, orc.FILTER_FIR], orc.PGRAM_WELCH),
                                               ([orc.FILTER_BUTTER], orc.DFT_RFFT),
                                               ([orc.FILTER_FIR, orc.FILTER_BUTTER], orc.PGRAM_WELCH)])
@pytest.mark.parametrize('irregular', [False, True])
def test_design_cache_is_bit_identical_to_fresh_designs(methods, transform, irregular):
    """The fs-keyed design cache (hits on regular timestamps; all-distinct rates, table overflow, own-slot fallback and the
    clear-on-thrash path on jittered ones with 300 streams x 4 jobs > 256 slots) returns exactly the bits of per-job designs."""
    from bpv import synth
    from bpv.engine import BatchedSignalProcessor
    S, T, W, steps = 300, 4, 140, 9
    rng = np.random.default_rng(5)
    ts = np.stack([synth.timestamps(rng, T * steps, 30.0, irregular=irregular, drop=0.02 if irregular else 0.0,
                                    origin=rng.uniform(0, 3) if irregular else 0.0) for _ in range(S)])
    raw = np.stack([synth.raw_signals(rng, ts[s], R=2, p_nan=0.02).T for s in range(S)])
    outs = []
    for cache in (False, True):
        eng = BatchedSignalProcessor(S, 2, signal_max_samples=W, max_frames_per_step=T, processing_methods=methods,
                                     spectrum_transform=transform, design_cache=cache, store_arrays=True, fir_taps=63)
        run = []
        for k in range(steps):
            res = eng.step_signals(torch.from_numpy(raw[:, k * T:(k + 1) * T].copy()).cuda(), torch.from_numpy(ts[:, k * T:(k + 1) * T].copy()).cuda())
            run.append((_snap(res), res.arrays['proc_y'].clone()))
        outs.append(run)
    for (a, pa), (b, pb) in zip(*outs):
        assert _same(a, b)
        assert torch.equal(pa.view(torch.int64), pb.view(torch.int64))


def test_design_cache_is_dropped_when_filter_parameters_change():
    """The table is keyed by fs only; the engine empties it when the band edges / orders it was filled under change (the
    drop-in SignalProcessor lets callers edit them between frames)."""
    S, T = 8, 3
    feed = _signal_steps(31, S, T, 24)
    a = _engine(S, 40, T, design_cache=True)
    b = _engine(S, 40, T, design_cache=False)
    for k, f in enumerate(feed):
        if k == 12:
            for e in (a, b):
                e.kw = dict(e.kw, min_freq=1.1, fir_df=0.25)
        assert _same(_snap(a.step_signals(*f)), _snap(b.step_signals(*f))), k


@pytest.mark.parametrize('R,W,T,store', [(2, 48, 4, False), (2, 300, 3, True), (3, 64, 4, False), (2, 250, 2, False), (2, 400, 2, False)])
def test_fused_welch_xcorr_grid_equals_the_two_launches(R, W, T, store):
    """overlap bit 4 (include/bpv.h bpv_window_welch_xcorr): Welch and xcorr CTAs interleaved in ONE grid give the bits of
    the two stand-alone launches — warm-up windows, holes, irregular timestamps, three ROIs (3 pairs per job: another CTA
    ratio), stored arrays, and a window over 320 samples (the entry point then runs the two launches itself)."""
    from bpv import synth
    from bpv.engine import BatchedSignalProcessor
    S, steps = 7, (W + 40) // T
    rng = np.random.default_rng(1000 * R + W)
    ts = np.stack([synth.timestamps(rng, T * steps, 30.0, irregular=True, drop=0.03, origin=rng.uniform(0, 9)) for _ in range(S)])
    raw = np.stack([synth.raw_signals(rng, ts[s], R=R, p_nan=0.03).T for s in range(S)])
    keys = ('peak_freq', 'peak_idx', 'peak_mag', 'lag_sec', 'lag_idx', 'lag_corr', 'status')
    runs = []
    for ov in (0, 4, 7):
        eng = BatchedSignalProcessor(S, R, signal_max_samples=W, max_frames_per_step=T, color_channel=orc.CHROM_GREEN,
                                     processing_methods=[orc.DETREND_LINEAR, orc.FILTER_FIR], spectrum_transform=orc.PGRAM_WELCH,
                                     store_arrays=store, overlap=ov)
        out = []
        for k in range(steps):
            res = eng.step_signals(torch.from_numpy(raw[:, k * T:(k + 1) * T].copy()).cuda(),
                                   torch.from_numpy(ts[:, k * T:(k + 1) * T].copy()).cuda())
            snap = {k2: getattr(res, k2).clone() for k2 in keys}
            if store:
                nb, nl = res.arrays['num_bins'], res.arrays['num_lags']
                snap.update(num_bins=nb.clone(), num_lags=nl.clone())
                # entries past num_bins / num_lags are undefined: compare the defined ones
                mb = torch.arange(res.arrays['mags'].shape[-1], device='cuda')[None, None, :] < nb[..., None]
                ml = torch.arange(res.arrays['corr'].shape[-1], device='cuda')[None, None, :] < nl[..., None]
                for name, m in (('freqs', mb), ('mags', mb), ('lags', ml), ('corr', ml)):
                    snap[name] = torch.where(m, res.arrays[name], torch.zeros_like(res.arrays[name])).view(torch.int32).clone()
            out.append(snap)
        torch.cuda.synchronize()
        runs.append(out)
    for other in runs[1:]:
        assert all(_same(x, y) for x, y in zip(runs[0], other))
    assert any(bool(torch.isfinite(x['lag_sec']).any()) for x in runs[0]) and any(bool((x['peak_idx'] >= 0).any()) for x in runs[0])
