"""GPU: ragged steps of the batched engine (per-stream frame counts, per-stream reset).  Stream s of a ragged engine must
equal its own one-stream engine fed only its frames, bit for bit, and that engine is pinned to the oracle and the golden
files by tests/test_engine_gpu.py."""
import pickle

import numpy as np
import pytest
import torch

from oracle import bpv_oracle as orc
from tests import helpers as h

pytestmark = pytest.mark.gpu

S, R, W, T = 7, 2, 48, 5
CFGS = {
    'fir_welch': dict(methods=[orc.DETREND_LINEAR, orc.FILTER_FIR], transform=orc.PGRAM_WELCH),
    'butter_ls': dict(methods=[orc.FILTER_BUTTER], transform=orc.PGRAM_LS),
    'cubic_dft': dict(methods=[orc.INTERP_CUBIC, orc.FILTER_BUTTER], transform=orc.DFT_RFFT),   # tensor-core DFT
}
FIELDS = ('peak_freq', 'peak_idx', 'peak_mag', 'lag_sec', 'lag_idx', 'lag_corr', 'status')


def _engine(S_, cfg, **kw):
    from bpv.engine import BatchedSignalProcessor
    return BatchedSignalProcessor(S_, R, signal_max_samples=W, max_frames_per_step=T, processing_methods=cfg['methods'],
                                  spectrum_transform=cfg['transform'], peak_max_samples=8, **kw)


def _data(seed, n_total):
    from bpv import synth
    rng = np.random.default_rng(seed)
    ts = np.stack([synth.timestamps(rng, n_total, 30.0 if s % 2 else 60.0, irregular=True, drop=0.03,
                                    origin=rng.uniform(0, 50)) for s in range(S)])
    ys = np.stack([synth.raw_signals(rng, ts[s], R=R, p_nan=0.03) for s in range(S)]).transpose(0, 2, 1)   # [S, n, R]
    return ts, np.ascontiguousarray(ys)


def _schedule(seed, steps=25):
    rng = np.random.default_rng(seed)
    n = rng.integers(0, T + 1, (steps, S))
    n[3] = 0                      # a step in which no stream takes a frame
    n[7] = T                      # every stream takes T
    n[9:14, 4] = 0                # a stream that idles for several steps
    n[:6, 6] = 0                  # a stream that joins late
    return n


def _host(res):
    out = {k: getattr(res, k).cpu().numpy() for k in FIELDS}
    out.update({k: v.cpu().numpy() for k, v in res.means.items()})
    out.update({k: v.cpu().numpy() for k, v in res.arrays.items()})
    return out


def _rows_equal(a, b, tag):
    """Bit-for-bit equality of per-job rows (NaN == NaN); spectra / correlations compared over their valid entries."""
    for k in b:
        x, y = a[k], b[k]
        if k in ('freqs', 'mags'):
            x, y = _valid(x, a['num_bins']), _valid(y, b['num_bins'])
        elif k in ('lags', 'corr'):
            x, y = _valid(x, a['num_lags']), _valid(y, b['num_lags'])
        assert x.shape == y.shape, (tag, k, x.shape, y.shape)
        xv, yv = x.view(np.uint8) if x.dtype.kind == 'f' else x, y.view(np.uint8) if y.dtype.kind == 'f' else y
        if x.dtype.kind == 'f':
            same = (x == y) | (np.isnan(x) & np.isnan(y))
            assert same.all(), (tag, k, np.argwhere(~same)[:5])
        else:
            assert np.array_equal(xv, yv), (tag, k)


def _valid(a, counts):
    a = a.copy()
    idx = np.arange(a.shape[-1])
    a[idx >= counts[..., None]] = 0
    return a


def _run_split(cfg, sched, ts, ys, reset_at=None, reset_streams=(), **kw):
    """The ragged engine, and per stream a one-stream engine fed only its frames (fresh after a reset of that stream)."""
    eng = _engine(S, cfg, **kw)
    singles = [_engine(1, cfg, **kw) for _ in range(S)]
    pos = np.zeros(S, dtype=np.int64)
    checked = 0
    for k, n in enumerate(sched):
        if k == reset_at:
            eng.reset(streams=list(reset_streams))
            for s in reset_streams:
                singles[s] = _engine(1, cfg, **kw)
        smp = np.full((S, T, R), np.nan)
        tst = np.full((S, T), np.nan)
        for s in range(S):
            smp[s, :n[s]] = ys[s, pos[s]:pos[s] + n[s]]
            tst[s, :n[s]] = ts[s, pos[s]:pos[s] + n[s]]
        res = eng.step_signals(torch.from_numpy(smp).cuda(), torch.from_numpy(tst).cuda(), frame_counts=n)
        assert res.jobs_per_stream is None or (n == T).all()
        off = res.job_offsets
        jobs = n if eng.windows == 'every_frame' else (n > 0).astype(int)
        assert np.array_equal(np.diff(off), jobs)
        assert np.array_equal(res.job_stream.cpu().numpy(), np.repeat(np.arange(S), jobs))
        got = _host(res)
        for s in range(S):
            if n[s] == 0:
                continue
            ref = _host(singles[s].step_signals(torch.from_numpy(ys[s:s + 1, pos[s]:pos[s] + n[s]].copy()).cuda(),
                                                torch.from_numpy(ts[s:s + 1, pos[s]:pos[s] + n[s]].copy()).cuda()))
            _rows_equal({kk: v[off[s]:off[s + 1]] for kk, v in got.items()}, ref, (k, s))
            checked += 1
        pos += n
    assert np.array_equal(eng.counts, [e.count for e in singles])
    return checked


@pytest.mark.parametrize('overlap', [0, 3])
@pytest.mark.parametrize('cache', [True, False], ids=['cache', 'nocache'])
@pytest.mark.parametrize('windows', ['every_frame', 'last'])
@pytest.mark.parametrize('cfg', list(CFGS))
def test_ragged_equals_independent_engines(cfg, windows, cache, overlap):
    sched = _schedule(1)
    ts, ys = _data(2, int(sched.sum(axis=0).max()) + 1)
    store = cache and overlap == 3              # stored arrays on a quarter of the cases keeps the run short
    assert _run_split(CFGS[cfg], sched, ts, ys, windows=windows, design_cache=cache, overlap=overlap, store_arrays=store) > 100


FH, FW = 48, 80                   # frame size of the step() tests


@pytest.mark.parametrize('overlap,ingest', [(1, 'plain'), (3, 'plain'), (4, 'plain'), (3, 'view'), (3, 'masked'), (0, 'plain')])
def test_ragged_step_with_frames_equals_independent_engines(overlap, ingest):
    """step(frames, boxes, ts, frame_counts=...): F1 on the frames, the ragged design-ahead schedule (overlap bit 1: timestamp
    push, job map and filter design on the side stream), the fused Welch + xcorr grid (bit 4), and frame_counts forwarded
    through the cropped-view and masked ingest.  Each stream equals a one-stream engine driven through step() with only its
    frames, bit for bit."""
    from bpv import synth
    cfg = CFGS['fir_welch']
    sched = _schedule(12, steps=14)
    ts, _ = _data(13, int(sched.sum(axis=0).max()) + 1)
    rng = np.random.default_rng(14)
    nf = ts.shape[1]
    frames = np.stack([synth.frames(rng, ts[s], FH, FW, f_pulse=1.0 + 0.2 * s) for s in range(S)])        # [S, nf, FH, FW, 3]
    bw = 60 if ingest == 'view' else FW
    boxes = np.stack([synth.roi_boxes(rng, nf, FH, bw, p_none=0.03) for _ in range(S)])                 # [S, nf, R, 4]
    masks = rng.integers(0, 3, (S, nf, FH, FW), dtype=np.uint8)
    kw = dict(overlap=overlap, store_arrays=True)
    extra = {}
    if ingest == 'view':
        extra = dict(view=(60, FH, 10, True))
    eng = _engine(S, cfg, **kw)
    singles = [_engine(1, cfg, **kw) for _ in range(S)]
    pos = np.zeros(S, dtype=np.int64)
    checked = 0
    for k, n in enumerate(sched):
        fr = np.zeros((S, T, FH, FW, 3), np.uint8)
        bx = np.full((S, T, R, 4), 0, np.int32)
        bx[..., 0] = synth.NO_BOX                                   # rows a stream does not take: no box, nothing sampled
        tst = np.full((S, T), np.nan)
        mk = np.zeros((S, T, FH, FW), np.uint8)
        for s in range(S):
            sl = slice(pos[s], pos[s] + n[s])
            fr[s, :n[s]], bx[s, :n[s]], tst[s, :n[s]], mk[s, :n[s]] = frames[s, sl], boxes[s, sl], ts[s, sl], masks[s, sl]
        if ingest == 'masked':
            extra = dict(masks=torch.from_numpy(mk).cuda(), mask_category=[1, 2])
        res = eng.step(torch.from_numpy(fr).cuda(), torch.from_numpy(bx).cuda(), torch.from_numpy(tst).cuda(), frame_counts=n, **extra)
        got, off = _host(res), res.job_offsets
        smp = res.samples.cpu().numpy() if res.samples is not None else None
        for s in range(S):
            if n[s] == 0:
                continue
            sl = slice(pos[s], pos[s] + n[s])
            ex1 = dict(extra)
            if ingest == 'masked':
                ex1 = dict(masks=torch.from_numpy(masks[s:s + 1, sl].copy()).cuda(), mask_category=[1, 2])
            r1 = singles[s].step(torch.from_numpy(frames[s:s + 1, sl].copy()).cuda(), torch.from_numpy(boxes[s:s + 1, sl].copy()).cuda(),
                                 torch.from_numpy(ts[s:s + 1, sl].copy()).cuda(), **ex1)
            assert h.same(smp[s, :n[s]], r1.samples.cpu().numpy()[0]), (k, s)
            _rows_equal({kk: v[off[s]:off[s + 1]] for kk, v in got.items()}, _host(r1), (k, s))
            checked += 1
        pos += n
    assert np.array_equal(eng.counts, [e.count for e in singles]) and checked > 40


def test_ragged_matches_oracle_on_full_windows():
    """Checked directly against the oracle: once a stream's window is full, every job of a ragged step equals the oracle's
    processing of that stream's own last W samples."""
    cfg = CFGS['fir_welch']
    sched = _schedule(3, steps=12)
    sched[0] = T
    ts, ys = _data(4, W + int(sched.sum(axis=0).max()) + 1)
    eng = _engine(S, cfg, store_arrays=True)
    # fill every window first: W frames per stream in level steps
    pos = np.zeros(S, dtype=np.int64)
    while pos[0] < W:
        k = min(T, W - int(pos[0]))
        eng.step_signals(torch.from_numpy(ys[:, pos[0]:pos[0] + k].copy()).cuda(), torch.from_numpy(ts[:, pos[0]:pos[0] + k].copy()).cuda())
        pos += k
    checked = 0
    for n in sched:
        smp, tst = np.full((S, T, R), np.nan), np.full((S, T), np.nan)
        for s in range(S):
            smp[s, :n[s]], tst[s, :n[s]] = ys[s, pos[s]:pos[s] + n[s]], ts[s, pos[s]:pos[s] + n[s]]
        res = eng.step_signals(torch.from_numpy(smp).cuda(), torch.from_numpy(tst).cuda(), frame_counts=n)
        a = _host(res)
        off = res.job_offsets
        for s in range(S):
            for t in range(n[s]):
                j, g = off[s] + t, pos[s] + t
                tw, yw = ts[s, g - W + 1:g + 1], ys[s, g - W + 1:g + 1]
                proc = [orc.preprocess(tw, yw[:, r], cfg['methods']) for r in range(R)]
                for r in range(R):
                    assert h.close(a['proc_y'][j, r], proc[r][1], rtol=1e-6, atol_frac=1e-7), (s, g, r)
                    ef, em = orc.spectrum(proc[r][0], proc[r][1], cfg['transform'])
                    assert a['peak_idx'][j, r] == orc.peak(ef, em)[2], (s, g, r)
                el, ec = orc.xcorr(proc[0][0], proc[0][1], proc[1][1])
                assert a['lag_idx'][j, 0] == orc.peak(el, ec)[2], (s, g)
                checked += 1
        pos += n
    assert checked > 50


@pytest.mark.parametrize('windows', ['every_frame', 'last'])
def test_level_counts_cannot_tell_the_paths_apart(windows):
    """frame_counts = [T] * S is the lockstep step; level counts forced through the job map give the same bits and layout."""
    cfg = CFGS['butter_ls']
    ts, ys = _data(5, 8 * T)
    engs = [_engine(S, cfg, windows=windows) for _ in range(3)]
    engs[2].force_jobmap = True
    for k in range(8):
        smp, tst = torch.from_numpy(ys[:, k * T:(k + 1) * T].copy()).cuda(), torch.from_numpy(ts[:, k * T:(k + 1) * T].copy()).cuda()
        r0 = engs[0].step_signals(smp, tst)
        r1 = engs[1].step_signals(smp, tst, frame_counts=[T] * S)
        r2 = engs[2].step_signals(smp, tst)
        assert r0.jobs_per_stream is not None and r1.jobs_per_stream == r0.jobs_per_stream and r2.jobs_per_stream is None
        assert engs[1].launches_per_step == engs[0].launches_per_step
        a = _host(r0)
        for r in (r1, r2):
            assert np.array_equal(r.job_offsets, r0.job_offsets)
            assert torch.equal(r.job_stream, r0.job_stream)
            _rows_equal(_host(r), a, k)
            assert torch.equal(r.packed32(), r0.packed32())
    assert engs[2].count == engs[0].count == 8 * T


def test_per_stream_reset():
    """reset(streams=[2, 5]) mid-run: those streams equal fresh one-stream engines fed the later frames (their running means
    start over); every other stream equals the run that never reset."""
    cfg = CFGS['fir_welch']
    sched = _schedule(6, steps=16)
    ts, ys = _data(7, int(sched.sum(axis=0).max()) + 1)
    _run_split(cfg, sched, ts, ys, reset_at=8, reset_streams=(2, 5))
    # the untouched streams against an engine that never reset
    a, b = _engine(S, cfg), _engine(S, cfg)
    pos = np.zeros(S, dtype=np.int64)
    for k, n in enumerate(sched):
        if k == 8:
            b.reset(streams=[2, 5])
            assert b.counts[2] == b.counts[5] == 0 and np.array_equal(np.delete(b.counts, [2, 5]), np.delete(a.counts, [2, 5]))
        smp, tst = np.full((S, T, R), np.nan), np.full((S, T), np.nan)
        for s in range(S):
            smp[s, :n[s]], tst[s, :n[s]] = ys[s, pos[s]:pos[s] + n[s]], ts[s, pos[s]:pos[s] + n[s]]
        ra = _host(a.step_signals(torch.from_numpy(smp).cuda(), torch.from_numpy(tst).cuda(), frame_counts=n))
        res = b.step_signals(torch.from_numpy(smp).cuda(), torch.from_numpy(tst).cuda(), frame_counts=n)
        rb, off = _host(res), res.job_offsets
        for s in set(range(S)) - {2, 5}:
            _rows_equal({kk: v[off[s]:off[s + 1]] for kk, v in rb.items()}, {kk: v[off[s]:off[s + 1]] for kk, v in ra.items()}, (k, s))
        pos += n
    ring_a, ring_b = a.ring_y.cpu().numpy(), b.ring_y.cpu().numpy()
    keep = [s for s in range(S) if s not in (2, 5)]
    assert ring_a[keep].tobytes() == ring_b[keep].tobytes()


def test_ragged_resume_from_state_dict():
    """A ragged run cut at step k, pickled through state_dict() and loaded into a new engine, equals the uninterrupted run;
    a version-1 state (one level count) still loads."""
    cfg = CFGS['butter_ls']
    sched = _schedule(8, steps=14)
    ts, ys = _data(9, int(sched.sum(axis=0).max()) + 1)
    a, b = _engine(S, cfg), _engine(S, cfg)
    pos = np.zeros(S, dtype=np.int64)
    for k, n in enumerate(sched):
        if k == 6:
            state = pickle.loads(pickle.dumps(b.state_dict()))
            assert state['version'] == 2 and np.array_equal(state['counts'], b.counts)
            b = _engine(S, cfg)
            b.load_state_dict(state)
        smp, tst = np.full((S, T, R), np.nan), np.full((S, T), np.nan)
        for s in range(S):
            smp[s, :n[s]], tst[s, :n[s]] = ys[s, pos[s]:pos[s] + n[s]], ts[s, pos[s]:pos[s] + n[s]]
        ra = _host(a.step_signals(torch.from_numpy(smp).cuda(), torch.from_numpy(tst).cuda(), frame_counts=n))
        rb = _host(b.step_signals(torch.from_numpy(smp).cuda(), torch.from_numpy(tst).cuda(), frame_counts=n))
        _rows_equal(rb, ra, k)
        pos += n
    # version 1: what state_dict() wrote before per-stream counts
    c = _engine(S, cfg)
    c.step_signals(torch.from_numpy(ys[:, :T].copy()).cuda(), torch.from_numpy(ts[:, :T].copy()).cuda())
    st = c.state_dict()
    v1 = dict(st, version=1, count=T, mean_count=T)
    del v1['counts'], v1['mean_counts']
    d = _engine(S, cfg)
    d.load_state_dict(v1)
    assert d.count == T and np.array_equal(d.counts, [T] * S)


def test_bad_frame_counts_raise_before_anything_is_enqueued():
    cfg = CFGS['butter_ls']
    eng = _engine(S, cfg)
    ts, ys = _data(10, T)
    smp, tst = torch.from_numpy(ys[:, :T].copy()).cuda(), torch.from_numpy(ts[:, :T].copy()).cuda()
    for bad in ([T] * (S - 1), [-1] + [T] * (S - 1), [T + 1] + [0] * (S - 1), torch.full((S,), T, device='cuda'),
                [0.5] * S):
        with pytest.raises(ValueError):
            eng.step_signals(smp, tst, frame_counts=bad)
    assert eng.count == 0 and eng._turn == 0 and torch.isnan(eng.ring_t).all()
    # J = 0: nothing enqueued, nothing changed
    res = eng.step_signals(smp, tst, frame_counts=np.zeros(S, dtype=np.int32))
    assert res.peak_freq.shape == (0, R) and res.job_stream.numel() == 0 and eng.count == 0 and eng.launches_per_step == 0
    assert torch.isnan(eng.ring_t).all()
    # a CPU tensor is accepted
    res = eng.step_signals(smp, tst, frame_counts=torch.tensor([T, 0, 1, 2, 3, 4, 5]))
    assert np.array_equal(eng.counts, [T, 0, 1, 2, 3, 4, 5]) and res.peak_freq.shape == (20, R)
    with pytest.raises(ValueError):
        eng.count


def test_stream_jobs_scan_at_full_scale():
    """bpv_stream_jobs at 65 536 streams against numpy; a num_jobs that disagrees with the counts writes no job map."""
    from bpv import ops
    rng = np.random.default_rng(11)
    Sx = 65536
    for last_only in (False, True):
        n = rng.integers(0, 9, Sx).astype(np.int32)
        g0 = rng.integers(0, 10 ** 6, Sx).astype(np.int64)
        jobs = (n > 0).astype(np.int64) if last_only else n.astype(np.int64)
        J = int(jobs.sum())
        js = torch.full((J + 5,), -7, dtype=torch.int32, device='cuda')
        jh = torch.full((J + 5,), -7, dtype=torch.int64, device='cuda')
        sj0 = torch.empty(Sx + 1, dtype=torch.int32, device='cuda')
        g1 = torch.full((Sx,), -7, dtype=torch.int64, device='cuda')
        gd, nd = torch.from_numpy(g0).cuda(), torch.from_numpy(n).cuda()
        ops.stream_jobs(gd, nd, last_only, J, js, jh, sj0, g1)
        off = np.concatenate([[0], np.cumsum(jobs)])
        assert np.array_equal(sj0.cpu().numpy(), off)
        stream = np.repeat(np.arange(Sx), jobs)
        head = (g0[stream] + n[stream] - 1) if last_only else np.concatenate([g0[s] + np.arange(n[s]) for s in range(Sx)])
        assert np.array_equal(js.cpu().numpy()[:J], stream) and np.array_equal(jh.cpu().numpy()[:J], head)
        assert (js.cpu().numpy()[J:] == -7).all()
        assert np.array_equal(g1.cpu().numpy(), g0 + n)
        # mismatch: the error status is stream_job0[S] != num_jobs, and nothing else is written
        js.fill_(-7); g1.fill_(-7)
        ops.stream_jobs(gd, nd, last_only, J - 1, js, jh, sj0, g1)
        assert int(sj0[Sx]) == J and (js.cpu().numpy() == -7).all() and (g1.cpu().numpy() == -7).all()
