"""GPU: window cadences of the batched engine (window_stride / window_phase).  Every job of a strided engine must equal, bit
for bit, the row with the same stream and head of an 'every_frame' engine fed the same input; with its running means it
must equal a one-stream engine fed the stream's samples in chunks that end at its cadence heads.  The 'every_frame' engine
is pinned to the oracle by tests/test_engine_gpu.py and tests/test_ragged_gpu.py."""
import pickle

import numpy as np
import pytest
import torch

from oracle import bpv_oracle as orc

pytestmark = pytest.mark.gpu

S, R, W, T = 7, 2, 48, 5
CFGS = {
    'fir_welch': dict(methods=[orc.DETREND_LINEAR, orc.FILTER_FIR], transform=orc.PGRAM_WELCH),
    'butter_ls': dict(methods=[orc.FILTER_BUTTER], transform=orc.PGRAM_LS),
    'cubic_dft': dict(methods=[orc.INTERP_CUBIC, orc.FILTER_BUTTER], transform=orc.DFT_RFFT),   # tensor-core DFT
}
FIELDS = ('peak_freq', 'peak_idx', 'peak_mag', 'lag_sec', 'lag_idx', 'lag_corr', 'status')
# uniform k and phase run the lockstep kernels with head_step = k (level steps); the others build the strided job map
CADENCES = {
    'k2': (2, 1), 'k3': (3, 2), 'kT': (T, 0), 'kT+2': (T + 2, 3),
    'per_stream': ([2, 1, 3, 7, 4, 5, 11], [1, 0, 2, 5, 0, 3, 10]),
    'staggered': (4, [s % 4 for s in range(S)]),
}


def _engine(S_, cfg, T_=T, **kw):
    from bpv.engine import BatchedSignalProcessor
    return BatchedSignalProcessor(S_, R, signal_max_samples=W, max_frames_per_step=T_, processing_methods=cfg['methods'],
                                  spectrum_transform=cfg['transform'], peak_max_samples=8, **kw)


def _data(seed, n_total):
    from bpv import synth
    rng = np.random.default_rng(seed)
    ts = np.stack([synth.timestamps(rng, n_total, 30.0 if s % 2 else 60.0, irregular=True, drop=0.03,
                                    origin=rng.uniform(0, 50)) for s in range(S)])
    ys = np.stack([synth.raw_signals(rng, ts[s], R=R, p_nan=0.03) for s in range(S)]).transpose(0, 2, 1)   # [S, n, R]
    return ts, np.ascontiguousarray(ys)


def _schedule(seed, steps=25, level=0):
    """Frame counts per step: `level` lockstep steps (None: every stream takes T), then random counts."""
    rng = np.random.default_rng(seed)
    n = rng.integers(0, T + 1, (steps, S))
    n[3] = 0                      # a step in which no stream takes a frame
    n[7] = T                      # every stream takes T from uneven counts
    n[9:14, 4] = 0
    return [None] * level + list(n)


def _host(res, means=True):
    out = {k: getattr(res, k).cpu().numpy() for k in FIELDS}
    if means:
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


def _cadence(eng):
    k, ph = (np.broadcast_to(np.asarray(v, dtype=np.int64), (eng.S,)) for v in (eng.window_stride, eng.window_phase))
    return k, ph


def _inputs(n, pos, ts, ys):
    """Step inputs [S, T] in which stream s takes its next n[s] samples (n = None: T each)."""
    nn = np.full(S, T) if n is None else n
    smp, tst = np.full((S, T, R), np.nan), np.full((S, T), np.nan)
    for s in range(S):
        smp[s, :nn[s]], tst[s, :nn[s]] = ys[s, pos[s]:pos[s] + nn[s]], ts[s, pos[s]:pos[s] + nn[s]]
    return torch.from_numpy(smp).cuda(), torch.from_numpy(tst).cuda(), nn


def _step_pair(a, b, smp, tst, n, tag):
    """One step of a strided engine `a` and an 'every_frame' engine `b` on the same input: a's rows, layout and every field
    but the running means equal b's rows of the same heads.  Returns a's result and the expected (jobs, heads)."""
    from bpv.engine import cadence_jobs
    c = a.counts
    assert np.array_equal(c, b.counts)
    nn = np.full(S, smp.shape[1]) if n is None else np.asarray(n)
    k, ph = _cadence(a)
    jobs, J, first = cadence_jobs(c, nn.astype(np.int64), k, ph)
    ra = a.step_signals(smp, tst, frame_counts=n)
    rb = b.step_signals(smp, tst, frame_counts=n)
    assert ra.peak_freq.shape[0] == J, tag
    assert np.array_equal(np.diff(ra.job_offsets), jobs), tag
    assert np.array_equal(ra.job_stream.cpu().numpy(), np.repeat(np.arange(S), jobs)), tag
    off_b = rb.job_offsets
    heads = [first[s] + np.arange(jobs[s]) * k[s] for s in range(S)]
    rows = np.concatenate([off_b[s] + (heads[s] - c[s]) for s in range(S)]).astype(np.int64)
    hb = _host(rb, means=False)
    _rows_equal(_host(ra, means=False), {kk: v[rows] for kk, v in hb.items()}, tag)
    assert np.array_equal(a.counts, b.counts)
    return ra, jobs, heads


@pytest.mark.parametrize('cache,overlap', [(True, 3), (False, 0), (True, 4)], ids=['cache-ov3', 'nocache-ov0', 'cache-ov4'])
@pytest.mark.parametrize('cadence', list(CADENCES))
@pytest.mark.parametrize('cfg', list(CFGS))
def test_strided_rows_equal_every_frame_rows(cfg, cadence, cache, overlap):
    """Eight level steps (the lockstep path for a uniform cadence), then random frame counts (the strided job map)."""
    k, ph = CADENCES[cadence]
    sched = _schedule(1, steps=16, level=8)
    ts, ys = _data(2, 8 * T + int(np.sum(sched[8:], axis=0).max()) + 1)
    kw = dict(design_cache=cache, overlap=overlap, store_arrays=overlap == 3)
    a = _engine(S, CFGS[cfg], window_stride=k, window_phase=ph, **kw)
    b = _engine(S, CFGS[cfg], **kw)
    pos = np.zeros(S, dtype=np.int64)
    total = 0
    for i, n in enumerate(sched):
        smp, tst, nn = _inputs(n, pos, ts, ys)
        res, jobs, _ = _step_pair(a, b, smp, tst, n, (i, cadence))
        if n is None and not isinstance(k, list) and not isinstance(ph, list):
            assert res.jobs_per_stream == jobs[0]                # the lockstep path with head_step = k
        total += int(jobs.sum())
        pos += nn
    assert total > 60


@pytest.mark.parametrize('cadence', ['k3', 'per_stream'])
@pytest.mark.parametrize('cfg', list(CFGS))
def test_strided_stream_equals_one_stream_engine_fed_to_its_heads(cfg, cadence):
    """Stream s of a strided engine, running means included, equals its own one-stream windows='last' engine fed the
    stream's samples in chunks that end exactly at its cadence heads."""
    k, ph = CADENCES[cadence]
    kk = np.broadcast_to(np.asarray(k), (S,))
    sched = _schedule(3, steps=18, level=4)
    ts, ys = _data(4, 4 * T + int(np.sum(sched[4:], axis=0).max()) + 1)
    eng = _engine(S, CFGS[cfg], window_stride=k, window_phase=ph, store_arrays=True)
    singles = [_engine(1, CFGS[cfg], T_=int(kk.max()), windows='last', store_arrays=True) for _ in range(S)]
    from bpv.engine import cadence_jobs
    pos = np.zeros(S, dtype=np.int64)
    fed = np.zeros(S, dtype=np.int64)
    checked = 0
    for i, n in enumerate(sched):
        smp, tst, nn = _inputs(n, pos, ts, ys)
        kc, pc = _cadence(eng)
        jobs, _, first = cadence_jobs(eng.counts, nn.astype(np.int64), kc, pc)
        res = eng.step_signals(smp, tst, frame_counts=n)
        got, off = _host(res), res.job_offsets
        for s in range(S):
            for q in range(jobs[s]):
                hd = int(first[s] + q * kc[s])
                ref = singles[s].step_signals(torch.from_numpy(ys[s:s + 1, fed[s]:hd + 1].copy()).cuda(),
                                              torch.from_numpy(ts[s:s + 1, fed[s]:hd + 1].copy()).cuda())
                _rows_equal({kx: v[off[s] + q:off[s] + q + 1] for kx, v in got.items()}, _host(ref), (i, s, q))
                fed[s] = hd + 1
                checked += 1
        pos += nn
    assert checked > 40


FH, FW = 48, 80                   # frame size of the step() tests
RH, RW = 36, 60                   # the frame size the resizing ingest samples from


@pytest.mark.parametrize('path', ['lockstep', 'jobmap'])
def test_zero_job_steps_push_their_frames(path):
    """T = 1 and k = 5: four steps in five have no job, yet sample and push their frames and advance the counts; the fifth
    equals the every-frame row.  The job map gets there through force_jobmap."""
    cfg = CFGS['butter_ls']
    ts, ys = _data(5, 40)
    a = _engine(S, cfg, T_=1, window_stride=5, window_phase=2)
    b = _engine(S, cfg, T_=1)
    a.force_jobmap = path == 'jobmap'
    pos = np.zeros(S, dtype=np.int64)
    for i in range(20):
        smp, tst, nn = _inputs(None, pos, ts, ys)
        smp, tst = smp[:, :1].contiguous(), tst[:, :1].contiguous()
        res, jobs, _ = _step_pair(a, b, smp, tst, None, i)
        assert np.array_equal(a.counts, [i + 1] * S)
        if (i + 1 + 2) % 5:
            assert jobs.sum() == 0 and res.peak_freq.shape == (0, R) and not res.job_offsets.any()
            assert res.samples is not None and torch.equal(res.samples.nan_to_num(), smp.nan_to_num())
            assert a.launches_per_step == (1 if path == 'lockstep' else 2)        # push (+ the job map)
            if path == 'lockstep':
                assert res.jobs_per_stream == 0 and res.job_stream.numel() == 0
        else:
            assert jobs.sum() == S
        pos += 1
    assert torch.equal(a.ring_y.isnan(), b.ring_y.isnan()) and torch.equal(a.ring_y.nan_to_num(), b.ring_y.nan_to_num())


@pytest.mark.parametrize('ingest,stagger', [('plain', False), ('plain', True), ('view', False), ('masked', True),
                                            ('nv12', False), ('resize', True)])
def test_step_with_frames_honours_the_cadence(ingest, stagger):
    """step(frames, boxes, ts): F1, the design-ahead schedule (overlap bit 1) on the lockstep (one phase) and job-map
    (staggered phases) paths, zero-job steps and their launch counts, the cropped-view, masked, NV12 and resizing ingest.
    Rows equal an every-frame engine's."""
    from bpv import synth
    cfg = CFGS['fir_welch']
    nf = 24
    ts, _ = _data(13, nf + 1)
    rng = np.random.default_rng(14)
    frames = np.stack([synth.frames(rng, ts[s], FH, FW, f_pulse=1.0 + 0.2 * s) for s in range(S)])        # [S, nf, FH, FW, 3]
    bh, bw = {'view': (FH, 60), 'resize': (RH, RW)}.get(ingest, (FH, FW))
    boxes = np.stack([synth.roi_boxes(rng, nf, bh, bw, p_none=0.03) for _ in range(S)])
    masks = rng.integers(0, 3, (S, nf, FH, FW), dtype=np.uint8)
    if ingest == 'nv12':
        frames = rng.integers(0, 256, (S, nf, FH * 3 // 2, FW), dtype=np.uint8)           # decoder buffers, pitch = FW
    ph = [s % 2 for s in range(S)] if stagger else 1        # two of the three residues: some steps still have no job
    a = _engine(S, cfg, T_=1, window_stride=3, window_phase=ph, overlap=3, store_arrays=True)
    b = _engine(S, cfg, T_=1, overlap=3, store_arrays=True)
    from bpv.engine import cadence_jobs
    zero = 0
    for i in range(nf):
        sl = slice(i, i + 1)
        fr, bx, tst = (torch.from_numpy(x[:, sl].copy()).cuda() for x in (frames, boxes, ts))
        extra = {}
        if ingest == 'view':
            extra = dict(view=(60, FH, 10, True))
        elif ingest == 'masked':
            extra = dict(masks=torch.from_numpy(masks[:, sl].copy()).cuda(), mask_category=[1, 2])
        elif ingest == 'nv12':
            extra = dict(nv12_size=(FH, FW))
        elif ingest == 'resize':
            extra = dict(resize_to=(RH, RW))
        c = a.counts
        k, p = _cadence(a)
        jobs, J, first = cadence_jobs(c, np.ones(S, dtype=np.int64), k, p)
        ra = a.step(fr, bx, tst, **extra)
        rb = b.step(fr, bx, tst, **extra)
        assert torch.equal(ra.samples.nan_to_num(), rb.samples.nan_to_num())
        assert np.array_equal(np.diff(ra.job_offsets), jobs)
        rows = np.flatnonzero(jobs)                          # T = 1: the every-frame row of stream s is row s
        _rows_equal(_host(ra, means=False), {kk: v[rows] for kk, v in _host(rb, means=False).items()}, i)
        if J == 0:
            zero += 1
            assert a.launches_per_step == 1 + (ingest == 'view') + 1 + (0 if not stagger else 1)   # F1 (+ view) + push (+ map)
    assert np.array_equal(a.counts, [nf] * S) and zero >= nf // 3


def test_changing_settings_reset_and_resume():
    """k / phase reassigned mid-run (uniform -> per stream), reset(streams=[2, 5]) restarts those streams' cadence, and a
    state_dict() taken mid-cycle and loaded into a fresh engine continues the run bit for bit, running means included."""
    cfg = CFGS['fir_welch']
    sched = _schedule(6, steps=24, level=3)
    ts, ys = _data(7, 3 * T + int(np.sum(sched[3:], axis=0).max()) + 1)
    a = _engine(S, cfg, window_stride=3, window_phase=1)
    b = _engine(S, cfg)
    c = None
    pos = np.zeros(S, dtype=np.int64)
    for i, n in enumerate(sched):
        if i == 8:
            a.window_stride, a.window_phase = [2, 3, 4, 5, 6, 7, 8], np.array([1, 2, 3, 4, 5, 6, 7])
        if i == 12:
            a.reset(streams=[2, 5])
            b.reset(streams=[2, 5])
            assert a.counts[2] == a.counts[5] == 0
        if i == 17:
            state = pickle.loads(pickle.dumps(a.state_dict()))
            assert state['version'] == 2
            c = _engine(S, cfg, window_stride=a.window_stride, window_phase=a.window_phase)
            c.load_state_dict(state)
        smp, tst, nn = _inputs(n, pos, ts, ys)
        if c is not None:
            rc = _host(c.step_signals(smp, tst, frame_counts=n))
        ra, _, heads = _step_pair(a, b, smp, tst, n, i)
        if i == 12:
            assert list(heads[2]) == [g for g in range(int(nn[2])) if (g + 1 + 3) % 4 == 0]     # count restarted at 0
        if c is not None:
            _rows_equal(rc, _host(ra), i)
            assert np.array_equal(c.counts, a.counts)
        pos += nn


def test_bad_cadence_raises_before_anything_is_enqueued():
    from bpv.engine import BatchedSignalProcessor
    cfg = CFGS['butter_ls']
    eng = _engine(S, cfg)
    ts, ys = _data(10, T)
    smp, tst = torch.from_numpy(ys[:, :T].copy()).cuda(), torch.from_numpy(ts[:, :T].copy()).cuda()
    bad = [(0, 0), (-2, 0), (2.5, 0), (2, 0.5), ([2] * (S - 1), 0), (2, [0] * (S + 1)), (3, 3), (3, -1), ([3] * S, [0, 1, 2, 3, 0, 1, 2]),
           (torch.full((S,), 2, dtype=torch.int32, device='cuda'), 0), (2, torch.zeros(S, dtype=torch.int32, device='cuda')),
           ('2', 0), (2 ** 31, 0)]
    for k, ph in bad:
        eng.window_stride, eng.window_phase = k, ph
        with pytest.raises(ValueError):
            eng.step_signals(smp, tst)
        with pytest.raises(ValueError):
            eng.step_signals(smp, tst, frame_counts=[T, 1, 0, 2, 3, 4, 5])
    assert eng.count == 0 and eng._turn == 0 and torch.isnan(eng.ring_t).all()
    # a stride needs windows='every_frame'
    with pytest.raises(ValueError):
        BatchedSignalProcessor(S, R, signal_max_samples=W, max_frames_per_step=T, windows='last', window_stride=2)
    last = _engine(S, cfg, windows='last')
    last.window_stride = 4
    with pytest.raises(ValueError):
        last.step_signals(smp, tst)
    assert last.count == 0 and torch.isnan(last.ring_t).all()
    # valid forms: a CPU tensor, numpy arrays, integral floats; the counts move only now
    eng.window_stride, eng.window_phase = torch.tensor([2] * S), np.arange(S) % 2
    eng.step_signals(smp, tst)
    eng.window_stride, eng.window_phase = 3.0, 0
    eng.step_signals(smp, tst)
    assert eng.count == 2 * T


def test_stream_jobs_strided_scan_at_full_scale():
    """bpv_stream_jobs_strided at 65 536 streams against the host planning; out-of-range strides / phases read as documented
    (a stride below 1 as 1, a phase modulo the stride); a num_jobs that disagrees with the counts writes no job map."""
    from bpv import ops
    from bpv.engine import cadence_jobs
    rng = np.random.default_rng(11)
    Sx = 65536
    n = rng.integers(0, 9, Sx).astype(np.int32)
    g0 = rng.integers(0, 10 ** 6, Sx).astype(np.int64)
    g0[:1000] += 2 ** 45                                     # long-running streams
    k = rng.integers(1, 70, Sx).astype(np.int32)
    ph = (rng.integers(0, 2 ** 30, Sx) % k).astype(np.int32)
    k[5:9], ph[9:13] = [0, -3, 0, -2 ** 31], [-1, 70, -2 ** 31, 2 ** 31 - 1]
    kh = np.maximum(k.astype(np.int64), 1)
    phh = ph.astype(np.int64) % kh                           # Python / numpy modulo: in [0, k)
    for stride, phase in ((k, ph), (None, None)):
        ke, pe = (kh, phh) if stride is not None else (np.ones(Sx, np.int64), np.zeros(Sx, np.int64))
        jobs, J, first = cadence_jobs(g0, n.astype(np.int64), ke, pe)
        js = torch.full((J + 5,), -7, dtype=torch.int32, device='cuda')
        jh = torch.full((J + 5,), -7, dtype=torch.int64, device='cuda')
        sj0 = torch.empty(Sx + 1, dtype=torch.int32, device='cuda')
        g1 = torch.full((Sx,), -7, dtype=torch.int64, device='cuda')
        gd, nd = torch.from_numpy(g0).cuda(), torch.from_numpy(n).cuda()
        kd = None if stride is None else torch.from_numpy(stride).cuda()
        pd = None if phase is None else torch.from_numpy(phase).cuda()
        ops.stream_jobs_strided(gd, nd, kd, pd, J, js, jh, sj0, g1)
        off = np.concatenate([[0], np.cumsum(jobs)])
        assert np.array_equal(sj0.cpu().numpy(), off)
        stream = np.repeat(np.arange(Sx), jobs)
        head = first[stream] + (np.arange(J) - off[stream]) * ke[stream]
        assert np.array_equal(js.cpu().numpy()[:J], stream) and np.array_equal(jh.cpu().numpy()[:J], head)
        assert (js.cpu().numpy()[J:] == -7).all() and (jh.cpu().numpy()[J:] == -7).all()
        assert np.array_equal(g1.cpu().numpy(), g0 + n)
        # mismatch: stream_job0[S] reports the device's sum, nothing else is written
        js.fill_(-7); jh.fill_(-7); g1.fill_(-7)
        ops.stream_jobs_strided(gd, nd, kd, pd, J + 1, js, jh, sj0, g1)
        assert int(sj0[Sx]) == J and (js.cpu().numpy() == -7).all() and (jh.cpu().numpy() == -7).all()
        assert (g1.cpu().numpy() == -7).all()


def _kernels(fn):
    """Number of kernels a call enqueues, by a torch.profiler trace (copies and fills are not launches)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(e.count for e in prof.key_averages()
               if e.device_type.name == 'CUDA' and not e.key.startswith(('Memcpy', 'Memset')))


@pytest.mark.parametrize('cfg', ['butter_ls', 'fir_welch'])
def test_launches_per_step_match_a_trace(cfg):
    """launches_per_step of a lockstep strided step, a job-map strided step and zero-job steps on both paths (step_signals
    and step with frames) equals the kernels a torch.profiler trace of that step shows."""
    from bpv import synth
    ts, ys = _data(15, 60)
    rng = np.random.default_rng(16)
    frames = np.stack([synth.frames(rng, ts[s, :8], FH, FW) for s in range(S)])
    boxes = np.stack([synth.roi_boxes(rng, 8, FH, FW) for _ in range(S)])
    lock = _engine(S, CFGS[cfg], window_stride=2, window_phase=1)
    jmap = _engine(S, CFGS[cfg], window_stride=[2, 3, 1, 4, 2, 5, 3], window_phase=[0, 1, 0, 2, 1, 4, 0])
    zero = _engine(S, CFGS[cfg], T_=1, window_stride=6)
    zmap = _engine(S, CFGS[cfg], T_=1, window_stride=6, window_phase=[0, 0, 0, 0, 0, 0, 1])
    pos = np.zeros(S, dtype=np.int64)
    for i in range(3):
        smp, tst, nn = _inputs(None, pos, ts, ys)
        for eng in (lock, jmap):
            eng.step_signals(smp, tst)                          # warm-up: pinned staging, side streams, design cache
            got = _kernels(lambda: eng.step_signals(smp, tst))
            assert got == eng.launches_per_step and got > 4, (cfg, i, got, eng.launches_per_step)
        pos += nn
    assert lock.step_signals(smp, tst).jobs_per_stream is not None
    assert jmap.step_signals(smp, tst).jobs_per_stream is None
    for eng, want in ((zero, 2), (zmap, 3)):                    # F1 + push (+ the job map)
        for i in range(4):                                      # counts 0 .. 3: no stream reaches a cadence point
            fr, bx = torch.from_numpy(frames[:, i:i + 1].copy()).cuda(), torch.from_numpy(boxes[:, i:i + 1].copy()).cuda()
            tst = torch.from_numpy(ts[:, i:i + 1].copy()).cuda()
            res = None

            def run():
                nonlocal res
                res = eng.step(fr, bx, tst)
            got = _kernels(run)
            assert res.peak_freq.shape[0] == 0 and got == eng.launches_per_step == want, (cfg, i, got, eng.launches_per_step)
