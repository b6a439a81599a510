"""CPU: the host planning of a batched-engine step (engine.plan_jobs): which steps run lockstep and which build a job map,
and the jobs, heads and offsets of each, against a brute-force walk over every stream's samples."""
import numpy as np
import pytest

S, T = 6, 5


def _heads(c, n, k, ph, last=False):
    """Newest-sample indices of the windows stream s evaluates while its count goes from c to c + n."""
    if last:
        return [c + n - 1] if n else []
    return [m - 1 for m in range(c + 1, c + n + 1) if (m + ph) % k == 0]


def _check(plan, counts, n, k, ph, last=False):
    """Jobs, heads and job_offsets of a plan equal the brute-force walk, on either path."""
    c = np.broadcast_to(np.asarray(counts, dtype=np.int64), (S,))
    nn = np.full(S, T) if n is None else n
    kk, pp = (np.ones(S, np.int64), np.zeros(S, np.int64)) if k is None else (k, ph)
    heads = [_heads(int(c[s]), int(nn[s]), int(kk[s]), int(pp[s]), last) for s in range(S)]
    assert plan.T == T and plan.J == sum(map(len, heads))
    if plan.lock:
        assert isinstance(plan.jobs, int) and plan.n is None and plan.off is None
        for h in heads:
            assert h == [plan.head0 + i * plan.head_step for i in range(plan.jobs)]
    else:
        assert np.array_equal(plan.n, nn) and np.array_equal(plan.jobs, [len(h) for h in heads])
        assert np.array_equal(plan.off, np.concatenate([[0], np.cumsum([len(h) for h in heads])]))


LEVEL, RAGGED = None, np.array([T, 0, 3, T, 1, 2], dtype=np.int64)
UNIFORM = (np.full(S, 3, np.int64), np.full(S, 1, np.int64))
PER_STREAM = (np.array([2, 3, 1, 4, 2, 7], np.int64), np.array([1, 0, 0, 3, 0, 6], np.int64))
CASES = {   # (counts, mean counts, frames, cadence, last, force_jobmap) -> lockstep?
    'level': (9, 4, LEVEL, None, False, False, True),
    'level_as_array': (9, 4, np.full(S, T, np.int64), None, False, False, True),
    'ragged': (9, 4, RAGGED, None, False, False, False),
    'uneven_counts': (np.arange(S, dtype=np.int64), 0, LEVEL, None, False, False, False),
    'uneven_mean_counts': (9, np.arange(S, dtype=np.int64), LEVEL, None, False, False, False),
    'forced': (9, 4, LEVEL, None, False, True, False),
    'last': (9, 4, LEVEL, None, True, False, True),
    'last_ragged': (9, 4, RAGGED, None, True, False, False),
    'uniform_cadence': (9, 4, LEVEL, UNIFORM, False, False, True),
    'uniform_cadence_ragged': (9, 4, RAGGED, UNIFORM, False, False, False),
    'uniform_cadence_forced': (9, 4, LEVEL, UNIFORM, False, True, False),
    'per_stream_cadence': (9, 4, LEVEL, PER_STREAM, False, False, False),
    'per_stream_cadence_ragged': (np.arange(S, dtype=np.int64) * 7, 4, RAGGED, PER_STREAM, False, False, False),
}


@pytest.mark.parametrize('case', list(CASES))
def test_plan_jobs_decision_table(case):
    from bpv.engine import plan_jobs
    counts, mcounts, n, cad, last, force, lock = CASES[case]
    k, ph = cad if cad is not None else (None, None)
    plan = plan_jobs(S, counts, mcounts, n, T, cad, last=last, force_jobmap=force)
    assert plan.lock == lock, case
    _check(plan, counts, n, k, ph, last)


@pytest.mark.parametrize('force', [False, True])
def test_zero_job_strided_steps(force):
    """k = 20 > T: a step pushes its frames without reaching a cadence point; J = 0 on both paths, and the step after
    the point is reached has one job per stream."""
    from bpv.engine import plan_jobs
    k, ph = np.full(S, 20, np.int64), np.full(S, 4, np.int64)
    for c, want in ((0, 0), (5, 0), (15, S), (20, 0)):
        plan = plan_jobs(S, c, 0, None, T, (k, ph), force_jobmap=force)
        assert plan.lock == (not force) and plan.J == want, (c, force)
        _check(plan, c, None, k, ph)
        if plan.lock:
            assert plan.jobs == want // S
        else:
            assert int(plan.jobs.sum()) == want


@pytest.mark.parametrize('cad', [None, PER_STREAM], ids=['default', 'per_stream'])
def test_a_step_without_frames_has_no_plan(cad):
    """A step in which no stream takes a frame has no plan, whatever the counts and cadence: it enqueues nothing."""
    from bpv.engine import plan_jobs
    for counts in (9, np.arange(S, dtype=np.int64)):
        for force in (False, True):
            assert plan_jobs(S, counts, 4, np.zeros(S, np.int64), T, cad, force_jobmap=force) is None
    assert plan_jobs(S, 9, 4, np.array([0, 0, 0, 1, 0, 0]), T, cad) is not None
