"""CPU: the host planning of window cadences (engine.cadence_jobs) against a brute-force walk over the samples, and the
argument checks of bpv_stream_jobs_strided (include/bpv.h) — every case returns before the first CUDA call."""
import ctypes as C

import numpy as np
import pytest

from bpv import _cabi


@pytest.fixture(scope='module')
def lib():
    from bpv import build
    build.build()
    return _cabi.lib()


def _brute(c, n, k, ph):
    """Heads of the windows a stream evaluates while its count goes from c to c + n: after its m-th sample (global index
    m - 1) exactly when (m + ph) % k == 0."""
    return [m - 1 for m in range(c + 1, c + n + 1) if (m + ph) % k == 0]


@pytest.mark.parametrize('huge', [False, True])
def test_cadence_jobs_matches_brute_force(huge):
    from bpv.engine import cadence_jobs
    rng = np.random.default_rng(3 + huge)
    S = 400
    base = 2 ** 52 if huge else 0
    c = base + rng.integers(0, 10 ** 4, S)
    n = rng.integers(0, 70, S)
    k = rng.choice([1, 2, 3, 7, 15, 30, 60, 64, 65, 100], S)
    ph = (rng.integers(0, 2 ** 20, S) % k)
    c[:3], n[:3], k[:3], ph[:3] = base, 0, 5, 4                       # nothing taken: no job
    jobs, J, first = cadence_jobs(c.astype(np.int64), n.astype(np.int64), k.astype(np.int64), ph.astype(np.int64))
    assert J == int(jobs.sum())
    for s in range(S):
        heads = _brute(int(c[s]), int(n[s]), int(k[s]), int(ph[s]))
        assert jobs[s] == len(heads), s
        assert heads == [int(first[s]) + i * int(k[s]) for i in range(len(heads))], s


def test_cadence_jobs_on_scalars_and_the_default_cadence():
    from bpv.engine import cadence_jobs
    # k = 1, phase 0: a job after every frame, heads c .. c + n - 1
    assert cadence_jobs(17, 5, 1, 0) == (5, 5, 17)
    # k = 5, T = 1: one step in five has a job, and a stream's phase picks which
    seq = [cadence_jobs(c, 1, 5, 2)[0] for c in range(10)]
    assert seq == [0, 0, 1, 0, 0, 0, 0, 1, 0, 0] and cadence_jobs(2, 1, 5, 2)[2] == 2
    # the phase carries across steps of any size: the union of the heads of split steps is the heads of one step
    for k, ph in ((4, 1), (7, 6), (3, 0)):
        heads, c = [], 11
        for n in (1, 5, 0, 9, 2, 13):
            q, _, h0 = cadence_jobs(c, n, k, ph)
            heads += [h0 + i * k for i in range(q)]
            c += n
        assert heads == _brute(11, c - 11, k, ph)


def test_stream_jobs_strided_rejects_bad_arguments(lib):
    a = C.cast((C.c_uint8 * 64)(), C.c_void_p)
    f = lib.bpv_stream_jobs_strided
    assert f(0, a, a, a, a, 0, a, a, a, a, None) == -1                       # no streams
    assert f(65537, a, a, a, a, 0, a, a, a, a, None) == -1                   # more than one launch serves
    assert f(4, a, a, a, a, -1, a, a, a, a, None) == -1                      # negative num_jobs
    assert f(4, a, a, a, a, 2 ** 31, a, a, a, a, None) == -1
    assert f(4, a, a, a, a, 3, None, a, a, a, None) == -1                    # jobs without a map
    assert f(4, a, a, a, a, 3, a, None, a, a, None) == -1
    assert f(4, None, a, a, a, 0, a, a, a, a, None) == -1                    # no counts
    assert f(4, a, None, a, a, 0, a, a, a, a, None) == -1
    assert f(4, a, a, a, a, 0, a, a, None, a, None) == -1                    # no offsets
    assert f(4, a, a, a, a, 0, a, a, a, None, None) == -1                    # no advanced counts
    assert b'bpv_stream_jobs_strided' in lib.bpv_last_error()
