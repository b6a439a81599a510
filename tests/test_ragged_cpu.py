"""CPU: argument checks of the ragged-step C entry points (include/bpv.h) — every case returns before the first CUDA call —
and the host side of the job-map params."""
import ctypes as C

import pytest

from bpv import _cabi, ops


@pytest.fixture(scope='module')
def lib():
    from bpv import build
    build.build()
    return _cabi.lib()


def _params(S=2, methods=(_cabi.FILTER_FIR,)):
    return ops.make_params(S, 2, 33, 32, 31, 1, 1, list(methods), _cabi.PGRAM_LS)


def test_ring_push_ragged_rejects_bad_arguments(lib):
    a = C.cast((C.c_uint8 * 64)(), C.c_void_p)
    assert lib.bpv_ring_push_ragged(a, a, 2, 2, 33, None, a, 4, a, a, None) == -1          # no counts
    assert lib.bpv_ring_push_ragged(a, a, 2, 2, 33, a, None, 4, a, a, None) == -1
    assert lib.bpv_ring_push_ragged(a, a, 2, 2, 33, a, a, 4, None, None, None) == -1         # nothing to push
    assert b'bpv_ring_push_ragged' in lib.bpv_last_error()
    assert lib.bpv_ring_push_ragged(a, a, 0, 2, 33, a, a, 4, a, a, None) == -1
    assert lib.bpv_ring_push_ragged(a, a, 2, 2, 33, a, a, 34, a, a, None) == -1              # T > cap


def test_stream_jobs_rejects_bad_sizes(lib):
    a = C.cast((C.c_uint8 * 64)(), C.c_void_p)
    assert lib.bpv_stream_jobs(0, a, a, 0, 0, a, a, a, a, None) == -1
    assert lib.bpv_stream_jobs(65537, a, a, 0, 0, a, a, a, a, None) == -1
    assert lib.bpv_stream_jobs(4, a, a, 0, -1, a, a, a, a, None) == -1
    assert lib.bpv_stream_jobs(4, a, a, 0, 2 ** 31, a, a, a, a, None) == -1
    assert lib.bpv_stream_jobs(4, a, a, 0, 3, None, a, a, a, None) == -1                      # jobs without a map
    assert lib.bpv_stream_jobs(4, None, a, 0, 0, a, a, a, a, None) == -1
    assert b'bpv_stream_jobs' in lib.bpv_last_error()


def test_window_jobs_entry_points_reject_bad_arguments(lib):
    a = C.cast((C.c_uint8 * 4096)(), C.c_void_p)
    p = _params()
    design = lambda q, js, jh, nj, ws=None, nb=0: lib.bpv_window_design_jobs(a, C.byref(q), ws, nb, None, 0, js, jh, nj, None)
    filt = lambda q, js, jh, nj, ws=None, nb=0: lib.bpv_window_filter_jobs(a, a, C.byref(q), ws, nb, None, 0, a, a, a, js, jh, nj, None)
    pre = lambda q, js, jh, nj: lib.bpv_window_preprocess_jobs(a, a, C.byref(q), None, 0, a, a, a, js, jh, nj, None)
    for call in (design, filt, pre):
        assert call(p, a, a, -1) == -1                               # negative job count
        assert call(p, None, a, 3) == -1                             # no job map
        assert call(p, a, None, 3) == -1
        assert call(p, None, None, 0) == 0                           # nothing to do
    assert b'job map' in lib.bpv_last_error()
    assert design(_params(S=0), a, a, 3) == -1                       # rings of no stream
    # the workspace holds the designs of num_jobs jobs: bpv_window_workspace_bytes of params with S * jobs_per_stream >= num_jobs
    need3 = lib.bpv_window_workspace_bytes(C.byref(_params(S=3)))
    assert need3 > lib.bpv_window_workspace_bytes(C.byref(_params(S=2)))
    assert design(p, a, a, 3, a, need3 - 1) == -1 and b'workspace' in lib.bpv_last_error()
    assert filt(p, a, a, 3, a, need3 - 1) == -1 and b'workspace' in lib.bpv_last_error()
    q = _params(); q.fir_taps = 128
    assert filt(q, a, a, 3) == -3


def test_running_mean_jobs_rejects_bad_arguments(lib):
    a = C.cast((C.c_uint8 * 64)(), C.c_void_p)
    assert lib.bpv_running_mean_jobs(a, 2, 2, 129, a, a, a, 60.0, a, a, None) == -1         # history > 128
    assert lib.bpv_running_mean_jobs(a, 2, 2, 8, None, a, a, 60.0, a, a, None) == -1
    assert lib.bpv_running_mean_jobs(a, 2, 2, 8, a, None, a, 60.0, a, a, None) == -1
    assert lib.bpv_running_mean_jobs(a, 2, 2, 8, a, a, a, 60.0, None, None, None) == -1
    assert lib.bpv_running_mean_jobs(a, 0, 2, 8, a, a, a, 60.0, a, a, None) == -1


def test_jobs_params_describe_the_job_list():
    p = ops.make_params(7, 2, 53, 48, 100, 1, 5, [_cabi.FILTER_BUTTER], _cabi.PGRAM_LS)
    q = ops.jobs_params(p, 23)
    assert (q.S, q.jobs_per_stream, q.head0, q.head_step) == (23, 1, 0, 0)
    assert (q.R, q.cap, q.window, q.num_methods, q.methods[0]) == (2, 53, 48, 1, _cabi.FILTER_BUTTER)
    assert (p.S, p.jobs_per_stream, p.head0) == (7, 5, 100)          # the ring params are left alone
