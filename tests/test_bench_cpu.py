"""CPU: bench.py's argument checks and its --dump-outputs writer (the timed GPU path itself needs a device)."""
import dataclasses
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_steps_must_be_at_least_one():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '0'], capture_output=True, text=True,
                       timeout=120)
    assert r.returncode == 2 and '--steps must be at least 1' in r.stderr, r.stderr[-2000:]


def test_dump_fields_are_step_result_fields():
    import bench
    from bpv.engine import StepResult
    assert set(bench.DUMP_FIELDS) <= {f.name for f in dataclasses.fields(StepResult)}


def test_dump_outputs_writes_every_result_field_as_finite_float64(tmp_path):
    import bench
    from bpv.engine import StepResult
    S, T, R, P = 3, 4, 2, 1
    J = S * T
    g = torch.Generator().manual_seed(0)
    f64 = lambda *shape: torch.randn(*shape, generator=g, dtype=torch.float64)
    i32 = lambda *shape: torch.randint(-300, 300, shape, generator=g, dtype=torch.int32)
    res = StepResult(jobs_per_stream=T, samples=f64(S, T, R), peak_freq=f64(J, R), peak_idx=i32(J, R), peak_mag=f64(J, R),
                     lag_sec=f64(J, P), lag_idx=i32(J, P), lag_corr=f64(J, P), status=i32(J, R))
    res.samples[0, 1, 0] = float('nan')                 # a missed detection
    res.peak_freq[5] = float('nan')                     # a window without a peak
    res.lag_corr[2, 0], res.lag_corr[3, 0] = float('inf'), float('-inf')
    out = tmp_path / 'out'
    bench.dump_outputs(res, str(out))
    floats = [k for k in bench.DUMP_FIELDS if getattr(res, k).is_floating_point()]
    assert floats == ['samples', 'peak_freq', 'peak_mag', 'lag_sec', 'lag_corr']
    assert sorted(os.listdir(out)) == sorted([f'{k}.npy' for k in bench.DUMP_FIELDS] + [f'{k}_nonfinite.npy' for k in floats])
    for f in os.listdir(out):
        a = np.load(out / f)
        assert a.dtype == np.float64 and np.isfinite(a).all(), f
    for k in bench.DUMP_FIELDS:
        want = getattr(res, k).numpy().astype(np.float64)
        got = np.load(out / f'{k}.npy')
        if k in floats:                                 # the value and its code rebuild the output exactly
            code = np.load(out / f'{k}_nonfinite.npy')
            assert np.array_equal(code != 0, ~np.isfinite(want)) and np.all(got[code != 0] == 0), k
            got = np.select([code == 1, code == 2, code == 3], [np.nan, np.inf, -np.inf], got)
        assert np.array_equal(got, want, equal_nan=True), k
    assert np.load(out / 'samples_nonfinite.npy')[0, 1, 0] == 1 and np.load(out / 'samples.npy')[0, 1, 0] == 0
    assert np.load(out / 'lag_corr_nonfinite.npy')[2:4, 0].tolist() == [2.0, 3.0]
