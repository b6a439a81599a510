"""CPU: host-side logic of the drop-in modules (no compute calls into the CUDA library) and the C-ABI surface."""
import importlib.util
import os
import pickle
import re
import sys

import numpy as np
import pytest

from oracle import bpv_oracle as orc
from tests import helpers as h

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = h.REFERENCE


def test_cabi_exports_every_declared_symbol():
    """libbpv.so loads and exports exactly the entry points include/bpv.h declares."""
    from bpv import _cabi, build
    build.build()
    hdr = open(os.path.join(ROOT, 'include', 'bpv.h')).read()
    hdr = re.sub(r'/\*.*?\*/', '', hdr, flags=re.S)
    declared = set(re.findall(r'\b(bpv_[a-z0-9_]+)\s*\(', hdr))
    assert len(declared) >= 12
    lib = _cabi.lib()
    for name in declared:
        assert hasattr(lib, name), f'{name} declared in bpv.h but not exported'
    assert declared == set(_cabi.EXPORTS), declared ^ set(_cabi.EXPORTS)
    assert lib.bpv_version() == 100
    import ctypes
    assert ctypes.sizeof(_cabi.WindowParams) == lib.bpv_sizeof_window_params() == 120


def test_ctypes_signatures_follow_the_header():
    """Every prototype of include/bpv.h and its ctypes binding agree on the number of arguments and on which of them
    are pointers / 64-bit / 32-bit / double (a mismatch would corrupt the call silently)."""
    import ctypes
    from bpv import _cabi
    hdr = open(os.path.join(ROOT, 'include', 'bpv.h')).read()
    hdr = re.sub(r'/\*.*?\*/', '', hdr, flags=re.S)
    protos = re.findall(r'\b([a-z_0-9]+(?:\s*\*)?)\s*\b(bpv_[a-z0-9_]+)\s*\(([^)]*)\)\s*;', hdr)
    assert {n for _, n, _ in protos} == set(_cabi.EXPORTS)

    def kind(decl):
        decl = decl.strip()
        if '*' in decl:
            return 'p'
        base = decl.rsplit(' ', 1)[0] if ' ' in decl else decl
        return {'int64_t': 'q', 'int32_t': 'i', 'int': 'i', 'double': 'd'}[base.replace('const', '').strip()]

    ckind = {ctypes.c_void_p: 'p', ctypes.c_char_p: 'p', ctypes.c_int64: 'q', ctypes.c_int32: 'i', ctypes.c_int: 'i',
             ctypes.c_double: 'd'}
    for _, name, args in protos:
        want = [] if args.strip() in ('', 'void') else [kind(a) for a in args.split(',')]
        _, bound = _cabi._SIGS[name]
        got = ['p' if (isinstance(t, type) and issubclass(t, ctypes._Pointer)) else ckind[t] for t in bound]
        assert got == want, (name, got, want)


def test_no_cpu_fallback_without_library(monkeypatch):
    from bpv import _cabi
    monkeypatch.setattr(_cabi, '_lib', None)
    monkeypatch.setattr(_cabi, 'LIB_PATH', '/nonexistent/libbpv.so')
    with pytest.raises(_cabi.BpvError):
        _cabi.lib()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, 'bp-from-video_b200')
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh')):
                src = open(os.path.join(dp, f)).read()
                assert 'oracle' not in src.replace('bpv_oracle', 'oracle') or f == 'nothing', (dp, f)
                assert '/root/reference' not in src, (dp, f)


def test_roi_module_surface():
    import model
    import roi
    assert [c.landmark_indices for c in roi.SELECTED_ROI_CONFIGS] == [[151], [0, 9]]
    assert roi.FACE_FOREHEAD_CONFIG.relative_bbox == (-0.00, -0.10, 0.20, 0.05)
    assert roi.HAND_PALM_CONFIG.relative_bbox == (-0.10, -0.10, 0.10, 0.10)
    assert roi.FACE_CHEEK_CONFIG.model_type is model.ModelType.FACE_LANDMARKER
    assert roi.HAND_WRIST_CONFIG.model_type is model.ModelType.HAND_LANDMARKER and roi.HAND_WRIST_CONFIG.landmark_indices == [0]
    assert roi.FACE_EYEBROW_CONFIG.relative_bbox == (-0.10, -0.15, 0.25, 0.00)
    assert model.ModelType.FACE_LANDMARKER == 'face_landmarker'


def test_signal_basic_semantics():
    import signal_data as sd
    s = sd.Signal(s_maxlen=4)
    assert len(s.x) == 4 and np.isnan(s.x).all() and not s.v.any() and np.isnan(s.range_x).all()
    for t, y in [(0.0, 1.0), (0.1, np.nan), (0.2, 5.0), (0.3, 2.0), (0.4, 5.0)]:
        s.add_sample(t, y)
    assert np.allclose(s.x, [0.1, 0.2, 0.3, 0.4]) and s.w.tolist() == [False, True, True, True]
    assert s.range_y == (2.0, 5.0) and np.isclose(s.get_fs(), 10.0)
    assert s.get_peak() == (0.2, 5.0)                      # first maximum wins
    assert np.isclose(s.get_mean(), 4.0) and s.get_mean(as_int=True) == 4
    e = sd.Signal([], [], s_maxlen=0)
    assert e.get_peak() == (np.nan, np.nan) or all(np.isnan(v) for v in e.get_peak())
    r = sd.Signal(yi=(np.nan,) * 6, s_maxlen=2)
    assert r.y.shape == (2, 6) and np.isnan(r.get_mean(as_int=True)).all()
    r.add_sample(1.0, (10, 21, 1, 2, 3, 4))
    r.add_sample(2.0, (11, 22, 2, 3, 4, 5))
    assert r.get_mean(as_int=True).tolist() == [10, 22, 2, 2, 4, 4]      # half-to-even: 10.5->10, 21.5->22
    g = sd.SignalGroup(2, s_maxlen=3)
    g.add_samples(1.0, [1.0, 2.0])
    g.add_samples(2.0, [3.0, np.nan])
    assert g.range_y == (1.0, 3.0) and [len(s.x) for s in g] == [3, 3]
    pickle.loads(pickle.dumps(g))


def _load_ref(name):
    spec = importlib.util.spec_from_file_location(f'ref_{name}', os.path.join(REF, f'{name}.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _eq(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return a.shape == b.shape and np.array_equal(a, b, equal_nan=True)


@pytest.mark.skipif(not os.path.isdir(REF), reason=h.NO_REFERENCE)
def test_signal_data_differential_vs_reference():
    """Random operation sequences on our Signal/SignalGroup and the reference's must agree on everything."""
    import warnings
    warnings.simplefilter('ignore')
    import signal_data as ours
    ref = _load_ref('signal_data')
    rng = np.random.default_rng(0)
    for trial in range(80):
        maxlen = int(rng.integers(1, 7))
        vec = trial % 3 == 0
        yi = (np.nan,) * 6 if vec else np.nan
        a, b = ours.SignalGroup(2, yi=yi, s_maxlen=maxlen), ref.SignalGroup(2, yi=yi, s_maxlen=maxlen)
        for step in range(12):
            t = float(step) * 0.1 if rng.uniform() > 0.1 else np.nan
            ys = []
            for _ in range(2):
                if rng.uniform() < 0.25:
                    ys.append((np.nan,) * 6 if vec else np.nan)
                elif not vec and rng.uniform() < 0.08:
                    ys.append(float(rng.choice([np.inf, -np.inf])))      # non-finite but not NaN: masked out, yet seen by the ranges
                else:
                    ys.append(tuple(int(v) for v in rng.integers(0, 50, 6)) if vec else float(rng.integers(0, 5)))
            a.add_samples(t, ys)
            b.add_samples(t, ys)
            assert _eq(a.range_x, b.range_x) and _eq(a.range_y, b.range_y)
            for sa, sb in zip(a, b):
                assert _eq(sa.x, np.array(sb.x)) and _eq(sa.y, np.array(sb.y)) and _eq(sa.v, sb.v) and _eq(sa.w, sb.w)
                assert _eq(sa.range_x, sb.range_x) and _eq(sa.range_y, sb.range_y)
                assert _eq(sa.get_fs(), sb.get_fs()) and _eq(sa.get_fs(True), sb.get_fs(True)) if not vec else True
                assert _eq(sa.get_mean(), sb.get_mean()) and _eq(sa.get_mean(True), sb.get_mean(True))
                if not vec:
                    pa, pb = sa.get_peak(), sb.get_peak()
                    assert _eq(pa[0], pb[0]) and _eq(pa[1], pb[1])
                    pa, pb = sa.get_peak(0.2, 0.9), sb.get_peak(0.2, 0.9)
                    assert _eq(pa[0], pb[0]) and _eq(pa[1], pb[1])
            assert all(_eq(x, y) for x, y in zip(a.get_means(True), b.get_means(True)))
    # list construction + range clobbering behaviour (SURVEY 8a "range clobbering")
    xs, ys = [0.5, 1.0, 2.0, 3.0], [0.1, 0.9, np.nan, 0.4]
    sa, sb = ours.Signal(xs, ys, s_maxlen=4), ref.Signal(xs, ys, s_maxlen=4)
    sa.set_range((0.8, 4.0), (0, 1)); sb.set_range((0.8, 4.0), (0, 1))
    assert sa.get_peak() == sb.get_peak()
    ga, gb = ours.SignalGroup(signals=[sa]), ref.SignalGroup(signals=[sb])
    assert sa.range_x == sb.range_x == (0.5, 3.0) and ga.range_x == gb.range_x


def test_calc_rois_matches_reference_rounding():
    """calc_rois is host logic: anchors and corners incl. half-to-even rounding and missing detections."""
    import signal_processor as sp
    proc = sp.SignalProcessor()

    class Out:
        def __init__(self, d): self.detections = d

    class Res:
        def __init__(self, f, hd): self.face_landmarker, self.hand_landmarker = Out(f), Out(hd)
    for name in ('c1_butter_ls', 'lin_const_fir_dft'):
        g = h.load_case(name)
        for i in range(len(g['ts'])):
            face, hand = [], []
            if g['present'][i, 0]:
                pts = np.zeros((478, 2), np.int64); pts[151] = g['face_pt'][i]
                face = [(tuple(int(v) for v in g['face_bbox'][i]), pts)]
            if g['present'][i, 1]:
                pts = np.zeros((21, 2), np.int64); pts[0], pts[9] = g['hand_pts'][i, 0], g['hand_pts'][i, 1]
                hand = [(tuple(int(v) for v in g['hand_bbox'][i]), pts)]
            got = proc.calc_rois(Res(face, hand))
            exp = h.case_rois(g, i)
            for a, b in zip(got, exp):
                assert _eq(a, b), (name, i, a, b)

    class Bad:
        model_type, landmark_indices, relative_bbox = 'person_segmenter', [0], (0, 0, 1, 1)
    with pytest.raises(NotImplementedError):
        sp.SignalProcessor([Bad()]).calc_rois(Res([], []))


def test_signal_processor_surface_matches_reference_signature():
    import inspect
    import signal_processor as sp
    sig = inspect.signature(sp.SignalProcessor.__init__)
    names = list(sig.parameters)
    assert names[:5] == ['self', 'selected_roi_configs', 'roi_max_samples', 'signal_max_samples', 'peak_max_samples']
    for kw, default in dict(butter_order=16, butter_min_bw=0.1, fir_taps=127, fir_df=0.3, min_freq=0.8, max_freq=4.0,
                            min_mag=0.0, max_mag=1.0, min_lag=-0.5, max_lag=0.5, min_corr=-1.0, max_corr=1.0).items():
        assert sig.parameters[kw].default == default and sig.parameters[kw].kind is inspect.Parameter.KEYWORD_ONLY
    for m in ('calc_rois', 'make_filter', 'sample_signal', 'sample_signals', 'process_signal', 'process_signals',
              'transform_signal', 'transform_signals', 'correlate_signal_pair', 'correlate_signals', 'process', 'run', 'cleanup'):
        assert callable(getattr(sp.SignalProcessor, m))
    assert [m.name for m in sp.SignalProcessingMethod] == ['DIFF_1', 'DIFF_2', 'INTERP_LINEAR', 'INTERP_CUBIC', 'DETREND_CONST',
                                                          'DETREND_LINEAR', 'FILTER_BUTTER', 'FILTER_FIR']
    assert [m.value for m in sp.SignalSpectrumTransform] == [orc.DFT_RFFT, orc.PGRAM_WELCH, orc.PGRAM_LS]
    st = sp.SignalStore(2, 1, 250, 50)
    assert [len(s.x) for s in st.sg_raw] == [250, 250] and st.sg_corr.num_signals == 1 and st.sg_roi.signals[0].y.shape == (1, 6)
    pickle.loads(pickle.dumps(st.snapshot()))


@pytest.mark.skipif(not os.path.isdir(REF), reason=h.NO_REFERENCE)
def test_reference_modules_import_on_top_of_the_drop_in():
    """PYTHONPATH=<ours>:<reference>: the reference's own video_reader must import against OUR profiler/exceptions,
    and `signal_processor` / `roi` / `signal_data` must resolve to the drop-in (INTEGRATION.md §1)."""
    import subprocess
    code = ("import sys, video_reader, signal_processor, roi, signal_data, profiler, exceptions;"
            "assert 'bp-from-video_b200' in signal_processor.__file__ and 'bp-from-video_b200' in roi.__file__;"
            f"assert 'bp-from-video_b200' in profiler.__file__ and video_reader.__file__.startswith({REF!r});"
            "assert issubclass(exceptions.CaptureError, RuntimeError);"
            "p = signal_processor.SignalProcessor(); assert p.num_signals == 2 and p.store.sg_corr.num_signals == 1;"
            "print('ok')")
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, 'bp-from-video_b200') + ':' + REF)
    r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, env=env, timeout=120)
    assert r.returncode == 0 and 'ok' in r.stdout, r.stderr[-2000:]


def test_cabi_rejects_bad_arguments_before_touching_the_gpu():
    """Argument validation of the C ABI (include/bpv.h error codes): every case below returns before the first CUDA call,
    so it runs without a GPU.  -1 = BPV_E_INVALID, -2 = BPV_E_UNSUPPORTED (the reference's NotImplementedError,
    signal_processor.py:185/238/262), -3 = BPV_E_TOO_LARGE; bpv_last_error() names the entry point."""
    import ctypes as C
    from bpv import _cabi, ops
    lib = _cabi.lib()
    buf = (C.c_uint8 * 4096)()
    a = C.cast(buf, C.c_void_p)        # a non-NULL address that is never dereferenced
    # F1: NULL frames, NULL boxes, bad sizes, short row stride, unknown channel, too many ROIs, empty batch
    assert lib.bpv_roi_sample_u8(None, None, 0, 24, 8, 8, 1, a, 1, 0, None, a, 0, None) == -1
    assert b'bpv_roi_sample_u8' in lib.bpv_last_error()
    assert lib.bpv_roi_sample_u8(a, None, 192, 24, 8, 8, 1, None, 1, 0, None, a, 0, None) == -1
    assert lib.bpv_roi_sample_u8(a, None, 192, 24, 0, 8, 1, a, 1, 0, None, a, 0, None) == -1
    assert lib.bpv_roi_sample_u8(a, None, 192, 23, 8, 8, 1, a, 1, 0, None, a, 0, None) == -1
    assert lib.bpv_roi_sample_u8(a, None, 192, 24, 8, 8, 1, a, 1, 7, None, a, 0, None) == -2
    assert b'NotImplementedError' in lib.bpv_last_error()
    assert lib.bpv_roi_sample_u8(a, None, 192, 24, 8, 8, 2 ** 31, a, 2, 0, None, a, 0, None) == -3
    assert lib.bpv_roi_sample_u8(a, None, 192, 24, 8, 8, 0, a, 1, 0, None, a, 0, None) == 0          # empty batch: nothing to do
    # NV12 wants even sizes and pitch >= W; the fused resize wants positive target sizes
    assert lib.bpv_roi_sample_nv12(a, 96, 8, 7, 8, 1, a, 1, 0, None, a, None) == -1
    assert lib.bpv_roi_sample_nv12(a, 96, 6, 8, 8, 1, a, 1, 0, None, a, None) == -1
    assert lib.bpv_roi_sample_nv12(a, 96, 8, 8, 8, 0, a, 1, 0, None, a, None) == 0
    assert lib.bpv_roi_sample_resized_u8(a, 192, 24, 8, 8, 0, 4, 1, a, 1, 0, None, a, None) == -1
    assert lib.bpv_roi_sample_resized_u8(a, 192, 24, 8, 8, 4, 4, 1, a, 1, 9, None, a, None) == -2
    # window pipeline: NULL params, filter limits, unknown method / transform, window > cap, missing workspace
    assert lib.bpv_window_workspace_bytes(None) == -1
    assert lib.bpv_window_preprocess(a, a, None, None, 0, a, a, a, None) == -1
    good = dict(butter_order=16, butter_min_bw=0.1, fir_taps=127, fir_df=0.3, min_freq=0.8, max_freq=4.0, ls_num_freqs=0)

    def params(methods, transform=_cabi.PGRAM_LS, W=32, cap=33, **kw):
        return ops.make_params(1, 2, cap, W, W - 1, 1, 1, methods, transform, **{**good, **kw})
    pre = lambda p, ws=None, nbytes=0: lib.bpv_window_preprocess(a, a, C.byref(p), ws, nbytes, a, a, a, None)
    assert pre(params([], butter_order=17)) == -3
    assert pre(params([], fir_taps=128)) == -3                      # even / > 127 taps
    assert pre(params([], W=40, cap=33)) == -1                      # window longer than the ring
    p = params([_cabi.DIFF_1]); p.methods[0] = 42
    assert pre(p) == -2 and b'NotImplementedError' in lib.bpv_last_error()
    assert pre(params([_cabi.FILTER_FIR])) == -1                    # filter design needs the caller's workspace
    assert b'workspace' in lib.bpv_last_error()
    need = lib.bpv_window_workspace_bytes(C.byref(params([_cabi.FILTER_FIR])))
    assert need == 1 * ((16 * 6 + 520) * 8 + 8 + 16)            # per job: sos | taps [128] | zi [128] | merged taps [264] | cache ref | miss entry
    assert pre(params([_cabi.FILTER_FIR]), a, need - 1) == -1
    p = params([], transform=9)
    assert lib.bpv_window_spectrum(a, a, C.byref(p), 64, None, 0, None, None, a, a, a, a, None) == -2
    assert lib.bpv_window_spectrum(None, a, C.byref(params([])), 64, None, 0, None, None, a, a, a, a, None) == -1
    assert lib.bpv_window_xcorr(None, a, C.byref(params([])), None, None, None, a, a, a, None) == -1
    assert lib.bpv_window_xcorr(a, a, C.byref(params([])), a, None, None, a, a, a, None) == -1      # corr_lag without corr_val
    assert lib.bpv_butter_sos_design(None, 4, C.byref(params([])), a, None) == -1
    assert lib.bpv_firls_design(a, 0, C.byref(params([])), a, None) == 0                              # nothing to design
    assert lib.bpv_dft256_tc(None, 1, a, None) == -1
