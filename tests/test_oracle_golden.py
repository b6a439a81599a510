"""CPU: the oracle (oracle/bpv_oracle.py) must reproduce, bit for bit, what the unmodified
reference produced for the committed golden fixtures (tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest

from oracle import bpv_oracle as orc
from tests import helpers as h


@pytest.mark.parametrize('name', list(h.CASES))
def test_process_matches_reference(name):
    _replay(h.CASES[name], h.load_case(name), name)


@pytest.mark.skipif(not os.path.isdir(h.REFERENCE), reason=h.NO_REFERENCE)
def test_live_differential_vs_reference(tmp_path):
    """Beyond the frozen fixtures: run the UNMODIFIED reference now, in a subprocess, on cases that are not committed
    (other method chains, filter orders, tap counts, frame rates, ROI smoothing lengths) and demand exact equality."""
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(h.GOLDEN, 'make_golden.py'), '--live', str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and 'live ok' in r.stdout, r.stderr[-2000:]
    for name, case in h.LIVE_CASES.items():
        g = np.load(os.path.join(str(tmp_path), f'{name}.npz'))
        _replay(case, {k: g[k] for k in g.files}, name)


def _replay(case, g, name):
    channel, methods, transform, window, n, fps, irregular, p_none, roi_ms, kw = case
    frames = h.case_frames(g)
    st = orc.OracleStream(2, roi_ms, window, 50, h.CHANNEL[channel], [h.METHOD[m] for m in methods],
                          h.TRANSFORM[transform], **kw)
    full_at = set(int(i) for i in g['full_at'])
    for i in range(n):
        out = st.process(frames[i], float(g['ts'][i]), h.case_rois(g, i))
        assert h.same(np.array([np.asarray(b, dtype=float) for b in out['boxes']]), g['boxes'][i]), (name, i)
        assert h.same(out['samples'], g['raw'][i]), (name, i)
        assert h.same(out['bpm'], g['bpm'][i]), (name, i)
        assert h.same(out['ptt'], g['ptt'][i]), (name, i)
        if i in full_at:
            for r in range(2):
                assert h.same(out['proc_x'][r], g[f'f{i}_proc_x{r}'])
                assert h.same(out['proc_y'][r], g[f'f{i}_proc_y{r}'])
                assert h.same(out['freqs'][r], g[f'f{i}_spec_x{r}'])
                assert h.same(out['mags'][r], g[f'f{i}_spec_y{r}'])
            assert h.same(out['lags'][0], g[f'f{i}_corr_x0'])
            assert h.same(out['corr'][0], g[f'f{i}_corr_y0'])


def test_roi_sample_matches_reference():
    g = np.load(os.path.join(h.GOLDEN, 'roi_sample.npz'))
    rng = np.random.default_rng(int(g['seed']))
    frame = rng.integers(0, 256, (int(g['H']), int(g['W']), 3), dtype=np.uint8)
    n_empty = 0
    for k, box in enumerate(g['boxes']):
        sroi = (0, 0, *[int(v) for v in box])
        sB, sG, sR, n = orc.roi_sums(frame, box)
        n_empty += n == 0
        for c in (orc.GREEN, orc.CHROM_GREEN):
            ref = g['values'][c, k]
            assert h.same(orc.roi_sample(frame, sroi, c), ref)
            assert h.same(orc.value_from_sums(sB, sG, sR, n, c), ref), (k, box, c)
    assert 0 < n_empty < len(g['boxes'])


def test_nv12_conversion_matches_opencv():
    """The oracle's NV12 -> BGR restatement against OpenCV itself (cv2 is the decoder-side converter the reference sits
    behind, video_reader.py:93): bit-exact on random planes, extreme values and odd plane sizes."""
    cv2 = pytest.importorskip('cv2')
    rng = np.random.default_rng(12)
    for H, W in [(2, 2), (6, 10), (48, 64), (270, 480)]:
        nv = rng.integers(0, 256, (H * 3 // 2, W), dtype=np.uint8)
        assert np.array_equal(orc.nv12_to_bgr(nv, H, W), cv2.cvtColor(nv, cv2.COLOR_YUV2BGR_NV12)), (H, W)
    for fill in (0, 16, 128, 235, 255):
        nv = np.full((12, 8), fill, np.uint8)
        nv[8:] = rng.choice([0, 255, 128], size=(4, 8)).astype(np.uint8)
        assert np.array_equal(orc.nv12_to_bgr(nv, 8, 8), cv2.cvtColor(nv, cv2.COLOR_YUV2BGR_NV12)), fill


def test_resize_restatement_matches_opencv():
    """The oracle's cv2.resize (INTER_LINEAR, uint8) restatement against OpenCV itself: bit-exact for down- and
    up-scaling, mixed, identity, exact 2x decimation (area fast path) and tiny images."""
    cv2 = pytest.importorskip('cv2')
    rng = np.random.default_rng(21)
    for (sh, sw), (dh, dw) in [((48, 64), (30, 40)), ((48, 64), (96, 128)), ((270, 480), (180, 320)), ((37, 53), (50, 31)),
                               ((100, 100), (333, 77)), ((64, 64), (32, 32)), ((64, 64), (32, 33)), ((5, 7), (50, 70)),
                               ((90, 160), (90, 160)), ((216, 384), (54, 96))]:
        src = rng.integers(0, 256, (sh, sw, 3), dtype=np.uint8)
        assert np.array_equal(orc.resize_linear_u8(src, dw, dh), cv2.resize(src, (dw, dh))), ((sh, sw), (dh, dw))


def test_resize_and_nv12_restatements_fuzzed_against_opencv():
    """Seeded fuzz of the two ingest restatements against cv2 over random geometries (down / up / mixed scaling, 1-pixel
    targets, 2-pixel sources; even NV12 sizes): every output byte equal."""
    cv2 = pytest.importorskip('cv2')
    rng = np.random.default_rng(99)
    for _ in range(200):
        sh, sw = int(rng.integers(2, 120)), int(rng.integers(2, 160))
        dh, dw = int(rng.integers(1, 200)), int(rng.integers(1, 260))
        src = rng.integers(0, 256, (sh, sw, 3), dtype=np.uint8)
        assert np.array_equal(orc.resize_linear_u8(src, dw, dh), cv2.resize(src, (dw, dh))), ((sh, sw), (dh, dw))
    for _ in range(40):
        H, W = 2 * int(rng.integers(1, 60)), 2 * int(rng.integers(1, 80))
        nv = rng.integers(0, 256, (H * 3 // 2, W), dtype=np.uint8)
        assert np.array_equal(orc.nv12_to_bgr(nv, H, W), cv2.cvtColor(nv, cv2.COLOR_YUV2BGR_NV12)), (H, W)
