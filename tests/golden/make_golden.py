"""Generate golden vectors by running the UNMODIFIED reference, the checkout of the upstream bp-from-video project at
__graft_entry__.REFERENCE.  Run:  python tests/golden/make_golden.py   (writes tests/golden/*.npz)

The reference has no tests/golden vectors of its own, so these fixtures are the parity pin for
`oracle/bpv_oracle.py` (tests/test_oracle_golden.py demands exact equality) and, through the
oracle, for the CUDA path.  Frames are regenerated from the stored seed by `bpv.synth.frames`
(numpy PCG64 streams are stable), everything else (timestamps, detections, outputs) is stored.
Nothing here is needed at run time on the GPU box.
"""
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, 'bp-from-video_b200'))
from bpv import synth  # noqa: E402


def load_reference():
    """Import the reference's modules without letting our drop-in modules shadow them."""
    for name in ('roi', 'signal_data', 'signal_processor', 'model', 'profiler', 'exceptions'):
        sys.modules.pop(name, None)
    sys.path.insert(0, REF)
    import signal_processor as sp  # noqa
    import profiler  # noqa
    profiler.profiler.enabled = False  # as pbp.py:11
    sys.path.remove(REF)
    assert sp.__file__.startswith(REF), sp.__file__
    return sp


class _Out:
    def __init__(self, detections):
        self.detections = detections


class _Results:
    def __init__(self, face, hand):
        self.face_landmarker = _Out(face)
        self.hand_landmarker = _Out(hand)


class _Frame:
    def __init__(self, frame, ts):
        self.frame, self.timestamp = frame, ts


def make_detections(rng, n, H, W, p_none):
    """Per frame: face (bbox, anchor point 151) and hand (bbox, points 0 and 9)."""
    face_bbox = np.empty((n, 4), np.int64)
    hand_bbox = np.empty((n, 4), np.int64)
    face_pt = np.empty((n, 2), np.int64)
    hand_pts = np.empty((n, 2, 2), np.int64)
    for i in range(n):
        cx, cy = 0.45 * W + rng.integers(-2, 3), 0.30 * H + rng.integers(-2, 3)
        bw, bh = 0.25 * W + rng.integers(-1, 2), 0.40 * H + rng.integers(-1, 2)
        face_bbox[i] = np.rint([cx - bw / 2, cy - bh / 2, cx + bw / 2, cy + bh / 2])
        face_pt[i] = np.rint([cx - 0.1 * bw, cy - 0.2 * bh])
        cx, cy = 0.70 * W + rng.integers(-2, 3), 0.72 * H + rng.integers(-2, 3)
        bw, bh = 0.20 * W + rng.integers(-1, 2), 0.33 * H + rng.integers(-1, 2)
        hand_bbox[i] = np.rint([cx - bw / 2, cy - bh / 2, cx + bw / 2, cy + bh / 2])
        hand_pts[i, 0] = np.rint([cx - 3, cy + 4])
        hand_pts[i, 1] = np.rint([cx + 2 + rng.integers(0, 2), cy - 3])  # odd sums exercise .5 rounding
    present = rng.uniform(size=(n, 2)) >= p_none
    return face_bbox, face_pt, hand_bbox, hand_pts, present


def stub_results(i, d):
    face_bbox, face_pt, hand_bbox, hand_pts, present = d
    face, hand = [], []
    if present[i, 0]:
        pts = np.zeros((478, 2), np.int64)
        pts[151] = face_pt[i]
        face = [(tuple(int(v) for v in face_bbox[i]), pts)]
    if present[i, 1]:
        pts = np.zeros((21, 2), np.int64)
        pts[0], pts[9] = hand_pts[i, 0], hand_pts[i, 1]
        hand = [(tuple(int(v) for v in hand_bbox[i]), pts)]
    return _Results(face, hand)


def sig_arrays(group):
    return [np.asarray(s.x, dtype=float) for s in group], [np.asarray(s.y, dtype=float) for s in group]


sys.path.insert(0, ROOT)
from tests.helpers import CASES, LIVE_CASES, SEEDS, IMG_H as H, IMG_W as W, REFERENCE as REF  # noqa: E402  (single source of the case tables)



def run_case(sp, name, seed, table=CASES):
    channel, methods, transform, window, n, fps, irregular, p_none, roi_ms, kw = table[name]
    rng = np.random.default_rng(seed)
    ts = synth.timestamps(rng, n, fps, irregular=irregular, drop=0.05 if irregular else 0.0, origin=3.0)
    det = make_detections(rng, n, H, W, p_none)
    frames = synth.frames(np.random.default_rng(seed + 1000), ts, H, W, f_pulse=1.3)
    proc = sp.SignalProcessor(None, roi_ms, window, 50,
                              color_channel=sp.SignalColorChannel[channel],
                              processing_methods=[sp.SignalProcessingMethod[m] for m in methods],
                              spectrum_transform=sp.SignalSpectrumTransform[transform], **kw)
    full_at = sorted(set([0, 1, 2, 3, 4, 7, window - 1, window, n - 1]) & set(range(n)))
    out = dict(seed=seed, ts=ts, face_bbox=det[0], face_pt=det[1], hand_bbox=det[2], hand_pts=det[3], present=det[4],
               full_at=np.array(full_at), boxes=np.full((n, 2, 6), np.nan), raw=np.full((n, 2), np.nan),
               bpm=np.full((n, 2), np.nan), ptt=np.full((n, 1), np.nan))
    for i in range(n):
        store = proc.process(_Frame(frames[i], float(ts[i])), stub_results(i, det))
        out['boxes'][i] = np.array([np.asarray(b, dtype=float) for b in store.sg_roi.get_means(as_int=True)])
        out['raw'][i] = [s.y[-1] for s in store.sg_raw]
        out['bpm'][i] = [s.y[-1] for s in store.sg_bpm]
        out['ptt'][i] = [s.y[-1] for s in store.sg_ptt]
        if i in full_at:
            px, py = sig_arrays(store.sg_proc)
            fx, fy = sig_arrays(store.sg_spec)
            cx, cy = sig_arrays(store.sg_corr)
            for r in range(2):
                out[f'f{i}_proc_x{r}'], out[f'f{i}_proc_y{r}'] = px[r], py[r]
                out[f'f{i}_spec_x{r}'], out[f'f{i}_spec_y{r}'] = fx[r], fy[r]
            out[f'f{i}_corr_x0'], out[f'f{i}_corr_y0'] = cx[0], cy[0]
    return out


def roi_case(sp, seed=7):
    """sample_signal on random + edge-case boxes (negative wrap, clamp, empty) for both channels."""
    rng = np.random.default_rng(seed)
    Hh, Ww = 48, 64
    frame = rng.integers(0, 256, (Hh, Ww, 3), dtype=np.uint8)
    boxes = rng.integers(-Ww - 8, Ww + 24, (256, 4))
    edge = [(60, 40, 70, 50), (-10, -10, 30, 30), (-50, -40, -10, -10), (10, 10, 10, 30), (20, 30, 10, 40),
            (0, 0, Ww, Hh), (0, 0, 1, 1), (Ww - 1, Hh - 1, Ww, Hh), (-Ww, -Hh, Ww, Hh), (5, 5, 6, 40), (3, 7, 61, 8)]
    boxes = np.concatenate([np.array(edge), boxes])
    vals = np.empty((2, len(boxes)))
    for c, ch in enumerate((sp.SignalColorChannel.GREEN, sp.SignalColorChannel.CHROM_GREEN)):
        p = sp.SignalProcessor(color_channel=ch)
        for k, (x0, y0, x1, y1) in enumerate(boxes):
            vals[c, k] = p.sample_signal(frame, (0, 0, int(x0), int(y0), int(x1), int(y1)))
    return dict(seed=seed, H=Hh, W=Ww, boxes=boxes.astype(np.int64), values=vals)


def main():
    warnings.simplefilter('ignore')
    if not os.path.isdir(REF):
        sys.exit(f'no checkout of the upstream bp-from-video project at {REF}')
    sp = load_reference()
    if len(sys.argv) == 3 and sys.argv[1] == '--live':     # the non-committed differential cases, into a scratch directory
        for k, name in enumerate(LIVE_CASES):
            np.savez_compressed(os.path.join(sys.argv[2], f'{name}.npz'), **run_case(sp, name, 500 + k, LIVE_CASES))
        print('live ok')
        return
    for k, name in enumerate(CASES):
        out = run_case(sp, name, seed=SEEDS[name])
        np.savez_compressed(os.path.join(HERE, f'{name}.npz'), **out)
        print(name, 'ok', sum(v.nbytes for v in out.values() if isinstance(v, np.ndarray)) // 1024, 'KiB')
    np.savez_compressed(os.path.join(HERE, 'roi_sample.npz'), **roi_case(sp))
    print('roi_sample ok')


if __name__ == '__main__':
    main()
