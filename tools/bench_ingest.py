"""Development micro-benchmark of the ingest variants of F1 (SURVEY 8f row 2): NV12 planes and fused cv2.resize, next to
the plain BGR kernel on the same boxes (config-2 geometry).  Not a judged number."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'bp-from-video_b200'))
from bpv import ops, synth  # noqa: E402

N, H, W = int(os.environ.get('INGEST_FRAMES', 8192)), 1080, 1920      # 8192 frames: 51 GB of BGR / 25 GB of NV12 in HBM, far beyond L2
PEAK = 6466.5                                                           # measured copy bandwidth (MEASURED_PEAKS.json), GB/s
rng = np.random.default_rng(0)
boxes_np = synth.roi_boxes(rng, N, H, W)
boxes = torch.from_numpy(boxes_np).cuda()
px = 0
for f in range(N):
    for r in range(2):
        b = boxes_np[f, r]
        if b[0] != synth.NO_BOX:
            px += max(0, min(b[2], W) - max(b[0], 0)) * max(0, min(b[3], H) - max(b[1], 0))


def timeit(fn, iters=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(iters + 1)]
    ev[0].record()
    for i in range(iters):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    return float(np.median([ev[i].elapsed_time(ev[i + 1]) for i in range(iters)]))


bgr = torch.empty((N, H, W, 3), dtype=torch.uint8, device='cuda')
for i in range(0, N, 64):
    bgr[i:i + 64].random_(0, 256)
t = timeit(lambda: ops.roi_sample(bgr, boxes, 1, roi_pixels_hint=5800))
t_bgr = t
print(f'BGR      {N} frames: {t*1e3:8.1f} us  {3*px/t/1e6:8.1f} GB/s of ROI bytes = {3*px/t/1e6/PEAK:.3f} of the copy peak  {N/t*1e3/1e6:6.2f} M frames/s')
nv = torch.empty((N, H * 3 // 2, W), dtype=torch.uint8, device='cuda').random_(0, 256)
t = timeit(lambda: ops.roi_sample_nv12(nv, H, W, boxes, 1))
print(f'NV12     {N} frames: {t*1e3:8.1f} us  {1.5*px/t/1e6:8.1f} GB/s of ROI bytes (1.5 B/px) = {1.5*px/t/1e6/PEAK:.3f} of the copy peak  {N/t*1e3/1e6:6.2f} M frames/s  = {t/t_bgr:.2f} x the BGR kernel per frame')
t = timeit(lambda: ops.roi_sample_nv12(nv, H, W, boxes, 0))
print(f'NV12 GREEN {N} frames: {t*1e3:8.1f} us  = {t/t_bgr:.2f} x the BGR kernel per frame')
del nv
# VideoReader target_res: 1080p source sampled as if resized to 720p; boxes scaled to the 720p frame
dh, dw = 720, 1280
b720 = boxes_np.copy()
ok = b720[..., 0] != synth.NO_BOX
b720[ok] = np.rint(b720[ok] * (dw / W)).astype(np.int32)
b720_d = torch.from_numpy(b720).cuda()
t = timeit(lambda: ops.roi_sample_resized(bgr, dh, dw, b720_d, 1))
print(f'resized  {N} frames (1080p -> 720p boxes): {t*1e3:8.1f} us  {N/t*1e3/1e6:6.2f} M frames/s  = {t/t_bgr:.2f} x the BGR kernel per frame')
t = timeit(lambda: ops.roi_sample_resized(bgr, dh, dw, b720_d, 0))
print(f'resized GREEN {N} frames: {t*1e3:8.1f} us  = {t/t_bgr:.2f} x the BGR kernel per frame')
