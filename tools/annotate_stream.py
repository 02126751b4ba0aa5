"""GPU-box demo / probe: the whole device-resident chain of the lane path through the public API -- frames rasterised on the
GPU, lanes detected with two batches in flight, the lane overlay and the offset indicator drawn on the GPU -- and its rate.

    python tools/annotate_stream.py [batches] [frames_per_batch] [width] [height] [i420]

With ``i420`` the chain ends as annotated video would: every annotated batch is converted to I420 on the device
(``bgr_to_i420(view, out=pinned)``) and lands in pinned host memory, ready for an encoder (``ffmpeg -f rawvideo
-pix_fmt yuv420p``); the check of the first batch is then on those I420 bytes.

What demo.py does per frame on the CPU (detect -> draw_lanes -> get_lane_center_offset -> draw_lane_offset_indicator,
/root/reference/demo.py:108-128, app.py:124-180), here per batch and without the frames ever leaving HBM.  Prints one JSON
line; checks the first batch against the cv2 call sequence."""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import cv2
import numpy as np
import torch

from draw_util import cv2_draw_lanes, cv2_offset_indicator
from multimodal_autonomous_driving_perception_and_planning_b200 import (LaneDetector, OverlayRenderer, SyntheticDataGenerator,
                                                                        bgr_to_i420)

batches = int(sys.argv[1]) if len(sys.argv) > 1 else 8
n = int(sys.argv[2]) if len(sys.argv) > 2 else 256
w = int(sys.argv[3]) if len(sys.argv) > 3 else 1920
h = int(sys.argv[4]) if len(sys.argv) > 4 else 1080
i420 = len(sys.argv) > 5 and sys.argv[5] == "i420"

gen = SyntheticDataGenerator(w, h)
t0 = time.perf_counter()
stream = [gen.generate_batch_device(n) for _ in range(batches)]          # consecutive stretches of one camera stream
torch.cuda.synchronize()
t_gen = time.perf_counter() - t0

det, ov = LaneDetector(max_batch=n), OverlayRenderer()
pinned = torch.empty((n, h * 3 // 2, w), dtype=torch.uint8).pin_memory() if i420 else None


def run(keep_first=False):
    first = None
    for i, lanes in enumerate(det.detect_batches(stream)):
        view = stream[i].clone() if keep_first and i == 0 else stream[i]   # annotate in place (the demo overwrites its frame too)
        det.draw_lanes_batch(view, lanes)
        offs = [det.get_lane_center_offset(w, l, r) for l, r in lanes]
        ov.draw_lane_offset_indicator_batch(view, offs)
        if i420:
            bgr_to_i420(view, out=pinned)          # blocking: the I420 bytes of the batch are in host memory
        if keep_first and i == 0:
            first = (pinned.numpy().copy() if i420 else view, lanes, offs)
    torch.cuda.synchronize()
    return first


clean0 = stream[0].clone()
first = run(keep_first=True)                                               # warm-up + the batch that is checked
view, lanes, offs = first
host = clean0.cpu().numpy()
for k in range(0, n, max(1, n // 8)):
    l, r = lanes[k]
    ref = cv2_offset_indicator(cv2_draw_lanes(host[k].copy(), None if l is None else l.points, None if r is None else r.points), offs[k])
    if i420:
        assert np.array_equal(cv2.cvtColor(ref, cv2.COLOR_BGR2YUV_I420), view[k]), k
    else:
        assert np.array_equal(ref, view[k].cpu().numpy()), k
stream = [gen.generate_batch_device(n, start_frame=i * n) for i in range(batches)]
det.reset()
torch.cuda.synchronize()
t0 = time.perf_counter()
run()
dt = time.perf_counter() - t0
print(json.dumps({"resolution": [w, h], "batches": batches, "frames_per_batch": n,
                  "generate_frames_per_s": batches * n / t_gen,
                  ("detect_draw_indicator_i420_to_host_frames_per_s" if i420 else "detect_draw_indicator_frames_per_s"):
                      batches * n / dt,
                  "checked_against_cv2": "first batch, every %d-th frame" % max(1, n // 8)}))
