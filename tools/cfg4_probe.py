"""GPU-box probe: config 4 (128 x 3840x2160) stage times, for A/B of PPHT kernel choices (LANE_B200_K4=v2, or
another build of the library through LANE_B200_LIB)."""
import json, os, sys, time
sys.path.insert(0, '.')
import numpy as np, torch
from multimodal_autonomous_driving_perception_and_planning_b200 import LaneDetector, SyntheticDataGenerator
n = 128
base = SyntheticDataGenerator(3840, 2160).generate_batch_device(4, start_frame=0)
dev = base.repeat(n // 4, 1, 1, 1).contiguous()
det = LaneDetector(max_batch=n)
ctx = det._context(2160, 3840, n)
pf, pv = np.zeros((1, 2, 3)), np.zeros((1, 2), np.uint8)
for _ in range(2):
    ctx.detect(dev.data_ptr(), n, True, None, 1, pf, pv, 0.7, 0.3)
ctx.set_profiling(True)
tot = {}
for _ in range(3):
    recs = ctx.detect(dev.data_ptr(), n, True, None, 1, pf, pv, 0.7, 0.3)
    ms, _ = ctx.stage_ms()
    for k, v in ms.items():
        tot[k] = tot.get(k, 0) + v / 3
print(json.dumps({"env": {k: os.environ.get(k) for k in ("LANE_B200_K4", "LANE_B200_LIB")}, "paths": ctx.last_paths(),
                  "stage_ms": {k: round(v, 4) for k, v in tot.items()}, "segments_mean": float(recs["n_segments"].mean())}))
