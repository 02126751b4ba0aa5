"""GPU-box probe of what a per-camera ROI costs and buys on an 8-camera 1080p rig.  Prints one JSON line, with the
card's name and power limit beside the numbers.

    python tools/rig_roi_probe.py [steps]

- ``throughput``: frames/s of 8 cameras x 32 device-resident frames per batch, two batches in flight
  (``LaneContext.enqueue`` twice, then collect / enqueue alternately), over ``steps`` batches (default 40) for
  (a) one context with one shared ROI, (b) one context with 8 distinct ROIs (``lane_set_roi_masks``) and (c) 8
  single-ROI contexts of 32 frames each, one after another, each with its own two batches in flight.
- ``latency``: p50 / p99 in ms of one tick of 8 x 1 host frames (one frame per camera, blocking call in, records out)
  for the same three setups; (c) is 8 blocking calls of one frame.
Before anything is timed, the records of (b) and (c) are compared: they must be equal byte for byte."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import numpy as np
import torch

from multimodal_autonomous_driving_perception_and_planning_b200 import _native, multi_camera_batch
from test_gpu_stream_roi import rig_masks

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 40
H, W, CAMS, PER_CAM = 1080, 1920, 8, 32
if not torch.cuda.is_available():
    sys.exit("rig_roi_probe: no CUDA device (the probe measures the GPU; there is nothing to fall back to)")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        return q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi unavailable: {e}"


masks = rig_masks(H, W)
cams = multi_camera_batch(CAMS, PER_CAM, W, H, period=8)                  # [8, 32, H, W, 3], 1.6 GB: more than L2
rig_order = np.array([(s, t) for t in range(PER_CAM) for s in range(CAMS)])  # tick-major: cameras interleaved
rig_ids = rig_order[:, 0].astype(np.int32)
rig_dev = torch.from_numpy(np.stack([cams[s, t] for s, t in rig_order])).cuda()
cam_dev = torch.from_numpy(cams.reshape(CAMS * PER_CAM, H, W, 3)).cuda()   # camera-major for (c)
torch.cuda.synchronize()
FB = H * W * 3
N = CAMS * PER_CAM


class Pipe:
    """A context with up to two batches in flight, state carried on the device."""

    def __init__(self, mask, n, S):
        self.ctx = _native.LaneContext(H, W, n, mask)
        self.n, self.S = n, S
        self.fit, self.valid = np.zeros((S, 2, 3)), np.zeros((S, 2), np.uint8)
        self.started = False

    def push(self, ptr, ids):
        out = self.ctx.collect(self.fit, self.valid) if len(self.ctx._inflight) == 2 else None
        if self.started:
            self.ctx.enqueue(ptr, self.n, ids, self.S, None, None, 0.7, 0.3)
        else:
            self.ctx.enqueue(ptr, self.n, ids, self.S, self.fit, self.valid, 0.7, 0.3)
            self.started = True
        return out

    def drain(self):
        out = []
        while self.ctx._inflight:
            out.append(self.ctx.collect(self.fit, self.valid))
        return out


def setups():
    a = [Pipe(masks[0], N, CAMS)]
    b = [Pipe(masks, N, CAMS)]
    c = [Pipe(masks[s], PER_CAM, 1) for s in range(CAMS)]
    return {"a_shared_roi": (a, lambda p, k: p.push(rig_dev.data_ptr(), rig_ids)),
            "b_rig_rois": (b, lambda p, k: p.push(rig_dev.data_ptr(), rig_ids)),
            "c_8_contexts": (c, lambda p, k: p.push(cam_dev.data_ptr() + k * PER_CAM * FB, None))}


def check_b_equals_c(S):
    b, c = S["b_rig_rois"][0][0], S["c_8_contexts"][0]
    b.push(rig_dev.data_ptr(), rig_ids)
    rb = b.drain()[0]
    for k, p in enumerate(c):
        p.push(cam_dev.data_ptr() + k * PER_CAM * FB, None)
        rc = p.drain()[0]
        for t in range(PER_CAM):
            i = int(np.nonzero((rig_order[:, 0] == k) & (rig_order[:, 1] == t))[0][0])
            assert rb[i].tobytes() == rc[t].tobytes(), (k, t)


def throughput(pipes, push):
    for p in pipes:                                          # warm-up: every shape, both result slots
        for _ in range(3):
            push(p, pipes.index(p))
        p.drain()
        p.started = False
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        for k, p in enumerate(pipes):
            push(p, k)
    for p in pipes:
        p.drain()
    dt = time.perf_counter() - t0
    return round(steps * N / dt, 1)


def latency(ctxs, ticks=300):
    tick_frames = np.ascontiguousarray(cams[:, 0])           # one host frame per camera
    ids = np.arange(CAMS, dtype=np.int32)
    ts = []
    for i in range(ticks + 20):
        t0 = time.perf_counter()
        if len(ctxs) == 1:
            fit, valid = np.zeros((CAMS, 2, 3)), np.zeros((CAMS, 2), np.uint8)
            ctxs[0].detect(tick_frames, CAMS, False, ids, CAMS, fit, valid, 0.7, 0.3)
        else:
            for s, c in enumerate(ctxs):
                fit, valid = np.zeros((1, 2, 3)), np.zeros((1, 2), np.uint8)
                c.detect(tick_frames[s:s + 1], 1, False, None, 1, fit, valid, 0.7, 0.3)
        if i >= 20:
            ts.append((time.perf_counter() - t0) * 1e3)
    return {"p50_ms": round(float(np.percentile(ts, 50)), 3), "p99_ms": round(float(np.percentile(ts, 99)), 3)}


S = setups()
check_b_equals_c(S)
for pipes, _ in S.values():
    for p in pipes:
        p.ctx.close()
S = setups()
result = {"probe": "rig_roi", "card": card(), "device": torch.cuda.get_device_name(), "frames": f"{CAMS}x{PER_CAM} {W}x{H}",
          "steps": steps, "throughput_fps": {}, "latency_8x1": {}}
for name, (pipes, push) in S.items():
    result["throughput_fps"][name] = throughput(pipes, push)
for name, (pipes, _) in S.items():
    lat_ctxs = [_native.LaneContext(H, W, CAMS, masks[0] if name.startswith("a") else masks)] if len(pipes) == 1 \
        else [_native.LaneContext(H, W, 1, masks[s]) for s in range(CAMS)]
    result["latency_8x1"][name] = latency(lat_ctxs)
    for c in lat_ctxs:
        c.close()
    for p in pipes:
        p.ctx.close()
print(json.dumps(result), flush=True)
