"""GPU-box probe of a mixed rig: eight cameras of different sizes and decoder layouts detected at 640x480.  Prints one
JSON line, with the card's name and power limit beside the numbers.

    python tools/rig_ingest_probe.py [ticks] [steps]

The rig: 1 x 3840x2160 NV12 (front), 4 x 1936x1216 NV12 (surround), 2 x 1280x720 I420 (software-decoded), 1 x
1920x1080 BGR; the generator's scenes converted with bgr_to_nv12 / bgr_to_i420.  Three setups:
  (a) ``LaneDetector.detect_rig``: one call, one ingest launch for every camera;
  (b) eight single-camera detectors with ``target_size``, one after another;
  (c) ``FrameIngest`` per camera into a device tensor, ``torch.cat``, then one ``detect_streams``.
- ``latency_8x1``: p50 / p99 in ms of one tick of one pinned host frame per camera, blocking call in, lanes out, over
  ``ticks`` ticks (default 1000) after 50 warm-up ticks.  For (c) the host frames are copied to the device first.
- ``throughput_fps``: frames/s with 32 device-resident frames per camera (256 per step), over ``steps`` steps
  (default 30) after two warm-up steps; the frames (1.3 GB) are more than L2 holds.
- ``ingest_kernel_ms``: device time of k0_rig_ingest for the 256 frames, against the sum of the per-camera ingest
  kernels (k0_ingest_resize / k0_resize) for the same frames, from torch.profiler's CUDA activity in a pass of its own,
  averaged over 10 calls.
Before anything is timed, (a) and (b) are compared: every camera's records must be equal byte for byte."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

from bgr_yuv420 import bgr_to_i420, bgr_to_nv12
from multimodal_autonomous_driving_perception_and_planning_b200 import FrameIngest, LaneDetector
from util import gen_frames

ticks = int(sys.argv[1]) if len(sys.argv) > 1 else 1000
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 30
if not torch.cuda.is_available():
    sys.exit("rig_ingest_probe: no CUDA device (the probe measures the GPU; there is nothing to fall back to)")

RIG = [("nv12", 3840, 2160)] + [("nv12", 1936, 1216)] * 4 + [("i420", 1280, 720)] * 2 + [("bgr", 1920, 1080)]
LAYOUTS = [lay for lay, _, _ in RIG]
TARGET = (640, 480)
PER_CAM, DISTINCT = 32, 8
CAMS = len(RIG)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        return q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi unavailable: {e}"


def camera(s, lay, w, h):
    bgr = gen_frames(w, h, DISTINCT, start=1000 * s)
    frames = bgr if lay == "bgr" else [(bgr_to_nv12 if lay == "nv12" else bgr_to_i420)(f) for f in bgr]
    return np.stack([frames[t % DISTINCT] for t in range(PER_CAM)])


cams = [camera(s, *c) for s, c in enumerate(RIG)]
dev = [torch.from_numpy(c).cuda() for c in cams]
pinned = []
for c in cams:
    t = torch.empty((1,) + c.shape[1:], dtype=torch.uint8).pin_memory()
    t.numpy()[...] = c[:1]
    pinned.append(t)
tick_frames = [t.numpy() for t in pinned]
torch.cuda.synchronize()
N = CAMS * PER_CAM


def single(det, lay, frames):
    fn = {"bgr": det.detect_batch, "nv12": det.detect_batch_nv12, "i420": det.detect_batch_i420}[lay]
    return fn(frames, target_size=TARGET)


class Ingest:
    """(c): every camera through FrameIngest into a device tensor, one torch.cat, one detect_streams."""

    def __init__(self, max_batch):
        self.ing = FrameIngest(TARGET)
        self.det = LaneDetector(max_batch=max_batch)

    def __call__(self, frames):
        conv = {"bgr": self.ing.resize_batch, "nv12": self.ing.from_nv12, "i420": self.ing.from_i420}
        out = [conv[lay](f) for lay, f in zip(LAYOUTS, frames)]
        ids = np.concatenate([np.full(len(f), s, np.int32) for s, f in enumerate(frames)])
        return self.det.detect_streams(torch.cat(out), stream_ids=ids)


def check_a_equals_b():
    a = LaneDetector(max_batch=N)
    a.detect_rig(dev, LAYOUTS, target_size=TARGET)
    off = 0
    for s, lay in enumerate(LAYOUTS):
        b = LaneDetector(max_batch=PER_CAM)
        single(b, lay, dev[s])
        assert a.last_records[off:off + PER_CAM].tobytes() == b.last_records.tobytes(), s
        off += PER_CAM
        b.close()
    a.close()


def latency():
    a = LaneDetector(max_batch=CAMS)
    bs = [LaneDetector(max_batch=1) for _ in range(CAMS)]
    c = Ingest(CAMS)
    arms = {
        "a_detect_rig": lambda: a.detect_rig(tick_frames, LAYOUTS, target_size=TARGET),
        "b_8_detectors": lambda: [single(bs[s], lay, tick_frames[s]) for s, lay in enumerate(LAYOUTS)],
        "c_ingest_cat_streams": lambda: c([p.cuda(non_blocking=True) for p in pinned]),
    }
    out = {}
    for name, fn in arms.items():
        ts = []
        for i in range(ticks + 50):
            t0 = time.perf_counter()
            fn()
            if i >= 50:
                ts.append((time.perf_counter() - t0) * 1e3)
        out[name] = {"p50_ms": round(float(np.percentile(ts, 50)), 3), "p99_ms": round(float(np.percentile(ts, 99)), 3)}
    return out


def throughput():
    a = LaneDetector(max_batch=N)
    bs = [LaneDetector(max_batch=PER_CAM) for _ in range(CAMS)]
    c = Ingest(N)
    arms = {
        "a_detect_rig": lambda: a.detect_rig(dev, LAYOUTS, target_size=TARGET),
        "b_8_detectors": lambda: [single(bs[s], lay, dev[s]) for s, lay in enumerate(LAYOUTS)],
        "c_ingest_cat_streams": lambda: c(dev),
    }
    out = {}
    for name, fn in arms.items():
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
        out[name] = round(steps * N / (time.perf_counter() - t0), 1)
    return out


def ingest_kernels(calls=10):
    from torch.profiler import ProfilerActivity, profile
    a = LaneDetector(max_batch=N)
    ing = FrameIngest(TARGET)
    conv = {"bgr": ing.resize_batch, "nv12": ing.from_nv12, "i420": ing.from_i420}
    a.detect_rig(dev, LAYOUTS, target_size=TARGET)
    [conv[lay](f) for lay, f in zip(LAYOUTS, dev)]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            a.detect_rig(dev, LAYOUTS, target_size=TARGET)
            [conv[lay](f) for lay, f in zip(LAYOUTS, dev)]
        torch.cuda.synchronize()
    rig_us = per_cam_us = 0.0
    for e in prof.key_averages():
        if "k0_rig_ingest" in e.key:
            rig_us += e.device_time_total
        elif "k0_ingest_resize" in e.key or "k0_resize" in e.key:
            per_cam_us += e.device_time_total
    return {"k0_rig_ingest": round(rig_us / calls / 1e3, 4), "per_camera_sum": round(per_cam_us / calls / 1e3, 4)}


check_a_equals_b()
result = {"probe": "rig_ingest", "card": card(), "device": torch.cuda.get_device_name(),
          "rig": [f"{lay} {w}x{h}" for lay, w, h in RIG], "target": TARGET, "ticks": ticks, "steps": steps,
          "latency_8x1": latency(), "throughput_fps": throughput(), "ingest_kernel_ms": ingest_kernels()}
print(json.dumps(result), flush=True)
