"""GPU-box probe of a mixed rig streamed two ticks deep (``LaneDetector.detect_rig_stream``) against ``detect_rig``
called tick after tick.  Prints one JSON line, with the card's name and power limit read in the same run.

    python tools/rig_stream_probe.py [ticks] [steps]

The rig of ``tools/rig_ingest_probe.py``: 1 x 3840x2160 NV12, 4 x 1936x1216 NV12, 2 x 1280x720 I420, 1 x 1920x1080 BGR,
all detected at 640x480.
  (a) ``device_fps``: frames/s with 32 device-resident frames per camera per tick (256 per tick; 1.3 GB of sources,
      more than L2 holds), over ``steps`` ticks (default 30) after two warm-up ticks.
  (b) ``pinned_8x1``: ticks of one pinned host frame per camera, over ``ticks`` ticks (default 1000) after 50 warm-up
      ticks: ticks/s of either form, and for the stream p50 / p99 in ms from handing a tick to the generator to getting
      its lanes back.
  (c) ``numpy_8x1``: the same with ordinary numpy ticks, which the stream first copies into its pinned buffers.
Before anything is timed, the stream's records of every form are compared with ``detect_rig``'s, byte for byte."""
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
from multimodal_autonomous_driving_perception_and_planning_b200 import LaneDetector
from util import gen_frames

ticks = int(sys.argv[1]) if len(sys.argv) > 1 else 1000
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 30
if not torch.cuda.is_available():
    sys.exit("rig_stream_probe: no CUDA device (the probe measures the GPU; there is nothing to fall back to)")

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


def pinned(a):
    t = torch.empty(a.shape, dtype=torch.uint8).pin_memory()
    t.numpy()[...] = a
    return t


# host ticks of one frame per camera: DISTINCT different ticks, used round robin
host_ticks = [[np.ascontiguousarray(c[k:k + 1]) for c in cams] for k in range(DISTINCT)]
pinned_ticks = [[pinned(f) for f in tick] for tick in host_ticks]
torch.cuda.synchronize()


def rig_call(det, tick):
    return det.detect_rig(tick, LAYOUTS, target_size=TARGET)


def stream(det, seq):
    return det.detect_rig_stream(seq, LAYOUTS, target_size=TARGET)


def check():
    """Every form's streamed records equal detect_rig's, tick after tick, on fresh detectors."""
    forms = {"device": ([dev] * 3, CAMS * PER_CAM), "pinned": (pinned_ticks[:4], CAMS), "numpy": (host_ticks[:4], CAMS)}
    for name, (seq, mb) in forms.items():
        a, b = LaneDetector(max_batch=mb), LaneDetector(max_batch=mb)
        want = []
        for tick in seq:
            rig_call(a, [t.numpy() if isinstance(t, torch.Tensor) and not t.is_cuda else t for t in tick])
            want.append(a.last_records.copy())
        got = []
        for _ in stream(b, seq):
            got.append(b.last_records.copy())
        assert [r.tobytes() for r in got] == [r.tobytes() for r in want], name
        assert a._stream_fit.tobytes() == b._stream_fit.tobytes(), name
        a.close()
        b.close()


def device_fps():
    out = {}
    a, b = LaneDetector(max_batch=CAMS * PER_CAM), LaneDetector(max_batch=CAMS * PER_CAM)
    for _ in range(2):
        rig_call(a, dev)
    for _ in stream(b, [dev] * 2):
        pass
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        rig_call(a, dev)
    torch.cuda.synchronize()
    out["detect_rig"] = round(steps * CAMS * PER_CAM / (time.perf_counter() - t0), 1)
    t0 = time.perf_counter()
    for _ in stream(b, [dev] * steps):
        pass
    torch.cuda.synchronize()
    out["detect_rig_stream"] = round(steps * CAMS * PER_CAM / (time.perf_counter() - t0), 1)
    a.close()
    b.close()
    return out


def host_8x1(seq_ticks, blocking_ticks):
    a, b = LaneDetector(max_batch=CAMS), LaneDetector(max_batch=CAMS)
    for i in range(50):
        rig_call(a, blocking_ticks[i % DISTINCT])
    t0 = time.perf_counter()
    for i in range(ticks):
        rig_call(a, blocking_ticks[i % DISTINCT])
    blocking_tps = ticks / (time.perf_counter() - t0)

    handed = []

    def source(n):
        for i in range(n):
            handed.append(time.perf_counter())
            yield seq_ticks[i % DISTINCT]

    for _ in stream(b, source(50)):
        pass
    handed.clear()
    lat = []
    t0 = time.perf_counter()
    for k, _ in enumerate(stream(b, source(ticks))):
        lat.append((time.perf_counter() - handed[k]) * 1e3)
    stream_tps = ticks / (time.perf_counter() - t0)
    a.close()
    b.close()
    return {"detect_rig_ticks_per_s": round(blocking_tps, 1), "detect_rig_stream_ticks_per_s": round(stream_tps, 1),
            "stream_p50_ms": round(float(np.percentile(lat, 50)), 3),
            "stream_p99_ms": round(float(np.percentile(lat, 99)), 3)}


check()
pinned_as_numpy = [[t.numpy() for t in tick] for tick in pinned_ticks]      # detect_rig's form of the pinned ticks
result = {"probe": "rig_stream", "card": card(), "device": torch.cuda.get_device_name(),
          "rig": [f"{lay} {w}x{h}" for lay, w, h in RIG], "target": TARGET, "ticks": ticks, "steps": steps,
          "a_device_fps": device_fps(), "b_pinned_8x1": host_8x1(pinned_ticks, pinned_as_numpy),
          "c_numpy_8x1": host_8x1(host_ticks, host_ticks)}
print(json.dumps(result), flush=True)
