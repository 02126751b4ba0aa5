"""GPU-box probe of frame egress (K8, ``bgr_to_i420``): annotated BGR frames in HBM -> I420, on the device and off to
the host.  Prints one JSON line, with the card's name and power limit beside the numbers.

    python tools/egress_probe.py [frames] [width] [height]

- ``kernel``: CUDA-event time of the conversion of ``frames`` device frames (256 x 1080p by default: 1.6 GB in,
  0.8 GB out, more than L2) into a device tensor; achieved GB/s at 4.5 B/px, and its share of a device-to-device copy
  of the same frames measured in this run (the way DESIGN.md section 6 measures its copy bandwidth).
- ``d2h``: frames/s of four routes from the device frames to host memory: I420 into pinned memory, I420 into pageable
  (numpy) memory, a plain pinned copy of the BGR frames, and a plain pinned copy of the I420 byte count.  The first over
  the last is the PCIe fraction of the I420 route.
- ``annotate``: the chain of tools/annotate_stream.py (``detect_batches`` -> ``draw_lanes_batch`` -> offset indicator)
  in frames/s, once with the frames left in HBM and once ending in ``bgr_to_i420(view, out=pinned)``.
Sampled frames of every route are compared with cv2.cvtColor(f, COLOR_BGR2YUV_I420) before anything is timed."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import cv2
import numpy as np
import torch

from multimodal_autonomous_driving_perception_and_planning_b200 import (LaneDetector, OverlayRenderer, SyntheticDataGenerator,
                                                                        bgr_to_i420)

n = int(sys.argv[1]) if len(sys.argv) > 1 else 256
w = int(sys.argv[2]) if len(sys.argv) > 2 else 1920
h = int(sys.argv[3]) if len(sys.argv) > 3 else 1080
if not torch.cuda.is_available():
    sys.exit("egress_probe: no CUDA device (the probe measures the GPU; there is nothing to fall back to)")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        return q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi unavailable: {e}"


def event_ms(fn, reps):
    for _ in range(3):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / reps


def wall_s(fn, reps):
    fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps


def check(got, frames, every):
    for k in range(0, n, every):
        want = cv2.cvtColor(frames[k].cpu().numpy(), cv2.COLOR_BGR2YUV_I420)
        assert np.array_equal(np.asarray(got[k].cpu() if torch.is_tensor(got) else got[k]), want), k


gen = SyntheticDataGenerator(w, h)
frames = gen.generate_batch_device(n)
i420_shape = (n, h * 3 // 2, w)
px = n * h * w

# ---- kernel
dev_out = torch.empty(i420_shape, dtype=torch.uint8, device="cuda")
bgr_to_i420(frames, out=dev_out)
check(dev_out, frames, max(1, n // 16))
k_ms = event_ms(lambda: bgr_to_i420(frames, out=dev_out), 20)
copy_dst = torch.empty_like(frames)
c_ms = event_ms(lambda: copy_dst.copy_(frames), 20)
k_gbs = px * 4.5 / (k_ms * 1e-3) / 1e9
c_gbs = 2 * frames.numel() / (c_ms * 1e-3) / 1e9
del copy_dst

# ---- device -> host
pinned = torch.empty(i420_shape, dtype=torch.uint8).pin_memory()
pageable = np.empty(i420_shape, np.uint8)
pinned_bgr = torch.empty(frames.shape, dtype=torch.uint8).pin_memory()
flat = frames.view(-1)
i420_bytes = pinned.numel()
bgr_to_i420(frames, out=pinned)
bgr_to_i420(frames, out=pageable)
check(pinned.numpy(), frames, max(1, n // 8))
check(pageable, frames, max(1, n // 8))
routes = {
    "i420_pinned": wall_s(lambda: bgr_to_i420(frames, out=pinned), 5),
    "i420_pageable": wall_s(lambda: bgr_to_i420(frames, out=pageable), 5),
    "bgr_plain_pinned_copy": wall_s(lambda: pinned_bgr.copy_(frames), 5),
    "i420_bytes_plain_pinned_copy": wall_s(lambda: pinned.view(-1).copy_(flat[:i420_bytes]), 5),
}
d2h = {k: {"frames_per_s": n / s, "gb_per_s": (i420_bytes if "i420" in k else frames.numel()) / s / 1e9}
       for k, s in routes.items()}
d2h["i420_pinned_pcie_frac"] = routes["i420_bytes_plain_pinned_copy"] / routes["i420_pinned"]
d2h["i420_over_bgr_copy"] = routes["bgr_plain_pinned_copy"] / routes["i420_pinned"]
del pinned_bgr, pageable, dev_out

# ---- the annotate chain
batches = 4
stream = [gen.generate_batch_device(n, start_frame=i * n) for i in range(batches)]
det, ov = LaneDetector(max_batch=n), OverlayRenderer()


def chain(to_host):
    for i, lanes in enumerate(det.detect_batches(stream)):
        view = stream[i]
        det.draw_lanes_batch(view, lanes)
        ov.draw_lane_offset_indicator_batch(view, [det.get_lane_center_offset(w, l, r) for l, r in lanes])
        if to_host:
            bgr_to_i420(view, out=pinned)
    torch.cuda.synchronize()


chain(True)                                                                # warm-up (annotates the frames once more)
annotate = {}
for name, to_host in (("hbm_frames_per_s", False), ("i420_to_pinned_host_frames_per_s", True)):
    for i in range(batches):                                               # fresh, unannotated frames
        gen.generate_batch_device(n, start_frame=i * n, out=stream[i])
    det.reset()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    chain(to_host)
    annotate[name] = batches * n / (time.perf_counter() - t0)
det.close()

print(json.dumps({
    "card_name_power_limit": card(), "resolution": [w, h], "frames": n,
    "kernel": {"ms": k_ms, "gb_per_s_at_4_5_bytes_per_px": k_gbs, "frames_per_s": n / (k_ms * 1e-3),
               "d2d_copy_gb_per_s": c_gbs, "share_of_d2d_copy": k_gbs / c_gbs},
    "d2h": d2h, "annotate": dict(annotate, batches=batches),
    "checked_against_cv2": "sampled frames of the device, pinned and pageable outputs"}))
