"""Decoder output at camera resolution into the lane path, on the GPU: one JSON line per measurement.

1. Kernel: 256 x 1080p NV12 -> 640x480 BGR, device-resident, the fused kernel (FrameIngest((640, 480)).from_nv12)
   against k0_nv12 + k0_resize (FrameIngest(None).from_nv12, then resize_batch), CUDA events, the two alternated in one
   process.  Touched bytes = NV12 bytes of the source rows / columns the taps read + the destination; the source
   (796 MB) is larger than L2.
2. End to end: detect_batch_nv12(pinned host 1080p NV12, target_size=(640, 480)) frames/s against a plain pinned copy
   of the same bytes (pcie_frac) and against the host route without the fused call (numpy NV12 -> full-size BGR on
   the host -> resized frame on the host -> detect_batch: 17.4 MB over PCIe per frame instead of 3.1 MB).
3. Whether the first batch matched cv2: the fused kernel's frames byte for byte, and the records of the e2e call
   against detect_batch of the cv2-prepared frames on a fresh detector.

Every line carries the device name and power limit read in the same run.
"""
import json
import os
import subprocess
import sys
import time

import cv2
import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multimodal_autonomous_driving_perception_and_planning_b200 import FrameIngest, LaneDetector  # noqa: E402
from multimodal_autonomous_driving_perception_and_planning_b200.generators import SyntheticDataGenerator  # noqa: E402
from oracle import nv12 as onv  # noqa: E402

HBM_GBS = 6556.0                      # measured HBM3e copy bandwidth of one B200 (DESIGN.md)
SW, SH, DW, DH, N = 1920, 1080, 640, 480, 256


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        out = "unknown"
    return {"device": name, "power_limit": out or "unknown"}


def emit(info, **kw):
    print(json.dumps({**kw, **info}), flush=True)


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    info = device_info()
    g = SyntheticDataGenerator(SW, SH)
    base = np.stack([onv.bgr_to_nv12_for_tests(g.generate_frame_with_vehicles()) for _ in range(16)])
    host = np.concatenate([base] * (N // len(base)))
    want = np.stack([cv2.resize(cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12), (DW, DH)) for f in host[:16]])

    # ---- 1. fused kernel vs the two-kernel composition, device-resident
    src = torch.from_numpy(host).cuda()
    fused, conv, rsz = FrameIngest((DW, DH)), FrameIngest(None), FrameIngest((DW, DH))
    run_fused = lambda: fused.from_nv12(src)                       # noqa: E731
    run_two = lambda: rsz.resize_batch(conv.from_nv12(src))        # noqa: E731
    out_f, out_t = run_fused(), run_two()
    torch.cuda.synchronize()
    match_kernel = bool(np.array_equal(out_f[:16].cpu().numpy(), want) and torch.equal(out_f, out_t))
    for _ in range(3):
        run_fused(), run_two()
    ms_f, ms_t = [], []
    for _ in range(5):                                            # alternate the two
        ms_f.append(timed(run_fused, 10))
        ms_t.append(timed(run_two, 10))
    rows, cols = min(SH, 2 * DH), min(SW, 2 * DW)
    touched = N * (rows * cols * 3 // 2 + DH * DW * 3)
    t_f, t_t = float(np.median(ms_f)), float(np.median(ms_t))
    emit(info, probe="ingest_kernel", shape=f"{N} x {SW}x{SH} NV12 -> {DW}x{DH} BGR", fused_ms=t_f, two_kernel_ms=t_t,
         fused_ms_all=ms_f, two_kernel_ms_all=ms_t, speedup=t_t / t_f, touched_bytes=touched,
         fused_GBps=touched / (t_f / 1e3) / 1e9, frac_of_measured_hbm=touched / (t_f / 1e3) / 1e9 / HBM_GBS,
         bit_exact_vs_cv2=match_kernel)
    del src, out_f, out_t
    torch.cuda.empty_cache()

    # ---- 2. end to end from pinned host memory
    pinned_t = torch.empty(host.shape, dtype=torch.uint8).pin_memory()
    pinned = pinned_t.numpy()
    pinned[...] = host
    dev = torch.empty(host.shape, dtype=torch.uint8, device="cuda")
    copy_ms = float(np.median([timed(lambda: dev.copy_(pinned_t, non_blocking=True), 5) for _ in range(3)]))

    det = LaneDetector(max_batch=128)
    det.detect_batch_nv12(pinned[:128], target_size=(DW, DH))     # warm-up: contexts, tap tables, staging
    det.reset()
    first = det.detect_batch_nv12(pinned[:16], target_size=(DW, DH))
    got_first = det.last_records.copy()
    ref = LaneDetector(max_batch=16)
    ref.detect_batch(want)
    match_e2e = bool(got_first.tobytes() == ref.last_records.tobytes()) and len(first) == 16
    walls = []
    for _ in range(5):
        t0 = time.perf_counter()
        det.detect_batch_nv12(pinned, target_size=(DW, DH))
        walls.append(time.perf_counter() - t0)
    wall = float(np.median(walls))

    # the host route before the fused call: convert (NV12 in, full-size BGR out), resize (BGR in, target out), detect
    old = LaneDetector(max_batch=128)
    old_route = lambda frames: old.detect_batch(rsz.resize_batch(conv.from_nv12(frames)))   # noqa: E731
    old_route(host[:128])
    old_walls = []
    for _ in range(3):
        t0 = time.perf_counter()
        old_route(host)
        old_walls.append(time.perf_counter() - t0)
    old_wall = float(np.median(old_walls))
    fps, copy_fps, old_fps = N / wall, N / (copy_ms / 1e3), N / old_wall
    emit(info, probe="ingest_e2e", shape=f"{N} x {SW}x{SH} NV12 pinned host -> detect at {DW}x{DH}",
         frames_per_s=fps, wall_s_all=walls, plain_pinned_copy_frames_per_s=copy_fps, pcie_frac=fps / copy_fps,
         old_route="numpy: FrameIngest(None).from_nv12, FrameIngest(target).resize_batch, detect_batch", old_route_frames_per_s=old_fps,
         speedup_vs_old_route=fps / old_fps, first_batch_matches_cv2=match_e2e, dense_reruns=det.dense_reruns)
    det.close()
    old.close()
    ref.close()


if __name__ == "__main__":
    main()
