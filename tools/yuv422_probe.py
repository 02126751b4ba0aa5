"""Packed YUV 4:2:2 camera frames into the lane path, on the GPU: prints one JSON line with the card's name and power
limit.

    python tools/yuv422_probe.py [--parent-lib PATH]

1. ``kernel``: device time (CUDA events, median of alternated rounds) of 64 device-resident 1080p UYVY frames through
   - UYVY -> BGR at 1080p (k0_yuv422_vec) and UYVY -> 640x480 (k0_yuv422_resize),
   - NV12 -> BGR at 1080p (k0_nv12) and NV12 -> 640x480 (k0_yuv420_resize),
   against a device-to-device copy that moves 5 B per 1080p pixel (reads 2.5 B/px and writes 2.5 B/px: the traffic of
   UYVY -> BGR at the same size, 2 B/px in and 3 B/px out).  The UYVY sources (265 MB) are larger than L2.
2. ``e2e``: frames/s of ``detect_batch_yuv422`` / ``detect_batch_nv12`` / ``detect_batch`` (BGR) on 128 pinned host
   1080p frames detected at 640x480, and of a plain pinned host-to-device copy of the UYVY bytes.  Before timing, the
   first 16 UYVY frames' records are compared with ``detect_batch`` of the cv2-prepared frames.
3. ``rig_ingest``: device time of k0_rig_ingest (torch.profiler) on the mixed rig of tools/rig_ingest_probe.py (1 x 4K
   NV12, 4 x 1936x1216 NV12, 2 x 720p I420, 1 x 1080p BGR; 32 frames each; no 4:2:2 camera) at 640x480, with this
   tree's library and, given ``--parent-lib``, with a build of the parent commit, in alternated child processes.
"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

if not torch.cuda.is_available():
    sys.exit("yuv422_probe: no CUDA device (the probe measures the GPU; there is nothing to fall back to)")

from multimodal_autonomous_driving_perception_and_planning_b200 import _native  # noqa: E402

if os.environ.get("YUV422_PROBE_PARENT"):
    _native._PROTOS.pop("lane_yuv422_to_bgr_batch")        # the parent's library has no 4:2:2 entry

from bgr_yuv420 import bgr_to_i420, bgr_to_nv12  # noqa: E402
from multimodal_autonomous_driving_perception_and_planning_b200 import FrameIngest, LaneDetector  # noqa: E402
from util import gen_frames  # noqa: E402

SW, SH, DW, DH = 1920, 1080, 640, 480


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        return q.stdout.strip() or q.stderr.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi unavailable: {e}"


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def scenes(n):
    import cv2
    bgr = np.stack(gen_frames(SW, SH, 16, start=700))
    bgr = np.concatenate([bgr] * (n // 16))
    return bgr, np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2YUV_UYVY) for f in bgr]), np.stack([bgr_to_nv12(f) for f in bgr])


def kernels():
    n = 64
    _, uyvy, nv12 = scenes(n)
    uyvy_d, nv12_d = torch.from_numpy(uyvy).cuda(), torch.from_numpy(nv12).cuda()
    copy_src = torch.empty(n * SH * SW * 5 // 2, dtype=torch.uint8, device="cuda")
    copy_dst = torch.empty_like(copy_src)
    full, small = FrameIngest(None), FrameIngest((DW, DH))
    arms = {
        "uyvy_1080p_same_size": lambda: full.from_yuv422(uyvy_d, "uyvy"),
        "uyvy_1080p_to_640x480": lambda: small.from_yuv422(uyvy_d, "uyvy"),
        "nv12_1080p_same_size": lambda: full.from_nv12(nv12_d),
        "nv12_1080p_to_640x480": lambda: small.from_nv12(nv12_d),
        "d2d_copy_5B_per_px": lambda: copy_dst.copy_(copy_src),
    }
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in arms}
    for _ in range(7):
        for k, fn in arms.items():
            ms[k].append(timed(fn, 5))
    med = {k: float(np.median(v)) for k, v in ms.items()}
    copy = med["d2d_copy_5B_per_px"]
    out = {"frames": n, "ms_per_batch": {k: round(v, 4) for k, v in med.items()},
           "copy_GBps": round(n * SH * SW * 5 / (copy / 1e3) / 1e9, 1),
           "share_of_copy": {k: round(copy / v, 3) for k, v in med.items() if k != "d2d_copy_5B_per_px"}}
    del uyvy_d, nv12_d, copy_src, copy_dst
    torch.cuda.empty_cache()
    return out


def e2e():
    import cv2
    n = 128
    bgr, uyvy, nv12 = scenes(n)
    want = np.stack([cv2.resize(cv2.cvtColor(f, cv2.COLOR_YUV2BGR_UYVY), (DW, DH)) for f in uyvy[:16]])
    ref = LaneDetector(max_batch=16)
    ref.detect_batch(want)
    check = LaneDetector(max_batch=16)
    check.detect_batch_yuv422(uyvy[:16], "uyvy", target_size=(DW, DH))
    match = check.last_records.tobytes() == ref.last_records.tobytes()
    ref.close()
    check.close()
    pinned = {}
    for k, a in (("uyvy", uyvy), ("nv12", nv12), ("bgr", bgr)):
        t = torch.empty(a.shape, dtype=torch.uint8).pin_memory()
        t.numpy()[...] = a
        pinned[k] = t
    dev = torch.empty(uyvy.shape, dtype=torch.uint8, device="cuda")
    copy_ms = float(np.median([timed(lambda: dev.copy_(pinned["uyvy"], non_blocking=True), 5) for _ in range(5)]))
    det = LaneDetector(max_batch=n)
    arms = {
        "uyvy": lambda: det.detect_batch_yuv422(pinned["uyvy"].numpy(), "uyvy", target_size=(DW, DH)),
        "nv12": lambda: det.detect_batch_nv12(pinned["nv12"].numpy(), target_size=(DW, DH)),
        "bgr": lambda: det.detect_batch(pinned["bgr"].numpy(), target_size=(DW, DH)),
    }
    for fn in arms.values():
        fn()
    walls = {k: [] for k in arms}
    for _ in range(5):
        for k, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            walls[k].append(time.perf_counter() - t0)
    fps = {k: round(n / float(np.median(v)), 1) for k, v in walls.items()}
    copy_fps = n / (copy_ms / 1e3)
    det.close()
    return {"frames": n, "frames_per_s": fps, "plain_pinned_copy_of_uyvy_frames_per_s": round(copy_fps, 1),
            "uyvy_share_of_copy": round(fps["uyvy"] / copy_fps, 3), "h2d_GBps": round(uyvy.nbytes / (copy_ms / 1e3) / 1e9, 1),
            "first_16_match_cv2_prepared": bool(match), "dense_reruns": det.dense_reruns}


def rig_kernel_ms(calls=10):
    """k0_rig_ingest device time per call on tools/rig_ingest_probe.py's rig (this process's library)."""
    from torch.profiler import ProfilerActivity, profile
    rig = [("nv12", 3840, 2160)] + [("nv12", 1936, 1216)] * 4 + [("i420", 1280, 720)] * 2 + [("bgr", 1920, 1080)]
    cams = []
    for s, (lay, w, h) in enumerate(rig):
        bgr = gen_frames(w, h, 8, start=1000 * s)
        frames = bgr if lay == "bgr" else [(bgr_to_nv12 if lay == "nv12" else bgr_to_i420)(f) for f in bgr]
        cams.append(torch.from_numpy(np.stack([frames[t % 8] for t in range(32)])).cuda())
    layouts = [lay for lay, _, _ in rig]
    det = LaneDetector(max_batch=256)
    det.detect_rig(cams, layouts, target_size=(DW, DH))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            det.detect_rig(cams, layouts, target_size=(DW, DH))
        torch.cuda.synchronize()
    us = sum(e.device_time_total for e in prof.key_averages() if "k0_rig_ingest" in e.key)
    recs = det.last_records.copy()
    det.close()
    return us / calls / 1e3, recs


def rig_ingest(parent_lib):
    """Alternated child processes, each timing k0_rig_ingest with one library."""
    libs = {"this_tree": None}
    if parent_lib:
        libs["parent"] = parent_lib
    ms, recs = {k: [] for k in libs}, {}
    for _ in range(3):
        for k, lib in libs.items():
            env = dict(os.environ)
            if lib:
                env["LANE_B200_LIB"], env["YUV422_PROBE_PARENT"] = os.path.abspath(lib), "1"
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--rig-child"], env=env, capture_output=True,
                                 text=True, timeout=900)
            if out.returncode:
                raise RuntimeError(out.stderr[-3000:])
            r = json.loads(out.stdout.strip().splitlines()[-1])
            ms[k].append(r["k0_rig_ingest_ms"])
            recs[k] = r["records_sha"]
    med = {k: float(np.median(v)) for k, v in ms.items()}
    out = {"k0_rig_ingest_ms": {k: round(v, 4) for k, v in med.items()}, "k0_rig_ingest_ms_all": ms,
           "records_equal": len(set(recs.values())) == 1}
    if "parent" in med:
        out["change_vs_parent"] = round(med["this_tree"] / med["parent"] - 1, 4)
    return out


def main():
    if "--rig-child" in sys.argv:
        import hashlib
        ms, recs = rig_kernel_ms()
        print(json.dumps({"k0_rig_ingest_ms": ms, "records_sha": hashlib.sha256(recs.tobytes()).hexdigest()}))
        return
    parent = sys.argv[sys.argv.index("--parent-lib") + 1] if "--parent-lib" in sys.argv else None
    result = {"probe": "yuv422", "card": card(), "device": torch.cuda.get_device_name(), "kernel": kernels(), "e2e": e2e(),
              "rig_ingest": rig_ingest(parent)}
    print(json.dumps(result), flush=True)


if __name__ == "__main__":
    main()
