"""Camera frames of one layout into the lane path, on the GPU: prints one JSON line with the card's name and power
limit.

    python tools/layout_probe.py --layout bayer_rggb|bayer_bggr|bayer_grbg|bayer_gbrg|uyvy|yuyv [--parent-lib PATH]

1. ``kernel``: device time (CUDA events, median of alternated rounds) of 64 device-resident 1080p frames through
   - the layout -> BGR at 1080p (Bayer: k0_ingest_resize on identity taps; 4:2:2: k0_yuv422_vec) and the layout ->
     640x480 (k0_ingest_resize),
   - NV12 -> BGR at 1080p (k0_nv12) and NV12 -> 640x480 (k0_ingest_resize),
   each against a device-to-device copy that moves the bytes of the layout -> BGR at the same size per 1080p pixel
   (Bayer 4 B: 1 B/px in and 3 B/px out; 4:2:2 5 B), half read and half written.  The sources (133 MB Bayer, 265 MB
   4:2:2, 199 MB NV12) are larger than L2.
2. ``e2e``: frames/s of ``detect_batch_bayer`` / ``detect_batch_yuv422``, ``detect_batch_nv12`` and ``detect_batch``
   (BGR) on 128 pinned host 1080p frames detected at 640x480, and of a plain pinned host-to-device copy of the layout's
   bytes.  Before timing, the first 16 frames' records are compared with ``detect_batch`` of the cv2-prepared frames.
3. ``rig_ingest``: device time of k0_rig_ingest (torch.profiler) on the mixed rig of tools/rig_ingest_probe.py (1 x 4K
   NV12, 4 x 1936x1216 NV12, 2 x 720p I420, 1 x 1080p BGR; 32 frames each) at 640x480.
The kernel and rig arms run with this tree's library and, given ``--parent-lib``, with a build of the parent commit,
in alternated child processes (3 each); ``kernel`` reports this tree's medians and every child's.
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
    sys.exit("layout_probe: no CUDA device (the probe measures the GPU; there is nothing to fall back to)")

from bgr_yuv420 import bgr_to_i420, bgr_to_nv12  # noqa: E402
from multimodal_autonomous_driving_perception_and_planning_b200 import FrameIngest, LaneDetector  # noqa: E402
from util import gen_frames  # noqa: E402

SW, SH, DW, DH = 1920, 1080, 640, 480
LAYOUT = sys.argv[sys.argv.index("--layout") + 1]
BAYER = LAYOUT.startswith("bayer_")
if LAYOUT not in ("bayer_rggb", "bayer_bggr", "bayer_grbg", "bayer_gbrg", "uyvy", "yuyv"):
    sys.exit(f"layout_probe: --layout {LAYOUT!r} is not a Bayer or 4:2:2 layout")
PATTERN = LAYOUT.removeprefix("bayer_")
ARM = "bayer" if BAYER else LAYOUT                       # the JSON's name of the layout's arms
COPY_BPP = 4 if BAYER else 5                             # bytes per pixel of the layout -> BGR at the same size


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


def cv2_code(kind):
    import cv2
    if BAYER:
        return getattr(cv2, "COLOR_Bayer" + PATTERN.upper() + "2BGR")
    return {"uyvy": (cv2.COLOR_BGR2YUV_UYVY, cv2.COLOR_YUV2BGR_UYVY),
            "yuyv": (cv2.COLOR_BGR2YUV_YUY2, cv2.COLOR_YUV2BGR_YUY2)}[LAYOUT][kind == "to_bgr"]


def scenes(n):
    import cv2
    from oracle import bayer as ob
    bgr = np.stack(gen_frames(SW, SH, 16, start=700))
    bgr = np.concatenate([bgr] * (n // 16))
    cam = [ob.mosaic_of_bgr(f, PATTERN) if BAYER else cv2.cvtColor(f, cv2_code("from_bgr")) for f in bgr]
    return bgr, np.stack(cam), np.stack([bgr_to_nv12(f) for f in bgr])


def convert(ing, frames):
    return ing.from_bayer(frames, PATTERN) if BAYER else ing.from_yuv422(frames, LAYOUT)


def detect(det, frames, **kw):
    return det.detect_batch_bayer(frames, PATTERN, **kw) if BAYER else det.detect_batch_yuv422(frames, LAYOUT, **kw)


def kernels():
    n = 64
    _, cam, nv12 = scenes(n)
    cam_d, nv12_d = torch.from_numpy(cam).cuda(), torch.from_numpy(nv12).cuda()
    copy_src = torch.empty(n * SH * SW * COPY_BPP // 2, dtype=torch.uint8, device="cuda")
    copy_dst = torch.empty_like(copy_src)
    full, small = FrameIngest(None), FrameIngest((DW, DH))
    arms = {
        f"{ARM}_1080p_same_size": lambda: convert(full, cam_d),
        f"{ARM}_1080p_to_640x480": lambda: convert(small, cam_d),
        "nv12_1080p_same_size": lambda: full.from_nv12(nv12_d),
        "nv12_1080p_to_640x480": lambda: small.from_nv12(nv12_d),
        f"d2d_copy_{COPY_BPP}B_per_px": lambda: copy_dst.copy_(copy_src),
    }
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in arms}
    for _ in range(7):
        for k, fn in arms.items():
            ms[k].append(timed(fn, 5))
    med = {k: float(np.median(v)) for k, v in ms.items()}
    del cam_d, nv12_d, copy_src, copy_dst
    torch.cuda.empty_cache()
    return med


def kernel_summary(meds):
    """``kernel``'s JSON from every child's medians per library: this tree's median over its children, and each child's
    values for the spread."""
    n, copy_key = 64, f"d2d_copy_{COPY_BPP}B_per_px"
    med = {k: float(np.median([m[k] for m in meds["this_tree"]])) for k in meds["this_tree"][0]}
    copy = med[copy_key]
    return {"frames": n, "ms_per_batch": {k: round(v, 4) for k, v in med.items()},
            "copy_GBps": round(n * SH * SW * COPY_BPP / (copy / 1e3) / 1e9, 1),
            "share_of_copy": {k: round(copy / v, 3) for k, v in med.items() if k != copy_key},
            "ms_per_batch_all": {lib: {k: [round(m[k], 4) for m in ms] for k in ms[0]} for lib, ms in meds.items()}}


def e2e():
    import cv2
    n = 128
    bgr, cam, nv12 = scenes(n)
    want = np.stack([cv2.resize(cv2.cvtColor(f, cv2_code("to_bgr")), (DW, DH)) for f in cam[:16]])
    ref = LaneDetector(max_batch=16)
    ref.detect_batch(want)
    check = LaneDetector(max_batch=16)
    detect(check, cam[:16], target_size=(DW, DH))
    match = check.last_records.tobytes() == ref.last_records.tobytes()
    ref.close()
    check.close()
    pinned = {}
    for k, a in ((ARM, cam), ("nv12", nv12), ("bgr", bgr)):
        t = torch.empty(a.shape, dtype=torch.uint8).pin_memory()
        t.numpy()[...] = a
        pinned[k] = t
    dev = torch.empty(cam.shape, dtype=torch.uint8, device="cuda")
    copy_ms = float(np.median([timed(lambda: dev.copy_(pinned[ARM], non_blocking=True), 5) for _ in range(5)]))
    det = LaneDetector(max_batch=n)
    arms = {
        ARM: lambda: detect(det, pinned[ARM].numpy(), target_size=(DW, DH)),
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
    return {"frames": n, "frames_per_s": fps, f"plain_pinned_copy_of_{ARM}_frames_per_s": round(copy_fps, 1),
            f"{ARM}_share_of_copy": round(fps[ARM] / copy_fps, 3), "h2d_GBps": round(cam.nbytes / (copy_ms / 1e3) / 1e9, 1),
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


def alternated(parent_lib):
    """Alternated child processes, each timing the kernel arms and k0_rig_ingest with one library: ``kernel`` and
    ``rig_ingest``'s JSON."""
    libs = {"this_tree": None}
    if parent_lib:
        libs["parent"] = parent_lib
    ms, kern, recs = {k: [] for k in libs}, {k: [] for k in libs}, {}
    for _ in range(3):
        for k, lib in libs.items():
            env = dict(os.environ)
            if lib:
                env["LANE_B200_LIB"] = os.path.abspath(lib)
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "--layout", LAYOUT, "--child"], env=env,
                                 capture_output=True, text=True, timeout=900)
            if out.returncode:
                raise RuntimeError(out.stderr[-3000:])
            r = json.loads(out.stdout.strip().splitlines()[-1])
            kern[k].append(r["kernel_ms"])
            ms[k].append(r["k0_rig_ingest_ms"])
            recs[k] = r["records_sha"]
    med = {k: float(np.median(v)) for k, v in ms.items()}
    rig = {"k0_rig_ingest_ms": {k: round(v, 4) for k, v in med.items()}, "k0_rig_ingest_ms_all": ms,
           "records_equal": len(set(recs.values())) == 1}
    if "parent" in med:
        rig["change_vs_parent"] = round(med["this_tree"] / med["parent"] - 1, 4)
    return kernel_summary(kern), rig


def main():
    if "--child" in sys.argv:
        import hashlib
        kern = kernels()
        ms, recs = rig_kernel_ms()
        print(json.dumps({"kernel_ms": kern, "k0_rig_ingest_ms": ms,
                          "records_sha": hashlib.sha256(recs.tobytes()).hexdigest()}))
        return
    parent = sys.argv[sys.argv.index("--parent-lib") + 1] if "--parent-lib" in sys.argv else None
    kernel, rig = alternated(parent)
    result = {"probe": LAYOUT, "card": card(), "device": torch.cuda.get_device_name(), "kernel": kernel, "e2e": e2e(),
              "rig_ingest": rig}
    print(json.dumps(result), flush=True)


if __name__ == "__main__":
    main()
