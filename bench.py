#!/usr/bin/env python
"""Headline benchmark: 1080p lane-detect frames/s on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the whole hot path (K1 blur+hist, K2 Canny+hysteresis, ROI compaction,
K4 HoughLinesP, K5 fit/EMA/offset, result copy-back) over one batch of synthetic 1920x1080 frames
per GPU (BASELINE config 2: 256 frames on one B200).  Scaling is weak: every rank processes its own
camera streams with no collective on the data path; the per-frame records are gathered to rank 0
with one NCCL gather per step (BASELINE config 3 semantics).

value   frames/s with the frames already resident in HBM when the timed region starts.
e2e     frames/s through the public API (LaneDetector.detect_batch) with HOST (pinned) frames:
        host->device copy and device->host records inside the timed region.  e2e.pcie_frac relates the bytes/s it moves to
        a plain pinned cudaMemcpyAsync of the same payload measured in the same process (with every rank copying at the
        same time): the host->device link is what bounds it.  e2e_nv12 is the same leg with the frames in a video
        decoder's NV12 layout (1.5 B/px over the link, converted to BGR on the device, bit-exact vs cv2).
roofline  the EDGE PATH -- everything from BGR frames to the Canny edge map and ROI point list: k1_probe + k1_fused
        (gray + blur + histogram + Sobel + NMS), k2t_threshold, k2_canny_cluster -- algorithmic 4 B/px (3 B/px BGR read +
        1 B/px edge-map write, SURVEY.md 8d) over its CUDA-event time measured live on the launching stream;
        roofline.k1_fused is the same figure for the fused kernel's stage alone.
cpu_baseline  the reference's OpenCV path (oracle/cv2_pipeline.py: the reference call sequence on
        the same cv2/numpy) on this box's host cores, bounded sample.
--config3  BASELINE config 3 instead of the weak-scaling default: an 8-camera 1080p rig, --frames-per-stream frames per
        camera, whole streams sharded over the N ranks (8/N cameras per GPU, strong scaling), records gathered to rank 0.
--dump-outputs DIR  after the timed steps, rank 0 writes what its last timed step returned to the caller (the per-frame
        records of every native batch of that step, and the smoothing state after it) as DIR/<name>.npy, float64.  The
        inputs are seeded, so two builds run with the same arguments can be compared array for array.
"""
import argparse
import collections
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

H, W = 1080, 1920
ALGO_BYTES_PER_FRAME = 4 * H * W          # SURVEY.md 8(d)
DUMP_BYTES = 64 << 20                     # --dump-outputs: larger outputs are written as a seeded sample of frames


# ------------------------------------------------------------------------------------ outputs
def dump_outputs(path, recs, state_fit, state_valid, limit=DUMP_BYTES):
    """Write the records ``recs`` (RECORD_DTYPE, one per frame) field by field as ``path/<field>.npy`` (the fields of
    ``side`` as ``side_<field>.npy``, shaped [frames, 2, ...]), plus ``frame_index.npy`` (which records were written) and
    the smoothing state ``state_fit.npy`` / ``state_valid.npy``; every array float64 (the int32 fields convert exactly).
    If all frames would exceed ``limit`` bytes, a fixed seeded sample of frames is written instead."""
    cols = {f"side_{k}": recs["side"][k] for k in recs.dtype["side"].base.names}
    cols.update((k, recs[k]) for k in recs.dtype.names if k != "side")
    per_frame = 8 * (1 + sum(int(np.prod(a.shape[1:], dtype=np.int64)) for a in cols.values()))
    fixed = 8 * (state_fit.size + state_valid.size) + 1024 * (len(cols) + 3)      # + room for the .npy headers
    keep = max(0, min(len(recs), (limit - fixed) // per_frame))
    idx = np.arange(len(recs))
    if keep < len(recs):
        idx = np.sort(np.random.default_rng(0).choice(len(recs), keep, replace=False))
    os.makedirs(path, exist_ok=True)
    out = dict(((k, a[idx]) for k, a in cols.items()), frame_index=idx, state_fit=state_fit, state_valid=state_valid)
    for k, a in out.items():
        np.save(os.path.join(path, k + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


# ------------------------------------------------------------------------------------ CPU arm
def _cpu_worker(args):
    """One host core: the reference's cv2 path over its own camera stream (cv2 threads = 1)."""
    stream, n_frames, width, height = args
    import cv2
    cv2.setNumThreads(1)
    from multimodal_autonomous_driving_perception_and_planning_b200.generators import SyntheticDataGenerator
    from oracle.cv2_pipeline import Cv2LaneOracle
    distinct = min(n_frames, 16)
    frames = SyntheticDataGenerator(width, height).generate_batch(distinct, start_frame=stream * 1000)
    det = Cv2LaneOracle()
    for i in range(3):
        det.detect(frames[i % distinct])
    det.reset()
    t0 = time.perf_counter()
    found = 0
    for i in range(n_frames):
        lf, rf = det.detect(frames[i % distinct])
        det.offset(width, lf, rf)
        found += (lf is not None) + (rf is not None)
    return n_frames, time.perf_counter() - t0, found


def cpu_reference_fps(frames_per_worker, workers=None):
    import multiprocessing as mp
    workers = workers or os.cpu_count() or 1
    ctx = mp.get_context("fork")
    with ctx.Pool(workers) as pool:
        res = pool.map(_cpu_worker, [(s, frames_per_worker, W, H) for s in range(workers)])
    total = sum(r[0] for r in res)
    slowest = max(r[1] for r in res)
    return total / slowest, workers, total, slowest


def cpu_info():
    model = "unknown"
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    import cv2
    return {"cpu_model": model, "os_cpu_count": os.cpu_count(), "cv2": cv2.__version__, "numpy": np.__version__}


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    # the sample's own timestamp is used (lines reach the pipe in bursts, so arrival time is not sampling time)
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "20",
                 "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        import datetime
        skew = time.perf_counter() - time.time()          # wall clock -> perf_counter
        for line in self.proc.stdout:
            line = line.strip()
            stamp, _, rest = line.partition(",")
            try:
                t = datetime.datetime.strptime(stamp.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp() + skew
            except ValueError:
                t = time.perf_counter()
            self.lines.append((t, rest.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        rows = [l for (t, l) in self.lines if t0 <= t <= t1] or [l for (_, l) in self.lines[-3:]]
        for l in rows:
            p = [x.strip() for x in l.split(",")]
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


class NvmlSampler:
    """SM clock and clock-event reasons straight from NVML every ~2 ms (nvidia-smi's loop cannot go below ~20 ms, which is
    as long as the whole timed region): the samples that fall inside the timed region itself."""

    def __init__(self, index):
        self.samples, self.stop_flag, self.ok = [], False, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
        except Exception:
            self.ok = False

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                t = time.perf_counter()
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.samples.append((t, sm, rs))
            except Exception:
                pass
            time.sleep(0.002)

    def window(self, t0, t1):
        self.stop_flag = True
        if not self.ok:
            return None
        nv = self.nv
        rows = [(sm, rs) for (t, sm, rs) in self.samples if t0 <= t <= t1]
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        reasons = sorted(k for k, bit in names.items() if any(rs & bit for _, rs in rows))
        return {"samples": len(rows), "sm_mhz": float(np.median([sm for sm, _ in rows])) if rows else None,
                "sm_min_mhz": min((sm for sm, _ in rows), default=None), "sm_max_mhz": self.max_sm, "reasons": reasons,
                "source": "NVML polled every ~2 ms"}


# ------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=256, help="frames per GPU per step")
    ap.add_argument("--distinct", type=int, default=64, help="distinct generator frames per stream (tiled in time)")
    ap.add_argument("--cpu-frames", type=int, default=1024, help="CPU baseline sample: frames per host core")
    ap.add_argument("--skip-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--skip-e2e", action="store_true", help="skip the e2e leg (profiling runs)")
    ap.add_argument("--config3", action="store_true", help="BASELINE config 3: 8 cameras sharded by stream (strong scaling)")
    ap.add_argument("--frames-per-stream", type=int, default=512, help="config 3: frames per camera per step")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        args.gpus = world

    base = {"metric": "1080p lane-detect frames/s", "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "data": "synthetic (SyntheticDataGenerator 1920x1080, per-stream phase 1000, rasterised on the device)"}
    workload = (f"batch of {args.frames} synthetic 1920x1080 frames per GPU (BASELINE configs[1]; "
                f"{args.distinct} distinct generator frames per stream tiled in time), full detect path")

    # ---------------------------------------------------------------- reference arm (CPU, rank 0 only)
    if args.impl == "reference":
        if rank != 0:
            return
        for _ in range(min(args.warmup, 1)):
            cpu_reference_fps(8)
        vals = []
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fps, cores, total, slowest = cpu_reference_fps(128)    # bounded: ~1.5 s of 16-core work per step
            vals.append((fps, total, slowest))
        fps = sum(v[1] for v in vals) / sum(v[2] for v in vals)
        sample = (f"{vals[0][1]} frames/step ({vals[0][1] // cores} per core) of the same 1080p generator streams, "
                  f"{cores} processes x cv2.setNumThreads(1), sequential detect() per stream")
        base["data"] = "synthetic (SyntheticDataGenerator 1920x1080, per-stream phase 1000, drawn by cv2 on the host: the same frames)"
        out = dict(base, impl="reference", value=fps, ms_per_step=1e3 * sum(v[2] for v in vals) / args.steps,
                   dtype="u8/int32/f64", config={"workload": workload, "host": cpu_info()},
                   cpu_baseline={"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
                   e2e={"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                   wall_s=time.perf_counter() - t0)
        print(json.dumps(out))
        return

    # ---------------------------------------------------------------- CPU baseline first (before CUDA init)
    cpu_baseline = None
    if rank == 0 and args.gpus == 1 and not args.skip_cpu:
        fps, cores, total, slowest = cpu_reference_fps(args.cpu_frames)
        cpu_baseline = {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                        "sample": f"{total} frames ({args.cpu_frames} per core x {cores} processes, cv2 threads=1 each) "
                                  f"of the same 1080p generator streams in {slowest:.1f} s; "
                                  f"oracle/cv2_pipeline.py = the reference call sequence on cv2 {cpu_info()['cv2']}",
                        "host": cpu_info()}

    import torch
    import torch.distributed as dist
    from multimodal_autonomous_driving_perception_and_planning_b200 import LaneDetector, _native

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    # ---- inputs: this rank's camera stream(s), generated on the device (no host rasterisation, no upload)
    from multimodal_autonomous_driving_perception_and_planning_b200 import SyntheticDataGenerator, bgr_to_nv12
    from multimodal_autonomous_driving_perception_and_planning_b200.distributed import RecordGatherer, streams_of_rank

    def make_stream(cam, t):
        """t frames of camera `cam` in HBM: --distinct generator frames (phase cam * 1000) rasterised ON THE DEVICE by
        k7_draw (bit-identical to the host cv2 generator: tests/test_gpu_draw.py), tiled in time."""
        d = min(args.distinct, t)
        base = SyntheticDataGenerator(W, H).generate_batch_device(d, start_frame=cam * 1000, device=local)
        idx = torch.arange(t, device=dev) % d
        return base.index_select(0, idx).contiguous()

    if args.config3:
        cams = streams_of_rank(8, world, rank)               # whole cameras per rank: 8/N each
        n = args.frames_per_stream                           # frames per native call = one camera's sequence
    else:
        cams = [rank]
        n = args.frames
    S = len(cams)
    t_gen = time.perf_counter()
    dev_streams = [make_stream(c, n) for c in cams]
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t_gen
    pinned = dev_streams[0][:min(n, args.frames)].cpu().pin_memory()                 # the e2e leg's host batch
    torch.cuda.synchronize()
    frames_step = S * n                                      # frames this rank processes per step

    det = LaneDetector(device=local, max_batch=n)
    ctx = det._context(H, W, n)                              # native context for n frames per call
    stream = torch.cuda.ExternalStream(ctx.stream(), device=dev)
    prev_fit = np.zeros((S, 2, 3), np.float64)
    prev_valid = np.zeros((S, 2), np.uint8)
    rec_bytes = _native.RECORD_DTYPE.itemsize * frames_step
    gatherer = RecordGatherer(n, dev) if world > 1 else None
    sids = [np.full(n, k, np.int32) for k in range(S)]

    # Streaming form of the C ABI: a step is one native batch per camera of this rank.  Batches are enqueued two deep with the
    # EMA state carried on the device (exactly the state chain of calling detect() frame after frame on one detector
    # per camera), so the GPU goes from one batch's last kernel to the next batch's first without waiting for the host; all
    # batches run in order on one stream.  The records of every batch are gathered to rank 0 (the path's only
    # collective, NCCL over NVLink) straight from the context's device copy: lane_ctx_records_device stays valid until the
    # batch after next is enqueued, and the context's stream waits for the gather before that slot is reused.
    state = {"queued": 0, "next": 0, "first": True, "last_recs": None, "last_bufs": None,
             "step_recs": collections.deque(maxlen=S)}                # the batches of the last step, camera order

    def enqueue_next():
        k = state["next"] % S
        if state["first"]:
            ctx.enqueue(dev_streams[k].data_ptr(), n, sids[k], S, prev_fit, prev_valid, 0.7, 1 - 0.7)   # explicit state
            state["first"] = False
        else:
            ctx.enqueue(dev_streams[k].data_ptr(), n, sids[k], S, None, None, 0.7, 1 - 0.7)            # state on the device
        state["next"] += 1
        state["queued"] += 1

    def run_batches(total, on_collect=None):
        """total batches through the two-deep queue; every collected batch is gathered (N > 1)."""
        done = 0
        issued = 0
        while issued < min(2, total):
            enqueue_next(); issued += 1
        while done < total:
            recs = ctx.collect(prev_fit, prev_valid)
            state["queued"] -= 1
            done += 1
            state["last_recs"] = recs
            state["step_recs"].append(recs)
            if on_collect:
                on_collect()
            if gatherer is not None:
                state["last_bufs"] = gatherer.gather_device(ctx.records_device_ptr(), to_host=False)
                # only the fit kernel that next writes this result slot waits for the collective (not the edge kernels)
                ctx.fence_records(torch.cuda.current_stream(dev).cuda_stream)
            if issued < total:
                enqueue_next(); issued += 1
        if gatherer is not None:
            stream.wait_stream(torch.cuda.current_stream(dev))   # timing events on the context's stream see the gathers
        state["first"] = True                                # the next run starts from the host copy of the state again

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    nvml_sampler = NvmlSampler(local) if rank == 0 else None
    t_load0 = time.perf_counter()
    run_batches(max(args.warmup, 3) * S)
    found = int(state["last_recs"]["side"]["valid"].sum())

    # ---- timed region: value (device-resident inputs).  No stage events here: outside profiling mode the context runs the
    # back half of a batch (PPHT, fit, record copies) on a second stream, so that the edge kernels of the next queued batch
    # fill the SMs the PPHT's last wave of frames leaves idle; events between the stages would serialise the two streams.
    stage_sum = {k: 0.0 for k in _native.STAGE_NAMES}
    launches = [0]

    def account():
        ms, ln = ctx.stage_ms()
        for k in stage_sum:
            stage_sum[k] += ms[k]
        launches[0] += sum(ln.values())

    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record(stream)
    run_batches(args.steps * S)              # every batch has been collected (host waited for its last copy) on return
    e1.record(stream)
    barrier()
    t1 = time.perf_counter()
    timed_window = (t0, t1)
    dev_ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, np.concatenate(state["step_recs"]), prev_fit, prev_valid)
    # ---- the same K steps once more with CUDA events between the stages (one stream): stage split, launch count and the
    # edge-path roofline come from this pass; its step time is reported beside the overlapped one
    ctx.set_profiling(True)
    barrier()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record(stream)
    run_batches(args.steps * S, account)
    p1.record(stream)
    barrier()
    serial_ms = p0.elapsed_time(p1)
    ctx.set_profiling(False)
    if world > 1:
        tm = torch.tensor([dev_ms], device=dev)
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        dev_ms = float(tm.item())
    total_frames = frames_step * args.steps
    if world > 1:
        tf = torch.tensor([total_frames], device=dev, dtype=torch.int64)
        dist.all_reduce(tf)
        total_frames = int(tf.item())
    value = total_frames / (dev_ms / 1e3)

    # ---- the same device-resident batches through the public Python API (LaneDetector.detect_batches: two batches in flight,
    # LaneLine objects built for every frame); reported beside `value`, which drives the C ABI's streaming calls directly
    api_fps = None
    if not args.config3:
        det.reset()
        reps = max(args.steps, 4)
        for _ in det.detect_batches([dev_streams[0]] * 3):
            pass
        barrier()
        ta = time.perf_counter()
        n_lanes = 0
        for lanes in det.detect_batches([dev_streams[0]] * reps):
            n_lanes += len(lanes)
        barrier()
        api_fps = n_lanes / (time.perf_counter() - ta)
        if world > 1:
            tt = torch.tensor([api_fps], device=dev)
            dist.all_reduce(tt)
            api_fps = float(tt.item())
        det.reset()

    # ---- multi-GPU correctness, outside the timed region: did rank 0 receive every rank's records?
    gather_verified, lanes_per_rank = None, None
    if world > 1:
        import hashlib
        local_hash = int.from_bytes(hashlib.sha256(state["last_recs"].tobytes()).digest()[:7], "little")
        hashes = [torch.zeros(1, dtype=torch.int64, device=dev) for _ in range(world)]
        dist.all_gather(hashes, torch.tensor([local_hash], dtype=torch.int64, device=dev))
        if rank == 0:
            got = [b.cpu().numpy().view(_native.RECORD_DTYPE) for b in state["last_bufs"]]
            mine = [int.from_bytes(hashlib.sha256(g.tobytes()).digest()[:7], "little") for g in got]
            gather_verified = mine == [int(h.item()) for h in hashes]
            lanes_per_rank = [int(g["side"]["valid"].sum()) for g in got]

    # ---- e2e: public API with host (pinned) frames, H2D + records D2H inside the timed region
    host_frames = pinned.numpy()
    ne = host_frames.shape[0]
    e2e_steps = 0 if args.skip_e2e else args.steps

    def e2e_leg(call, arg):
        det.reset()
        for _ in range(2 if e2e_steps else 0):
            call(arg)
        barrier()
        t = time.perf_counter()
        last = None
        for _ in range(e2e_steps):
            lanes = call(arg)
            last = det.get_lane_center_offset(W, *lanes[-1])
        barrier()
        sec = max(time.perf_counter() - t, 1e-9)
        if world > 1:
            tt = torch.tensor([sec], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            sec = float(tt.item())
        return args.gpus * ne * e2e_steps / sec, sec, last

    e2e_val, e2e_s, off = e2e_leg(det.detect_batch, host_frames)
    # the same leg with the frames in a decoder's NV12 layout: half the bytes over the link, converted on the device
    nv12_val, nv12_bytes = None, 0
    if e2e_steps:
        nv12 = torch.from_numpy(bgr_to_nv12(host_frames)).pin_memory().numpy()
        nv12_bytes = int(nv12.nbytes)
        nv12_val, _, _ = e2e_leg(det.detect_batch_nv12, nv12)
        del nv12
    # the step after the path (SURVEY 8f rank 3): draw_lanes + offset indicator for the whole batch in HBM, through the public
    # API (host lists of LaneLine in, annotated frames left on the device); reported beside the path, not part of `value`
    draw = None
    if e2e_steps and rank == 0:
        from multimodal_autonomous_driving_perception_and_planning_b200 import OverlayRenderer
        det.reset()
        lanes = det.detect_batch(dev_streams[0][:ne])
        offs = [det.get_lane_center_offset(W, l, r) for l, r in lanes]
        ov = OverlayRenderer()
        canvas = dev_streams[0][:ne].clone()
        det.draw_lanes_batch(canvas, lanes)
        ov.draw_lane_offset_indicator_batch(canvas, offs)
        torch.cuda.synchronize()
        reps = 5
        td = time.perf_counter()
        for _ in range(reps):
            det.draw_lanes_batch(canvas, lanes)
            ov.draw_lane_offset_indicator_batch(canvas, offs)
        torch.cuda.synchronize()
        draw = {"value": ne * reps / (time.perf_counter() - td), "unit": "frames/s",
                "api": "LaneDetector.draw_lanes_batch + OverlayRenderer.draw_lane_offset_indicator_batch (frames in HBM, "
                       "bit-exact vs cv2: tests/test_gpu_draw.py)"}
        del canvas
    # the roof of the e2e leg: a plain pinned copy of the same payload, every rank copying at the same time
    pcie_gbs = None
    if e2e_steps:
        dst = torch.empty(host_frames.nbytes, dtype=torch.uint8, device=dev)
        src = pinned.view(-1)
        quarter = (src.numel() + 3) // 4

        def plain_copy():
            for a in range(0, src.numel(), quarter):
                dst[a:a + quarter].copy_(src[a:a + quarter], non_blocking=True)

        for _ in range(2):
            plain_copy()
        barrier()
        tc = time.perf_counter()
        reps = max(3, e2e_steps // 2)
        for _ in range(reps):
            plain_copy()
        barrier()
        sec = max(time.perf_counter() - tc, 1e-9)
        if world > 1:
            tt = torch.tensor([sec], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            sec = float(tt.item())
        pcie_gbs = host_frames.nbytes * reps / sec / 1e9        # per GPU, with all N ranks copying
        del dst
    clocks = None
    if sampler:
        # nvidia-smi samples every 20 ms: the timed region alone is tens of ms, so the record spans everything that ran
        # under load (warm-up, timed region, e2e legs) and says how many samples fell inside the timed region itself
        clocks = sampler.stop(t_load0, time.perf_counter())
        clocks["window"] = "warm-up + timed region + e2e legs"
        clocks["samples_in_timed_region"] = sum(1 for (t, _) in sampler.lines if timed_window[0] <= t <= timed_window[1])
        if nvml_sampler is not None:
            clocks["timed_region"] = nvml_sampler.window(*timed_window)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        batches = args.steps * S
        k1_ms = stage_sum["blur_hist"] / batches             # per native batch of n frames
        canny_ms = (stage_sum["canny"] + stage_sum["compact"]) / batches
        edge_ms = k1_ms + canny_ms
        algo = n * ALGO_BYTES_PER_FRAME
        edge_achieved = algo / (edge_ms / 1e3) / 1e9 if edge_ms > 0 else 0.0
        k1_achieved = algo / (k1_ms / 1e3) / 1e9 if k1_ms > 0 else 0.0
        # dram__bytes_read.sum + dram__bytes_write.sum of the edge-path kernels of one 256 x 1080p batch, exported from the
        # committed ncu capture (profiles/r2_edge_traffic.json names the report and the per-kernel figures)
        traffic, traffic_src = None, None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "r2_edge_traffic.json")))
            if n == tr.get("frames_per_launch") and (W, H) == tuple(tr.get("resolution", ())):
                traffic, traffic_src = float(tr["edge_path_dram_bytes"]), "profiles/r2_edge_traffic.json"
        except (OSError, ValueError, KeyError):
            pass
        e2e_bytes_s = ne * ALGO_BYTES_PER_FRAME * 0.75 * e2e_steps / e2e_s if e2e_steps else 0.0   # 3 B/px per GPU
        out = dict(base, value=value, ms_per_step=dev_ms / args.steps, dtype="u8/int32/f64",
                   scaling="strong" if args.config3 else "weak",
                   config={"workload": workload if not args.config3 else
                           (f"BASELINE configs[2]: 8-camera 1920x1080 rig, {n} frames per camera per step ({args.distinct} "
                            f"distinct generator frames per camera tiled in time), whole cameras sharded over the GPUs, "
                            f"records gathered to rank 0, full detect path"),
                           "frames_per_gpu_per_step": frames_step, "frames_per_native_batch": n, "resolution": [W, H],
                           "l2_policy": "inputs larger than L2 (1.6 GB of frames per 256-frame batch vs 126 MB L2)",
                           "parallelism": f"stream-sharded x{args.gpus}, NCCL gather of records only"},
                   roofline={"bound": "hbm",
                             "kernel": "edge path: k1_probe + k1_fused (gray, 5x5 blur, histogram, Sobel, NMS) + k2t_threshold + "
                                       "k2_canny_cluster (hysteresis, ROI, point list)",
                             "achieved": edge_achieved, "peak": peak, "unit": "GB/s", "frac": edge_achieved / peak,
                             "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 (of fallback)",
                             "traffic": traffic, "traffic_source": traffic_src,
                             "ms_per_launch": edge_ms, "algorithmic_bytes_per_launch": algo,
                             "frac_of_nominal_8TBs": edge_achieved / 8000.0,
                             "k1_fused": {"ms": k1_ms, "achieved": k1_achieved, "frac": k1_achieved / peak}},
                   stage_ms_per_batch={k: v / batches for k, v in stage_sum.items()},
                   stage_pass={"ms_per_step": serial_ms / args.steps,
                               "note": "second pass of the same steps, one stream with events between the stages; `value` "
                                       "is the first pass (back half of each batch on a second stream)"},
                   e2e={"value": e2e_val, "unit": "frames/s", "h2d_bytes_per_step": int(host_frames.nbytes),
                        "d2h_bytes_per_step": int(_native.RECORD_DTYPE.itemsize * ne),
                        "api": "LaneDetector.detect_batch(numpy pinned)",
                        "pcie_gbs_plain_copy_per_gpu": pcie_gbs,
                        "pcie_frac": (e2e_bytes_s / 1e9 / pcie_gbs) if pcie_gbs else None},
                   e2e_nv12={"value": nv12_val, "unit": "frames/s", "h2d_bytes_per_step": nv12_bytes,
                             "api": "LaneDetector.detect_batch_nv12(numpy pinned): NV12 -> BGR on the device, bit-exact vs cv2"},
                   value_public_api={"value": api_fps, "unit": "frames/s",
                                     "api": "LaneDetector.detect_batches(CUDA tensors): pipelined detect_batch, LaneLine objects "
                                            "for every frame, wall clock"},
                   draw=draw,
                   input_generation={"seconds": t_gen, "frames": int(sum(min(args.distinct, n) for _ in cams)),
                                     "api": "SyntheticDataGenerator.generate_batch_device (k7_draw)"},
                   gpu_launches=launches[0], clocks=clocks, lanes_found_last_batch=found,
                   last_offset=None if off is None else float(off))
        if world > 1:
            out["gather_verified"] = gather_verified
            out["lanes_found_per_rank_at_rank0"] = lanes_per_rank
        if cpu_baseline:
            out["cpu_baseline"] = cpu_baseline
        print(json.dumps(out))
    det.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
