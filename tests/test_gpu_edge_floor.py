"""The fused edge kernel's exact-floor redo pass (k1_fused, DESIGN.md §4 K1F), reached on purpose.

A trap frame (edge_floor.trap_frame) makes k1_probe's floor far higher than the frame's true Canny low: the first pass
misses almost every edge pixel, and only the redo pass (launch_fused_edge_redo + the second cluster pass) restores them.
Trap frames are mixed into batches at every position, size and shape, through every detect entry point; every frame's
thresholds, counts, CLASS / EDGES / POINTS / SEGMENTS taps must equal the stage oracle bit for bit and its fits must
match at the bars of test_gpu_parity.py.

Child processes run the same batches with LANE_B200_SYNC_DEBUG=1, which prints "N of M frames redone" for every chunk
with a redo: the counts must be the restated probe's prediction, chunk by chunk.  Other children force the floor with
LANE_K1F_PRE (read once per process): 0 (no floor), 255 (every frame redone), and the low and low + 1 of generator frames
with final edge pixels at exactly mag == low + 1, which pin the comparisons `low < pre` and `M > pre`.
"""
import functools
import json
import os
import re
import subprocess
import sys

if __name__ == "__main__":                     # child process (run_child): the paths tests/conftest.py sets up
    _tests = os.path.dirname(os.path.abspath(__file__))
    sys.path[:0] = [os.path.dirname(_tests), _tests, os.path.join(_tests, "golden")]

import numpy as np  # noqa: E402
import pytest  # noqa: E402

pytestmark = pytest.mark.gpu

from edge_floor import probe_floor, trap_frame  # noqa: E402
from multimodal_autonomous_driving_perception_and_planning_b200 import LaneDetector, _native  # noqa: E402
from oracle import stages as S  # noqa: E402
from util import gen_frames  # noqa: E402

# generator frames with final edge pixels at exactly mag == low + 1, by their low (the "boundary" scenario's frames)
BOUNDARY = {99: [("gen", 640, 480, 4, 7, 2), ("gen", 640, 480, 4, 7, 3)], 97: [("gen", 1920, 1080, 4, 7, 0)]}
SHAPES = [(480, 640), (135, 480), (32, 640), (1080, 1920)]
SIZES = [1, 3, 17, 64]
CAM_POLY = np.array([[(0, 479), (120, 250), (520, 250), (639, 479)]], np.int32)      # the trap camera's own ROI


# ---- frames, named by hashable specs so that a child process can rebuild them --------------------------------------
@functools.lru_cache(maxsize=None)
def _gen(w, h, n, start):
    return gen_frames(w, h, n, start)


@functools.lru_cache(maxsize=None)
def frame(spec):
    """("trap", h, w, seed, lattice value) | ("gen", w, h, n, start, i): frame i of gen_frames(w, h, n, start) |
    ("noise", h, w, seed, saturated left half)."""
    kind, *a = spec
    if kind == "trap":
        f = trap_frame(*a)
    elif kind == "gen":
        f = _gen(*a[:4])[a[4]]
    else:
        h, w, seed, sat = a
        f = np.random.default_rng(seed).integers(0, 256, (h, w, 3), dtype=np.uint8)
        if sat:
            f[:, : w // 2] = 255
    f.flags.writeable = False
    return f


def trap(h, w, i):
    return ("trap", h, w, i % 4, 240)


def normal(h, w, i):
    return ("gen", w, h, 8, 0, i % 8)


def arrangements(n):
    """Trap positions of a batch of n frames, by name; arrangements that coincide at this size are kept once."""
    out = {}
    for name, pos in (("first", {0}), ("middle", {n // 2}), ("last", {n - 1}), ("alternating", set(range(0, n, 2))),
                      ("all", set(range(n))), ("none", set())):
        if pos not in out.values():
            out[name] = pos
    return out


def mixed(h, w, n, traps):
    return tuple(trap(h, w, i) if i in traps else normal(h, w, i) for i in range(n))


# ---- the stage oracle, per frame and ROI, and the fit chain ------------------------------------------------------
@functools.lru_cache(maxsize=None)
def oracle(spec, roi_key=None):
    f = frame(spec)
    h, w = f.shape[:2]
    b = S.blur5(S.gray(f))
    low, high, m2 = S.thresholds(b)
    t = S.canny(b, low, high)
    roi = None if roi_key is None else np.array([roi_key], np.int32)
    masked = t.edges & S.roi_mask(h, w, roi)
    ys, xs = np.nonzero(masked)
    return dict(m2=m2, low=low, high=high, cls=t.cls, edges=t.edges, n_edges=int((t.edges != 0).sum()),
                points=np.stack([xs, ys], 1).astype(np.int32), lines=S.houghp(masked))


def roi_key(poly):
    return None if poly is None else tuple(map(tuple, np.asarray(poly).reshape(-1, 2).tolist()))


def check(recs, specs, state, roi=None, ctx=None):
    """Records of `specs` in order (and the context's taps when given) against the oracle.  `state` = [prev_left,
    prev_right] of the frames' stream before them, advanced in place."""
    from test_gpu_parity import _check_side
    key = roi_key(roi)
    for i, spec in enumerate(specs):
        o, r = oracle(spec, key), recs[i]
        h = frame(spec).shape[0]
        w = frame(spec).shape[1]
        assert (r["median_x2"], r["low"], r["high"]) == (o["m2"], o["low"], o["high"]), (i, spec)
        assert (r["n_edges"], r["n_roi_points"], r["n_segments"]) == (o["n_edges"], len(o["points"]), len(o["lines"])), \
            (i, spec)
        if ctx is not None:
            assert np.array_equal(ctx.tap(_native.TAP_CLASS, i), o["cls"]), (i, spec)
            assert np.array_equal(ctx.tap(_native.TAP_EDGES, i), o["edges"]), (i, spec)
            if len(o["points"]):
                assert np.array_equal(ctx.tap(_native.TAP_POINTS, i), o["points"]), (i, spec)
            assert np.array_equal(ctx.tap(_native.TAP_SEGMENTS, i), o["lines"]), (i, spec)
        sides = S.separate(o["lines"], w)
        fits = [S.fit_side(sides[s], h, state[s]) for s in (0, 1)]
        for s, fit in enumerate(fits):
            assert bool(r["side"][s]["valid"]) == (fit is not None), (i, spec, s)
            if fit is not None:
                _check_side(r["side"][s], fit.coeffs, fit.points, fit.confidence, h)
                state[s] = fit.coeffs
        off = S.center_offset(w, *fits)
        assert bool(r["offset_valid"]) == (off is not None)
        if off is not None:
            assert abs(r["offset"] - off) <= 0.5


def same_lanes(a, b):
    for x, y in zip(a, b):
        for s in (0, 1):
            assert (x[s] is None) == (y[s] is None)
            if x[s] is not None:
                assert np.array_equal(x[s].polynomial, y[s].polynomial) and np.array_equal(x[s].points, y[s].points)


def same_state(a, b):
    for p in ("prev_left_fit", "prev_right_fit"):
        assert (getattr(a, p) is None) == (getattr(b, p) is None)
        if getattr(a, p) is not None:
            assert np.array_equal(getattr(a, p), getattr(b, p))


# ---- scenarios: batches of detect_batch calls that a child process can replay ------------------------------------
def host_chunk(n):
    """Frames per chunk of a host batch (lane_abi.cu): the redo count is printed per chunk."""
    return max(1, min(64, (n + 3) // 4))


def scenario(name):
    """[(label, specs, on_device, max_segments)]: detect_batch calls on a fresh LaneDetector(max_batch=len(specs))."""
    if name == "mixed":
        return [(f"{h}x{w}/{n}/{a}" + ("/cuda" if dev else ""), mixed(h, w, n, pos), dev, 256)
                for h, w in SHAPES for n in SIZES for a, pos in arrangements(n).items()
                for dev in ((False, True) if n >= 17 else (False,))]
    calls = [("gen640", tuple(normal(480, 640, i) for i in range(6)), False, 256),
             ("trap", mixed(480, 640, 17, set(range(1, 17, 3))), False, 256)]
    calls += [(f"noise{h}x{w}", tuple(("noise", h, w, h + w + k, k == 2) for k in range(3)), False, 4096)
              for h, w in [(16, 16), (48, 64), (135, 480), (271, 976), (137, 1936), (1080, 1920)]]
    if name == "boundary":
        calls = [("gen640@7", tuple(("gen", 640, 480, 4, 7, i) for i in range(4)), False, 256),
                 ("gen1080@7", tuple(("gen", 1920, 1080, 4, 7, i) for i in range(2)), True, 256)]
    return calls


@functools.lru_cache(maxsize=None)
def redone(spec, forced=None):
    """Whether the first pass lists the frame for the redo pass: its true low is below the floor it runs with."""
    return oracle(spec)["low"] < (probe_floor(frame(spec)) if forced is None else forced)


def expected_redo_lines(calls, forced=None):
    """{label: [(redone, chunk frames)]} for every chunk that redoes at least one frame, from the restated probe."""
    out = {}
    for label, specs, on_device, _ in calls:
        step = len(specs) if on_device else host_chunk(len(specs))
        lines = []
        for a in range(0, len(specs), step):
            chunk = specs[a:a + step]
            k = sum(redone(s, forced) for s in chunk)
            if k:
                lines.append((k, len(chunk)))
        out[label] = lines
    return out


def play(calls, check_taps):
    """Run the calls, each after a marker line on stderr, checking records (and taps) against the oracle."""
    import torch
    for label, specs, on_device, max_segments in calls:
        sys.stderr.write(f"@call {label}\n")
        sys.stderr.flush()
        frames = np.stack([frame(s) for s in specs])
        det = LaneDetector(max_batch=len(specs), max_segments=max_segments, debug=check_taps)
        det.detect_batch(torch.from_numpy(frames).cuda() if on_device else frames)
        check(det.last_records, specs, [None, None], ctx=det._ctx if check_taps else None)
        det.close()
        sys.stderr.flush()


def run_child(name, forced=None):
    """Replay scenario `name` in a fresh process with LANE_B200_SYNC_DEBUG=1 (and LANE_K1F_PRE=forced): returns the
    calls and {label: [(redone, chunk frames)]} parsed from its stderr."""
    env = dict(os.environ, LANE_B200_SYNC_DEBUG="1")
    env.pop("LANE_K1F_PRE", None)
    if forced is not None:
        env["LANE_K1F_PRE"] = str(forced)
    args = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + [os.path.abspath(__file__), name]
    p = subprocess.run(args, env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-4000:]
    got, label = {}, None
    for line in p.stderr.splitlines():
        if line.startswith("@call "):
            label = line[6:]
            got[label] = []
        m = re.search(r"lane_b200: (\d+) of (\d+) frames redone", line)
        if m:
            got[label].append((int(m.group(1)), int(m.group(2))))
    return scenario(name), got


# ---- mixed batches ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", SHAPES)
def test_mixed_batches_equal_the_oracle(shape):
    """Trap frames first, in the middle, last, alternating, all or none, in host batches of 1, 3, 17 and 64 frames (traps
    land in every host chunk, of 1, 5 or 16 frames): every tap and record bit-exact.  Batches of 17 and 64 also run from
    the device as one chunk, whose first pass cuts its last n / 8 frames into thinner tail bands."""
    import torch
    h, w = shape
    for n in SIZES:
        det = LaneDetector(max_batch=n, debug=True)
        for name, pos in arrangements(n).items():
            det.reset()
            specs = mixed(h, w, n, pos)
            frames = np.stack([frame(s) for s in specs])
            det.detect_batch(frames)
            check(det.last_records, specs, [None, None], ctx=det._ctx)
            if n >= 17:
                want = det.last_records.copy()
                det.reset()
                det.detect_batch(torch.from_numpy(frames).cuda())
                assert det.last_records.tobytes() == want.tobytes(), (n, name)
        det.close()


def test_redo_counts_per_chunk_equal_the_probe_prediction():
    calls, got = run_child("mixed")
    want = expected_redo_lines(calls)
    assert sum(k for lines in want.values() for k, _ in lines) > 100      # the trap frames do reach the redo pass
    assert got == want
    print("redo lines per call:", json.dumps({k: v for k, v in got.items() if v}))


# ---- every entry point, with trap frames mixed in ---------------------------------------------------------------
def test_host_and_device_batches_with_traps_in_later_chunks():
    import torch
    h, w = 480, 640
    specs = mixed(h, w, 12, {4, 7, 8, 11})          # host_chunk(12) = 3: traps in chunks 1, 2 and 3, none in chunk 0
    frames = np.stack([frame(s) for s in specs])
    a, b = LaneDetector(max_batch=12, debug=True), LaneDetector(max_batch=12, debug=True)
    la = a.detect_batch(frames)
    check(a.last_records, specs, [None, None], ctx=a._ctx)
    lb = b.detect_batch(torch.from_numpy(frames).cuda())
    check(b.last_records, specs, [None, None], ctx=b._ctx)
    assert a.last_records.tobytes() == b.last_records.tobytes()
    same_lanes(la, lb)
    a.close(); b.close()


@pytest.mark.parametrize("pattern", ["consecutive", "alternate"])
def test_two_deep_batches_equal_blocking_calls(pattern):
    """detect_batches keeps two batches in flight (the Hough half of one under the edge kernels of the next): redone
    frames there must give the records, lanes and prev_*_fit of detect_batch batch after batch."""
    import torch
    h, w, n = 1080, 1920, 6
    traps = [{1}, {0, 5}, set(), set(), {2, 3}, {5}] if pattern == "consecutive" else \
        [{0, 2, 4}, set(), {5}, set(), {1}, set()]
    batches = [tuple(trap(h, w, 3 * b + i) if i in t else normal(h, w, 3 * b + i) for i in range(n))
               for b, t in enumerate(traps)]
    dev = [torch.from_numpy(np.stack([frame(s) for s in specs])).cuda() for specs in batches]
    ref = LaneDetector(max_batch=n)
    want, state = [], [None, None]
    for specs, fr in zip(batches, dev):
        lanes = ref.detect_batch(fr)
        check(ref.last_records, specs, state)
        want.append((lanes, ref.last_records.copy(), ref.prev_left_fit, ref.prev_right_fit))
    det = LaneDetector(max_batch=n)
    for k, lanes in enumerate(det.detect_batches(dev)):
        same_lanes(lanes, want[k][0])
        assert det.last_records.tobytes() == want[k][1].tobytes(), k
        assert np.array_equal(det.prev_left_fit, want[k][2]) and np.array_equal(det.prev_right_fit, want[k][3])
    same_state(det, ref)
    ref.close(); det.close()


def test_streams_with_a_trap_camera_roi_equal_single_roi_detectors():
    """Multi-ROI context: the redo pass reads each listed frame's own ROI plane.  Camera 1 sends trap frames and has
    its own polygon; every camera's records equal a single-ROI detector's and the oracle with that camera's ROI."""
    h, w, t = 480, 640, 3
    polys = [None, CAM_POLY, None]
    cams = [[normal(h, w, i) for i in range(t)], [trap(h, w, i) for i in range(t)],
            [normal(h, w, 4 + i) for i in range(t)]]
    order = [(s, k) for k in range(t) for s in (2, 1, 0)]
    specs = [cams[s][k] for s, k in order]
    det = LaneDetector(max_batch=len(order), debug=True)
    lanes = det.detect_streams(np.stack([frame(x) for x in specs]), stream_ids=[s for s, _ in order], stream_rois=polys)
    assert det._ctx.n_roi == 3
    recs = det.last_records
    for s, poly in enumerate(polys):
        ks = [k for k, (c, _) in enumerate(order) if c == s]
        single = LaneDetector(poly, max_batch=t, debug=True)
        single.detect_batch(np.stack([frame(x) for x in cams[s]]))
        assert recs[ks].tobytes() == single.last_records.tobytes(), s
        check(single.last_records, cams[s], [None, None], roi=poly, ctx=single._ctx)
        for j, k in enumerate(ks):
            o = oracle(cams[s][j], roi_key(poly))
            if len(o["points"]):
                assert np.array_equal(det._ctx.tap(_native.TAP_POINTS, k), o["points"]), (s, j)
        single.close()
    det.close()


@pytest.mark.parametrize("where", ["host", "cuda"])
def test_rig_with_a_trap_camera_at_the_target_size_equals_detect_batch(where):
    """detect_rig: a BGR trap camera already at the target size next to NV12 / I420 cameras the device resizes.  Host
    rigs run in host chunks of two frames; a CUDA rig is one chunk whose redo list is frames 2..4 of 6."""
    import torch
    from bgr_yuv420 import bgr_to_i420, bgr_to_nv12
    h, w = 480, 640
    traps = [trap(h, w, i) for i in range(3)]
    bgr = np.stack([frame(x) for x in traps])
    big = np.stack(gen_frames(1280, 720, 2, start=50))
    rig = [np.stack([bgr_to_nv12(f) for f in big]), bgr, np.stack([bgr_to_i420(f) for f in big[:1]])]
    if where == "cuda":
        rig = [torch.from_numpy(c).cuda() for c in rig]
    det = LaneDetector(max_batch=8)
    got = det.detect_rig(rig, ["nv12", "bgr", "i420"], target_size=(w, h))
    recs = det.last_records
    single = LaneDetector(max_batch=3)
    want = single.detect_batch(bgr)
    assert recs[2:5].tobytes() == single.last_records.tobytes()
    same_lanes(got[1], want)
    check(single.last_records, traps, [None, None])
    det.close(); single.close()


def test_trap_frames_in_a_chunk_that_is_rerun_dense():
    """A 1080p noise frame overflows the segment lists: its chunk, trap frames included, is re-run on the dense
    context, whose first pass redoes the trap frames again."""
    import torch
    h, w = 1080, 1920
    specs = (trap(h, w, 0), ("noise", h, w, 7, False), normal(h, w, 0), trap(h, w, 1))
    frames = np.stack([frame(s) for s in specs])
    for src in (frames, torch.from_numpy(frames).cuda()):
        det = LaneDetector(max_batch=4)
        det.detect_batch(src)
        assert det.dense_reruns == 1 and not det.last_records["flags"].any()
        check(det.last_records, specs, [None, None])
        det.close()


# ---- forced floors, one process per value -------------------------------------------------------------------------
@pytest.mark.parametrize("forced", [0, 255])
def test_forced_floor(forced):
    """No floor (every NMS candidate queued) and a floor above every low (every frame redone): generator taps, the
    fused kernel's noise shapes with full Canny taps, and a trap batch."""
    calls, got = run_child("forced", forced)
    want = expected_redo_lines(calls, forced)
    lines = [km for v in want.values() for km in v]
    if forced == 0:
        assert not lines
    else:                                        # every chunk of every call redoes all its frames
        assert all(k == m for k, m in lines) and sum(k for k, _ in lines) == sum(len(c[1]) for c in calls)
    assert got == want


@pytest.mark.parametrize("forced", [97, 98, 99, 100])
def test_forced_floor_at_low_and_low_plus_one(forced):
    """Generator frames whose final edges include pixels at exactly mag == low + 1 (low 99 at 640x480, 97 at 1080p):
    with pre == low they are not redone and the first pass must keep those pixels (M > pre); with pre == low + 1 they
    must be redone (low < pre).  Either comparison off by one loses them."""
    calls, got = run_child("boundary", forced)
    low = forced if forced in BOUNDARY else forced - 1
    for s in BOUNDARY[low]:
        o = oracle(s)
        mag = S.canny(S.blur5(S.gray(frame(s))), o["low"], o["high"]).mag
        assert o["low"] == low and ((o["edges"] != 0) & (mag == low + 1)).any(), s
        assert redone(s, forced) == (forced == low + 1)
    assert got == expected_redo_lines(calls, forced)


if __name__ == "__main__":
    play(scenario(sys.argv[1]), check_taps=sys.argv[1] != "mixed")
