"""A rig streamed two ticks deep (``LaneDetector.detect_rig_stream``, ``lane_rig_enqueue``).

Every tick's records, the per-camera smoothing state after it and ``last_records`` must equal, byte for byte, those of
``detect_rig`` called tick after tick on a fresh detector, for CUDA, pinned-tensor and numpy ticks, including ticks with
absent cameras, uneven counts, an overflowing camera and ticks the pipeline cannot take."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import torch  # noqa: E402

from bgr_yuv420 import bgr_to_i420, bgr_to_nv12  # noqa: E402
from multimodal_autonomous_driving_perception_and_planning_b200 import LaneDetector, _native  # noqa: E402
from test_gpu_stream_roi import rig_polys  # noqa: E402
from util import gen_frames  # noqa: E402

# (layout, width, height): a 4K front camera, two automotive surround sensors, a 720p software-decoded camera and a
# 1080p BGR camera
RIG = [("nv12", 3840, 2160), ("nv12", 1936, 1216), ("nv12", 1936, 1216), ("i420", 1280, 720), ("bgr", 1920, 1080)]
LAYOUTS = [lay for lay, *_ in RIG]
NOISE_CAM = 4                                        # the BGR camera; its ROI is the full frame
TARGETS = [(640, 480), (1280, 720)]
# frames per camera in each tick (0: no frame; None: the camera is absent from the tick)
COUNTS = [[1, 1, 1, 1, 1], [2, 0, 1, None, 1], [1, 2, 2, 1, 2], [None, 1, 0, 2, 1], [2, 1, 1, 1, 1], [1, 1, 2, 2, 0],
          [1, None, 1, 1, 2]]
NOISE_TICK = 4


def encode(bgr, layout):
    if layout == "bgr":
        return bgr
    return np.stack([(bgr_to_nv12 if layout == "nv12" else bgr_to_i420)(f) for f in bgr])


@pytest.fixture(scope="module")
def rig():
    """Camera s's frames in its layout: four of the generator's scenes at its size."""
    return [encode(np.stack(gen_frames(w, h, 4, start=1000 * s)), lay) for s, (lay, w, h) in enumerate(RIG)]


def polys_for(target):
    p = rig_polys(target[1], target[0])
    return [p[1], p[2], p[3], None, p[6]]


def numpy_ticks(rig, counts=COUNTS, noise_tick=NOISE_TICK):
    ticks = []
    for k, row in enumerate(counts):
        tick = []
        for s, t in enumerate(row):
            if t is None:
                tick.append(None)
            elif s == NOISE_CAM and k == noise_tick:
                tick.append(np.random.default_rng(k).integers(0, 256, (t, 1080, 1920, 3), dtype=np.uint8))
            else:
                tick.append(np.ascontiguousarray(np.roll(rig[s], -k, axis=0)[:t]))
        ticks.append(tick)
    return ticks


def pinned(a):
    t = torch.empty(a.shape, dtype=torch.uint8).pin_memory()
    t.numpy()[...] = a
    return t


def as_kind(ticks, kind):
    conv = {"numpy": lambda a: a, "pinned": pinned, "cuda": lambda a: torch.from_numpy(a).cuda()}[kind]
    return [[None if c is None else conv(c) for c in tick] for tick in ticks]


def blocking(ticks, target, polys, **kw):
    """detect_rig tick after tick on a fresh detector: (lanes, records, state after) per tick."""
    det = LaneDetector(**kw)
    out = []
    for tick in ticks:
        lanes = det.detect_rig(tick, LAYOUTS, target_size=target, stream_rois=polys)
        out.append((lanes, det.last_records.copy(), det._stream_fit.copy(), det._stream_valid.copy()))
    det.close()
    return out


def assert_same(got, want):
    """got / want: (lanes, records, fit, valid) per tick."""
    assert len(got) == len(want)
    for k, ((gl, gr, gf, gv), (wl, wr, wf, wv)) in enumerate(zip(got, want)):
        assert [len(c) for c in gl] == [len(c) for c in wl], k
        assert gr.tobytes() == wr.tobytes(), k
        assert gf.tobytes() == wf.tobytes() and gv.tobytes() == wv.tobytes(), k


def streamed(det, ticks, target, polys):
    out = []
    for lanes in det.detect_rig_stream(ticks, LAYOUTS, target_size=target, stream_rois=polys):
        out.append((lanes, det.last_records.copy(), det._stream_fit.copy(), det._stream_valid.copy()))
    return out


@pytest.mark.parametrize("target", TARGETS)
@pytest.mark.parametrize("kind", ["cuda", "pinned", "numpy"])
def test_stream_equals_detect_rig_tick_after_tick(rig, kind, target):
    polys = polys_for(target)
    ticks = numpy_ticks(rig)
    want = blocking(ticks, target, polys, max_batch=8, max_segments=8)
    det = LaneDetector(max_batch=8, max_segments=8)
    got = streamed(det, as_kind(ticks, kind), target, polys)
    assert_same(got, want)
    assert det.dense_reruns >= 1 and not det._ctx._inflight
    assert max(want[NOISE_TICK][1]["n_segments"]) > 8                    # the noise camera did overflow
    det.close()


def test_state_carries_from_detect_rig_through_the_stream_into_detect_streams(rig):
    """detect_rig, then detect_rig_stream, then detect_streams on one detector equals the all-blocking sequence."""
    target = (640, 480)
    polys = polys_for(target)
    ticks = numpy_ticks(rig)[:4]
    frames = np.stack(gen_frames(640, 480, len(RIG), start=77))
    ids = np.arange(len(RIG), dtype=np.int32)

    def run(stream):
        det = LaneDetector(max_batch=8)
        det.detect_rig(ticks[0], LAYOUTS, target_size=target, stream_rois=polys)
        out = [det.last_records.copy()]
        rest = as_kind(ticks[1:], "cuda")
        if stream:
            for _ in det.detect_rig_stream(rest, LAYOUTS, target_size=target, stream_rois=polys):
                out.append(det.last_records.copy())
        else:
            for t in rest:
                det.detect_rig(t, LAYOUTS, target_size=target, stream_rois=polys)
                out.append(det.last_records.copy())
        det.detect_streams(frames, stream_ids=ids, stream_rois=polys)
        out.append(det.last_records.copy())
        state = (det._stream_fit.copy(), det._stream_valid.copy())
        det.close()
        return out, state

    (got, gs), (want, ws) = run(True), run(False)
    assert [r.tobytes() for r in got] == [r.tobytes() for r in want]
    assert gs[0].tobytes() == ws[0].tobytes() and gs[1].tobytes() == ws[1].tobytes()


def test_ticks_the_pipeline_cannot_take_go_through_detect_rig(rig):
    """CUDA ticks with a numpy tick, a tick larger than max_batch and a tick without frames in the middle: still equal
    to detect_rig tick after tick."""
    target = (640, 480)
    polys = polys_for(target)
    counts = [[1, 1, 1, 1, 1], [1, 2, 1, 1, 1], [2, 2, 2, 2, 2], [0, None, 0, 0, 0], [1, 1, 1, 1, 1], [1, 1, 0, 1, 1]]
    ticks = numpy_ticks(rig, counts, noise_tick=-1)
    mixed = as_kind(ticks, "cuda")
    mixed[1] = ticks[1]                                                   # a numpy tick between CUDA ticks
    det = LaneDetector(max_batch=8)
    got = []
    for k, lanes in enumerate(det.detect_rig_stream(mixed, LAYOUTS, target_size=target, stream_rois=polys)):
        if k == 3:
            assert lanes == [[] for _ in RIG]
        got.append((lanes, det.last_records.copy(), det._stream_fit.copy(), det._stream_valid.copy()))
    ref = LaneDetector(max_batch=8)
    want = []
    for tick in ticks:
        lanes = ref.detect_rig(tick, LAYOUTS, target_size=target, stream_rois=polys)
        want.append((lanes, ref.last_records.copy(), ref._stream_fit.copy(), ref._stream_valid.copy()))
    assert_same(got, want)
    assert sum(len(c) for c in want[2][0]) == 10                           # more than max_batch: chunked
    det.close()
    ref.close()


@pytest.mark.parametrize("kind", ["pinned", "numpy"])
def test_host_staging_is_not_reused_while_a_tick_reads_it(rig, kind):
    """The caller's source of tick i is overwritten as soon as tick i is yielded, while tick i+1 is in flight; the
    ticks behind it keep their records."""
    target = (640, 480)
    polys = polys_for(target)
    ticks = numpy_ticks(rig, COUNTS, noise_tick=-1)
    want = blocking(ticks, target, polys, max_batch=8)
    src = as_kind(ticks, kind)
    det = LaneDetector(max_batch=8)
    got = []
    for k, lanes in enumerate(det.detect_rig_stream(src, LAYOUTS, target_size=target, stream_rois=polys)):
        got.append((lanes, det.last_records.copy(), det._stream_fit.copy(), det._stream_valid.copy()))
        assert len(det._ctx._inflight) == (1 if k + 1 < len(ticks) else 0)
        for cam in src[k]:
            if cam is not None:
                (cam.numpy() if kind == "pinned" else cam)[...] = 255
    assert_same(got, want)
    det.close()


def test_raw_rig_enqueue(rig):
    S = 8
    polys = rig_polys(480, 640)
    det, ref = LaneDetector(max_batch=8), LaneDetector(max_batch=8)
    ctx = det._context(480, 640, 8, stream_rois=polys, n_masks=S)
    rctx = ref._context(480, 640, 8, stream_rois=polys, n_masks=S)
    lib, P = _native.lib(), _native._ptr
    i420 = np.ascontiguousarray(rig[3][:2])
    dev = torch.from_numpy(i420).cuda()
    host = pinned(i420)
    bgr = torch.from_numpy(np.stack(gen_frames(640, 480, 2, start=5))).cuda()
    torch.cuda.synchronize()
    fit, valid = np.zeros((S, 2, 3)), np.zeros((S, 2), np.uint8)
    out = np.zeros(8, _native.RECORD_DTYPE)

    def enq(*srcs, on_device=1, pf=None, pv=None, n_streams=S):
        arr = (_native.LaneRigSource * max(len(srcs), 1))(*[_native.LaneRigSource(*s) for s in srcs])
        return lib.lane_rig_enqueue(ctx._h, arr if srcs else None, len(srcs), on_device, n_streams, P(pf), P(pv))

    def collect():
        assert lib.lane_detect_collect(ctx._h, P(fit), P(valid), P(out)) == 0
        return out.copy()

    ok_dev = (dev.data_ptr(), _native.INPUT_I420, 720, 1280, 2, 3)
    assert enq(ok_dev) == -4 and b"no state" in lib.lane_last_error(ctx._h)        # NULL state, none on the device
    # lane_detect_rig's validation
    assert enq() == -1                                                               # null sources
    assert enq((dev.data_ptr(), _native.INPUT_I420, 720, 1280, 0, 3), pf=fit, pv=valid) == -1   # no frame at all
    assert enq(ok_dev, ok_dev, ok_dev, ok_dev, ok_dev, pf=fit, pv=valid) == -1       # 10 frames, max_batch 8
    assert enq(ok_dev, (dev.data_ptr(), 0, 720, 1280, -1, 0), pf=fit, pv=valid) == -1   # negative n
    assert enq((dev.data_ptr(), 3, 720, 1280, 2, 0), pf=fit, pv=valid) == -1         # unknown format
    assert enq((dev.data_ptr(), _native.INPUT_I420, 0, 1280, 2, 0), pf=fit, pv=valid) == -1     # non-positive size
    assert enq((dev.data_ptr(), _native.INPUT_NV12, 720, 1279, 2, 0), pf=fit, pv=valid) == -1   # odd YUV width
    assert enq((dev.data_ptr(), _native.INPUT_I420, 720, 1280, 2, 8), pf=fit, pv=valid) == -1   # stream_id >= S
    assert enq((0, _native.INPUT_I420, 720, 1280, 2, 0), pf=fit, pv=valid) == -1     # null frames
    assert enq(ok_dev, pf=fit, pv=valid, n_streams=S + 1) == -1                      # more streams than masks
    # host sources must be page-locked
    assert enq((i420.ctypes.data, _native.INPUT_I420, 720, 1280, 2, 3), on_device=0, pf=fit, pv=valid) == -1
    assert b"source 0" in lib.lane_last_error(ctx._h) and b"page-locked" in lib.lane_last_error(ctx._h)
    assert not ctx._inflight

    # queue rules: explicit state with one tick in flight, a third tick with two in flight
    ok_host = (host.data_ptr(), _native.INPUT_I420, 720, 1280, 2, 3)
    assert enq(ok_host, on_device=0, pf=fit, pv=valid) == 0
    assert enq(ok_dev, pf=fit, pv=valid) == -4
    assert enq(ok_dev) == 0
    assert enq(ok_dev) == -4 and b"two batches" in lib.lane_last_error(ctx._h)
    got = [collect(), collect()]
    rfit, rvalid = np.zeros((S, 2, 3)), np.zeros((S, 2), np.uint8)
    for k in range(2):
        want = rctx.detect_rig([(i420, _native.INPUT_I420, (720, 1280), 2, 3)], False, S, rfit, rvalid, 0.7, 1 - 0.7)
        assert got[k][:2].tobytes() == want.tobytes(), k
    assert fit.tobytes() == rfit.tobytes() and valid.tobytes() == rvalid.tobytes()

    # a rig tick queued behind a lane_detect_enqueue batch, collected in order
    ctx.enqueue(bgr.data_ptr(), 2, None, S, fit, valid, 0.7, 1 - 0.7)
    assert enq(ok_dev) == 0
    first = ctx.collect(fit, valid)
    second = collect()[:2]
    want1 = rctx.detect(bgr.data_ptr(), 2, True, None, S, rfit, rvalid, 0.7, 1 - 0.7)
    want2 = rctx.detect_rig([(dev.data_ptr(), _native.INPUT_I420, (720, 1280), 2, 3)], True, S, rfit, rvalid, 0.7, 1 - 0.7)
    assert first.tobytes() == want1.tobytes() and second.tobytes() == want2.tobytes()
    assert fit.tobytes() == rfit.tobytes() and valid.tobytes() == rvalid.tobytes()
    det.close()
    ref.close()
