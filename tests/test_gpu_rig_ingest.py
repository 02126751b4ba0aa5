"""A rig of cameras with their own resolutions and decoder layouts in one batched call (``LaneDetector.detect_rig``,
``lane_detect_rig``, kernel k0_rig_ingest).

Every camera's records must equal, byte for byte, those of a fresh single-camera detector fed that camera's frames with
``target_size``; the ingest output (LANE_TAP_FRAME) must equal cv2's conversion and resize of every frame; lanes must
match the cv2 reference pipeline within the bars of test_gpu_parity.py."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import cv2  # noqa: E402

from bgr_yuv420 import bgr_to_i420, bgr_to_nv12  # noqa: E402
from multimodal_autonomous_driving_perception_and_planning_b200 import LaneDetector, _native  # noqa: E402
from oracle.cv2_pipeline import Cv2LaneOracle  # noqa: E402
from test_gpu_stream_roi import rig_polys  # noqa: E402
from util import gen_frames  # noqa: E402

# (layout, width, height, frames this tick): a 4K front camera, four automotive surround sensors, a 720p software-decoded
# camera, a 1080p BGR camera, and one whose rows and chroma rows are not 4-byte aligned
RIG = [("nv12", 3840, 2160, 2), ("nv12", 1936, 1216, 3), ("nv12", 1936, 1216, 1), ("nv12", 1936, 1216, 2),
       ("nv12", 1936, 1216, 2), ("i420", 1280, 720, 3), ("bgr", 1920, 1080, 1), ("nv12", 1282, 722, 2)]
CODES = {"nv12": cv2.COLOR_YUV2BGR_NV12, "i420": cv2.COLOR_YUV2BGR_I420}
TARGETS = [(640, 480), (1280, 720)]


def encode(bgr, layout):
    if layout == "bgr":
        return bgr
    return np.stack([(bgr_to_nv12 if layout == "nv12" else bgr_to_i420)(f) for f in bgr])


def prepare(frames, layout, target):
    """What VideoDataLoader with target_size hands LaneDetector.detect: cv2's conversion, then cv2.resize."""
    bgr = frames if layout == "bgr" else [cv2.cvtColor(f, CODES[layout]) for f in frames]
    return np.stack([cv2.resize(f, target) for f in bgr])


@pytest.fixture(scope="module")
def rig():
    """Camera s's frames in its layout: the generator's scenes at its size, three per camera (a tick uses the first T)."""
    return [encode(np.stack(gen_frames(w, h, 3, start=1000 * s)), lay) for s, (lay, w, h, _) in enumerate(RIG)]


def tick(rig, k=0, counts=None):
    counts = [c for *_, c in RIG] if counts is None else counts
    return [cam[k:k + t] if t else None for cam, t in zip(rig, counts)]


LAYOUTS = [lay for lay, *_ in RIG]


def single_camera(frames, layout, poly, target, **kw):
    """A fresh single-camera detector on one camera's frames: (records, detector)."""
    det = LaneDetector(poly, max_batch=max(len(frames), 1), **kw)
    fn = {"bgr": det.detect_batch, "nv12": det.detect_batch_nv12, "i420": det.detect_batch_i420}[layout]
    fn(frames, target_size=target)
    return det.last_records.copy(), det


def per_camera(recs, counts):
    out, a = [], 0
    for t in counts:
        out.append(recs[a:a + t])
        a += t
    return out


def assert_equals_single_cameras(got_recs, cams, target, polys, **kw):
    counts = [0 if c is None else len(c) for c in cams]
    for s, (got, cam) in enumerate(zip(per_camera(got_recs, counts), cams)):
        if cam is None:
            continue
        want, d = single_camera(cam, LAYOUTS[s], polys[s], target, **kw)
        assert got.tobytes() == want.tobytes(), (target, s)
        d.close()


def _pinned(a):
    import torch
    t = torch.empty(a.shape, dtype=torch.uint8).pin_memory()
    t.numpy()[...] = a
    return t, t.numpy()


@pytest.mark.parametrize("target", TARGETS)
@pytest.mark.parametrize("where", ["chunks", "staged", "pinned", "cuda"])
def test_rig_equals_single_camera_detectors(rig, where, target):
    """chunks: max_batch 5, so chunks straddle cameras; staged: one pageable native call of >= 24 MB (the staging ring);
    pinned host frames; CUDA tensors."""
    import torch
    cams = tick(rig)
    n = sum(len(c) for c in cams)
    polys = rig_polys(target[1], target[0])
    keep = []
    if where == "staged":
        assert sum(c.nbytes for c in cams) >= 24 << 20
    elif where == "pinned":
        keep = [_pinned(c) for c in cams]
        cams = [p for _, p in keep]
    elif where == "cuda":
        cams = [torch.from_numpy(c).cuda() for c in cams]
    det = LaneDetector(max_batch=5 if where == "chunks" else n)
    lanes = det.detect_rig(cams, LAYOUTS, target_size=target, stream_rois=polys)
    assert [len(x) for x in lanes] == [c for *_, c in RIG]
    assert (det._ctx.height, det._ctx.width) == (target[1], target[0]) and det._ctx.n_roi == len(RIG)
    assert_equals_single_cameras(det.last_records, tick(rig), target, polys)
    del keep
    det.close()


@pytest.mark.parametrize("target", TARGETS)
def test_frame_tap_is_cv2s_conversion_and_resize(rig, target):
    cams = tick(rig)
    det = LaneDetector(max_batch=sum(len(c) for c in cams))
    det.detect_rig(cams, LAYOUTS, target_size=target)
    k = 0
    for s, cam in enumerate(cams):
        want = prepare(cam, LAYOUTS[s], target)
        for i in range(len(cam)):
            assert np.array_equal(det._ctx.tap(_native.TAP_FRAME, k), want[i]), (target, s, i)
            k += 1
    det.close()


def test_cameras_already_at_the_target_size_pass_unchanged(rig):
    """Identity taps: the 1080p BGR camera's frames unchanged, a 1080p NV12 camera's frames exactly cv2.cvtColor."""
    bgr = rig[6][:1]
    nv12 = encode(np.stack(gen_frames(1920, 1080, 2, start=77)), "nv12")
    det = LaneDetector(max_batch=4)
    det.detect_rig([rig[5][:1], bgr, nv12], ["i420", "bgr", "nv12"], target_size=(1920, 1080))
    assert np.array_equal(det._ctx.tap(_native.TAP_FRAME, 1), bgr[0])
    for i in range(2):
        assert np.array_equal(det._ctx.tap(_native.TAP_FRAME, 2 + i), cv2.cvtColor(nv12[i], cv2.COLOR_YUV2BGR_NV12))
    det.close()


def test_lanes_match_the_cv2_pipeline(rig):
    target = (640, 480)
    polys = rig_polys(480, 640)
    cams = tick(rig)
    det = LaneDetector(max_batch=16)
    lanes = det.detect_rig(cams, LAYOUTS, target_size=target, stream_rois=polys)
    ys = np.linspace(480 * 0.6, 480, 50)
    for s, cam in enumerate(cams):
        ref = Cv2LaneOracle(roi_vertices=polys[s])
        for i, f in enumerate(prepare(cam, LAYOUTS[s], target)):
            lf, rf = ref.detect(f)
            for side, fit in enumerate((lf, rf)):
                lane = lanes[s][i][side]
                assert (lane is None) == (fit is None), (s, i, side)
                if fit is not None:
                    xw = np.polyval(fit.coeffs, ys)
                    assert np.abs(np.polyval(lane.polynomial, ys) - xw).max() <= 1e-6 * max(1.0, np.abs(xw).max())
                    assert np.abs(lane.points.astype(np.int64) - fit.points).max() <= 1
            off, want_off = det.get_lane_center_offset(640, *lanes[s][i]), Cv2LaneOracle.offset(640, lf, rf)
            assert (off is None) == (want_off is None) and (off is None or abs(off - want_off) <= 0.5)
    det.close()


def test_state_carries_across_rig_and_stream_calls(rig):
    """Tick 1 (every camera), tick 2 (camera 3 has no frame), then tick 3 through detect_streams on the cv2-prepared
    frames: every camera's records equal a single-camera detector fed only that camera's frames, call after call."""
    target = (640, 480)
    polys = rig_polys(480, 640)
    counts = [1] * len(RIG)
    t1, t2 = tick(rig, 0, counts), tick(rig, 1, [0 if s == 3 else 1 for s in range(len(RIG))])
    t3 = [prepare(rig[s][2:3], LAYOUTS[s], target) for s in range(len(RIG))]
    det = LaneDetector(max_batch=8)
    det.detect_rig(t1, LAYOUTS, target_size=target, stream_rois=polys)
    r1 = det.last_records.copy()
    fit3 = det._stream_fit[3].copy()
    det.detect_rig(t2, LAYOUTS, target_size=target, stream_rois=polys)
    r2 = det.last_records.copy()
    assert det._stream_fit[3].tobytes() == fit3.tobytes()
    det.detect_streams(np.concatenate(t3), stream_ids=np.arange(len(RIG)), stream_rois=polys)
    r3 = det.last_records.copy()
    k2 = 0
    for s in range(len(RIG)):
        ref = LaneDetector(polys[s], max_batch=1)
        fn = {"bgr": ref.detect_batch, "nv12": ref.detect_batch_nv12, "i420": ref.detect_batch_i420}[LAYOUTS[s]]
        fn(t1[s], target_size=target)
        assert r1[s].tobytes() == ref.last_records.tobytes(), s
        if t2[s] is not None:
            fn(t2[s], target_size=target)
            assert r2[k2].tobytes() == ref.last_records.tobytes(), s
            k2 += 1
        ref.detect_batch(t3[s])
        assert r3[s].tobytes() == ref.last_records.tobytes(), s
        ref.close()
    det.close()


def test_noise_camera_is_rerun_on_the_dense_context(rig):
    target = (1280, 720)
    polys = rig_polys(720, 1280)
    cams = tick(rig)
    cams[6] = np.random.default_rng(5).integers(0, 256, (2, 1080, 1920, 3), dtype=np.uint8)    # full-frame ROI
    det = LaneDetector(max_batch=8, max_segments=8)
    det.detect_rig(cams, LAYOUTS, target_size=target, stream_rois=polys)
    assert det.dense_reruns >= 1 and not det.last_records["flags"].any()
    counts = [len(c) for c in cams]
    for s, got in enumerate(per_camera(det.last_records, counts)):
        want, d = single_camera(cams[s], LAYOUTS[s], polys[s], target, max_segments=8)
        assert got.tobytes() == want.tobytes(), s
        if s == 6:
            assert d.dense_reruns >= 1 and max(got["n_segments"]) > 8
        d.close()
    det.close()


def test_raw_rig_call_error_codes(rig):
    polys = rig_polys(480, 640)
    det = LaneDetector(max_batch=4)
    ctx = det._context(480, 640, 4, stream_rois=polys, n_masks=len(polys))
    lib = _native.lib()
    cam = np.ascontiguousarray(rig[5][:2])                        # 2 x 1280x720 I420
    fit, valid = np.zeros((9, 2, 3)), np.zeros((9, 2), np.uint8)
    out = np.zeros(8, _native.RECORD_DTYPE)
    P = _native._ptr

    def call(*srcs, S=8, ctx_h=ctx._h, pf=fit, o=out):
        arr = (_native.LaneRigSource * max(len(srcs), 1))(*[_native.LaneRigSource(*s) for s in srcs])
        return lib.lane_detect_rig(ctx_h, arr if srcs else None, len(srcs), 0, S, P(pf), P(valid), P(o))

    ok = (cam.ctypes.data, _native.INPUT_I420, 720, 1280, 2, 5)
    assert call(ok) == 0
    assert call(ok, pf=None) == -1 and call(ok, o=None) == -1 and call() == -1      # null sources / state / out
    assert call((cam.ctypes.data, _native.INPUT_I420, 720, 1280, 0, 5)) == -1      # no frame at all
    assert call(ok, ok, ok) == -1                                                   # 6 frames, max_batch 4
    assert call(ok, (cam.ctypes.data, 0, 720, 1280, -1, 0)) == -1                   # negative n
    assert call((cam.ctypes.data, 3, 720, 1280, 2, 0)) == -1                        # unknown format
    assert call((cam.ctypes.data, _native.INPUT_I420, 0, 1280, 2, 0)) == -1         # non-positive size
    assert call((cam.ctypes.data, _native.INPUT_NV12, 720, 1279, 2, 0)) == -1       # odd YUV width
    assert call((cam.ctypes.data, _native.INPUT_NV12, 719, 1280, 2, 0)) == -1       # odd YUV height
    assert call((cam.ctypes.data, _native.INPUT_I420, 720, 1280, 2, 8)) == -1       # stream_id outside [0, 8)
    assert call((cam.ctypes.data, _native.INPUT_I420, 720, 1280, 2, -1)) == -1
    assert call(ok, S=9) == -1 and b"ROI masks" in lib.lane_last_error(ctx._h)      # more streams than masks
    assert call(ok) == 0                                                            # and the context still works
    det.close()
