"""One ROI per camera of a rig in one batched call: ``detect_streams(..., stream_rois=[...])`` and the native contexts
with several ROI masks (``lane_set_roi_masks``).

Every frame's records, taps and Hough outputs must equal, byte for byte, what a single-ROI detector built with that
camera's polygon gives on that camera's frames in order; lanes must match the cv2 reference pipeline with that polygon
within the bars of test_gpu_parity.py."""
import cv2
import numpy as np
import pytest

from cases import CUSTOM_ROI
from multimodal_autonomous_driving_perception_and_planning_b200 import LaneDetector, _native, multi_camera_batch
from oracle import stages as S
from oracle.cv2_pipeline import Cv2LaneOracle
from util import gen_frames

pytestmark = pytest.mark.gpu

N_CAMS = 8


def rig_polys(h, w):
    """Eight polygons in roi_vertices form: default (None), shifted, narrowed, non-convex, CUSTOM_ROI scaled, one that
    keeps only the sky (no lane in it), the full frame, and one wholly outside the frame (an empty mask)."""
    def poly(*pts):
        return np.array([pts], np.int32)
    dx = int(w * 0.08)
    return [
        None,
        poly((int(w * 0.1) + dx, h), (int(w * 0.4) + dx, int(h * 0.6)), (int(w * 0.6) + dx, int(h * 0.6)), (int(w * 0.9) + dx, h)),
        poly((int(w * 0.25), h), (int(w * 0.45), int(h * 0.62)), (int(w * 0.55), int(h * 0.62)), (int(w * 0.75), h)),
        poly((0, h - 1), (int(w * 0.3), int(h * 0.55)), (int(w * 0.5), int(h * 0.85)), (int(w * 0.7), int(h * 0.55)), (w - 1, h - 1)),
        (CUSTOM_ROI.astype(np.float64) * [w / 640, h / 480]).astype(np.int32),
        poly((0, 0), (w - 1, 0), (w - 1, int(h * 0.2)), (0, int(h * 0.2))),
        poly((0, 0), (w - 1, 0), (w - 1, h - 1), (0, h - 1)),
        poly((-40, -40), (-10, -40), (-10, -10)),
    ]


def rig_masks(h, w):
    return np.stack([S.roi_mask(h, w, p) for p in rig_polys(h, w)])


def interleaved(n_cams, t):
    """Frame order of a rig tick by tick, cameras rotated every tick: (camera, time) per position."""
    return [((s + k) % n_cams, k) for k in range(t) for s in range(n_cams)]


def rig_frames(h, w, t):
    """[S, T, H, W, 3] camera streams: the generator's scenes at 1080p, its frames one per camera at other sizes."""
    if (h, w) == (1080, 1920):
        return multi_camera_batch(N_CAMS, t, w, h)
    return np.stack([np.stack(gen_frames(w, h, t, start=1000 * s)) for s in range(N_CAMS)])


def single_roi_records(cams, polys, **kw):
    """What one single-ROI LaneDetector per camera returns for that camera's frames in order: (records, detector)."""
    out = []
    for s, poly in enumerate(polys):
        det = LaneDetector(poly, max_batch=cams.shape[1], **kw)
        det.detect_batch(cams[s])
        out.append((det.last_records.copy(), det))
    return out


def run_rig(cams, polys, max_batch, **kw):
    order = interleaved(cams.shape[0], cams.shape[1])
    frames = np.stack([cams[s, t] for s, t in order])
    det = LaneDetector(max_batch=max_batch, **kw)
    lanes = det.detect_streams(frames, stream_ids=[s for s, _ in order], stream_rois=polys)
    return det, lanes, order


def test_rig_1080p_equals_single_roi_detectors_and_cv2():
    h, w, t = 1080, 1920, 3
    cams, polys = rig_frames(h, w, t), rig_polys(h, w)
    det, lanes, order = run_rig(cams, polys, max_batch=10)          # 24 frames: three chunks, host frames
    recs = det.last_records
    print(f"lane_ctx_last_paths = {det._ctx.last_paths()} (PATH_ALL_FAST = {_native.PATH_ALL_FAST})")
    assert det._ctx.n_roi == N_CAMS
    want = single_roi_records(cams, polys)
    for k, (s, ti) in enumerate(order):
        assert recs[k].tobytes() == want[s][0][ti].tobytes(), (k, s, ti)
    ys = np.linspace(h * 0.6, h, 50)
    for s, poly in enumerate(polys):
        ref = Cv2LaneOracle(roi_vertices=poly)
        for ti in range(t):
            k = order.index((s, ti))
            lf, rf = ref.detect(cams[s, ti])
            for side, fit in enumerate((lf, rf)):
                lane = lanes[k][side]
                assert (lane is None) == (fit is None), (s, ti, side)
                if fit is not None:
                    xw = np.polyval(fit.coeffs, ys)
                    assert np.abs(np.polyval(lane.polynomial, ys) - xw).max() <= 1e-6 * max(1.0, np.abs(xw).max())
                    assert np.abs(lane.points.astype(np.int64) - fit.points).max() <= 1
            off, want_off = det.get_lane_center_offset(w, *lanes[k]), Cv2LaneOracle.offset(w, lf, rf)
            assert (off is None) == (want_off is None) and (off is None or abs(off - want_off) <= 0.5)
    # the empty ROI has no point and no lane
    assert all(recs[k]["n_roi_points"] == 0 and recs[k]["side"]["valid"].sum() == 0
               for k, (s, _) in enumerate(order) if s == 7)
    for _, d in want:
        d.close()
    det.close()


@pytest.mark.parametrize("shape", [(480, 640), (481, 643)])       # 643 columns: the generic-width byte-map kernels
def test_rig_taps_and_standard_hough_equal_single_roi(shape):
    h, w = shape
    t = 2
    cams, polys = rig_frames(h, w, t), rig_polys(h, w)
    n = N_CAMS * t
    det, _, order = run_rig(cams, polys, max_batch=n, debug=True)
    ctx, recs = det._ctx, det.last_records
    if w % 16:
        assert not ctx.last_paths() & _native.PATH_CLUSTER_CANNY
    want = single_roi_records(cams, polys, debug=True)
    thr = 5
    peaks, counts, acc, _ = ctx.hough_lines_batch(n, threshold=thr, max_peaks=1 << 15, with_accum=True)
    single_hough = [d._ctx.hough_lines_batch(t, threshold=thr, max_peaks=1 << 15, with_accum=True) for _, d in want]
    oracles = [S.StageOracle(roi_vertices=p) for p in polys]
    for k, (s, ti) in enumerate(order):
        assert recs[k].tobytes() == want[s][0][ti].tobytes(), (shape, k, s)
        tr = oracles[s].step(cams[s, ti])            # frames of a camera come in time order
        ys, xs = np.nonzero(tr.masked)
        got_pts = ctx.tap(_native.TAP_POINTS, k) if len(xs) else np.zeros((0, 2), np.int32)
        assert np.array_equal(got_pts, np.stack([xs, ys], 1).astype(np.int32).reshape(-1, 2)), (shape, k, s)
        assert np.array_equal(ctx.tap(_native.TAP_SEGMENTS, k), tr.lines), (shape, k, s)
        # batched standard Hough: the single-ROI context's output, and cv2's peaks of Canny & this camera's mask
        sp, sc, sa, _ = single_hough[s]
        assert counts[k] == sc[ti] and np.array_equal(peaks[k], sp[ti]) and np.array_equal(acc[k], sa[ti]), (shape, k, s)
        lines = cv2.HoughLinesWithAccumulator(tr.masked, 1, np.pi / 180, thr)
        if lines is None:
            assert counts[k] == 0
        else:
            lines = lines.reshape(-1, 3)
            assert np.array_equal(lines[:, 2].astype(np.int32), peaks[k][:, 2])
            assert np.allclose(lines[:, 0], peaks[k][:, 0] - (2 * (w + h)) * 0.5)
        # one-frame accumulator tap
        a1, p1, f1 = ctx.hough_accumulator(k, threshold=thr, max_peaks=1 << 16)
        a2, p2, f2 = want[s][1]._ctx.hough_accumulator(ti, threshold=thr, max_peaks=1 << 16)
        assert np.array_equal(a1, a2) and np.array_equal(p1, p2) and f1 == f2, (shape, k, s)
    for _, d in want:
        d.close()
    det.close()


def test_streaming_two_batches_in_flight_equals_blocking_calls():
    import torch
    h, w, n_batches = 1080, 1920, 6
    cams = multi_camera_batch(N_CAMS, n_batches, w, h)
    masks = rig_masks(h, w)
    rng = np.random.default_rng(1)
    ids = [rng.permutation(N_CAMS).astype(np.int32) for _ in range(n_batches)]       # one frame per camera per batch
    frames = torch.from_numpy(np.stack([cams[s, b] for b in range(n_batches) for s in ids[b]])).cuda()
    torch.cuda.synchronize()
    fbytes = h * w * 3

    blocking = _native.LaneContext(h, w, N_CAMS, masks)
    fit, valid = np.zeros((N_CAMS, 2, 3)), np.zeros((N_CAMS, 2), np.uint8)
    want = [blocking.detect(frames.data_ptr() + b * N_CAMS * fbytes, N_CAMS, True, ids[b], N_CAMS, fit, valid, 0.7, 0.3)
            for b in range(n_batches)]

    ctx = _native.LaneContext(h, w, N_CAMS, masks)
    fit2, valid2 = np.zeros((N_CAMS, 2, 3)), np.zeros((N_CAMS, 2), np.uint8)
    ptr = [frames.data_ptr() + b * N_CAMS * fbytes for b in range(n_batches)]
    ctx.enqueue(ptr[0], N_CAMS, ids[0], N_CAMS, fit2, valid2, 0.7, 0.3)
    ctx.enqueue(ptr[1], N_CAMS, ids[1], N_CAMS, None, None, 0.7, 0.3)
    got = []
    for b in range(2, n_batches):
        got.append(ctx.collect(fit2, valid2))
        ctx.enqueue(ptr[b], N_CAMS, ids[b], N_CAMS, None, None, 0.7, 0.3)
    got += [ctx.collect(fit2, valid2), ctx.collect(fit2, valid2)]
    for b in range(n_batches):
        assert got[b].tobytes() == want[b].tobytes(), b
    assert fit2.tobytes() == fit.tobytes() and np.array_equal(valid2, valid)
    ctx.close(); blocking.close()


def test_dense_camera_reruns_on_a_context_with_the_same_masks():
    h, w, t = 1080, 1920, 2
    cams, polys = rig_frames(h, w, t), rig_polys(h, w)
    cams[6] = np.random.default_rng(5).integers(0, 256, cams[6].shape, dtype=np.uint8)    # full-frame ROI, noise
    det, _, order = run_rig(cams, polys, max_batch=N_CAMS * t)
    assert det.dense_reruns >= 1 and not det.last_records["flags"].any()
    assert det._dense_ctx.n_roi == N_CAMS
    want = single_roi_records(cams, polys)
    assert want[6][1].dense_reruns >= 1
    for k, (s, ti) in enumerate(order):
        assert det.last_records[k].tobytes() == want[s][0][ti].tobytes(), (k, s)
    assert max(det.last_records["n_segments"]) > 256
    for _, d in want:
        d.close()
    det.close()


def _set_masks(ctx, masks):
    masks = np.ascontiguousarray(masks, np.uint8)
    ctx._check(_native.lib().lane_set_roi_masks(ctx._h, _native._ptr(masks), masks.shape[0]))


@pytest.mark.parametrize("shape", [(480, 640), (481, 643)])
def test_masks_set_again_on_a_live_context_equal_fresh_contexts(shape):
    h, w = shape
    cams = rig_frames(h, w, 1)
    frames = np.ascontiguousarray(cams[:, 0])
    ids = np.arange(N_CAMS, dtype=np.int32)[::-1].copy()
    frames = np.ascontiguousarray(frames[ids])
    rig, one = rig_masks(h, w), rig_masks(h, w)[3:4]

    def detect(ctx):
        fit, valid = np.zeros((N_CAMS, 2, 3)), np.zeros((N_CAMS, 2), np.uint8)
        recs = ctx.detect(frames, N_CAMS, False, ids, N_CAMS, fit, valid, 0.7, 0.3)
        return recs.tobytes() + fit.tobytes() + valid.tobytes()

    want = {}
    for name, m in (("rig", rig), ("one", one)):
        fresh = _native.LaneContext(h, w, N_CAMS, m)
        want[name] = detect(fresh)
        fresh.close()
    live = _native.LaneContext(h, w, N_CAMS, rig)
    for name, m in (("rig", rig), ("one", one), ("rig", rig)):
        _set_masks(live, m)
        assert detect(live) == want[name], (shape, name)
    # more streams than masks is refused, the context stays usable
    lib = _native.lib()
    fit, valid = np.zeros((N_CAMS + 1, 2, 3)), np.zeros((N_CAMS + 1, 2), np.uint8)
    out = np.zeros(N_CAMS, _native.RECORD_DTYPE)
    rc = lib.lane_detect_batch(live._h, _native._ptr(frames), 0, N_CAMS, _native._ptr(ids), N_CAMS + 1,
                               _native._ptr(fit), _native._ptr(valid), _native._ptr(out))
    assert rc == -1 and b"ROI masks" in lib.lane_last_error(live._h)
    assert detect(live) == want["rig"]
    assert lib.lane_set_roi_masks(live._h, _native._ptr(rig), 0) == -1
    live.close()
