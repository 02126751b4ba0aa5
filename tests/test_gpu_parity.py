"""Parity of the CUDA path (through the C ABI) against the oracle and the reference goldens.

Run on the B200 box: python -m pytest tests -m gpu.  Nothing here reads /root/reference.
Bars: integer/byte/index stages bit-exact (blur, histogram, thresholds, NMS classes, Canny map,
ROI point list, HoughLinesP segments, standard-Hough accumulator and peaks); fp64 tail within
1e-3 relative on coefficients (atol for the mathematically-zero ones), <= 1e-6 px on the
evaluated lane x positions, sample points within 1 px of the reference's truncated ints.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import cv2  # noqa: E402

from cases import CUSTOM_ROI, build_cases, custom_roi_frames  # noqa: E402
from multimodal_autonomous_driving_perception_and_planning_b200 import (  # noqa: E402
    LaneDetector, SyntheticDataGenerator, _native)
from oracle import stages as S  # noqa: E402
from oracle.cv2_pipeline import Cv2LaneOracle  # noqa: E402
from util import gen_frames, golden, h16, lines_of, unpack_edges  # noqa: E402

COEF_RTOL = 1e-3       # north_star: "within 1e-3 relative (or 0.5 px)"
X_ATOL_PX = 1e-6


def _sample_rows(h):
    return np.linspace(h * 0.6, h, 50)


def _check_side(rec_side, want_coeffs, want_points, want_conf, h):
    got = rec_side["coeffs"]
    xs_got = np.polyval(got, _sample_rows(h))
    xs_want = np.polyval(want_coeffs, _sample_rows(h))
    assert np.abs(xs_got - xs_want).max() <= X_ATOL_PX * max(1.0, np.abs(xs_want).max())
    scale = np.abs(want_coeffs) + np.array([1e-9, 1e-6, 1e-3])   # zero quadratic terms come back as 1e-15 noise
    assert (np.abs(got - want_coeffs) / scale).max() <= COEF_RTOL
    assert np.abs(rec_side["points"].astype(np.int64) - want_points).max() <= 1
    assert rec_side["confidence"] == want_conf


def _run_stage_checks(frames, roi=None, hough=False):
    """Every tap of every frame against the stage oracle (bit-exact), records against its fits."""
    h, w = frames[0].shape[:2]
    det = LaneDetector(roi, max_batch=len(frames), debug=True)
    lanes = det.detect_batch(np.stack(frames))
    recs, ctx = det.last_records, det._ctx
    so = S.StageOracle(roi_vertices=roi)
    for i, f in enumerate(frames):
        tr = so.step(f)
        assert np.array_equal(ctx.tap(_native.TAP_GRAY, i), tr.gray), i
        assert np.array_equal(ctx.tap(_native.TAP_BLUR, i), tr.blurred), i
        assert np.array_equal(ctx.tap(_native.TAP_HIST, i), S.hist256(tr.blurred)), i
        assert (recs[i]["median_x2"], recs[i]["low"], recs[i]["high"]) == (tr.median_x2, tr.low, tr.high), i
        assert np.array_equal(ctx.tap(_native.TAP_CLASS, i), tr.canny.cls), i
        edges = ctx.tap(_native.TAP_EDGES, i)
        assert np.array_equal(edges, tr.canny.edges), i
        assert recs[i]["n_edges"] == int((tr.canny.edges != 0).sum())
        ys, xs = np.nonzero(tr.masked)
        assert recs[i]["n_roi_points"] == len(xs)
        if len(xs):
            assert np.array_equal(ctx.tap(_native.TAP_POINTS, i), np.stack([xs, ys], 1).astype(np.int32)), i
        assert recs[i]["n_segments"] == len(tr.lines), (i, recs[i]["n_segments"], len(tr.lines))
        assert np.array_equal(ctx.tap(_native.TAP_SEGMENTS, i), tr.lines), i
        for s, fit in enumerate((tr.left, tr.right)):
            assert bool(recs[i]["side"][s]["valid"]) == (fit is not None), (i, s)
            assert (lanes[i][s] is None) == (fit is None)
            if fit is not None:
                _check_side(recs[i]["side"][s], fit.coeffs, fit.points, fit.confidence, h)
                assert recs[i]["side"][s]["n_lines"] == fit.n_lines
        assert bool(recs[i]["offset_valid"]) == (tr.offset is not None)
        if tr.offset is not None:
            assert abs(recs[i]["offset"] - tr.offset) <= 0.5
        if hough:
            acc, peaks, found = ctx.hough_accumulator(i, threshold=5, max_peaks=1 << 16)
            want = S.hough_accum(tr.masked)
            assert np.array_equal(acc, want), i
            assert np.array_equal(peaks, S.hough_peaks(want, h, w, 5)), i
    det.close()
    return recs


def test_stage_taps_generator_640x480():
    _run_stage_checks(gen_frames(640, 480, 6), hough=True)


# (8, 64) and (12, 1936): widths the fused kernel takes but fewer than 16 rows -> k1_tile + k2a_sobel_nms + the cluster
@pytest.mark.parametrize("shape", [(7, 9), (5, 5), (3, 3), (33, 65), (64, 64), (481, 643), (240, 320), (8, 64), (12, 1936)])
def test_stage_taps_noise(shape):
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    frames = [rng.integers(0, 256, shape + (3,), dtype=np.uint8) for _ in range(2)]
    _run_stage_checks(frames, hough=shape[0] >= 33)


@pytest.mark.parametrize("shape", [(16, 16), (48, 64), (135, 480), (271, 976), (137, 1936), (1080, 1920)])
def test_fused_kernel_blur_hist_thresholds_noise(shape):
    """Fused edge kernel (W % 16 == 0, H >= 16): blur plane, histogram and thresholds on uniform noise, every
    strip/band/edge-lane layout (1, 2, 3 and 5 strips; partial last strip; odd band heights)."""
    rng = np.random.default_rng(shape[0] + shape[1])
    frames = np.stack([rng.integers(0, 256, shape + (3,), dtype=np.uint8) for _ in range(3)])
    frames[2, :, : shape[1] // 2] = 255          # saturated half: counters and clipping
    det = LaneDetector(max_batch=3, debug=True)
    det.detect_batch(frames)
    for i in range(3):
        want = S.blur5(S.gray(frames[i]))
        assert np.array_equal(det._ctx.tap(_native.TAP_BLUR, i), want), (shape, i)
        assert np.array_equal(det._ctx.tap(_native.TAP_HIST, i), S.hist256(want))
        low, high, m2 = S.thresholds(want)
        r = det.last_records[i]
        assert (r["median_x2"], r["low"], r["high"]) == (m2, low, high)
    det.close()


def test_stage_taps_smooth_black_white_lines():
    rng = np.random.default_rng(11)
    smooth = cv2.GaussianBlur(rng.integers(0, 256, (300, 400, 3), dtype=np.uint8), (31, 31), 0)
    lines = np.zeros((300, 400, 3), np.uint8)
    for _ in range(30):
        p = rng.integers(0, 400, 4)
        cv2.line(lines, (int(p[0]), int(p[1] % 300)), (int(p[2]), int(p[3] % 300)),
                 tuple(int(v) for v in rng.integers(60, 256, 3)), int(rng.integers(1, 4)))
    _run_stage_checks([smooth, np.zeros((300, 400, 3), np.uint8), np.full((300, 400, 3), 255, np.uint8), lines],
                      hough=True)


def test_edge_cases_against_oracle_and_golden():
    for name, frames in build_cases(SyntheticDataGenerator).items():
        recs = _run_stage_checks(frames)
        gold = golden("case_" + name)
        for i in range(len(frames)):
            assert recs[i]["n_edges"] == gold["n_edges"][i] and recs[i]["n_roi_points"] == gold["n_roi"][i], name
            assert np.array_equal(recs[i]["side"]["valid"], gold["valid"][i]), name


def test_custom_roi():
    frames = custom_roi_frames(SyntheticDataGenerator)
    recs = _run_stage_checks(frames, roi=CUSTOM_ROI, hough=True)
    gold = golden("case_custom_roi")
    assert [r["n_roi_points"] for r in recs] == list(gold["n_roi"])


def _check_against_golden(frames, gold, max_batch):
    h, w = frames[0].shape[:2]
    det = LaneDetector(max_batch=max_batch, debug=True)
    lanes = det.detect_batch(np.stack(frames))
    recs = det.last_records
    exact_points = 0
    total_points = 0
    for i in range(len(frames)):
        assert (recs[i]["median_x2"], recs[i]["low"], recs[i]["high"]) == \
            (gold["median_x2"][i], gold["low"][i], gold["high"][i])
        assert recs[i]["n_edges"] == gold["n_edges"][i] and recs[i]["n_roi_points"] == gold["n_roi"][i]
        assert recs[i]["n_segments"] == len(lines_of(gold, i))
        for s in (0, 1):
            assert bool(recs[i]["side"][s]["valid"]) == bool(gold["valid"][i, s])
            if gold["valid"][i, s]:
                _check_side(recs[i]["side"][s], gold["poly"][i, s], gold["points"][i, s], gold["conf"][i, s], h)
                exact_points += int((lanes[i][s].points == gold["points"][i, s]).all())
                total_points += 1
        off = det.get_lane_center_offset(w, *lanes[i])
        assert (off is None) == bool(np.isnan(gold["offset"][i]))
        if off is not None:
            assert abs(off - gold["offset"][i]) <= 0.5
    assert exact_points >= 0.99 * total_points
    return det, recs


def test_config1_300_frames_vs_reference_golden():
    """BASELINE config 1: the demo's 300-frame 640x480 sequence, one stream, EMA carried through."""
    gold = golden("config1_640x480")
    frames = gen_frames(640, 480, 300)
    det, recs = _check_against_golden(frames, gold, max_batch=300)
    ctx = det._ctx
    for i in range(0, 300, 7):
        assert h16(ctx.tap(_native.TAP_BLUR, i)) == str(gold["blur_hash"][i])
        assert h16(ctx.tap(_native.TAP_EDGES, i)) == str(gold["edge_hash"][i])
        assert np.array_equal(ctx.tap(_native.TAP_SEGMENTS, i), lines_of(gold, i))
    det.close()


@pytest.mark.parametrize("name,w,h,n,start", [("hd1080_cam0", 1920, 1080, 4, 0), ("hd1080_cam1", 1920, 1080, 2, 1000),
                                               ("hd720", 1280, 720, 2, 0), ("uhd2160", 3840, 2160, 1, 0)])
def test_larger_resolutions_vs_reference_golden(name, w, h, n, start):
    gold = golden(name)
    frames = gen_frames(w, h, n, start)
    det, recs = _check_against_golden(frames, gold, max_batch=n)
    for i in range(n):
        assert np.array_equal(det._ctx.tap(_native.TAP_EDGES, i), unpack_edges(gold["edges_packed"][i], h, w))
        assert np.array_equal(det._ctx.tap(_native.TAP_SEGMENTS, i), lines_of(gold, i))
    acc, peaks, found = det._ctx.hough_accumulator(0, threshold=50, max_peaks=4096)
    masked = unpack_edges(gold["edges_packed"][0], h, w) & S.roi_mask(h, w)
    want = S.hough_accum(masked)
    assert np.array_equal(acc, want)
    assert np.array_equal(peaks, S.hough_peaks(want, h, w, 50))
    det.close()


def test_detect_equals_detect_batch_and_chunking():
    frames = gen_frames(640, 480, 24)
    a = LaneDetector(max_batch=24)
    b = LaneDetector(max_batch=5)      # forces chunked native calls
    c = LaneDetector()
    la = a.detect_batch(np.stack(frames))
    lb = b.detect_batch(np.stack(frames))
    lc = [c.detect(f) for f in frames]
    for x, y, z in zip(la, lb, lc):
        for s in (0, 1):
            assert (x[s] is None) == (y[s] is None) == (z[s] is None)
            if x[s] is not None:
                assert np.array_equal(x[s].polynomial, y[s].polynomial) and np.array_equal(x[s].polynomial, z[s].polynomial)
                assert np.array_equal(x[s].points, z[s].points) and x[s].side == ("left", "right")[s]
    assert np.array_equal(a.prev_left_fit, c.prev_left_fit) and c.prev_left_fit is lc[-1][0].polynomial
    for d in (a, b, c):
        d.close()


def test_state_semantics_hit_miss_hit_and_reset():
    """SURVEY A.10: a miss keeps prev_*_fit; the next hit is smoothed against it; reset clears it."""
    g = SyntheticDataGenerator()
    f0 = g.generate_frame_with_vehicles()
    f1 = g.generate_frame_with_vehicles()
    det = LaneDetector()
    l0, r0 = det.detect(f0)
    assert l0 is not None and r0 is not None
    keep = det.prev_left_fit.copy()
    assert det.detect(np.zeros_like(f0)) == (None, None)
    assert np.array_equal(det.prev_left_fit, keep)
    l1, _ = det.detect(f1)
    raw = det.last_records[0]["side"][0]["raw"]
    assert np.array_equal(l1.polynomial, 0.7 * keep + (1 - 0.7) * raw)
    det.reset()
    assert det.prev_left_fit is None and det.prev_right_fit is None
    l2, _ = det.detect(f1)
    assert np.array_equal(l2.polynomial, det.last_records[0]["side"][0]["raw"])   # first hit is unsmoothed
    assert det.get_lane_center_offset(640, l2, None) is None
    # input untouched, non-contiguous view accepted
    view = np.ascontiguousarray(np.repeat(f0, 2, axis=1))[:, ::2]
    before = view.copy()
    det.reset()
    lv, _ = det.detect(view)
    assert np.array_equal(view, before) and np.array_equal(lv.polynomial, l0.polynomial)
    det.close()


def test_error_behaviour_matches_reference():
    det = LaneDetector()
    with pytest.raises(cv2.error):
        det.detect(np.zeros((48, 64, 3), np.float32))
    with pytest.raises(cv2.error):
        det.detect(np.zeros((48, 64), np.uint8))
    with pytest.raises(cv2.error):
        det.detect_batch(np.zeros((2, 48, 64, 1), np.uint8))
    assert det.detect_batch(np.zeros((0, 48, 64, 3), np.uint8)) == []


def test_streams_equal_independent_detectors():
    """Config 3 semantics at small scale: S cameras interleaved, each with its own EMA."""
    from multimodal_autonomous_driving_perception_and_planning_b200 import multi_camera_batch
    batch = multi_camera_batch(3, 5, 640, 480)
    det = LaneDetector(max_batch=16)
    got = det.detect_streams(batch)
    # interleaved order with explicit ids must give the same per-frame answers
    order = np.array([s * 5 + t for t in range(5) for s in range(3)])
    det2 = LaneDetector(max_batch=4)
    got2 = det2.detect_streams(batch.reshape(15, 480, 640, 3)[order], stream_ids=order // 5)
    for s in range(3):
        ref = Cv2LaneOracle()
        for t in range(5):
            lf, rf = ref.detect(batch[s, t])
            for side, fit in enumerate((lf, rf)):
                lane = got[s * 5 + t][side]
                lane2 = got2[int(np.nonzero(order == s * 5 + t)[0][0])][side]
                assert (lane is None) == (fit is None) == (lane2 is None)
                if fit is not None:
                    assert np.array_equal(lane.polynomial, lane2.polynomial)
                    assert np.abs(np.polyval(lane.polynomial, _sample_rows(480)) -
                                  np.polyval(fit.coeffs, _sample_rows(480))).max() < 1e-6
    det.close(); det2.close()


def test_torch_cuda_input_matches_host_input():
    import torch
    frames = np.stack(gen_frames(640, 480, 4))
    a = LaneDetector(max_batch=4).detect_batch(frames)
    b = LaneDetector(max_batch=4).detect_batch(torch.from_numpy(frames).cuda())
    for x, y in zip(a, b):
        for s in (0, 1):
            assert np.array_equal(x[s].polynomial, y[s].polynomial)


def test_config2_full_size_properties():
    """BASELINE config 2 at full size (256 x 1080p on one GPU): size-independent properties.
    The batch tiles 8 distinct frames, so per-frame (pre-EMA) results must repeat with period 8,
    must equal the golden for frames 0..3, and the edge count must equal a popcount of the map."""
    from multimodal_autonomous_driving_perception_and_planning_b200 import multi_camera_batch
    batch = multi_camera_batch(1, 256, 1920, 1080, period=8)[0]
    det = LaneDetector(max_batch=256, debug=False)
    det.detect_batch(batch)
    recs = det.last_records
    gold = golden("hd1080_cam0")
    for k in ("median_x2", "low", "high", "n_edges", "n_roi_points", "n_segments"):
        assert np.array_equal(recs[k], np.tile(recs[k][:8], 32)), k
    assert np.array_equal(recs["side"]["raw"], np.tile(recs["side"]["raw"][:8], (32, 1, 1)))
    assert np.array_equal(recs["n_edges"][:4], gold["n_edges"]) and np.array_equal(recs["n_roi_points"][:4], gold["n_roi"])
    for i in (0, 100, 255):
        e = det._ctx.tap(_native.TAP_EDGES, i)
        assert int((e != 0).sum()) == recs[i]["n_edges"] and set(np.unique(e)) <= {0, 255}
        assert np.array_equal(e, unpack_edges(gold["edges_packed"][i % 8], 1080, 1920)) if i % 8 < 4 else True
    assert recs["side"]["valid"].all()
    det.close()


def test_road_layout_cues_match_cv2():
    """SURVEY 8(f) rank 2: SceneClassifier's Canny(gray, 50, 150) + HoughLinesP(100, 100, 10) on the whole frame
    (src/tagging/scene_classifier.py:145-161), same kernels with other parameters, bit-exact vs cv2."""
    from multimodal_autonomous_driving_perception_and_planning_b200.perception import RoadLayoutAnalyzer
    rng = np.random.default_rng(3)
    frames = gen_frames(640, 480, 3) + [rng.integers(0, 256, (480, 640, 3), dtype=np.uint8)]
    an = RoadLayoutAnalyzer(max_batch=4, max_segments=8192)
    cues = an.analyze_batch(np.stack(frames))
    for f, c in zip(frames, cues):
        gray = cv2.cvtColor(f, cv2.COLOR_BGR2GRAY)
        edges = cv2.Canny(gray, 50, 150)
        h, w = gray.shape
        center = edges[h // 3:2 * h // 3, w // 3:2 * w // 3]
        assert c.center_density == np.sum(center > 0) / center.size
        want = cv2.HoughLinesP(edges, 1, np.pi / 180, 100, minLineLength=100, maxLineGap=10)
        want = np.zeros((0, 4), np.int32) if want is None else want.reshape(-1, 4)
        assert np.array_equal(c.lines, want)
        if len(want):
            assert abs(c.avg_length - np.mean([np.sqrt((l[2] - l[0]) ** 2 + (l[3] - l[1]) ** 2) for l in want])) < 1e-9
    an.close()


def _random_scene(rng, h, w):
    """Random structured frame: background gradient, random lines / rectangles / circles, mild noise."""
    yy, xx = np.mgrid[0:h, 0:w]
    base = (rng.integers(20, 200) + rng.integers(-60, 60) * yy / h + rng.integers(-60, 60) * xx / w)
    img = np.clip(np.stack([base + rng.integers(-20, 20) for _ in range(3)], -1), 0, 255).astype(np.uint8)
    for _ in range(int(rng.integers(3, 25))):
        col = tuple(int(v) for v in rng.integers(0, 256, 3))
        p = rng.integers(-20, max(h, w) + 20, 4)
        kind = rng.integers(0, 3)
        if kind == 0:
            cv2.line(img, (int(p[0]), int(p[1])), (int(p[2]), int(p[3])), col, int(rng.integers(1, 6)))
        elif kind == 1:
            cv2.rectangle(img, (int(p[0]), int(p[1])), (int(p[2]), int(p[3])), col, int(rng.choice([-1, 1, 2])))
        else:
            cv2.circle(img, (int(p[0]) % w, int(p[1]) % h), int(rng.integers(3, 60)), col, int(rng.choice([-1, 1, 3])))
    if rng.random() < 0.5:
        img = np.clip(img.astype(np.int16) + rng.integers(-6, 7, img.shape), 0, 255).astype(np.uint8)
    return img


@pytest.mark.parametrize("seed", range(10))
def test_randomised_scenes_against_cv2(seed):
    """Property-style sweep: random sizes (aligned and not), random structured content; the Canny map, the masked
    point list and the HoughLinesP segments must equal what cv2 itself computes with the reference's calls."""
    rng = np.random.default_rng(1000 + seed)
    h = int(rng.integers(40, 420))
    w = int(rng.choice([rng.integers(3, 40) * 16, rng.integers(50, 640)]))
    frames = [_random_scene(rng, h, w) for _ in range(3)]
    # odd seeds use looser Hough literals so small frames still produce many segments
    thr, min_len, gap = (50, 50, 150) if seed % 2 == 0 else (int(rng.integers(8, 30)), int(rng.integers(5, 30)),
                                                              int(rng.integers(0, 40)))
    det = LaneDetector(max_batch=3, max_segments=4096, debug=True)
    det._context(h, w, 3).set_hough_params(thr, min_len, gap)
    det.detect_batch(np.stack(frames))
    ref = Cv2LaneOracle()
    for i, f in enumerate(frames):
        edges = ref.edges(ref.blurred(f))
        masked = ref.masked(edges)
        lines = cv2.HoughLinesP(masked, rho=1, theta=np.pi / 180, threshold=thr, minLineLength=min_len,
                                maxLineGap=gap)
        want = np.zeros((0, 4), np.int32) if lines is None else lines.reshape(-1, 4)
        assert np.array_equal(det._ctx.tap(_native.TAP_EDGES, i), edges), (seed, i, h, w)
        assert det.last_records[i]["n_roi_points"] == int((masked != 0).sum())
        assert np.array_equal(det._ctx.tap(_native.TAP_SEGMENTS, i), want), (seed, i, h, w, thr, min_len, gap)
    det.close()


# ---- frame ingest (SURVEY 8f rank 1): batched cv2.resize on the device -------------------------------------
RESIZE_CASES = [(1920, 1080, 640, 480), (1920, 1080, 1280, 720), (640, 480, 1920, 1080), (1000, 700, 333, 217),
                (333, 217, 1000, 700), (64, 48, 640, 480), (5, 7, 33, 21), (1280, 720, 1279, 719), (17, 9, 1, 1)]


@pytest.mark.parametrize("sw,sh,dw,dh", RESIZE_CASES)
@pytest.mark.parametrize("cn", [3, 1])
def test_resize_batch_matches_cv2_and_oracle(sw, sh, dw, dh, cn):
    from multimodal_autonomous_driving_perception_and_planning_b200 import FrameIngest
    from oracle import resize as orz
    rng = np.random.default_rng(sw + 3 * dh + cn)
    frames = rng.integers(0, 256, (3, sh, sw, cn), dtype=np.uint8)
    got = FrameIngest((dw, dh)).resize_batch(frames)
    want = np.stack([cv2.resize(f, (dw, dh)).reshape(dh, dw, cn) for f in frames])
    assert got.shape == want.shape and got.dtype == np.uint8
    assert np.array_equal(got, want)
    assert np.array_equal(got[0], orz.resize_linear(frames[0], (dw, dh)).reshape(dh, dw, cn))


def test_resize_on_device_feeds_detector_without_leaving_hbm():
    """1080p generator frames -> FrameIngest(640x480) on the device -> LaneDetector.detect_batch(CUDA tensor):
    the same lanes as cv2.resize + the cv2 reference pipeline frame by frame."""
    import torch
    from multimodal_autonomous_driving_perception_and_planning_b200 import FrameIngest
    from multimodal_autonomous_driving_perception_and_planning_b200 import multi_camera_batch
    big = multi_camera_batch(1, 6, 1920, 1080)[0]
    dev_small = FrameIngest((640, 480)).resize_batch(torch.from_numpy(big).cuda())
    assert dev_small.is_cuda and tuple(dev_small.shape) == (6, 480, 640, 3)
    small = np.stack([cv2.resize(f, (640, 480)) for f in big])
    assert np.array_equal(dev_small.cpu().numpy(), small)
    det = LaneDetector(max_batch=6)
    lanes = det.detect_batch(dev_small)
    ref = Cv2LaneOracle()
    for i, f in enumerate(small):
        lf, rf = ref.detect(f)
        for got, want in ((lanes[i][0], lf), (lanes[i][1], rf)):
            assert (got is None) == (want is None)
            if got is not None:
                assert np.allclose(got.polynomial, want.coeffs, rtol=1e-3, atol=1e-6)
    det.close()


def test_resize_errors():
    from multimodal_autonomous_driving_perception_and_planning_b200 import FrameIngest
    with pytest.raises(cv2.error):
        FrameIngest((8, 8)).resize_batch(np.zeros((1, 4, 4, 3), np.float32))
    with pytest.raises(cv2.error):
        FrameIngest((8, 8)).resize_batch(np.zeros((1, 4, 4, 2), np.uint8))
    assert FrameIngest(None).resize_batch(np.zeros((1, 4, 4, 3), np.uint8)).shape == (1, 4, 4, 3)


# ---- scene statistics (SURVEY 8f rank 2, second half) --------------------------------------------------------
def test_scene_stats_match_cv2_expressions():
    """avg_brightness, laplacian_var and green_ratio of SceneClassifier (scene_classifier.py:183-186, :237-254)."""
    import torch
    from multimodal_autonomous_driving_perception_and_planning_b200 import multi_camera_batch
    from multimodal_autonomous_driving_perception_and_planning_b200.perception.scene_stats import SceneStatsAnalyzer
    from oracle import scene_stats as oss
    rng = np.random.default_rng(5)
    batches = [multi_camera_batch(1, 3, 1920, 1080)[0], multi_camera_batch(1, 3, 640, 480)[0],
               rng.integers(0, 256, (2, 97, 131, 3), dtype=np.uint8), rng.integers(0, 256, (2, 1, 9, 3), dtype=np.uint8),
               rng.integers(0, 256, (2, 200, 1, 3), dtype=np.uint8)]
    grass = np.zeros((2, 130, 260, 3), np.uint8)
    grass[...] = (40, 160, 60)
    grass[:, ::3] = (90, 200, 30)
    grass[:, :, ::7] = (200, 200, 200)
    batches.append(grass)
    an = SceneStatsAnalyzer()
    for frames in batches:
        for got_all in (an.analyze_batch(frames), an.analyze_batch(torch.from_numpy(frames).cuda())):
            for f, got in zip(frames, got_all):
                want = oss.frame_sums(f)
                assert (got.sum_gray, got.sum_laplacian, got.sum_laplacian_sq, got.green_pixels) == \
                    (want.sum_gray, want.sum_laplacian, want.sum_laplacian_sq, want.green_pixels)
                gray = cv2.cvtColor(f, cv2.COLOR_BGR2GRAY)
                green = cv2.inRange(cv2.cvtColor(f, cv2.COLOR_BGR2HSV), (35, 40, 40), (85, 255, 255))
                assert got.avg_brightness == np.mean(gray)
                assert got.green_ratio == np.sum(green > 0) / green.size
                assert got.laplacian_var == pytest.approx(cv2.Laplacian(gray, cv2.CV_64F).var(), rel=1e-12, abs=1e-12)


def test_hysteresis_long_weak_chains_are_schedule_independent():
    """Low-contrast textured scenes make long weak chains that cross band and word boundaries: the hysteresis
    kernel's walks / dirty flags / boundary rounds must give cv2's edge map on every run."""
    rng = np.random.default_rng(77)
    frames = []
    for _ in range(3):
        img = _random_scene(rng, 1080, 1920)
        img = np.clip(img.astype(np.int16) + rng.integers(-14, 15, img.shape), 0, 255).astype(np.uint8)
        frames.append(cv2.GaussianBlur(img, (0, 0), 1.5))
    frames = np.stack(frames)
    ref = Cv2LaneOracle()
    want = [ref.edges(ref.blurred(f)) for f in frames]
    det = LaneDetector(max_batch=3, max_segments=4096, debug=True)
    for _ in range(3):
        det.detect_batch(frames)
        for i in range(3):
            assert np.array_equal(det._ctx.tap(_native.TAP_EDGES, i), want[i]), i
            assert det.last_records[i]["hysteresis_rounds"] >= 1
    det.close()


def test_pageable_and_pinned_host_frames_give_identical_records():
    """Ordinary numpy frames go through the context's pinned staging ring (32 MB pieces copied by worker threads);
    pinned frames go straight to the copy engine.  Same records either way, call after call."""
    import torch
    from multimodal_autonomous_driving_perception_and_planning_b200 import multi_camera_batch
    frames = np.concatenate([multi_camera_batch(1, 10, 1920, 1080)[0]] * 4)          # 249 MB: eight pieces, two chunks
    pinned = torch.from_numpy(frames).pin_memory().numpy()
    det = LaneDetector(max_batch=40)
    det.detect_batch(pinned)
    want = det.last_records.copy()
    for _ in range(2):
        det.reset()
        det.detect_batch(frames)
        assert det.last_records.tobytes() == want.tobytes()
    det.close()


def test_two_batches_in_flight_with_state_on_the_device():
    """enqueue / enqueue / collect / ... with the EMA state carried on the device gives the records of calling
    detect_batch batch after batch on one detector (the reference's frame-after-frame state chain)."""
    import torch
    from multimodal_autonomous_driving_perception_and_planning_b200 import multi_camera_batch
    frames = multi_camera_batch(1, 24, 640, 480)[0]
    chunks = [frames[i:i + 6] for i in range(0, 24, 6)]
    det = LaneDetector(max_batch=6)
    want = []
    for ch in chunks:
        det.detect_batch(ch)
        want.append(det.last_records.copy())
    want_state = (det.prev_left_fit.copy(), det.prev_right_fit.copy())
    det.close()

    det = LaneDetector(max_batch=6)
    ctx = det._context(480, 640, 6)
    dev = [torch.from_numpy(ch).cuda() for ch in chunks]
    pf, pv = np.zeros((1, 2, 3)), np.zeros((1, 2), np.uint8)
    ctx.enqueue(dev[0].data_ptr(), 6, None, 1, pf, pv, 0.7, 1 - 0.7)            # explicit (empty) state
    got = []
    for i in range(4):
        if i + 1 < 4:
            ctx.enqueue(dev[i + 1].data_ptr(), 6, None, 1, None, None, 0.7, 1 - 0.7)   # queued behind batch i
        got.append(ctx.collect(pf, pv))
    for a, b in zip(got, want):
        assert a.tobytes() == b.tobytes()
    assert np.array_equal(pf[0, 0], want_state[0]) and np.array_equal(pf[0, 1], want_state[1]) and pv.all()
    with pytest.raises(_native.LaneError):                                    # a third batch does not fit the queue
        ctx.enqueue(dev[0].data_ptr(), 6, None, 1, None, None, 0.7, 1 - 0.7)
        ctx.enqueue(dev[1].data_ptr(), 6, None, 1, None, None, 0.7, 1 - 0.7)
        ctx.enqueue(dev[2].data_ptr(), 6, None, 1, None, None, 0.7, 1 - 0.7)
    while ctx._inflight:
        ctx.collect(pf, pv)
    det.close()
