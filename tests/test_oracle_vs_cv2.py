"""Pin the C restatement (oracle/lane_oracle.c) against the real cv2 / numpy.

The reference ships no golden vectors, so the arithmetic contract is "what cv2 4.13 and
numpy 2.3 compute" (SURVEY.md section 8c).  Every stage is compared bit-exactly.
"""
import cv2
import numpy as np
import pytest

from oracle import stages as S
from util import gen_frames


def _frames():
    rng = np.random.default_rng(5)
    out = [("gen640", gen_frames(640, 480, 1)[0]), ("gen720", gen_frames(1280, 720, 1, 7)[0])]
    for shape in [(5, 5), (7, 9), (3, 3), (1, 8), (8, 1), (2, 2), (33, 65), (481, 643), (240, 320)]:
        out.append((f"noise{shape}", rng.integers(0, 256, shape + (3,), dtype=np.uint8)))
    out.append(("smooth", cv2.GaussianBlur(rng.integers(0, 256, (300, 400, 3), dtype=np.uint8), (31, 31), 0)))
    out.append(("black", np.zeros((120, 160, 3), np.uint8)))
    out.append(("white", np.full((120, 160, 3), 255, np.uint8)))
    lines = np.zeros((400, 600, 3), np.uint8)
    for _ in range(25):
        p = rng.integers(0, 600, 4)
        cv2.line(lines, (int(p[0]), int(p[1] % 400)), (int(p[2]), int(p[3] % 400)),
                 tuple(int(v) for v in rng.integers(60, 256, 3)), int(rng.integers(1, 4)))
    out.append(("lines", lines))
    return out


FRAMES = _frames()


@pytest.fixture(autouse=True)
def _cv2_single_thread():
    """cv2 4.13's multi-threaded 8-bit GaussianBlur races on frames 6 to 11 rows tall: the 7x9 noise frame comes back with
    a wrong row in a few percent of calls, with 8 threads or 128 alike.  On one thread its result is deterministic and
    equals the exact 5x5 kernel, which is what the oracle restates."""
    threads = cv2.getNumThreads()
    cv2.setNumThreads(1)
    yield
    cv2.setNumThreads(threads)


@pytest.mark.parametrize("name,frame", FRAMES, ids=[n for n, _ in FRAMES])
def test_gray_blur_median_canny(name, frame):
    g = S.gray(frame)
    assert np.array_equal(g, cv2.cvtColor(frame, cv2.COLOR_BGR2GRAY))
    b = S.blur5(g)
    assert np.array_equal(b, cv2.GaussianBlur(g, (5, 5), 0))
    med = np.median(b)
    low, high, m2 = S.thresholds(b)
    assert m2 == 2 * med
    assert low == int(max(0, 0.7 * med)) and high == int(min(255, 1.3 * med))
    taps = S.canny(b, low, high)
    assert np.array_equal(taps.edges, cv2.Canny(b, low, high))
    # fixed thresholds too (scene_classifier.py:145 uses 50/150) and swapped order
    assert np.array_equal(S.canny(b, 50, 150).edges, cv2.Canny(b, 50, 150))
    assert np.array_equal(S.canny(b, 150, 50).edges, cv2.Canny(b, 150, 50))
    # Sobel taps
    assert np.array_equal(taps.dx, cv2.Sobel(b, cv2.CV_16S, 1, 0, ksize=3, borderType=cv2.BORDER_REPLICATE))
    assert np.array_equal(taps.dy, cv2.Sobel(b, cv2.CV_16S, 0, 1, ksize=3, borderType=cv2.BORDER_REPLICATE))


def test_threshold_lut_samples():
    lo, hi = S.threshold_lut()
    for m, want in [(140, (98, 182)), (141.5, (99, 183)), (142, (99, 184)), (196, (137, 254)),
                    (196.5, (137, 255)), (0, (0, 0)), (255, (178, 255))]:
        assert (lo[int(2 * m)], hi[int(2 * m)]) == want


def test_median_even_and_odd():
    rng = np.random.default_rng(0)
    for n in (1, 2, 3, 10, 11, 1000, 1001):
        a = rng.integers(0, 256, n, dtype=np.uint8)
        assert S.median_x2(S.hist256(a), n) == 2 * np.median(a)


@pytest.mark.parametrize("name,frame", FRAMES, ids=[n for n, _ in FRAMES])
def test_houghp_and_standard_hough(name, frame):
    h, w = frame.shape[:2]
    if h < 3 or w < 3:
        pytest.skip("degenerate")
    b = S.blur5(S.gray(frame))
    low, high, _ = S.thresholds(b)
    edges = cv2.Canny(b, low, high)
    for img in (edges, edges & S.roi_mask(h, w)):
        for (thr, mn, gap) in [(50, 50, 150), (100, 100, 10), (10, 5, 2)]:
            want = cv2.HoughLinesP(img, 1, np.pi / 180, thr, minLineLength=mn, maxLineGap=gap)
            want = np.zeros((0, 4), np.int32) if want is None else want.reshape(-1, 4)
            got = S.houghp(img, thr, mn, gap, max_lines=1 << 16)
            assert np.array_equal(got, want), (name, thr)
        acc = S.hough_accum(img)
        assert acc.sum() == 180 * int((img != 0).sum())
        pk = S.hough_peaks(acc, h, w, 5)
        want = cv2.HoughLinesWithAccumulator(img, 1, np.pi / 180, 5)
        if want is None:
            assert len(pk) == 0
            continue
        want = want.reshape(-1, 3)
        assert len(want) == len(pk)
        nr = S.hough_numrho(h, w)
        assert np.array_equal((pk[:, 0] - (nr - 1) * 0.5).astype(np.float32), want[:, 0])
        assert np.array_equal(pk[:, 1].astype(np.float32) * np.float32(np.pi / 180), want[:, 1])
        assert np.array_equal(pk[:, 2], want[:, 2].astype(np.int32))


def test_cv2_pipeline_equals_stage_oracle():
    from oracle.cv2_pipeline import Cv2LaneOracle
    a, b = S.StageOracle(), Cv2LaneOracle()
    for f in gen_frames(640, 480, 12):
        tr = a.step(f)
        lf, rf = b.detect(f)
        for x, y in ((tr.left, lf), (tr.right, rf)):
            assert (x is None) == (y is None)
            if x is not None:
                assert np.array_equal(x.coeffs, y.coeffs) and np.array_equal(x.points, y.points)
        assert tr.offset == b.offset(640, lf, rf)
