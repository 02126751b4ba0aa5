"""Packed YUV 4:2:2 camera frames into the lane path, without a GPU: the CPU statement of the conversion
(oracle/yuv422.py) equals cv2.cvtColor(f, COLOR_YUV2BGR_UYVY | COLOR_YUV2BGR_YUY2) on every (Y, U, V) triple and at
camera sizes, its resize equals cv2.resize of cv2's frame, and every argument error of detect_batch_yuv422 / detect_rig
/ FrameIngest.from_yuv422 / the raw entry points is raised before any device work."""
import ctypes

import cv2
import numpy as np
import pytest

from multimodal_autonomous_driving_perception_and_planning_b200 import FrameIngest, LaneDetector, _native
from oracle import resize as orz
from oracle import yuv422 as oy
from test_oracle_ingest import SIZE_PAIRS

CODES = {"uyvy": cv2.COLOR_YUV2BGR_UYVY, "yuyv": cv2.COLOR_YUV2BGR_YUY2}
ENCODE = {"uyvy": cv2.COLOR_BGR2YUV_UYVY, "yuyv": cv2.COLOR_BGR2YUV_YUY2}
ORDERS = sorted(CODES)
SIZES = [(1, 2), (3, 6), (721, 1280), (1080, 1920), (1216, 1936), (2160, 3840)]        # (h, w)


def random_sizes(k=40, seed=29):
    """(h, w), w even, from 1x2 to 4K, small sizes over-represented."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(k):
        top = int(rng.choice([16, 300, 2160]))
        out.append((int(rng.integers(1, top + 1)), 2 * int(rng.integers(1, top * 8 // 9 + 1))))
    return out


def frame(h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (h, w, 2), dtype=np.uint8)


def every_triple(order):
    """One [4096, 4096, 2] frame holding every (U, V) pair with 128 Y pairs each, so all 2^24 (Y, U, V) triples."""
    k = np.arange(4096 * 2048, dtype=np.int64)            # the 4-byte groups in raster order
    uv, j = k // 128, k % 128
    y0i, ui, y1i, vi = oy.OFFSETS[order]
    g = np.empty((k.size, 4), np.uint8)
    g[:, y0i], g[:, y1i] = 2 * j, 2 * j + 1
    g[:, ui], g[:, vi] = uv >> 8, uv & 255
    return g.reshape(4096, 4096, 2)


def test_layout_constants():
    assert _native.YUV422 == {"uyvy": 8, "yuyv": 9}
    assert (_native.INPUT_UYVY, _native.INPUT_YUYV) == (8, 9)


@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("h,w", SIZES)
def test_oracle_equals_cv2(order, h, w):
    f = frame(h, w, h * 7 + w)
    assert np.array_equal(oy.yuv422_to_bgr(f, order), cv2.cvtColor(f, CODES[order]))


@pytest.mark.parametrize("order", ORDERS)
def test_oracle_equals_cv2_on_random_sizes(order):
    for k, (h, w) in enumerate(random_sizes()):
        f = frame(h, w, k)
        assert np.array_equal(oy.yuv422_to_bgr(f, order), cv2.cvtColor(f, CODES[order])), (h, w)


@pytest.mark.parametrize("order", ORDERS)
def test_oracle_equals_cv2_on_every_yuv_triple(order):
    f = every_triple(order)
    assert np.array_equal(oy.yuv422_to_bgr(f, order), cv2.cvtColor(f, CODES[order]))


@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("src,dst", SIZE_PAIRS + [((1280, 721), (640, 480))])
def test_oracle_resize_equals_cv2_resize(order, src, dst):
    w, h = src
    f = frame(h, w, w + dst[0])
    assert np.array_equal(orz.resize_linear(oy.yuv422_to_bgr(f, order), dst), cv2.resize(cv2.cvtColor(f, CODES[order]), dst))


def test_cv2_encodes_camera_like_frames_and_odd_widths_are_refused():
    bgr = np.random.default_rng(3).integers(0, 256, (6, 10, 3), dtype=np.uint8)
    for order in ORDERS:
        f = cv2.cvtColor(bgr, ENCODE[order])
        assert f.shape == (6, 10, 2) and f.dtype == np.uint8
        assert np.array_equal(oy.yuv422_to_bgr(f, order), cv2.cvtColor(f, CODES[order]))
        with pytest.raises(cv2.error):
            cv2.cvtColor(np.zeros((4, 5, 2), np.uint8), CODES[order])
        with pytest.raises(ValueError):
            oy.yuv422_to_bgr(np.zeros((4, 5, 2), np.uint8), order)


YUV = np.zeros((2, 48, 64, 2), np.uint8)
BAD_FRAMES = [YUV.astype(np.float32), YUV.astype(np.uint16), YUV[0], YUV[..., 0], np.zeros((2, 48, 64, 3), np.uint8),
              np.zeros((2, 48, 63, 2), np.uint8), np.zeros((2, 48, 64, 1), np.uint8)]


def test_detect_batch_yuv422_errors_raise_before_the_device():
    det = LaneDetector()
    for bad in BAD_FRAMES:
        with pytest.raises(cv2.error):
            det.detect_batch_yuv422(bad, "uyvy", target_size=(32, 24))
    for order in ("UYVY", "yuy2", "yvyu", "", None, 8):
        with pytest.raises(ValueError):
            det.detect_batch_yuv422(YUV, order)
    with pytest.raises(TypeError):
        det.detect_batch_yuv422(YUV)                       # the order has no default
    for bad in [(640,), (0, 480), (640.0, 480), "640x480"]:
        with pytest.raises(cv2.error):
            det.detect_batch_yuv422(YUV, "yuyv", target_size=bad)
    assert det.detect_batch_yuv422(YUV[:0], "yuyv", target_size=(32, 24)) == []
    assert det._ctx is None


@pytest.mark.parametrize("cams,layouts,exc,match", [
    ([np.zeros((1, 48, 64, 3), np.uint8)], ["uyvy"], ValueError, "needs frames \\[T,H,W,2\\]"),
    ([np.zeros((1, 48, 64), np.uint8)], ["yuyv"], ValueError, "needs frames \\[T,H,W,2\\]"),
    ([np.zeros((48, 64, 2), np.uint8)], ["uyvy"], ValueError, "needs frames \\[T,H,W,2\\]"),
    ([np.zeros((1, 48, 63, 2), np.uint8)], ["uyvy"], ValueError, "even width"),
    ([np.zeros((1, 48, 64, 2), np.uint8)], ["yvyu"], ValueError, "layout 'yvyu'"),
    ([np.zeros((1, 48, 64, 2), np.uint8)], ["UYVY"], ValueError, "layout 'UYVY'"),
    ([np.zeros((1, 48, 64, 2), np.float32)], ["yuyv"], cv2.error, "uint8"),
])
def test_bad_yuv422_rig_arguments_raise_before_any_native_call(cams, layouts, exc, match):
    det = LaneDetector()
    with pytest.raises(exc, match=match):
        det.detect_rig(cams, layouts, target_size=(64, 48))
    assert det._ctx is None


def test_yuv422_layouts_are_planned_at_two_bytes_per_pixel():
    from multimodal_autonomous_driving_perception_and_planning_b200.perception import lane_detector as L
    det = LaneDetector()
    cams = [np.zeros((2, 1080, 1920, 2), np.uint8), np.zeros((1, 1620, 1920), np.uint8),
            np.zeros((1, 721, 1280, 2), np.uint8), np.zeros((1, 5, 3), np.uint8), np.zeros((1, 3, 2, 2), np.uint8)]
    p = det._rig_plan(cams, ["uyvy", "nv12", "yuyv", "bayer_rggb", "uyvy"], (640, 480), None)
    assert p.sizes == [(1080, 1920), (1080, 1920), (721, 1280), (5, 3), (3, 2)] and (p.h, p.w) == (480, 640)
    assert p.fmts == [8, 1, 9, 16, 8]
    assert [L._frame_bytes(f, *hw) for f, hw in zip(p.fmts, p.sizes)] == [1080 * 1920 * 2, 1080 * 1920 * 3 // 2,
                                                                          721 * 1280 * 2, 15, 12]
    assert [L._frame_bytes(f, *hw) for f, hw in zip(p.fmts, p.sizes)] == [c[0].nbytes for c in cams]
    for fmt in (_native.INPUT_UYVY, _native.INPUT_YUYV):
        q = L._Plan.of_frames(cams[2], fmt)
        assert q.sizes == [(721, 1280)] and (q.h, q.w) == (721, 1280)
        assert L._frame_bytes(fmt, *q.sizes[0]) == cams[2][0].nbytes
        q = L._Plan.of_frames(cams[0], fmt, (640, 480))
        assert q.sizes == [(1080, 1920)] and (q.h, q.w) == (480, 640)


def test_frame_ingest_yuv422_errors_raise_before_the_device():
    ing = FrameIngest((320, 240))
    for bad in BAD_FRAMES:
        with pytest.raises(cv2.error):
            ing.from_yuv422(bad, "uyvy")
    for order in ("vyuy", None):
        with pytest.raises(ValueError):
            ing.from_yuv422(YUV, order)


def test_context_free_entry_reports_no_device_under_its_own_name():
    pytest.importorskip("torch")
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is visible")
    lib = _native.lib()
    src, dst = np.zeros(48 * 64 * 2, np.uint8), np.zeros(24 * 32 * 3, np.uint8)
    rc = lib.lane_yuv422_to_bgr_batch(_native._ptr(src), _native.INPUT_UYVY, 1, 48, 64, _native._ptr(dst), 24, 32, 0, 0,
                                      None)
    assert rc == -3 and lib.lane_last_error(None).startswith(b"lane_yuv422_to_bgr_batch: ")


def test_raw_entry_points_reject_bad_arguments_without_a_device():
    lib = _native.lib()
    src = np.zeros(48 * 64 * 2, np.uint8)
    dst = np.zeros(24 * 32 * 3, np.uint8)
    p, q = src.ctypes.data_as(ctypes.c_void_p), dst.ctypes.data_as(ctypes.c_void_p)
    U = _native.INPUT_UYVY
    for fmt in (3, 7, 10, _native.INPUT_NV12, _native.INPUT_BAYER_RGGB):                    # not a 4:2:2 layout
        assert lib.lane_yuv422_to_bgr_batch(p, fmt, 1, 48, 64, q, 24, 32, 0, 0, None) == -1
    assert lib.lane_yuv422_to_bgr_batch(p, U, 1, 48, 63, q, 24, 32, 0, 0, None) == -1          # odd width
    assert b"even width" in lib.lane_last_error(None)
    assert lib.lane_yuv422_to_bgr_batch(p, U, 0, 48, 64, q, 24, 32, 0, 0, None) == -1          # empty batch
    assert lib.lane_yuv422_to_bgr_batch(None, U, 1, 48, 64, q, 24, 32, 0, 0, None) == -1       # null source
    assert lib.lane_yuv422_to_bgr_batch(p, U, 1, 48, 64, q, 0, 32, 0, 0, None) == -1           # empty destination
    assert lib.lane_yuv422_to_bgr_batch(p, U, 1, 48, 64, q, 70000, 32, 0, 0, None) == -5       # beyond the grid
    assert lib.lane_yuv422_to_bgr_batch(p, U, 70000, 48, 64, q, 24, 32, 0, 0, None) == -5
    # the 4:2:0 and Bayer entries keep refusing everything but their own layouts
    for fmt in _native.YUV422.values():
        assert lib.lane_yuv420_to_bgr_batch(p, fmt, 1, 48, 64, q, 24, 32, 0, 0, None) == -1
        assert lib.lane_bayer_to_bgr_batch(p, fmt, 1, 48, 64, q, 24, 32, 0, 0, None) == -1
    # context calls with a null context are invalid
    assert lib.lane_detect_batch_ingest(None, p, 0, 1, U, 48, 64, None, 1, None, None, None) == -1
    fit, valid = np.zeros((1, 2, 3)), np.zeros((1, 2), np.uint8)
    out = np.zeros(1, _native.RECORD_DTYPE)
    for fmt in (U, _native.INPUT_YUYV):
        srcs = (_native.LaneRigSource * 1)(_native.LaneRigSource(src.ctypes.data, fmt, 48, 64, 1, 0))
        assert lib.lane_detect_rig(None, srcs, 1, 0, 1, _native._ptr(fit), _native._ptr(valid), _native._ptr(out)) == -1
        assert lib.lane_rig_enqueue(None, srcs, 1, 0, 1, None, None) == -1
