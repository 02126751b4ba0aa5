"""The CPU statement of the fused ingest kernel (csrc/k0_ingest.cu): oracle resize of the oracle NV12 / I420 conversion
equals cv2.resize(cv2.cvtColor(f, COLOR_YUV2BGR_NV12 | COLOR_YUV2BGR_I420), size) -- at camera resolutions, up and down,
odd and tiny destinations and random even sources -- and the ingest entry points reject bad arguments before any
device work (these run without a GPU)."""
import ctypes

import cv2
import numpy as np
import pytest

from multimodal_autonomous_driving_perception_and_planning_b200 import FrameIngest, LaneDetector, _native
from oracle import nv12 as onv
from oracle import resize as orz
from yuv420 import i420_to_bgr, nv12_to_i420

# (source w, h) -> (destination w, h)
SIZE_PAIRS = [((1920, 1080), (640, 480)), ((1920, 1080), (960, 540)), ((1920, 1080), (1280, 720)),
              ((1280, 720), (1920, 1080)), ((3840, 2160), (640, 480)), ((642, 482), (333, 217)),
              ((640, 480), (640, 480)), ((2, 2), (5, 3))]
LAYOUTS = [("nv12", cv2.COLOR_YUV2BGR_NV12), ("i420", cv2.COLOR_YUV2BGR_I420)]


def random_size_pairs(k=40, seed=11):
    rng = np.random.default_rng(seed)
    return [((2 * int(rng.integers(1, 200)), 2 * int(rng.integers(1, 200))),
             (int(rng.integers(1, 400)), int(rng.integers(1, 400)))) for _ in range(k)]


def random_frame(src, layout, seed):
    w, h = src
    nv12 = np.random.default_rng(seed).integers(0, 256, (h * 3 // 2, w), dtype=np.uint8)
    return nv12 if layout == "nv12" else nv12_to_i420(nv12)


def oracle_ingest(frame, layout, dsize):
    bgr = onv.nv12_to_bgr(frame) if layout == "nv12" else i420_to_bgr(frame)
    return orz.resize_linear(bgr, dsize)


@pytest.mark.parametrize("layout,code", LAYOUTS)
@pytest.mark.parametrize("src,dst", SIZE_PAIRS)
def test_oracle_composition_equals_cv2(layout, code, src, dst):
    f = random_frame(src, layout, src[0] + dst[1])
    assert np.array_equal(oracle_ingest(f, layout, dst), cv2.resize(cv2.cvtColor(f, code), dst))


@pytest.mark.parametrize("layout,code", LAYOUTS)
def test_oracle_composition_equals_cv2_on_random_sizes(layout, code):
    for k, (src, dst) in enumerate(random_size_pairs()):
        f = random_frame(src, layout, k)
        assert np.array_equal(oracle_ingest(f, layout, dst), cv2.resize(cv2.cvtColor(f, code), dst)), (src, dst)


def test_i420_and_nv12_of_the_same_samples_convert_alike():
    f = random_frame((642, 482), "nv12", 3)
    assert np.array_equal(cv2.cvtColor(nv12_to_i420(f), cv2.COLOR_YUV2BGR_I420), cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12))
    with pytest.raises(ValueError):
        i420_to_bgr(np.zeros((9, 7), np.uint8))


YUV = np.zeros((2, 720, 640), np.uint8)
BAD_TARGETS = [(640,), (640, 480, 3), (0, 480), (640, -1), (640.0, 480), ("640", 480), 640, (True, 480)]


@pytest.mark.parametrize("call", ["detect_batch_nv12", "detect_batch_i420"])
def test_detector_yuv_input_errors_raise_before_the_device(call):
    det = LaneDetector()
    fn = getattr(det, call)
    for bad in (YUV.astype(np.float32), YUV[0], YUV[..., None], np.zeros((2, 721, 640), np.uint8),
                np.zeros((2, 722, 640), np.uint8), np.zeros((2, 720, 641), np.uint8)):
        with pytest.raises(cv2.error):
            fn(bad, target_size=(320, 240))
    for bad in BAD_TARGETS:
        with pytest.raises(cv2.error):
            fn(YUV, target_size=bad)
    assert fn(YUV[:0], target_size=(320, 240)) == []


def test_detector_bgr_target_size_errors_raise_before_the_device():
    det = LaneDetector()
    frames = np.zeros((2, 48, 64, 3), np.uint8)
    for bad in BAD_TARGETS:
        with pytest.raises(cv2.error):
            det.detect_batch(frames, target_size=bad)
    with pytest.raises(cv2.error):
        det.detect_batch(frames.astype(np.uint16), target_size=(32, 24))
    with pytest.raises(cv2.error):
        det.detect_batch(frames[0], target_size=(32, 24))


def test_frame_ingest_i420_errors_raise_before_the_device():
    ing = FrameIngest((320, 240))
    for bad in (YUV.astype(np.int16), YUV[0], np.zeros((2, 721, 640), np.uint8), np.zeros((2, 720, 641), np.uint8)):
        with pytest.raises(cv2.error):
            ing.from_i420(bad)
        with pytest.raises(cv2.error):
            ing.from_nv12(bad)


def test_raw_entry_points_reject_bad_arguments_without_a_device():
    lib = _native.lib()
    src = np.zeros(720 * 640, np.uint8)
    dst = np.zeros(240 * 320 * 3, np.uint8)
    p = src.ctypes.data_as(ctypes.c_void_p)
    q = dst.ctypes.data_as(ctypes.c_void_p)
    assert lib.lane_yuv420_to_bgr_batch(p, 0, 1, 480, 640, q, 240, 320, 0, 0, None) == -1       # BGR is not YUV
    assert lib.lane_yuv420_to_bgr_batch(p, 3, 1, 480, 640, q, 240, 320, 0, 0, None) == -1       # unknown format
    assert lib.lane_yuv420_to_bgr_batch(p, 1, 1, 481, 640, q, 240, 320, 0, 0, None) == -1       # odd height
    assert lib.lane_yuv420_to_bgr_batch(p, 2, 1, 480, 639, q, 240, 320, 0, 0, None) == -1       # odd width
    assert lib.lane_yuv420_to_bgr_batch(p, 1, 0, 480, 640, q, 240, 320, 0, 0, None) == -1       # empty batch
    assert lib.lane_yuv420_to_bgr_batch(p, 1, 1, 480, 640, q, 0, 320, 0, 0, None) == -1         # empty destination
    assert lib.lane_yuv420_to_bgr_batch(p, 1, 1, 480, 640, q, 70000, 320, 0, 0, None) == -5     # beyond the grid
    assert b"65535" in lib.lane_last_error(None)
    assert lib.lane_detect_batch_ingest(None, p, 0, 1, 1, 480, 640, None, 1, None, None, None) == -1
