"""A rig of cameras with their own sizes and layouts (``LaneDetector.detect_rig`` / ``lane_detect_rig``): the argument
checks that run before any device work, so they hold without a GPU."""
import ctypes

import cv2
import numpy as np
import pytest

from multimodal_autonomous_driving_perception_and_planning_b200 import LaneDetector, _native


def bgr(t, h, w, c=3, dtype=np.uint8):
    return np.zeros((t, h, w, c), dtype)


def yuv(t, h, w):
    return np.zeros((t, h * 3 // 2, w), np.uint8)


def test_wrong_channel_count_or_dtype_is_a_cv2_error():
    det = LaneDetector()
    with pytest.raises(cv2.error):
        det.detect_rig([bgr(1, 48, 64, c=4)], target_size=(64, 48))
    with pytest.raises(cv2.error):
        det.detect_rig([bgr(1, 48, 64, dtype=np.float32)], target_size=(64, 48))
    with pytest.raises(cv2.error):
        det.detect_rig([yuv(1, 48, 64).astype(np.int16)], ["nv12"], target_size=(64, 48))
    assert det._ctx is None


@pytest.mark.parametrize("cams,layouts,kw,match", [
    ([yuv(1, 48, 64)], ["bgr"], {}, "layout 'bgr'"),                                   # layout and shape disagree
    ([bgr(1, 48, 64)], ["nv12"], {}, "layout 'nv12'"),
    ([np.zeros((1, 47, 64), np.uint8)], ["i420"], {}, "layout 'i420'"),                # rows not H*3/2
    ([yuv(1, 48, 64)], ["yuyv"], {}, "layout 'yuyv'"),                                 # unknown layout
    ([yuv(1, 48, 64)], ["nv12", "nv12"], {}, "layouts"),                               # one layout per camera
    ([np.zeros((1, 48 * 3 // 2, 63), np.uint8)], ["i420"], {}, "even"),                # odd width
    ([bgr(1, 48, 64), bgr(1, 32, 64)], None, {}, "target_size"),                      # sizes differ, no target
    ([bgr(1, 48, 64), bgr(1, 48, 64)], None, {"stream_rois": [None]}, "stream_rois"),  # too few ROIs
    ([bgr(1, 48, 64), [[1]]], None, {}, "numpy arrays or all CUDA"),                  # not an array
])
def test_bad_rig_arguments_raise_before_any_native_call(cams, layouts, kw, match):
    det = LaneDetector()
    with pytest.raises(ValueError, match=match):
        det.detect_rig(cams, layouts, **kw)
    assert det._ctx is None


def test_mixed_host_and_device_cameras_are_refused():
    torch = pytest.importorskip("torch")
    cams = [bgr(1, 48, 64), torch.zeros((1, 48, 64, 3), dtype=torch.uint8)]       # a CPU tensor is not a rig camera
    det = LaneDetector()
    with pytest.raises(ValueError, match="numpy arrays or all CUDA"):
        det.detect_rig(cams)
    assert det._ctx is None


def test_a_tick_without_frames_returns_an_empty_list_per_camera():
    det = LaneDetector()
    assert det.detect_rig([None, bgr(0, 48, 64), yuv(0, 720, 1280)], ["bgr", "bgr", "nv12"]) == [[], [], []]
    assert det._ctx is None and det._stream_fit is None


def test_raw_rig_call_without_a_context_is_invalid():
    lib = _native.lib()
    frames = bgr(2, 48, 64)
    src = (_native.LaneRigSource * 1)(_native.LaneRigSource(frames.ctypes.data, _native.INPUT_BGR, 48, 64, 2, 0))
    fit, valid = np.zeros((1, 2, 3)), np.zeros((1, 2), np.uint8)
    out = np.zeros(2, _native.RECORD_DTYPE)
    rc = lib.lane_detect_rig(None, src, 1, 0, 1, _native._ptr(fit), _native._ptr(valid), _native._ptr(out))
    assert rc == -1 and b"lane_detect_rig" in lib.lane_last_error(None)
    assert lib.lane_detect_rig(None, None, 0, 0, 1, None, None, None) == -1


def test_rig_source_mirror_matches_the_header():
    assert ctypes.sizeof(_native.LaneRigSource) == 32
    assert [f for f, _ in _native.LaneRigSource._fields_] == ["frames", "format", "src_h", "src_w", "n", "stream_id"]
    assert _native.LaneRigSource.format.offset == 8 and _native.LaneRigSource.stream_id.offset == 24
