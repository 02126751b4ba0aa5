"""The pipelined rig (``LaneDetector.detect_rig_stream`` / ``lane_rig_enqueue``): argument checks that run before any
device work, and the binding's prototype, so they hold without a GPU."""
import ctypes
import os
import re

import cv2
import numpy as np
import pytest

from multimodal_autonomous_driving_perception_and_planning_b200 import LaneDetector, _native

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bgr(t, h, w, c=3, dtype=np.uint8):
    return np.zeros((t, h, w, c), dtype)


def yuv(t, h, w):
    return np.zeros((t, h * 3 // 2, w), np.uint8)


@pytest.mark.parametrize("cams,layouts,kw,match", [
    ([yuv(1, 48, 64)], ["yuyv"], {}, "layout 'yuyv'"),                                 # unknown layout
    ([yuv(1, 48, 64)], ["nv12", "nv12"], {}, "layouts"),                               # one layout per camera
    ([bgr(1, 48, 64)], ["nv12"], {}, "layout 'nv12'"),                                 # layout and shape disagree
    ([bgr(1, 48, 64), bgr(1, 32, 64)], None, {}, "target_size"),                      # sizes differ, no target
    ([bgr(1, 48, 64), bgr(1, 48, 64)], None, {"stream_rois": [None]}, "stream_rois"),  # too few ROIs
    ([bgr(1, 48, 64), [[1]]], None, {}, "numpy arrays or all CUDA"),                  # not an array
])
def test_bad_arguments_raise_what_detect_rig_raises_before_any_native_call(cams, layouts, kw, match):
    det = LaneDetector()
    with pytest.raises(ValueError, match=match) as streamed:
        next(det.detect_rig_stream([cams], layouts, **kw))
    with pytest.raises(ValueError) as blocking:
        det.detect_rig(cams, layouts, **kw)
    assert str(streamed.value).startswith(str(blocking.value))
    assert det._ctx is None


def test_bad_dtype_channels_or_target_size_is_a_cv2_error():
    det = LaneDetector()
    with pytest.raises(cv2.error):
        next(det.detect_rig_stream([[bgr(1, 48, 64, dtype=np.float32)]], target_size=(64, 48)))
    with pytest.raises(cv2.error):
        next(det.detect_rig_stream([[bgr(1, 48, 64, c=4)]], target_size=(64, 48)))
    with pytest.raises(cv2.error):
        next(det.detect_rig_stream([[bgr(1, 48, 64)]], target_size=(0, 48)))
    assert det._ctx is None


def test_ticks_without_frames_yield_empty_lists_without_a_context():
    det = LaneDetector()
    got = list(det.detect_rig_stream([[None, yuv(0, 48, 64)], [bgr(0, 48, 64), yuv(0, 720, 1280)]], ["bgr", "nv12"]))
    assert got == [[[], []], [[], []]]
    assert det._ctx is None and det._stream_fit is None


def test_raw_rig_enqueue_without_a_context_is_invalid():
    lib = _native.lib()
    frames = bgr(2, 48, 64)
    src = (_native.LaneRigSource * 1)(_native.LaneRigSource(frames.ctypes.data, _native.INPUT_BGR, 48, 64, 2, 0))
    assert lib.lane_rig_enqueue(None, src, 1, 0, 1, None, None) == -1
    assert b"lane_rig_enqueue" in lib.lane_last_error(None)


def test_rig_enqueue_prototype_matches_the_header():
    text = open(os.path.join(ROOT, "include", "lane_b200.h")).read()
    decl = re.search(r"LANE_API\s+int\s+lane_rig_enqueue\s*\(([^)]*)\)", text)
    assert decl, "lane_rig_enqueue is not declared"
    params = [" ".join(p.split()) for p in decl.group(1).split(",")]
    assert params == ["lane_ctx *ctx", "const lane_rig_source *sources", "int n_sources", "int frames_on_device",
                      "int n_streams", "const double *prev_fit", "const uint8_t *prev_valid"]
    res, args = _native._PROTOS["lane_rig_enqueue"]
    c = ctypes
    assert res is c.c_int
    assert args == [c.c_void_p, c.c_void_p, c.c_int, c.c_int, c.c_int, c.c_void_p, c.c_void_p]
    fn = _native.lib().lane_rig_enqueue
    assert fn.restype is c.c_int and fn.argtypes == args
