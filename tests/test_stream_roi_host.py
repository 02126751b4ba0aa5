"""Per-camera ROIs: argument checks that run before any device work, so they hold without a GPU."""
import numpy as np
import pytest

from multimodal_autonomous_driving_perception_and_planning_b200 import LaneDetector, _native


def test_set_roi_masks_rejects_bad_arguments_without_a_device():
    lib = _native.lib()
    assert lib.lane_set_roi_masks(None, None, 1) == -1
    mask = np.ones((4, 4), np.uint8)
    assert lib.lane_set_roi_masks(None, _native._ptr(mask), 1) == -1
    assert lib.lane_set_roi_masks(None, _native._ptr(mask), 0) == -1


def test_stream_rois_needs_an_entry_per_stream():
    frames = np.zeros((3, 48, 64, 3), np.uint8)
    poly = np.array([[(0, 47), (0, 20), (63, 20), (63, 47)]], np.int32)
    det = LaneDetector()
    with pytest.raises(ValueError, match="stream_rois"):
        det.detect_streams(frames, stream_ids=[0, 2, 1], stream_rois=[poly, None])
    with pytest.raises(ValueError, match="stream_rois"):
        det.detect_streams(frames[None], stream_rois=[])
    assert det._ctx is None
