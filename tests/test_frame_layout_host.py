"""The frame layout table (loaders/frame_layout.py) against the native one and against every host check that reads it:
the context-free entries, detect_rig's plan and FrameIngest refuse exactly the shapes and sizes the table refuses, with
the exception types callers rely on.  No device needed: an entry that accepts its arguments reports that none is there."""
import cv2
import numpy as np
import pytest

from multimodal_autonomous_driving_perception_and_planning_b200 import FrameIngest, LaneDetector, _native
from multimodal_autonomous_driving_perception_and_planning_b200.loaders.frame_layout import LAYOUTS

SIZES = [(4, 6), (6, 4), (3, 3), (5, 6), (4, 7), (5, 7), (2, 6), (6, 2), (2, 2), (1, 1)]


def _arrays(layout):
    """Arrays [2, ...] of this layout's frames at every size it can express, and of wrong ranks and last dimensions."""
    shapes = {(2,) + layout.frame_shape(h, w) for h, w in SIZES}
    good = (2,) + layout.frame_shape(4, 6)
    shapes |= {good + (1,), good[:3] if len(good) == 4 else good[:2]}                          # wrong rank
    shapes |= {good[:3] + (1,), good[:3] + (4,)} if layout.channels else {(2, 7, 6), (2, 8, 6)}  # wrong last dim
    return [np.zeros(s, np.uint8) for s in sorted(shapes)]


def _accepted(layout, frames) -> bool:
    hw = layout.hw(frames.shape)
    return hw is not None and not layout.refuses(*hw)


@pytest.mark.parametrize("name", sorted(n for n in LAYOUTS if LAYOUTS[n].entry))        # BGR has no such entry
def test_native_entries_refuse_the_sizes_the_table_refuses(name):
    layout = LAYOUTS[name]
    entry = getattr(_native.lib(), layout.entry)
    dst = np.zeros((1, 4, 4, 3), np.uint8)
    for h, w in SIZES:
        src = np.zeros(max(layout.frame_bytes(h, w), 1), np.uint8)
        rc = entry(_native._ptr(src), layout.fmt, 1, h, w, _native._ptr(dst), 4, 4, 0, 0, None)
        assert rc in (-1, 0, -3), (name, h, w, rc)
        assert (rc == -1) == layout.refuses(h, w), (name, h, w, _native.lib().lane_last_error(None))
        if rc == -1:
            assert _native.lib().lane_last_error(None).startswith(layout.entry.encode() + b": ")


@pytest.mark.parametrize("name", sorted(LAYOUTS))
def test_plan_refuses_the_shapes_the_table_refuses(name):
    layout = LAYOUTS[name]
    for frames in _arrays(layout):
        det = LaneDetector()
        if _accepted(layout, frames):
            assert layout.frame_bytes(*layout.hw(frames.shape)) == frames[0].nbytes
            p = det._rig_plan([frames], [name], (8, 6), None)
            assert p.fmts == [layout.fmt] and p.sizes == [layout.hw(frames.shape)]
            continue
        # a BGR camera with four dimensions but not three channels fails like cv2.cvtColor; every other shape or
        # size is the rig's own argument error
        exc = cv2.error if name == "bgr" and frames.ndim == 4 else ValueError
        with pytest.raises(exc) as e:
            det._rig_plan([frames], [name], (8, 6), None)
        assert type(e.value) is exc, (name, frames.shape)
    with pytest.raises(cv2.error, match="uint8"):
        LaneDetector()._rig_plan([np.zeros((2,) + layout.frame_shape(4, 6), np.float32)], [name], (8, 6), None)


@pytest.mark.parametrize("name", sorted(n for n in LAYOUTS if n != "bgr"))
def test_frame_ingest_refuses_the_shapes_the_table_refuses(name):
    layout = LAYOUTS[name]
    ing = FrameIngest((8, 6), device=0)
    convert = {"nv12": ing.from_nv12, "i420": ing.from_i420}.get(name)
    if convert is None:
        names = _native.BAYER if name.startswith("bayer_") else _native.YUV422
        key = name.removeprefix("bayer_")
        assert names[key] == layout.fmt
        convert = lambda f: (ing.from_bayer if names is _native.BAYER else ing.from_yuv422)(f, key)    # noqa: E731
    for frames in _arrays(layout):
        if not _accepted(layout, frames):
            with pytest.raises(cv2.error):
                convert(frames)
            continue
        try:                                         # converted when a device is there, else refused by the library
            assert convert(frames).shape == (2, 6, 8, 3)
        except _native.LaneError as e:
            assert e.code == -3, (name, frames.shape, e)
