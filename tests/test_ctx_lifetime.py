"""Lifetimes of the native context's resources: a ROI set again on a live context gives what a new context with that ROI
gives, a create that runs out of device memory leaves none behind, and contexts created and destroyed in turn do not
accumulate device memory.  Through the raw C ABI where the Python layer has no call (setting the ROI again)."""
import ctypes as C

import numpy as np
import pytest

from multimodal_autonomous_driving_perception_and_planning_b200 import _native
from oracle import stages as S
from util import gen_frames

pytestmark = pytest.mark.gpu

LANE_ERR_CUDA = -2


def _set_roi(ctx, mask):
    mask = np.ascontiguousarray(mask, np.uint8)
    ctx._check(_native.lib().lane_set_roi_mask(ctx._h, _native._ptr(mask)))


def _detect(ctx, frames):
    """One batch from the same explicit EMA state every time: records, state after it, and the ROI point lists."""
    prev_fit, prev_valid = np.zeros((1, 2, 3)), np.zeros((1, 2), np.uint8)
    recs = ctx.detect(np.ascontiguousarray(frames), len(frames), False, None, 1, prev_fit, prev_valid, 0.7, 0.3)
    points = [ctx.tap(_native.TAP_POINTS, i) if recs[i]["n_roi_points"] else None for i in range(len(frames))]
    return recs, prev_fit, prev_valid, points


def _assert_same(got, want, what):
    (r0, f0, v0, p0), (r1, f1, v1, p1) = got, want
    assert r0.tobytes() == r1.tobytes(), what          # RECORD_DTYPE has no padding
    assert f0.tobytes() == f1.tobytes() and np.array_equal(v0, v1), what
    for i, (a, b) in enumerate(zip(p0, p1)):
        assert (a is None) == (b is None) and (a is None or np.array_equal(a, b)), (what, i)


@pytest.mark.parametrize("shape", [(480, 640), (481, 643)])     # 643 columns: the byte-map kernels, built lazily
def test_roi_set_again_on_a_live_context_equals_a_new_context(shape):
    h, w = shape
    frames = np.stack(gen_frames(w, h, 4))
    roi_a = S.roi_mask(h, w)
    roi_b = S.roi_mask(h, w, np.array([[(0, h - 1), (0, h // 3), (w - 1, h // 3), (w - 1, h - 1)]], np.int32))
    assert roi_b.sum() > roi_a.sum()
    want = {}
    for name, roi in (("A", roi_a), ("B", roi_b)):
        fresh = _native.LaneContext(h, w, len(frames), roi, debug=True)
        want[name] = _detect(fresh, frames)
        fresh.close()

    live = _native.LaneContext(h, w, len(frames), roi_a, debug=True)
    for name, roi in (("A", roi_a), ("B", roi_b), ("A", roi_a)):
        _set_roi(live, roi)
        _assert_same(_detect(live, frames), want[name], (shape, name))
        if w % 16:
            assert not live.last_paths() & _native.PATH_CLUSTER_CANNY
    live.close()


def test_failed_create_leaves_nothing_behind():
    import torch
    lib = _native.lib()
    h = C.c_void_p()
    assert lib.lane_ctx_create(0, 1080, 1920, 4, 0, C.byref(h)) == 0       # CUDA context and module load paid here
    lib.lane_ctx_destroy(h)
    free0 = torch.cuda.mem_get_info(0)[0]

    # 2^20 frames of 1080p edge planes: some 270 GB, more than the card holds
    h = C.c_void_p()
    assert lib.lane_ctx_create(0, 1080, 1920, 1 << 20, 0, C.byref(h)) == LANE_ERR_CUDA
    assert h.value is None
    assert lib.lane_last_error(None)
    assert abs(torch.cuda.mem_get_info(0)[0] - free0) <= 4 << 20

    assert lib.lane_ctx_create(0, 1080, 1920, 4, 0, C.byref(h)) == 0, lib.lane_last_error(None)
    lib.lane_ctx_destroy(h)


def test_no_device_memory_growth_across_context_lifetimes():
    import torch
    h, w, batch, n = 480, 640, 32, 4
    src_h, src_w = 720, 1280
    nv12 = np.random.default_rng(3).integers(0, 256, (n, src_h * 3 // 2, src_w), dtype=np.uint8)
    roi = S.roi_mask(h, w)
    footprint, free_after = [], []
    for cycle in range(10):
        before = torch.cuda.mem_get_info(0)[0]
        ctx = _native.LaneContext(h, w, batch, roi, debug=True)
        _set_roi(ctx, roi)
        # host NV12 at another size: source staging and the copy stream
        ctx.detect(nv12, n, False, None, 1, np.zeros((1, 2, 3)), np.zeros((1, 2), np.uint8), 0.7, 0.3,
                   fmt=_native.INPUT_NV12, src_hw=(src_h, src_w))
        for max_peaks in (16, 64 * (cycle + 1)):
            ctx.hough_lines_batch(n, threshold=50, max_peaks=max_peaks, with_accum=max_peaks > 16)
        ctx.hough_accumulator(0, threshold=5, max_peaks=64)
        for tap in (_native.TAP_BLUR, _native.TAP_HIST, _native.TAP_CLASS, _native.TAP_EDGES, _native.TAP_POINTS,
                    _native.TAP_SEGMENTS, _native.TAP_GRAY):
            ctx.tap(tap, n - 1)
        footprint.append(before - torch.cuda.mem_get_info(0)[0])
        ctx.close()
        free_after.append(torch.cuda.mem_get_info(0)[0])
    assert footprint[0] > 0
    assert abs(free_after[-1] - free_after[0]) <= footprint[0] // 2, (free_after, footprint)
