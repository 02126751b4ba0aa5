"""Decoder output at camera resolution straight into the lane path: the fused YUV 4:2:0 -> BGR -> cv2.resize kernel
(FrameIngest.from_nv12 / from_i420 with target_size) byte-equal to cv2 and the oracle, and
LaneDetector.detect_batch / detect_batch_nv12 / detect_batch_i420 with target_size equal to detect_batch on the
cv2-prepared frames: same records, same EMA chain, same prev_*_fit, over chunked, staged, pinned and device input.

Run on the B200 box: python -m pytest tests -m gpu.
"""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import cv2  # noqa: E402

from multimodal_autonomous_driving_perception_and_planning_b200 import FrameIngest, LaneDetector, _native  # noqa: E402
from oracle.cv2_pipeline import Cv2LaneOracle  # noqa: E402
from oracle import nv12 as onv  # noqa: E402
from test_oracle_ingest import SIZE_PAIRS, oracle_ingest, random_frame  # noqa: E402
from util import gen_frames  # noqa: E402
from yuv420 import nv12_to_i420  # noqa: E402

CODES = {"nv12": cv2.COLOR_YUV2BGR_NV12, "i420": cv2.COLOR_YUV2BGR_I420}
TARGET = (640, 480)


def cv2_ingest(frames, layout, dsize):
    return np.stack([cv2.resize(cv2.cvtColor(f, CODES[layout]), dsize) for f in frames])


# ---- the fused kernel through FrameIngest --------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["nv12", "i420"])
@pytest.mark.parametrize("src,dst", SIZE_PAIRS)
def test_fused_ingest_matches_cv2_and_oracle(layout, src, dst):
    import torch
    frames = np.stack([random_frame(src, layout, 7 * k + src[0] + dst[0]) for k in range(2)])
    want = cv2_ingest(frames, layout, dst)
    ing = FrameIngest(dst)
    conv = ing.from_nv12 if layout == "nv12" else ing.from_i420
    got_host = conv(frames)
    got_dev = conv(torch.from_numpy(frames).cuda())
    assert isinstance(got_host, np.ndarray) and got_host.shape == want.shape
    assert got_dev.is_cuda and tuple(got_dev.shape) == want.shape
    assert np.array_equal(got_host, want)
    assert np.array_equal(got_dev.cpu().numpy(), want)
    assert np.array_equal(got_host[0], oracle_ingest(frames[0], layout, dst))
    # a CUDA source at a misaligned offset: the byte loads and byte-store fallback of the same kernel
    flat = torch.zeros(frames.size + 1, dtype=torch.uint8, device="cuda")
    flat[1:] = torch.from_numpy(frames.reshape(-1)).cuda()
    got_odd = conv(flat[1:].view(frames.shape))
    assert np.array_equal(got_odd.cpu().numpy(), want)


@pytest.mark.parametrize("layout", ["nv12", "i420"])
def test_fused_ingest_on_random_even_sizes(layout):
    import torch
    from test_oracle_ingest import random_size_pairs
    for k, (src, dst) in enumerate(random_size_pairs()):
        frames = np.stack([random_frame(src, layout, 100 + k), random_frame(src, layout, 200 + k)])
        ing = FrameIngest(dst)
        conv = ing.from_nv12 if layout == "nv12" else ing.from_i420
        got = conv(torch.from_numpy(frames).cuda()).cpu().numpy()
        assert np.array_equal(got, cv2_ingest(frames, layout, dst)), (src, dst)


# ---- detection at target_size ----------------------------------------------------------------------------------------
def _rows(h):
    return np.linspace(h * 0.6, h, 50)


def _same_lanes(got, want, h):
    for g, w in zip(got, want):
        assert (g is None) == (w is None)
        if g is not None:
            assert np.abs(np.polyval(g.polynomial, _rows(h)) - np.polyval(w.coeffs, _rows(h))).max() < 1e-6
            assert np.abs(g.points.astype(np.int64) - w.points).max() <= 1
            assert g.confidence == w.confidence


def _state(det):
    return [None if p is None else np.asarray(p).tobytes() for p in (det.prev_left_fit, det.prev_right_fit)]


@pytest.fixture(scope="module")
def hd_sources():
    """12 generator frames at 1080p as BGR, NV12 and I420, and the cv2-prepared 640x480 BGR frames of each layout."""
    bgr = np.stack(gen_frames(1920, 1080, 12))
    nv12 = np.stack([onv.bgr_to_nv12_for_tests(f) for f in bgr])
    i420 = np.stack([nv12_to_i420(f) for f in nv12])
    prepared = {"bgr": np.stack([cv2.resize(f, TARGET) for f in bgr]),
                "nv12": cv2_ingest(nv12, "nv12", TARGET), "i420": cv2_ingest(i420, "i420", TARGET)}
    return {"bgr": bgr, "nv12": nv12, "i420": i420}, prepared


def _reference(prepared):
    ref = LaneDetector(max_batch=len(prepared))
    lanes = ref.detect_batch(prepared)
    return ref, lanes


def _detect(det, layout, frames, **kw):
    fn = {"bgr": det.detect_batch, "nv12": det.detect_batch_nv12, "i420": det.detect_batch_i420}[layout]
    return fn(frames, **kw)


def _pinned(a):
    import torch
    t = torch.empty(a.shape, dtype=torch.uint8).pin_memory()
    t.numpy()[...] = a
    return t, t.numpy()


@pytest.mark.parametrize("layout", ["bgr", "nv12", "i420"])
@pytest.mark.parametrize("where", ["chunks", "staged", "pinned", "cuda"])
def test_detect_at_target_size_equals_detect_batch_of_cv2_prepared_frames(hd_sources, layout, where):
    """max_batch < n (several native calls, several chunks each); pageable host input of >= 24 MB per native call (the
    staging ring); pinned host input; CUDA input."""
    import torch
    src, prepared = hd_sources
    frames = src[layout]
    ref, want_lanes = _reference(prepared[layout])
    keep = None
    if where == "chunks":
        det = LaneDetector(max_batch=5)
    elif where == "staged":
        det = LaneDetector(max_batch=12)
        assert frames[0].nbytes * 12 >= 24 << 20
    elif where == "pinned":
        det = LaneDetector(max_batch=12)
        keep, frames = _pinned(frames)
    else:
        det = LaneDetector(max_batch=12)
        frames = torch.from_numpy(frames).cuda()
    lanes = _detect(det, layout, frames, target_size=TARGET)
    assert det._ctx.height == 480 and det._ctx.width == 640
    assert det.last_records.tobytes() == ref.last_records.tobytes()
    assert _state(det) == _state(ref)
    assert len(lanes) == len(want_lanes)
    if where == "chunks":
        oracle = Cv2LaneOracle()
        for i, f in enumerate(prepared[layout]):
            _same_lanes(lanes[i], oracle.detect(f), 480)
    del keep
    det.close()
    ref.close()


def test_dense_rerun_from_the_same_source_frames():
    """Uniform-noise 1080p NV12 with a small segment cap: the chunk is re-run on the dense context from the same NV12
    frames (state restored first), and the records equal the cv2-prepared run."""
    rng = np.random.default_rng(9)
    calm = gen_frames(1920, 1080, 2)
    nv12 = np.stack([onv.bgr_to_nv12_for_tests(calm[0]), rng.integers(0, 256, (1620, 1920), dtype=np.uint8),
                     onv.bgr_to_nv12_for_tests(calm[1]), rng.integers(0, 256, (1620, 1920), dtype=np.uint8)])
    prepared = cv2_ingest(nv12, "nv12", TARGET)
    det = LaneDetector(max_batch=2, max_segments=4)
    det.detect_batch_nv12(nv12, target_size=TARGET)
    assert det.dense_reruns > 0
    ref = LaneDetector(max_batch=2, max_segments=4)
    ref.detect_batch(prepared)
    assert det.last_records.tobytes() == ref.last_records.tobytes()
    assert _state(det) == _state(ref)
    det.close()
    ref.close()


def test_one_detector_fed_several_source_sizes_chains_its_state():
    """1080p, then 720p, then 4K decoder frames with one target size: every call equals its cv2-prepared counterpart
    on a detector fed the prepared frames in the same order (the EMA state chains across calls and sizes)."""
    det = LaneDetector(max_batch=4)
    ref = LaneDetector(max_batch=4)
    for k, (w, h) in enumerate([(1920, 1080), (1280, 720), (3840, 2160)]):
        nv12 = np.stack([onv.bgr_to_nv12_for_tests(f) for f in gen_frames(w, h, 3, start=10 * k)])
        det.detect_batch_nv12(nv12, target_size=TARGET)
        ref.detect_batch(cv2_ingest(nv12, "nv12", TARGET))
        assert det.last_records.tobytes() == ref.last_records.tobytes(), (w, h)
        assert _state(det) == _state(ref)
    det.close()
    ref.close()


def test_target_equal_to_source_is_the_plain_call(hd_sources):
    src, _ = hd_sources
    for layout in ("bgr", "nv12", "i420"):
        a = LaneDetector(max_batch=6)
        _detect(a, layout, src[layout][:6], target_size=(1920, 1080))
        b = LaneDetector(max_batch=6)
        _detect(b, layout, src[layout][:6])
        assert a.last_records.tobytes() == b.last_records.tobytes(), layout
        a.close()
        b.close()
    # I420 and NV12 of the same samples detect alike
    c = LaneDetector(max_batch=6)
    c.detect_batch_nv12(src["nv12"][:6])
    d = LaneDetector(max_batch=6)
    d.detect_batch_i420(src["i420"][:6])
    assert c.last_records.tobytes() == d.last_records.tobytes()


def test_raw_ingest_calls_reject_bad_arguments():
    det = LaneDetector(max_batch=4)
    ctx = det._context(480, 640, 4)
    lib = _native.lib()
    src = np.zeros((8, 1620, 1920), np.uint8)
    pf, pv = np.zeros((1, 2, 3)), np.zeros((1, 2), np.uint8)
    out = np.zeros(8, _native.RECORD_DTYPE)
    p = src.ctypes.data_as(ctypes.c_void_p)

    def call(n, fmt, h, w):
        return lib.lane_detect_batch_ingest(ctx._h, p, 0, n, fmt, h, w, None, 1, pf.ctypes.data_as(ctypes.c_void_p),
                                            pv.ctypes.data_as(ctypes.c_void_p), out.ctypes.data_as(ctypes.c_void_p))
    assert call(2, 3, 1080, 1920) == -1                                # unknown format
    assert call(2, -1, 1080, 1920) == -1
    assert call(2, _native.INPUT_NV12, 1081, 1920) == -1               # odd YUV sizes
    assert call(2, _native.INPUT_I420, 1080, 1919) == -1
    assert call(2, _native.INPUT_NV12, 0, 1920) == -1                  # non-positive size
    assert call(5, _native.INPUT_NV12, 1080, 1920) == -1               # n > max_batch
    assert call(2, _native.INPUT_NV12, 1080, 1920) == 0                # and the context still works
    det.close()
