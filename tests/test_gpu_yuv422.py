"""Packed YUV 4:2:2 camera frames straight into the lane path: the conversion kernels (FrameIngest.from_yuv422) byte-equal
to cv2 and the oracle, LaneDetector.detect_batch_yuv422 equal to detect_batch on the cv2-prepared frames (records, EMA
chain, prev_*_fit), and UYVY / YUYV cameras in detect_rig / detect_rig_stream beside NV12, I420, Bayer and BGR cameras
equal to one single-camera detector per camera.

Test frames are cv2's UYVY / YUYV encodings of the generator's scenes, so the lanes are real.

Run on the B200 box: python -m pytest tests -m gpu.
"""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import cv2  # noqa: E402
import torch  # noqa: E402

from bgr_yuv420 import bgr_to_i420, bgr_to_nv12  # noqa: E402
from multimodal_autonomous_driving_perception_and_planning_b200 import FrameIngest, LaneDetector, _native  # noqa: E402
from oracle import bayer as ob  # noqa: E402
from oracle import resize as orz  # noqa: E402
from oracle import yuv422 as oy  # noqa: E402
from oracle.cv2_pipeline import Cv2LaneOracle  # noqa: E402
from test_gpu_stream_roi import rig_polys  # noqa: E402
from test_yuv422_host import CODES, ENCODE, ORDERS  # noqa: E402
from util import gen_frames  # noqa: E402

TARGET = (640, 480)
# (source w, h) -> (destination w, h); 1924 is even but not a multiple of 8 (the generic same-size kernel)
PAIRS = [((1920, 1080), (640, 480)), ((1936, 1216), (640, 480)), ((3840, 2160), (640, 480)), ((1280, 720), (1920, 1080)),
         ((1280, 721), (640, 480)), ((1920, 1080), (1920, 1080)), ((1924, 1080), (1924, 1080)), ((2, 1), (5, 3))]


def encode(bgr, order):
    return np.stack([cv2.cvtColor(f, ENCODE[order]) for f in bgr])


def cv2_ingest(frames, order, dsize):
    return np.stack([cv2.resize(cv2.cvtColor(f, CODES[order]), dsize) for f in frames])


def pinned(a):
    t = torch.empty(a.shape, dtype=torch.uint8).pin_memory()
    t.numpy()[...] = a
    return t


def scene_frames(w, h, n, seed, order):
    """cv2's 4:2:2 of generator scenes where they are large enough to draw, random bytes below that."""
    if w >= 64 and h >= 48:
        return encode(np.stack(gen_frames(w, h, n, start=seed)), order)
    return np.random.default_rng(seed).integers(0, 256, (n, h, w, 2), dtype=np.uint8)


# ---- the conversion kernels through FrameIngest ------------------------------------------------------------------------
@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("src,dst", PAIRS)
def test_from_yuv422_matches_cv2_and_oracle(order, src, dst):
    frames = scene_frames(*src, 2, src[0] + dst[1], order)
    want = cv2_ingest(frames, order, dst)
    ing = FrameIngest(dst)
    got_host = ing.from_yuv422(frames, order)
    assert isinstance(got_host, np.ndarray) and np.array_equal(got_host, want)
    assert np.array_equal(got_host[1], orz.resize_linear(oy.yuv422_to_bgr(frames[1], order), dst))
    got_dev = ing.from_yuv422(torch.from_numpy(frames).cuda(), order)
    assert got_dev.is_cuda and np.array_equal(got_dev.cpu().numpy(), want)
    # a CUDA source misaligned by one byte
    flat = torch.zeros(frames.size + 1, dtype=torch.uint8, device="cuda")
    flat[1:] = torch.from_numpy(frames.reshape(-1)).cuda()
    assert np.array_equal(ing.from_yuv422(flat[1:].view(frames.shape), order).cpu().numpy(), want)
    # pinned host frames
    assert np.array_equal(ing.from_yuv422(pinned(frames).numpy(), order), want)
    if src == dst:
        assert np.array_equal(FrameIngest(None).from_yuv422(frames, order), want)      # no target: the conversion


@pytest.mark.parametrize("order", ORDERS)
def test_from_yuv422_of_a_pageable_batch_above_24_mb(order):
    """A host batch this large goes through the device's staging ring both ways."""
    frames = encode(np.stack(gen_frames(1920, 1080, 4, start=40)), order)
    frames = np.concatenate([frames] * 2)
    assert frames.nbytes >= 24 << 20
    for dst in ((640, 480), (1920, 1080)):
        got = FrameIngest(dst).from_yuv422(frames, order)
        assert got.nbytes >= 24 << 20 or dst == (640, 480)
        assert np.array_equal(got, cv2_ingest(frames, order, dst)), dst


# ---- detection at target_size ----------------------------------------------------------------------------------------
def _state(det):
    return [None if p is None else np.asarray(p).tobytes() for p in (det.prev_left_fit, det.prev_right_fit)]


N_HD = 14                                                 # 14 x 1080p 4:2:2 = 58 MB: one native call goes through staging


@pytest.fixture(scope="module")
def hd():
    """14 generator scenes at 1080p, and per order their 4:2:2 frames and the cv2-prepared 640x480 BGR frames."""
    bgr = np.stack(gen_frames(1920, 1080, N_HD, start=300))
    src = {o: encode(bgr, o) for o in ORDERS}
    return src, {o: cv2_ingest(src[o], o, TARGET) for o in ORDERS}


def test_reference_finds_lanes_on_the_4_2_2_frames(hd):
    """The comparisons below are not of empty records: cv2's pipeline finds both lanes on most frames."""
    _, prepared = hd
    for o in ORDERS:
        oracle = Cv2LaneOracle()
        both = sum(all(s is not None for s in oracle.detect(f)) for f in prepared[o])
        assert both >= 0.7 * N_HD, (o, both)


@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("where", ["chunks", "staged", "pinned", "cuda"])
def test_detect_batch_yuv422_equals_detect_batch_of_cv2_prepared_frames(hd, order, where):
    src, prepared = hd
    frames, keep = src[order], None
    ref = LaneDetector(max_batch=N_HD)
    ref.detect_batch(prepared[order])
    if where == "chunks":
        det = LaneDetector(max_batch=5)
    elif where == "staged":
        det = LaneDetector(max_batch=N_HD)
        assert frames.nbytes >= 24 << 20
    elif where == "pinned":
        det = LaneDetector(max_batch=N_HD)
        keep = pinned(frames)
        frames = keep.numpy()
    else:
        det = LaneDetector(max_batch=N_HD)
        frames = torch.from_numpy(frames).cuda()
    lanes = det.detect_batch_yuv422(frames, order, target_size=TARGET)
    assert (det._ctx.height, det._ctx.width) == (480, 640) and len(lanes) == N_HD
    assert det.last_records.tobytes() == ref.last_records.tobytes()
    assert _state(det) == _state(ref)
    del keep
    det.close()
    ref.close()


def test_yuv422_at_the_detection_size_is_the_conversion(hd):
    src, _ = hd
    for o in ORDERS:
        a = LaneDetector(max_batch=4)
        a.detect_batch_yuv422(src[o][:4], o)
        assert (a._ctx.height, a._ctx.width) == (1080, 1920)
        for i in range(4):
            assert np.array_equal(a._ctx.tap(_native.TAP_FRAME, i), cv2.cvtColor(src[o][i], CODES[o])), (o, i)
        b = LaneDetector(max_batch=4)
        b.detect_batch(np.stack([cv2.cvtColor(f, CODES[o]) for f in src[o][:4]]))
        assert a.last_records.tobytes() == b.last_records.tobytes() and _state(a) == _state(b)
        a.close()
        b.close()


# ---- a rig with 4:2:2 cameras --------------------------------------------------------------------------------------
# (layout, width, height, frames this tick): 1080p UYVY and 720p YUYV cameras, a 640x480 UYVY camera (at the 640x480
# target: identity taps in k0_rig_ingest), an odd-height YUYV camera, beside NV12, I420, Bayer and BGR cameras
RIG = [("uyvy", 1920, 1080, 2), ("nv12", 1936, 1216, 1), ("yuyv", 1280, 720, 2), ("i420", 1280, 720, 1),
       ("bayer_rggb", 1920, 1080, 1), ("uyvy", 640, 480, 2), ("yuyv", 1280, 721, 1), ("bgr", 1920, 1080, 1)]
LAYOUTS = [lay for lay, *_ in RIG]
NOISE_CAM = 0                                        # a UYVY camera; its ROI is the full frame


def encode_layout(bgr, layout):
    if layout == "bgr":
        return bgr
    if layout in CODES:
        return encode(bgr, layout)
    if layout.startswith("bayer_"):
        return np.stack([ob.mosaic_of_bgr(f, layout[6:]) for f in bgr])
    return np.stack([(bgr_to_nv12 if layout == "nv12" else bgr_to_i420)(f) for f in bgr])


def single_camera(frames, layout, poly, target, **kw):
    det = LaneDetector(poly, max_batch=max(len(frames), 1), **kw)
    if layout in CODES:
        det.detect_batch_yuv422(frames, layout, target_size=target)
    elif layout.startswith("bayer_"):
        det.detect_batch_bayer(frames, layout[6:], target_size=target)
    else:
        {"bgr": det.detect_batch, "nv12": det.detect_batch_nv12, "i420": det.detect_batch_i420}[layout](
            frames, target_size=target)
    return det.last_records.copy(), det


@pytest.fixture(scope="module")
def rig():
    return [encode_layout(np.stack(gen_frames(w, h, 3, start=500 * s)), lay) for s, (lay, w, h, _) in enumerate(RIG)]


def tick(rig, k=0, counts=None):
    counts = [c for *_, c in RIG] if counts is None else counts
    return [cam[k:k + t] if t else None for cam, t in zip(rig, counts)]


def polys_for(target):
    p = rig_polys(target[1], target[0])
    return [p[6], p[1], p[2], None, p[3], p[4], p[0], p[5]]


@pytest.mark.parametrize("target", [(640, 480), (1280, 720)])
@pytest.mark.parametrize("where", ["chunks", "staged", "pinned", "cuda"])
def test_rig_with_yuv422_cameras_equals_single_camera_detectors(rig, where, target):
    cams, keep = tick(rig), []
    n = sum(len(c) for c in cams)
    polys = polys_for(target)
    if where == "staged":
        assert sum(c.nbytes for c in cams) >= 24 << 20
    elif where == "pinned":
        keep = [pinned(c) for c in cams]
        cams = [t.numpy() for t in keep]
    elif where == "cuda":
        cams = [torch.from_numpy(c).cuda() for c in cams]
    det = LaneDetector(max_batch=4 if where == "chunks" else n)
    lanes = det.detect_rig(cams, LAYOUTS, target_size=target, stream_rois=polys)
    assert [len(x) for x in lanes] == [c for *_, c in RIG]
    a = 0
    for s, cam in enumerate(tick(rig)):
        want, d = single_camera(cam, LAYOUTS[s], polys[s], target)
        assert det.last_records[a:a + len(cam)].tobytes() == want.tobytes(), (target, s)
        a += len(cam)
        d.close()
    del keep
    det.close()


@pytest.mark.parametrize("target", [(640, 480), (1280, 720)])
def test_rig_frame_tap_is_cv2s_conversion_and_resize(rig, target):
    cams = tick(rig)
    det = LaneDetector(max_batch=sum(len(c) for c in cams))
    det.detect_rig(cams, LAYOUTS, target_size=target)
    k = 0
    for s, cam in enumerate(cams):
        for f in cam:
            if LAYOUTS[s] in CODES:
                want = cv2.resize(cv2.cvtColor(f, CODES[LAYOUTS[s]]), target)
                assert np.array_equal(det._ctx.tap(_native.TAP_FRAME, k), want), s
            k += 1
    det.close()


def test_noise_uyvy_camera_is_rerun_on_the_dense_context(rig):
    target = (640, 480)
    polys = polys_for(target)
    cams = tick(rig)
    cams[NOISE_CAM] = np.random.default_rng(5).integers(0, 256, (2, 1080, 1920, 2), dtype=np.uint8)
    det = LaneDetector(max_batch=11, max_segments=8)
    det.detect_rig(cams, LAYOUTS, target_size=target, stream_rois=polys)
    assert det.dense_reruns >= 1 and not det.last_records["flags"].any()
    a = 0
    for s, cam in enumerate(cams):
        want, d = single_camera(cam, LAYOUTS[s], polys[s], target, max_segments=8)
        assert det.last_records[a:a + len(cam)].tobytes() == want.tobytes(), s
        if s == NOISE_CAM:
            assert d.dense_reruns >= 1 and max(want["n_segments"]) > 8
            # and the cv2 pipeline on cv2's frames agrees
            ref = LaneDetector(polys[s], max_batch=2, max_segments=8)
            ref.detect_batch(cv2_ingest(cam, "uyvy", target))
            assert ref.last_records.tobytes() == want.tobytes()
            ref.close()
        a += len(cam)
        d.close()
    det.close()


COUNTS = [[1, 1, 1, 1, 1, 1, 1, 1], [2, 0, 1, None, 1, 1, 0, 1], [1, 1, 2, 1, 0, None, 1, 2], [0, 1, 1, 2, 1, 2, 1, 0]]


@pytest.mark.parametrize("kind", ["cuda", "pinned", "numpy"])
def test_stream_with_yuv422_cameras_equals_detect_rig_tick_after_tick(rig, kind):
    target = (640, 480)
    polys = polys_for(target)
    ticks = [[None if t is None else np.ascontiguousarray(np.roll(rig[s], -k, axis=0)[:t]) for s, t in enumerate(row)]
             for k, row in enumerate(COUNTS)]
    ref = LaneDetector(max_batch=9)
    want = []
    for t in ticks:
        ref.detect_rig(t, LAYOUTS, target_size=target, stream_rois=polys)
        want.append((ref.last_records.copy(), ref._stream_fit.copy(), ref._stream_valid.copy()))
    conv = {"numpy": lambda a: a, "pinned": pinned, "cuda": lambda a: torch.from_numpy(a).cuda()}[kind]
    src = [[None if c is None else conv(c) for c in t] for t in ticks]
    det = LaneDetector(max_batch=9)
    got = []
    for _ in det.detect_rig_stream(src, LAYOUTS, target_size=target, stream_rois=polys):
        got.append((det.last_records.copy(), det._stream_fit.copy(), det._stream_valid.copy()))
    assert len(got) == len(want)
    for k, (g, w) in enumerate(zip(got, want)):
        assert all(a.tobytes() == b.tobytes() for a, b in zip(g, w)), k
    assert not det._ctx._inflight
    det.close()
    ref.close()


def test_raw_yuv422_error_codes(rig):
    det = LaneDetector(max_batch=4)
    ctx = det._context(480, 640, 4)
    lib, P = _native.lib(), _native._ptr
    cam = np.ascontiguousarray(rig[0][:2])                        # 2 x 1080p UYVY
    fit, valid = np.zeros((1, 2, 3)), np.zeros((1, 2), np.uint8)
    out = np.zeros(4, _native.RECORD_DTYPE)
    U, Y = _native.INPUT_UYVY, _native.INPUT_YUYV

    def ingest(fmt, h, w, n=2):
        return lib.lane_detect_batch_ingest(ctx._h, P(cam), 0, n, fmt, h, w, None, 1, P(fit), P(valid), P(out))

    def rig_call(fmt, h, w, n=2):
        arr = (_native.LaneRigSource * 1)(_native.LaneRigSource(cam.ctypes.data, fmt, h, w, n, 0))
        return lib.lane_detect_rig(ctx._h, arr, 1, 0, 1, P(fit), P(valid), P(out))

    for call in (ingest, rig_call):
        assert call(10, 1080, 1920) == -1                                    # unknown format
        assert call(7, 1080, 1920) == -1
        assert call(U, 1080, 1919) == -1 and b"even width" in lib.lane_last_error(ctx._h)
        assert call(Y, 1080, 1921) == -1
        assert call(U, 1080, 1920, n=5) == -1                                # n > max_batch
        assert call(U, 1081, 1918) == 0                                      # an odd height is fine for 4:2:2
        assert call(U, 1080, 1920) == 0
        assert call(Y, 1080, 1920) == 0
    dev = torch.from_numpy(cam).cuda()
    arr = (_native.LaneRigSource * 1)(_native.LaneRigSource(cam.ctypes.data, U, 1080, 1920, 2, 0))
    assert lib.lane_rig_enqueue(ctx._h, arr, 1, 0, 1, P(fit), P(valid)) == -1           # pageable host frames
    arr = (_native.LaneRigSource * 1)(_native.LaneRigSource(dev.data_ptr(), U, 1080, 1919, 2, 0))
    assert lib.lane_rig_enqueue(ctx._h, arr, 1, 1, 1, P(fit), P(valid)) == -1
    arr = (_native.LaneRigSource * 1)(_native.LaneRigSource(dev.data_ptr(), Y, 1080, 1920, 2, 0))
    torch.cuda.synchronize()
    assert lib.lane_rig_enqueue(ctx._h, arr, 1, 1, 1, P(fit), P(valid)) == 0
    assert lib.lane_detect_collect(ctx._h, P(fit), P(valid), P(out)) == 0
    # the context-free entry on the device
    src = torch.from_numpy(cam).cuda()
    dst = torch.empty((2, 480, 640, 3), dtype=torch.uint8, device="cuda")
    s, q = ctypes.c_void_p(src.data_ptr()), ctypes.c_void_p(dst.data_ptr())
    assert lib.lane_yuv422_to_bgr_batch(s, _native.INPUT_NV12, 2, 1080, 1920, q, 480, 640, 1, 0, None) == -1
    assert lib.lane_yuv422_to_bgr_batch(s, U, 2, 1080, 1919, q, 480, 640, 1, 0, None) == -1
    assert lib.lane_yuv422_to_bgr_batch(s, U, 2, 1080, 1920, q, 480, 640, 1, 99, None) == -1
    assert b"lane_yuv422_to_bgr_batch" in lib.lane_last_error(None)
    assert lib.lane_yuv422_to_bgr_batch(s, U, 2, 1080, 1920, q, 480, 640, 1, 0, None) == 0
    torch.cuda.synchronize()
    assert np.array_equal(dst.cpu().numpy(), cv2_ingest(cam, "uyvy", TARGET))
    # the 4:2:0 and Bayer entries refuse the 4:2:2 layouts on the device too
    assert lib.lane_yuv420_to_bgr_batch(s, U, 2, 1080, 1920, q, 480, 640, 1, 0, None) == -1
    assert lib.lane_bayer_to_bgr_batch(s, Y, 2, 1080, 1920, q, 480, 640, 1, 0, None) == -1
    det.close()


@pytest.mark.parametrize("order", ORDERS)
def test_context_free_entry_host_batch_above_24_mb_equals_the_cuda_result(order):
    """The checks tests/test_host_boundary.py makes of the older context-free entries."""
    lib = _native.lib()
    frames = encode(np.stack(gen_frames(1920, 1080, 4, start=70)), order)
    frames = np.concatenate([frames] * 2)
    assert frames.nbytes >= 24 << 20
    fmt = _native.YUV422[order]
    n = frames.shape[0]
    for dh, dw in ((1080, 1920), (480, 640)):
        host = np.empty((n, dh, dw, 3), np.uint8)
        assert lib.lane_yuv422_to_bgr_batch(_native._ptr(frames), fmt, n, 1080, 1920, _native._ptr(host), dh, dw, 0, 0,
                                            None) == 0
        src = torch.from_numpy(frames).cuda()
        dst = torch.empty((n, dh, dw, 3), dtype=torch.uint8, device="cuda")
        assert lib.lane_yuv422_to_bgr_batch(ctypes.c_void_p(src.data_ptr()), fmt, n, 1080, 1920,
                                            ctypes.c_void_p(dst.data_ptr()), dh, dw, 1, 0, None) == 0
        torch.cuda.synchronize()
        assert np.array_equal(host, dst.cpu().numpy()), (dh, dw)
    bad = torch.cuda.device_count()
    out = np.empty((n, 480, 640, 3), np.uint8)
    assert lib.lane_yuv422_to_bgr_batch(_native._ptr(frames), fmt, n, 1080, 1920, _native._ptr(out), 480, 640, 0, bad,
                                        None) == -1
    assert lib.lane_last_error(None).startswith(b"lane_yuv422_to_bgr_batch: ")
