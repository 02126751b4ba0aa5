"""Raw Bayer camera frames into the lane path, without a GPU: the CPU statement of the demosaic (oracle/bayer.py) equals
cv2.cvtColor(f, COLOR_Bayer<P>2BGR) for all four patterns, its resize equals cv2.resize of cv2's frame, and every
argument error of detect_batch_bayer / detect_rig / FrameIngest.from_bayer / the raw entry points is raised before any
device work."""
import ctypes

import cv2
import numpy as np
import pytest

from multimodal_autonomous_driving_perception_and_planning_b200 import FrameIngest, LaneDetector, _native
from oracle import bayer as ob
from oracle import resize as orz
from test_oracle_ingest import SIZE_PAIRS

CODES = {"rggb": cv2.COLOR_BayerRGGB2BGR, "bggr": cv2.COLOR_BayerBGGR2BGR, "grbg": cv2.COLOR_BayerGRBG2BGR,
         "gbrg": cv2.COLOR_BayerGBRG2BGR}
SIZES = [(3, 3), (4, 4), (5, 7), (8, 10), (17, 33), (64, 96), (1080, 1920), (1216, 1936), (2160, 3840)]   # (h, w)


def random_sizes(k=40, seed=23):
    """(h, w) from 3x3 to 4K, small sizes over-represented."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(k):
        top = int(rng.choice([16, 300, 2160]))
        out.append((int(rng.integers(3, top + 1)), int(rng.integers(3, top * 16 // 9 + 1))))
    return out


def raw(h, w, seed):
    return np.random.default_rng(seed).integers(0, 256, (h, w), dtype=np.uint8)


def test_cv2_codes_are_the_aliases_the_layouts_name():
    assert CODES == {"rggb": cv2.COLOR_BayerBG2BGR, "bggr": cv2.COLOR_BayerRG2BGR, "grbg": cv2.COLOR_BayerGB2BGR,
                     "gbrg": cv2.COLOR_BayerGR2BGR}
    assert _native.BAYER == {"rggb": 16, "bggr": 17, "grbg": 18, "gbrg": 19}


@pytest.mark.parametrize("pattern", sorted(CODES))
@pytest.mark.parametrize("h,w", SIZES)
def test_oracle_equals_cv2(pattern, h, w):
    f = raw(h, w, h * 7 + w)
    assert np.array_equal(ob.bayer_to_bgr(f, pattern), cv2.cvtColor(f, CODES[pattern]))


@pytest.mark.parametrize("pattern", sorted(CODES))
def test_oracle_equals_cv2_on_random_sizes(pattern):
    for k, (h, w) in enumerate(random_sizes()):
        f = raw(h, w, k)
        assert np.array_equal(ob.bayer_to_bgr(f, pattern), cv2.cvtColor(f, CODES[pattern])), (h, w)


@pytest.mark.parametrize("pattern", sorted(CODES))
@pytest.mark.parametrize("src,dst", SIZE_PAIRS)
def test_oracle_resize_equals_cv2_resize(pattern, src, dst):
    w, h = src
    if h < 3 or w < 3:                                   # the 2x2 YUV pair: a Bayer frame needs 3 x 3
        w, h = 3, 3
    f = raw(h, w, w + dst[0])
    assert np.array_equal(orz.resize_linear(ob.bayer_to_bgr(f, pattern), dst),
                          cv2.resize(cv2.cvtColor(f, CODES[pattern]), dst))


def test_mosaic_keeps_each_sites_channel():
    bgr = np.random.default_rng(1).integers(0, 256, (6, 8, 3), dtype=np.uint8)
    for pattern, (py, px) in ob.PHASE.items():
        m = ob.mosaic_of_bgr(bgr, pattern)
        for y in range(6):
            for x in range(8):
                ry, rx = (y + py) & 1, (x + px) & 1
                want = bgr[y, x, 2] if (ry, rx) == (0, 0) else bgr[y, x, 0] if (ry, rx) == (1, 1) else bgr[y, x, 1]
                assert m[y, x] == want
    with pytest.raises(ValueError):
        ob.bayer_to_bgr(np.zeros((2, 5), np.uint8), "rggb")


RAW = np.zeros((2, 48, 64), np.uint8)
BAD_FRAMES = [RAW.astype(np.float32), RAW.astype(np.uint16), RAW[0], RAW[..., None], np.zeros((2, 2, 64), np.uint8),
              np.zeros((2, 48, 2), np.uint8)]


def test_detect_batch_bayer_errors_raise_before_the_device():
    det = LaneDetector()
    for bad in BAD_FRAMES:
        with pytest.raises(cv2.error):
            det.detect_batch_bayer(bad, "rggb", target_size=(32, 24))
    for pattern in ("RGGB", "rgbg", "", None, 16):
        with pytest.raises(ValueError):
            det.detect_batch_bayer(RAW, pattern)
    with pytest.raises(TypeError):
        det.detect_batch_bayer(RAW)                       # the pattern has no default
    for bad in [(640,), (0, 480), (640.0, 480), "640x480"]:
        with pytest.raises(cv2.error):
            det.detect_batch_bayer(RAW, "bggr", target_size=bad)
    assert det.detect_batch_bayer(RAW[:0], "grbg", target_size=(32, 24)) == []
    assert det._ctx is None


@pytest.mark.parametrize("cams,layouts,exc,match", [
    ([np.zeros((1, 48, 64, 3), np.uint8)], ["bayer_rggb"], ValueError, "needs frames \\[T,H,W\\]"),
    ([np.zeros((1, 2, 64), np.uint8)], ["bayer_bggr"], ValueError, "at least 3 rows"),
    ([np.zeros((1, 48, 2), np.uint8)], ["bayer_gbrg"], ValueError, "at least 3 rows"),
    ([np.zeros((1, 48, 64), np.uint8)], ["bayer_rgbg"], ValueError, "layout 'bayer_rgbg'"),
    ([np.zeros((1, 48, 64), np.uint8)], ["rggb"], ValueError, "layout 'rggb'"),
    ([np.zeros((1, 48, 64), np.uint8)], ["yuyv"], ValueError, "layout 'yuyv'"),
    ([np.zeros((1, 48, 64), np.float32)], ["bayer_grbg"], cv2.error, "uint8"),
])
def test_bad_bayer_rig_arguments_raise_before_any_native_call(cams, layouts, exc, match):
    det = LaneDetector()
    with pytest.raises(exc, match=match):
        det.detect_rig(cams, layouts, target_size=(64, 48))
    assert det._ctx is None


def test_bayer_rig_layouts_are_planned_at_one_byte_per_pixel():
    from multimodal_autonomous_driving_perception_and_planning_b200.perception import lane_detector as L
    det = LaneDetector()
    cams = [np.zeros((2, 1080, 1920), np.uint8), np.zeros((1, 1620, 1920), np.uint8), np.zeros((1, 5, 3), np.uint8)]
    p = det._rig_plan(cams, ["bayer_gbrg", "nv12", "bayer_rggb"], (640, 480), None)
    assert p.sizes == [(1080, 1920), (1080, 1920), (5, 3)] and p.fmts == [19, 1, 16] and (p.h, p.w) == (480, 640)
    assert [L._frame_bytes(f, *hw) for f, hw in zip(p.fmts, p.sizes)] == [1080 * 1920, 1080 * 1920 * 3 // 2, 15]
    q = L._Plan.of_frames(cams[0], _native.INPUT_BAYER_BGGR)
    assert q.sizes == [(1080, 1920)] and (q.h, q.w) == (1080, 1920)


def test_frame_ingest_bayer_errors_raise_before_the_device():
    ing = FrameIngest((320, 240))
    for bad in BAD_FRAMES:
        with pytest.raises(cv2.error):
            ing.from_bayer(bad, "rggb")
    with pytest.raises(ValueError):
        ing.from_bayer(RAW, "bgrg")


def test_context_free_entry_reports_no_device_under_its_own_name():
    pytest.importorskip("torch")
    import torch
    if torch.cuda.is_available():
        pytest.skip("a device is visible")
    lib = _native.lib()
    src, dst = np.zeros(48 * 64, np.uint8), np.zeros(24 * 32 * 3, np.uint8)
    rc = lib.lane_bayer_to_bgr_batch(_native._ptr(src), _native.INPUT_BAYER_RGGB, 1, 48, 64, _native._ptr(dst), 24, 32,
                                     0, 0, None)
    assert rc == -3 and lib.lane_last_error(None).startswith(b"lane_bayer_to_bgr_batch: ")


def test_raw_entry_points_reject_bad_arguments_without_a_device():
    lib = _native.lib()
    src = np.zeros(48 * 64, np.uint8)
    dst = np.zeros(24 * 32 * 3, np.uint8)
    p, q = src.ctypes.data_as(ctypes.c_void_p), dst.ctypes.data_as(ctypes.c_void_p)
    R = _native.INPUT_BAYER_RGGB
    assert lib.lane_bayer_to_bgr_batch(p, 3, 1, 48, 64, q, 24, 32, 0, 0, None) == -1            # unknown format
    assert lib.lane_bayer_to_bgr_batch(p, _native.INPUT_NV12, 1, 48, 64, q, 24, 32, 0, 0, None) == -1   # not Bayer
    assert lib.lane_bayer_to_bgr_batch(p, 20, 1, 48, 64, q, 24, 32, 0, 0, None) == -1
    assert lib.lane_bayer_to_bgr_batch(p, R, 1, 2, 64, q, 24, 32, 0, 0, None) == -1             # below 3 rows
    assert lib.lane_bayer_to_bgr_batch(p, R, 1, 48, 2, q, 24, 32, 0, 0, None) == -1             # below 3 columns
    assert b"3 rows" in lib.lane_last_error(None)
    assert lib.lane_bayer_to_bgr_batch(p, R, 0, 48, 64, q, 24, 32, 0, 0, None) == -1            # empty batch
    assert lib.lane_bayer_to_bgr_batch(None, R, 1, 48, 64, q, 24, 32, 0, 0, None) == -1         # null source
    assert lib.lane_bayer_to_bgr_batch(p, R, 1, 48, 64, q, 0, 32, 0, 0, None) == -1             # empty destination
    assert lib.lane_bayer_to_bgr_batch(p, R, 1, 48, 64, q, 70000, 32, 0, 0, None) == -5         # beyond the grid
    assert lib.lane_bayer_to_bgr_batch(p, R, 70000, 48, 64, q, 24, 32, 0, 0, None) == -5
    # the YUV entries keep refusing everything but their own layouts
    for fmt in _native.BAYER.values():
        assert lib.lane_yuv420_to_bgr_batch(p, fmt, 1, 48, 64, q, 24, 32, 0, 0, None) == -1
    # context calls with a null context, and the unknown format 3, are invalid
    assert lib.lane_detect_batch_ingest(None, p, 0, 1, R, 48, 64, None, 1, None, None, None) == -1
    fit, valid = np.zeros((1, 2, 3)), np.zeros((1, 2), np.uint8)
    out = np.zeros(1, _native.RECORD_DTYPE)
    for fmt in (R, 3):
        srcs = (_native.LaneRigSource * 1)(_native.LaneRigSource(src.ctypes.data, fmt, 48, 64, 1, 0))
        assert lib.lane_detect_rig(None, srcs, 1, 0, 1, _native._ptr(fit), _native._ptr(valid), _native._ptr(out)) == -1
        assert lib.lane_rig_enqueue(None, srcs, 1, 0, 1, None, None) == -1
