"""The egress direction, BGR -> YUV 4:2:0 (csrc/k8_egress.cu): the restatement in tests/bgr_yuv420.py equals
cv2.cvtColor(f, COLOR_BGR2YUV_I420) on random frames of many sizes and on every one of the 2^24 BGR values as the
top-left pixel of a 2x2 block (the pixel U and V are taken from); the NV12 re-layout equals the package's
bgr_to_nv12 and oracle/nv12.py's test-input helper; the public functions reject bad arguments before any native call,
and the C entry rejects them before touching a device."""
import ctypes

import cv2
import numpy as np
import pytest

from multimodal_autonomous_driving_perception_and_planning_b200 import _native, bgr_to_i420, bgr_to_nv12, generators
import bgr_yuv420 as egress
from oracle import nv12 as onv
from yuv420 import i420_to_nv12

# (H, W)
SIZES = [(2, 2), (2, 34), (6, 2), (482, 642), (480, 640), (720, 1280), (1080, 1920), (2160, 3840)]


def random_sizes(k=40, seed=5):
    rng = np.random.default_rng(seed)
    return [(2 * int(rng.integers(1, 300)), 2 * int(rng.integers(1, 500))) for _ in range(k)]


def random_bgr(hw, seed):
    return np.random.default_rng(seed).integers(0, 256, (*hw, 3), dtype=np.uint8)


@pytest.mark.parametrize("hw", SIZES)
def test_restatement_equals_cv2(hw):
    f = random_bgr(hw, hw[0] * 7 + hw[1])
    want = cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420)
    assert np.array_equal(egress.bgr_to_i420(f), want)
    assert np.array_equal(egress.bgr_to_nv12(f), i420_to_nv12(want))


def test_restatement_equals_cv2_on_random_even_sizes():
    for k, hw in enumerate(random_sizes()):
        f = random_bgr(hw, 1000 + k)
        assert np.array_equal(egress.bgr_to_i420(f), cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420)), hw


def test_every_bgr_value_as_the_chroma_pixel():
    """Value v = B | G << 8 | R << 16 is the top-left pixel of block v; the other three pixels of the block hold other
    values, so every Y is checked too.  16 slices of 2^20 blocks (1024 x 4096 frames)."""
    bh, bw = 512, 2048
    for s in range(16):
        v = np.arange(s << 20, (s + 1) << 20, dtype=np.uint32).reshape(bh, bw)
        f = np.empty((2 * bh, 2 * bw, 3), np.uint8)
        for (dy, dx), x in zip([(0, 0), (0, 1), (1, 0), (1, 1)], [v, v ^ 0x5A5A5A, ~v, v * 2654435761]):
            f[dy::2, dx::2, 0] = x & 0xFF
            f[dy::2, dx::2, 1] = (x >> 8) & 0xFF
            f[dy::2, dx::2, 2] = (x >> 16) & 0xFF
        assert np.array_equal(egress.bgr_to_i420(f), cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420)), s


def test_nv12_restatement_equals_the_package_and_the_test_helper():
    frames = np.stack([random_bgr((480, 642), k) for k in range(3)])
    want = np.stack([egress.bgr_to_nv12(f) for f in frames])
    assert np.array_equal(generators.bgr_to_nv12(frames), want)
    assert np.array_equal(bgr_to_nv12(frames), want)
    assert np.array_equal(np.stack([onv.bgr_to_nv12_for_tests(f) for f in frames]), want)
    assert np.array_equal(bgr_to_i420(frames), np.stack([egress.bgr_to_i420(f) for f in frames]))
    assert generators.bgr_to_nv12 is bgr_to_nv12


def test_host_path_with_out():
    frames = np.stack([random_bgr((6, 10), k) for k in range(2)])
    out = np.zeros((2, 9, 10), np.uint8)
    assert bgr_to_i420(frames, out=out) is out
    assert np.array_equal(out, np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420) for f in frames]))


def test_host_path_errors():
    with pytest.raises(ValueError):
        bgr_to_nv12(np.zeros((1, 5, 4, 3), np.uint8))
    with pytest.raises(ValueError):
        bgr_to_i420(np.zeros((1, 4, 7, 3), np.uint8))
    with pytest.raises(ValueError):
        bgr_to_i420(np.zeros((1, 4, 6, 3), np.uint8), out=np.zeros((1, 4, 6), np.uint8))
    with pytest.raises(ValueError):
        bgr_to_i420(np.zeros((1, 4, 6, 3), np.uint8), out=np.zeros((1, 6, 6), np.int16))


@pytest.mark.parametrize("fn", [bgr_to_i420, bgr_to_nv12])
def test_tensor_path_errors_raise_before_any_native_call(fn):
    """Tensors that are not on the CPU take the device path; meta tensors reach its checks without a device."""
    import torch

    def t(shape, dtype=torch.uint8):
        return torch.empty(shape, dtype=dtype, device="meta")
    for bad in (t((2, 5, 8, 3)), t((2, 4, 9, 3)), t((2, 0, 8, 3)), t((2, 4, 8, 4)), t((4, 8, 3)), t((2, 4, 8, 3), torch.int16)):
        with pytest.raises(cv2.error):
            fn(bad)
    for out in (np.zeros((2, 4, 8), np.uint8), np.zeros((2, 6, 8), np.int32), np.zeros((2, 6, 8), np.uint8)[:, ::-1],
                torch.zeros((2, 6, 9), dtype=torch.uint8), [0]):
        with pytest.raises(cv2.error):
            fn(t((2, 4, 8, 3)), out=out)
    with pytest.raises(cv2.error, match="CUDA"):                    # well-formed, but not on a CUDA device
        fn(t((2, 4, 8, 3)), out=np.zeros((2, 6, 8), np.uint8))


def test_raw_entry_rejects_bad_arguments_without_a_device():
    lib = _native.lib()
    buf = np.zeros(64, np.uint8)
    p = buf.ctypes.data_as(ctypes.c_void_p)

    def call(src, fmt, n, h, w, dst):
        return lib.lane_bgr_to_yuv420_batch(src, fmt, n, h, w, dst, 1, 0, None)
    I420, NV12 = _native.INPUT_I420, _native.INPUT_NV12
    assert call(None, I420, 1, 2, 2, p) == -1                      # null source
    assert call(p, I420, 1, 2, 2, None) == -1                      # null destination
    assert call(p, _native.INPUT_BGR, 1, 2, 2, p) == -1            # BGR is not an output layout
    assert call(p, 3, 1, 2, 2, p) == -1                            # unknown format
    assert call(p, NV12, -1, 2, 2, p) == -1                        # negative batch
    assert call(p, NV12, 1, 0, 2, p) == -1                         # non-positive sizes
    assert call(p, NV12, 1, 2, -2, p) == -1
    assert call(p, I420, 1, 3, 2, p) == -1                         # odd sizes
    assert call(p, I420, 1, 2, 5, p) == -1
    assert call(p, I420, 2 ** 31 - 1, 2 ** 30, 2 ** 30, p) == -1   # byte offsets beyond 2^62
    assert b"lane_bgr_to_yuv420_batch" in lib.lane_last_error(None)
    assert call(p, I420, 0, 2, 2, p) == 0                          # n = 0: nothing to do
