"""CPU restatement of ``cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)`` (uint8) and of its NV12 re-layout: the arithmetic of
the egress kernel (csrc/k8_egress.cu), pinned by tests/test_oracle_egress.py against cv2 on every one of the 2^24 BGR
values.  BT.601 limited range in 20-bit fixed point with a round-half constant (the inverse of oracle/nv12.py):

    Y = sat_u8(( 269484 R + 528482 G + 102760 B + (16 << 20)  + 2^19) >> 20)     every pixel
    U = sat_u8((-155188 R - 305135 G + 460324 B + (128 << 20) + 2^19) >> 20)     top-left pixel of each 2x2 block
    V = sat_u8(( 460324 R - 385875 G -  74448 B + (128 << 20) + 2^19) >> 20)     (no averaging)
    I420 layout uint8 [H * 3 / 2][W]: Y plane, then U [H/2][W/2], then V [H/2][W/2]; NV12: U and V interleaved
"""
import numpy as np

SHIFT = 20
EYR, EYG, EYB = 269484, 528482, 102760
EUR, EUG, EUB = -155188, -305135, 460324
EVR, EVG, EVB = 460324, -385875, -74448


def _planes(bgr: np.ndarray):
    bgr = np.asarray(bgr, dtype=np.uint8)
    if bgr.ndim != 3 or bgr.shape[2] != 3:
        raise ValueError("expected a uint8 [H, W, 3] BGR frame")
    h, w = bgr.shape[:2]
    if h < 2 or w < 2 or h % 2 or w % 2:
        raise ValueError("YUV 4:2:0 needs even, positive width and height")
    x = bgr.astype(np.int64)
    b, g, r = x[..., 0], x[..., 1], x[..., 2]
    half = 1 << (SHIFT - 1)
    y = (EYR * r + EYG * g + EYB * b + (16 << SHIFT) + half) >> SHIFT
    b, g, r = b[::2, ::2], g[::2, ::2], r[::2, ::2]
    u = (EUR * r + EUG * g + EUB * b + (128 << SHIFT) + half) >> SHIFT
    v = (EVR * r + EVG * g + EVB * b + (128 << SHIFT) + half) >> SHIFT
    return [np.clip(p, 0, 255).astype(np.uint8) for p in (y, u, v)]


def bgr_to_i420(bgr: np.ndarray) -> np.ndarray:
    """uint8 [H, W, 3] BGR (H, W even) -> uint8 [H*3/2, W] I420, i.e. cv2.cvtColor(bgr, cv2.COLOR_BGR2YUV_I420)."""
    y, u, v = _planes(bgr)
    h, w = y.shape
    return np.concatenate([y.ravel(), u.ravel(), v.ravel()]).reshape(h * 3 // 2, w)


def bgr_to_nv12(bgr: np.ndarray) -> np.ndarray:
    """uint8 [H, W, 3] BGR (H, W even) -> uint8 [H*3/2, W] NV12: the samples of bgr_to_i420, U and V interleaved."""
    y, u, v = _planes(bgr)
    h, w = y.shape
    return np.concatenate([y, np.stack([u, v], axis=-1).reshape(h // 2, w)])
