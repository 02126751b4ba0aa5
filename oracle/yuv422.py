"""TEST INFRASTRUCTURE ONLY -- CPU restatement of ``cv2.cvtColor(f, cv2.COLOR_YUV2BGR_UYVY | COLOR_YUV2BGR_YUY2)``
(uint8).

Most automotive GMSL / FPD-Link cameras deliver packed YUV 4:2:2 through their deserializer as UYVY, and a V4L2 USB
camera delivers YUYV (cv2's YUY2) by default: 2 B/px, every horizontal pixel pair sharing one (U, V), nothing shared
vertically.  cv2 takes such a frame as uint8 ``[H, W, 2]`` (W even) and converts it with the BT.601 limited-range
arithmetic of NV12 (``oracle/nv12.py``: same constants, same 20-bit fixed point); only the addressing differs.  Within
each 4-byte group:

    UYVY  U Y0 V Y1
    YUYV  Y0 U Y1 V

Pinned against cv2 by tests/test_yuv422_host.py; csrc/k0_common.cuh (k0_yuv422_resize_px) and csrc/k0_nv12.cu
(k0_yuv422_vec / k0_yuv422_generic) compute the same.

Only tests/, __graft_entry__.smoke() and the probes under tools/ may import this module.
"""
import numpy as np

from .nv12 import CUB, CUG, CVG, CVR, CY, SHIFT

# byte offsets of (Y0, U, Y1, V) within a 4-byte group
OFFSETS = {"uyvy": (1, 0, 3, 2), "yuyv": (0, 1, 2, 3)}


def yuv422_to_bgr(frame: np.ndarray, order: str) -> np.ndarray:
    """uint8 [H, W, 2] (W even) in byte order ``order`` ("uyvy" or "yuyv") -> uint8 [H, W, 3] BGR."""
    frame = np.asarray(frame, dtype=np.uint8)
    if frame.ndim != 3 or frame.shape[2] != 2 or frame.shape[1] % 2:
        raise ValueError(f"a YUV 4:2:2 frame needs shape [H, W, 2] with even W, got {frame.shape}")
    y0, u0, y1, v0 = OFFSETS[order]
    h, w = frame.shape[:2]
    g = frame.reshape(h, w // 2, 4).astype(np.int64)
    y = np.stack([g[..., y0], g[..., y1]], axis=-1).reshape(h, w)
    u = np.repeat(g[..., u0] - 128, 2, axis=1)
    v = np.repeat(g[..., v0] - 128, 2, axis=1)
    y = np.maximum(0, y - 16) * CY + (1 << (SHIFT - 1))
    r = (y + CVR * v) >> SHIFT
    gr = (y + CVG * v + CUG * u) >> SHIFT
    b = (y + CUB * u) >> SHIFT
    return np.clip(np.stack([b, gr, r], axis=-1), 0, 255).astype(np.uint8)
