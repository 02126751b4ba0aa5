"""I420 test helpers.  I420 (the ``yuv420p`` of software decoders) carries the same samples as NV12 -- a Y plane, then
a U plane and a V plane of H/2 x W/2 each, where NV12 interleaves U and V -- so its conversion is oracle/nv12.py's
after a re-layout of the chroma planes; tests/test_oracle_ingest.py pins that against cv2.COLOR_YUV2BGR_I420."""
import numpy as np

from oracle import nv12 as onv


def nv12_to_i420(nv12: np.ndarray) -> np.ndarray:
    """uint8 [H*3/2, W] NV12 -> the I420 frame of the same samples."""
    rows, w = nv12.shape
    h = rows * 2 // 3
    uv = nv12[h:].reshape(h // 2, w // 2, 2)
    return np.concatenate([nv12[:h].ravel(), uv[..., 0].ravel(), uv[..., 1].ravel()]).reshape(rows, w)


def i420_to_nv12(i420: np.ndarray) -> np.ndarray:
    rows, w = i420.shape
    h = rows * 2 // 3
    q = (h // 2) * (w // 2)
    flat = i420.reshape(-1)
    u = flat[h * w:h * w + q].reshape(h // 2, w // 2)
    v = flat[h * w + q:].reshape(h // 2, w // 2)
    out = np.empty_like(i420)
    out[:h] = i420[:h]
    out[h:] = np.stack([u, v], axis=-1).reshape(h // 2, w)
    return out


def i420_to_bgr(i420: np.ndarray) -> np.ndarray:
    """CPU restatement of ``cv2.cvtColor(i420, cv2.COLOR_YUV2BGR_I420)`` (uint8 [H*3/2, W], H and W even)."""
    i420 = np.asarray(i420, dtype=np.uint8)
    rows, w = i420.shape
    if rows % 3 or w % 2 or (rows * 2 // 3) % 2:
        raise ValueError("I420 needs even width and height")
    return onv.nv12_to_bgr(i420_to_nv12(i420))
