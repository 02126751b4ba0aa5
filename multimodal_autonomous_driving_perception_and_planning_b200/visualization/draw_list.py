"""cv2-shaped drawing calls recorded per frame and rasterised for the whole batch on the GPU (K7, ``csrc/k7_draw.cu``).

The reference draws with OpenCV on every frame: ``LaneDetector.draw_lanes``
(/root/reference/src/perception/lane_detector.py:220-251), ``OverlayRenderer.draw_lane_offset_indicator``
(/root/reference/src/visualization/overlays.py:103-148) and the synthetic generator (SURVEY.md Appendix B).  A
``DrawList`` records the same calls -- same names, argument order and meaning as ``cv2.line / rectangle / circle /
fillPoly / polylines`` -- for each frame of a batch, and ``execute`` runs them on frames resident in HBM through
``lane_draw_commands``; the pixels equal what the cv2 calls produce (OpenCV 4.13, uint8, LINE_8).

There is no CPU fallback: without the CUDA library / a GPU ``execute`` raises.
"""
from __future__ import annotations

import ctypes as C
import functools
from typing import Optional, Sequence

import numpy as np

from .. import _native

LINE, RECTANGLE, CIRCLE, FILLPOLY, POLYLINES, FILLPOLY_WEIGHTED, BITMAP, ROWS = 1, 2, 3, 4, 5, 6, 7, 8


@functools.lru_cache(maxsize=65536)
def _color_word(color: tuple) -> int:
    b, g, r = (int(min(255, max(0, round(float(c))))) for c in color[:3])
    return b | g << 8 | r << 16


def color_word(color: Sequence[int]) -> int:
    """(b, g, r) -> b | g << 8 | r << 16, each channel saturated to 0..255 as cv2's Scalar conversion does."""
    return _color_word(tuple(color))


def _f32_bits(v: float) -> int:
    return int(np.float32(v).view(np.int32))


class DrawList:
    """Drawing calls of ``n_frames`` frames.  ``frame`` selects the frame a call is recorded for; calls of one frame
    execute in the order they were recorded."""

    def __init__(self, n_frames: int):
        self.n_frames = int(n_frames)
        self._words = [[] for _ in range(self.n_frames)]      # python ints or numpy int32 arrays

    # ---- cv2-shaped calls
    def line(self, frame, pt1, pt2, color, thickness=1):
        self._words[frame].append((LINE, int(pt1[0]), int(pt1[1]), int(pt2[0]), int(pt2[1]), color_word(color), int(thickness)))

    def rectangle(self, frame, pt1, pt2, color, thickness=1):
        self._words[frame].append((RECTANGLE, int(pt1[0]), int(pt1[1]), int(pt2[0]), int(pt2[1]), color_word(color),
                                   int(thickness)))

    def circle(self, frame, center, radius, color, thickness=-1):
        if thickness >= 0:
            raise ValueError("only filled circles (thickness < 0) are on the reference's path")
        self._words[frame].append((CIRCLE, int(center[0]), int(center[1]), int(radius), color_word(color), int(thickness)))

    def fillPoly(self, frame, pts, color):
        p = np.asarray(pts, np.int32).reshape(-1, 2)
        self._words[frame].append(np.concatenate([np.array([FILLPOLY, color_word(color), len(p)], np.int32), p.ravel()]))

    def polylines(self, frame, pts, is_closed, color, thickness=1):
        p = np.asarray(pts, np.int32).reshape(-1, 2)
        self._words[frame].append(np.concatenate([np.array([POLYLINES, color_word(color), int(thickness), int(bool(is_closed)),
                                                            len(p)], np.int32), p.ravel()]))

    def fillPoly_weighted(self, frame, pts, color, alpha, beta, gamma=0.0):
        """``o = img.copy(); cv2.fillPoly(o, [pts], color); img = cv2.addWeighted(img, alpha, o, beta, gamma)``."""
        p = np.asarray(pts, np.int32).reshape(-1, 2)
        self._words[frame].append(np.concatenate([np.array([FILLPOLY_WEIGHTED, color_word(color), _f32_bits(alpha),
                                                            _f32_bits(beta), _f32_bits(gamma), len(p)], np.int32), p.ravel()]))

    def bitmap(self, frame, x, y, mask, color):
        """Pixels ``(x + i, y + j)`` with ``mask[j, i]`` set get ``color`` (text rendered once by ``cv2.putText``)."""
        m = np.asarray(mask).astype(bool)
        h, w = m.shape
        wpr = (w + 31) // 32
        padded = np.zeros((h, wpr * 32), np.uint8)
        padded[:, :w] = m
        words = np.packbits(padded.reshape(h, wpr, 32), axis=-1, bitorder="little").view("<u4").reshape(-1).astype(np.uint32)
        self._words[frame].append(np.concatenate([np.array([BITMAP, int(x), int(y), w, h, color_word(color)], np.int32),
                                                  words.view(np.int32)]))

    def rows(self, frame, y_start, x1, x2, colors):
        """``cv2.line(img, (x1, y), (x2, y), colors[y - y_start], 1)`` for ``len(colors)`` consecutive rows."""
        cw = np.array([color_word(c) for c in colors], np.int32)
        self._words[frame].append(np.concatenate([np.array([ROWS, int(y_start), len(cw), int(x1), int(x2)], np.int32), cw]))

    def extend(self, frame, words: np.ndarray):
        """Append an already encoded int32 command stream (e.g. the frame-independent part of a scene, encoded once)."""
        self._words[frame].append(np.asarray(words, np.int32))

    def encoded(self, frame) -> np.ndarray:
        parts = [np.asarray(w, np.int32).ravel() for w in self._words[frame]]
        return np.concatenate(parts) if parts else np.zeros(0, np.int32)

    # ---- execution
    def pack(self):
        per_frame = [self.encoded(f) for f in range(self.n_frames)]
        begin = np.zeros(self.n_frames + 1, np.int64)
        np.cumsum([len(w) for w in per_frame], out=begin[1:])
        words = np.concatenate(per_frame) if begin[-1] else np.zeros(1, np.int32)
        return np.ascontiguousarray(words, np.int32), begin

    def execute(self, frames, device: Optional[int] = None, return_ms: bool = False):
        """Draw in place.  ``frames``: uint8 ``[n_frames, H, W, 3]``, a CUDA torch tensor (drawn where it is, on torch's
        current stream) or a C-contiguous numpy array (copied to the device, drawn, copied back)."""
        if tuple(frames.shape[:1]) != (self.n_frames,) or len(frames.shape) != 4 or frames.shape[3] != 3:
            raise ValueError(f"expected uint8 frames [{self.n_frames}, H, W, 3], got {tuple(frames.shape)}")
        words, begin = self.pack()
        return run_commands(frames, words, begin, device, return_ms)


def run_commands(frames, words: np.ndarray, begin: np.ndarray, device: Optional[int] = None, return_ms: bool = False):
    lib = _native.lib()
    n, h, w = int(frames.shape[0]), int(frames.shape[1]), int(frames.shape[2])
    ms = C.c_float(0.0)
    if isinstance(frames, np.ndarray):
        if frames.dtype != np.uint8 or not frames.flags.c_contiguous:
            raise ValueError("numpy frames must be C-contiguous uint8")
        if device is None:
            import torch
            device = int(torch.cuda.current_device()) if torch.cuda.is_available() else 0
        rc = lib.lane_draw_commands(frames.ctypes.data_as(C.c_void_p), 0, n, h, w, words.ctypes.data_as(C.c_void_p),
                                    begin.ctypes.data_as(C.c_void_p), int(device), None, C.byref(ms))
    else:
        import torch
        if not frames.is_cuda or frames.dtype != torch.uint8 or not frames.is_contiguous():
            raise ValueError("torch frames must be a contiguous CUDA uint8 tensor")
        if device is not None and int(device) != frames.device.index:
            raise ValueError(f"device={device} but the frames are on {frames.device}")
        stream = torch.cuda.current_stream(frames.device).cuda_stream
        rc = lib.lane_draw_commands(C.c_void_p(frames.data_ptr()), 1, n, h, w, words.ctypes.data_as(C.c_void_p),
                                    begin.ctypes.data_as(C.c_void_p), frames.device.index, C.c_void_p(stream), C.byref(ms))
    _native.check_global(rc)
    return (frames, ms.value) if return_ms else frames
