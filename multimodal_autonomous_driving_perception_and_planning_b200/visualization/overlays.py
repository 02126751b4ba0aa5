"""Batched lane overlays on the GPU: the drawing step right after the lane path.

Mirrors, for a whole batch of frames resident in HBM and with identical pixels,

* ``LaneDetector.draw_lanes`` (/root/reference/src/perception/lane_detector.py:220-251) -> :func:`draw_lanes_batch`
* ``OverlayRenderer.draw_lane_offset_indicator`` (/root/reference/src/visualization/overlays.py:103-148)
  -> :meth:`OverlayRenderer.draw_lane_offset_indicator_batch`

The other ``OverlayRenderer`` panels (info panel, planning info, detection summary, tracking stats) consume the YOLO /
tracker / planner outputs, which are out of scope (SURVEY.md section 2), and are not rebuilt.

``cv2.putText`` is the one call that is not restated on the device: its glyph tables are data of the OpenCV build, so a
string is rendered once on the host by ``cv2.putText`` itself into a small bit mask (cached per distinct string) and
blitted by the kernel -- the same way the ROI polygon mask enters the lane path.

There is no CPU fallback: without the CUDA library / a GPU the calls raise.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import cv2
import numpy as np

from .. import _native
from .draw_list import DrawList

NUM_POINTS = _native.NUM_POINTS


def _lane_arrays(lanes):
    n = len(lanes)
    pts = np.zeros((2, n, NUM_POINTS, 2), np.int32)
    valid = np.zeros((2, n), np.uint8)
    for i, pair in enumerate(lanes):
        for s in (0, 1):
            lane = pair[s]
            if lane is not None:
                p = np.asarray(lane.points if hasattr(lane, "points") else lane, np.int32)
                if p.shape != (NUM_POINTS, 2):
                    raise ValueError(f"lane points must be int32[{NUM_POINTS}, 2], got {p.shape}")
                pts[s, i] = p
                valid[s, i] = 1
    return pts, valid


def draw_lanes_batch(frames, lanes: Sequence[Tuple[Optional[object], Optional[object]]], fill_lane: bool = True,
                     device: Optional[int] = None, return_ms: bool = False):
    """``LaneDetector.draw_lanes`` for every frame of a batch, IN PLACE.

    ``frames``: uint8 ``[N, H, W, 3]``, CUDA torch tensor (stays in HBM) or C-contiguous numpy array (round trip inside
    the call).  ``lanes``: ``N`` pairs ``(left, right)`` as ``detect_batch`` returns them (``LaneLine`` or ``None``; a
    plain int32 ``[50, 2]`` array is accepted in place of a ``LaneLine``).  Pixels equal
    ``detector.draw_lanes(frame, left, right, fill_lane)`` of the reference; note that the reference returns a new array
    when it fills and draws on its argument when it does not -- here the batch is always modified in place and
    returned."""
    if len(frames.shape) != 4 or frames.shape[3] != 3 or len(lanes) != frames.shape[0]:
        raise ValueError(f"expected uint8 frames [N, H, W, 3] and N lane pairs, got {tuple(frames.shape)} and {len(lanes)}")
    pts, valid = _lane_arrays(lanes)
    return draw_lanes_arrays(frames, pts[0], valid[0], pts[1], valid[1], fill_lane, device, return_ms)


def draw_lanes_arrays(frames, left_points, left_valid, right_points, right_valid, fill_lane=True, device=None,
                      return_ms=False):
    """Array form of :func:`draw_lanes_batch`: ``*_points`` int32 ``[N, 50, 2]``, ``*_valid`` uint8 ``[N]`` -- the fields
    ``side[s].points`` / ``side[s].valid`` of the native lane records, so a batch can be annotated straight from them."""
    lib = _native.lib()
    n, h, w = int(frames.shape[0]), int(frames.shape[1]), int(frames.shape[2])
    lp = np.ascontiguousarray(left_points, np.int32)
    rp = np.ascontiguousarray(right_points, np.int32)
    lv = np.ascontiguousarray(left_valid, np.uint8)
    rv = np.ascontiguousarray(right_valid, np.uint8)
    if lp.shape != (n, NUM_POINTS, 2) or rp.shape != (n, NUM_POINTS, 2) or lv.shape != (n,) or rv.shape != (n,):
        raise ValueError("lane arrays do not match the batch")
    ms = C.c_float(0.0)
    args = (lp.ctypes.data_as(C.c_void_p), lv.ctypes.data_as(C.c_void_p), rp.ctypes.data_as(C.c_void_p),
            rv.ctypes.data_as(C.c_void_p), int(bool(fill_lane)))
    if isinstance(frames, np.ndarray):
        if frames.dtype != np.uint8 or not frames.flags.c_contiguous:
            raise cv2.error("draw_lanes_batch: numpy frames must be C-contiguous uint8")
        if device is None:
            import torch
            device = int(torch.cuda.current_device()) if torch.cuda.is_available() else 0
        rc = lib.lane_draw_lanes_batch(frames.ctypes.data_as(C.c_void_p), 0, n, h, w, *args, int(device), None, C.byref(ms))
    else:
        import torch
        if not frames.is_cuda or frames.dtype != torch.uint8 or not frames.is_contiguous():
            raise cv2.error("draw_lanes_batch: torch frames must be a contiguous CUDA uint8 tensor")
        if device is not None and int(device) != frames.device.index:
            raise ValueError(f"device={device} but the frames are on {frames.device}")
        stream = torch.cuda.current_stream(frames.device).cuda_stream
        rc = lib.lane_draw_lanes_batch(C.c_void_p(frames.data_ptr()), 1, n, h, w, *args, frames.device.index,
                                       C.c_void_p(stream), C.byref(ms))
    _native.check_global(rc)
    return (frames, ms.value) if return_ms else frames


def draw_lanes_records(frames, records_device_ptr: int, fill_lane: bool = True):
    """``draw_lanes`` for a batch straight from the lane records ON THE DEVICE (``LaneContext.records_device_ptr()`` after a
    collect, i.e. ``lane_ctx_records_device``): neither the lanes nor the frames touch the host.  ``frames``: contiguous
    CUDA uint8 tensor ``[N, H, W, 3]``, drawn in place on torch's current stream (no synchronisation)."""
    import torch
    lib = _native.lib()
    if not frames.is_cuda or frames.dtype != torch.uint8 or not frames.is_contiguous() or len(frames.shape) != 4 or frames.shape[3] != 3:
        raise cv2.error("draw_lanes_records: frames must be a contiguous CUDA uint8 tensor [N, H, W, 3]")
    n, h, w = int(frames.shape[0]), int(frames.shape[1]), int(frames.shape[2])
    stream = torch.cuda.current_stream(frames.device).cuda_stream
    rc = lib.lane_draw_lanes_records(C.c_void_p(frames.data_ptr()), n, h, w, C.c_void_p(records_device_ptr), int(bool(fill_lane)),
                                     frames.device.index, C.c_void_p(stream))
    _native.check_global(rc)
    return frames


class OverlayRenderer:
    """The lane part of the reference's ``OverlayRenderer`` (src/visualization/overlays.py:16-24, :103-148), batched."""

    def __init__(self):
        self.font = cv2.FONT_HERSHEY_SIMPLEX
        self.font_scale = 0.5
        self.font_thickness = 1
        self._text_cache = {}

    def _text_mask(self, text: str, scale: float, thickness: int):
        """Bit mask of ``cv2.putText(img, text, org, self.font, scale, color, thickness)`` relative to ``org``:
        ``(dx, dy, mask)`` with ``mask[j, i]`` = pixel ``(org.x + dx + i, org.y + dy + j)`` is set."""
        key = (text, scale, thickness)
        hit = self._text_cache.get(key)
        if hit is None:
            (tw, th), base = cv2.getTextSize(text, self.font, scale, thickness)
            pad = 4 + thickness
            canvas = np.zeros((th + base + 2 * pad, tw + 2 * pad), np.uint8)
            org = (pad, pad + th)
            cv2.putText(canvas, text, org, self.font, scale, 255, thickness)
            ys, xs = np.nonzero(canvas)
            if len(ys) == 0:
                hit = (0, 0, np.zeros((1, 1), bool))
            else:
                y0, y1, x0, x1 = ys.min(), ys.max(), xs.min(), xs.max()
                hit = (int(x0 - org[0]), int(y0 - org[1]), canvas[y0:y1 + 1, x0:x1 + 1] > 0)
            self._text_cache[key] = hit
        return hit

    def put_text(self, dl: DrawList, frame: int, text: str, org, scale: float, color, thickness: int = 1,
                 frame_size: Optional[Tuple[int, int]] = None):
        """``cv2.putText(img, text, org, self.font, scale, color, thickness)`` recorded into ``dl``.  The rendered mask
        does not depend on where the string sits as long as it lies inside the image (putText places glyphs in whole
        pixels of ``org``); a string cut by the image border is rendered at its place instead, because cv2 clips each
        glyph stroke before rasterising it.  ``frame_size`` = (width, height) enables that check."""
        dx, dy, mask = self._text_mask(text, float(scale), int(thickness))
        x, y = int(org[0]) + dx, int(org[1]) + dy
        if frame_size is not None:
            w, h = frame_size
            if x < 0 or y < 0 or x + mask.shape[1] > w or y + mask.shape[0] > h:
                key = (text, float(scale), int(thickness), int(org[0]), int(org[1]), w, h)
                hit = self._text_cache.get(key)
                if hit is None:
                    canvas = np.zeros((h, w), np.uint8)
                    cv2.putText(canvas, text, (int(org[0]), int(org[1])), self.font, scale, 255, thickness)
                    ys, xs = np.nonzero(canvas)
                    hit = None if len(ys) == 0 else (int(xs.min()), int(ys.min()),
                                                     canvas[ys.min():ys.max() + 1, xs.min():xs.max() + 1] > 0)
                    self._text_cache[key] = hit if hit is not None else ()
                if not hit:
                    return
                x, y, mask = hit
        dl.bitmap(frame, x, y, mask, color)

    def record_lane_offset_indicator(self, dl: DrawList, frame: int, width: int, height: int, offset: Optional[float]):
        """The calls of ``draw_lane_offset_indicator`` (overlays.py:103-148) for one frame, recorded into ``dl``."""
        h, w = height, width
        indicator_w, indicator_h = 200, 30
        x_start = (w - indicator_w) // 2
        y_start = h - 50
        dl.rectangle(frame, (x_start, y_start), (x_start + indicator_w, y_start + indicator_h), (50, 50, 50), -1)
        dl.rectangle(frame, (x_start, y_start), (x_start + indicator_w, y_start + indicator_h), (100, 100, 100), 1)
        center_x = x_start + indicator_w // 2
        dl.line(frame, (center_x, y_start), (center_x, y_start + indicator_h), (255, 255, 255), 1)
        if offset is not None:
            max_offset = 100
            offset_px = int(np.clip(offset, -max_offset, max_offset))
            indicator_x = center_x + offset_px
            if abs(offset) < 20:
                color = (0, 255, 0)
            elif abs(offset) < 50:
                color = (0, 255, 255)
            else:
                color = (0, 0, 255)
            dl.circle(frame, (indicator_x, y_start + indicator_h // 2), 8, color, -1)
            self.put_text(dl, frame, f"Offset: {offset:.0f}px", (x_start + 5, y_start - 5), 0.4, (255, 255, 255), 1,
                          frame_size=(w, h))

    def _indicator_words(self, width: int, height: int, offset: Optional[float]) -> np.ndarray:
        """Encoded command stream of one frame's indicator; cached per (size, offset) -- a batch has few distinct offsets."""
        key = ("indicator", width, height, offset)
        words = self._text_cache.get(key)
        if words is None:
            tmp = DrawList(1)
            self.record_lane_offset_indicator(tmp, 0, width, height, offset)
            words = self._text_cache[key] = tmp.encoded(0)
            if len(self._text_cache) > 65536:
                self._text_cache.clear()
        return words

    def draw_lane_offset_indicator_batch(self, frames, offsets: Sequence[Optional[float]], device: Optional[int] = None):
        """``draw_lane_offset_indicator(frame, offset)`` for every frame of a batch, IN PLACE (uint8 ``[N, H, W, 3]``, CUDA
        tensor or numpy); ``offsets[i]`` is what ``get_lane_center_offset`` returned for frame ``i`` (``None`` allowed)."""
        from .draw_list import run_commands
        n, h, w = int(frames.shape[0]), int(frames.shape[1]), int(frames.shape[2])
        if len(offsets) != n:
            raise ValueError("one offset per frame")
        if len(frames.shape) != 4 or frames.shape[3] != 3:
            raise ValueError(f"expected uint8 frames [N, H, W, 3], got {tuple(frames.shape)}")
        parts = [self._indicator_words(w, h, None if off is None else float(off)) for off in offsets]
        begin = np.zeros(n + 1, np.int64)
        np.cumsum([len(p) for p in parts], out=begin[1:])
        return run_commands(frames, np.ascontiguousarray(np.concatenate(parts), np.int32), begin, device)

    def draw_lanes_batch(self, frames, lanes, fill_lane: bool = True, device: Optional[int] = None):
        return draw_lanes_batch(frames, lanes, fill_lane, device)
