"""Synthetic road-scene frames for the lane-detection path.

Re-creation of the reference's ``SyntheticDataGenerator`` whose source is gone from the
reference tree (only ``/root/reference/data/generators/__pycache__/synthetic_data.cpython-312.pyc``
survives; behavioural spec in SURVEY.md Appendix B).  Frames are bit-identical to that
bytecode's output (tests/test_generator.py checks sha256 fixtures taken from it).

All drawing uses cv2 on the host: the frames are the *input fixture* of the path, produced
once and uploaded; generation is never inside a timed region.  Pixel constants are absolute
(they do not scale with resolution), exactly as in the reference.

New here (BASELINE.json "data/generators: batched synthetic multi-camera frames"):
``generate_batch`` and ``multi_camera_batch`` return ``uint8[N,H,W,3]`` / ``uint8[S,T,H,W,3]``
stacks; camera ``s`` of a rig is the same scene generator started at ``frame_count = s*1000``.
"""
from __future__ import annotations

from typing import Iterator, Optional

import cv2
import numpy as np

_VEHICLE_COLORS = [(0, 100, 200), (200, 50, 50), (50, 200, 50), (200, 200, 50)]


class _Cv2Canvas:
    """The scene code draws through this: cv2 on a host image ..."""

    def __init__(self, img):
        self.img = img

    def line(self, p1, p2, color, thickness):
        cv2.line(self.img, p1, p2, color, thickness)

    def rectangle(self, p1, p2, color, thickness):
        cv2.rectangle(self.img, p1, p2, color, thickness)

    def circle(self, center, radius, color, thickness):
        cv2.circle(self.img, center, radius, color, thickness)

    def fillPoly(self, pts, color):
        cv2.fillPoly(self.img, [pts], color)

    def rows(self, y_start, x1, x2, colors):
        for i, c in enumerate(colors):
            cv2.line(self.img, (x1, y_start + i), (x2, y_start + i), c, 1)

    def cached(self, cache, key, paint):
        paint(self)


class _ListCanvas:
    """... or the same calls recorded into a DrawList for the device rasteriser (csrc/k7_draw.cu)."""

    def __init__(self, dl, frame):
        self.dl, self.frame = dl, frame

    def line(self, p1, p2, color, thickness):
        self.dl.line(self.frame, p1, p2, color, thickness)

    def rectangle(self, p1, p2, color, thickness):
        self.dl.rectangle(self.frame, p1, p2, color, thickness)

    def circle(self, center, radius, color, thickness):
        self.dl.circle(self.frame, center, radius, color, thickness)

    def fillPoly(self, pts, color):
        self.dl.fillPoly(self.frame, pts, color)

    def rows(self, y_start, x1, x2, colors):
        self.dl.rows(self.frame, y_start, x1, x2, colors)

    def cached(self, cache, key, paint):
        """Frame-independent layers (sky, ground, trees) are encoded once per generator and replayed as words."""
        words = cache.get(key)
        if words is None:
            from ..visualization.draw_list import DrawList
            tmp = DrawList(1)
            paint(_ListCanvas(tmp, 0))
            words = cache[key] = tmp.encoded(0)
        self.dl.extend(self.frame, words)


class SyntheticDataGenerator:
    def __init__(self, width: int = 640, height: int = 480, fps: float = 30.0):
        self.width = width
        self.height = height
        self.fps = fps
        self.dt = 1.0 / fps
        self.frame_count = 0
        self._static = {}            # encoded frame-independent layers of the device path

    # ------------------------------------------------------------------ scene layers
    def _paint_road(self, cv):
        w, h = self.width, self.height
        half = h // 2

        def backdrop(c):
            c.rows(0, 0, w, [(int(200 - 80 * (y / half)), int(180 - 60 * (y / half)), int(255 - 55 * (y / half)))
                             for y in range(half)])
            c.rectangle((0, half), (w, h), (60, 60, 60), -1)

        cv.cached(self._static, ("backdrop", w, h), backdrop)
        vp_x = w // 2 + int(20 * np.sin(self.frame_count * 0.02))
        vp_y = half
        road = np.array([[vp_x, vp_y], [50, h], [w - 50, h]], dtype=np.int32)
        cv.fillPoly(road, (80, 80, 80))
        self._draw_lane_markings(cv, vp_x, vp_y)
        cv.cached(self._static, ("environment", w, h), lambda c: self._draw_environment(c, half))

    def generate_road_frame(self) -> np.ndarray:
        img = np.zeros((self.height, self.width, 3), dtype=np.uint8)
        self._paint_road(_Cv2Canvas(img))
        return img

    def _draw_lane_markings(self, cv, vp_x, vp_y):
        h = self.height
        n = 10
        scroll = (self.frame_count * 5) % (h // n)

        def row(t):
            return min(int(vp_y + (h - vp_y) * t) + scroll, h)

        for i in range(n):
            ya, yb = row(i / n), row((i + 0.5) / n)
            if ya >= vp_y and yb >= vp_y:
                cv.line((vp_x, ya), (vp_x, yb), (255, 255, 200), 2)
        for side in (-1, 1):
            spread = side * 150
            for i in range(n):
                t1, t2 = i / n, (i + 0.6) / n
                cv.line((int(vp_x + spread * t1), row(t1)), (int(vp_x + spread * t2), row(t2)), (255, 255, 255), 2)

    def _draw_environment(self, cv, horizon_y):
        w, h = self.width, self.height
        for i in range(5):
            t = (i + 0.5) / 5
            base = int(horizon_y + (h - horizon_y) * t * 0.8)
            inset = int(30 + 50 * t)
            tall = int(30 + 40 * t)
            for x in (inset, w - inset):
                cv.line((x, base), (x, base - tall), (80, 50, 30), 2)
                cv.circle((x, base - tall - 10), int(15 * t + 5), (50, 120, 50), -1)

    @staticmethod
    def _paint_vehicle(cv, x, y, scale=1.0, color=(0, 100, 200)):
        bw, bh = int(60 * scale), int(40 * scale)
        cv.rectangle((x - bw // 2, y - bh // 2), (x + bw // 2, y + bh // 2), color, -1)
        cv.rectangle((x - bw // 2, y - bh // 2), (x + bw // 2, y + bh // 2), (0, 0, 0), 1)
        cv.rectangle((x - bw // 3, y - bh // 2), (x + bw // 3, y - bh // 4), (100, 100, 100), -1)
        rad = int(8 * scale)
        cv.circle((x - bw // 3, y + bh // 2), rad, (30, 30, 30), -1)
        cv.circle((x + bw // 3, y + bh // 2), rad, (30, 30, 30), -1)

    def generate_vehicle(self, frame, x, y, scale=1.0, color=(0, 100, 200)):
        self._paint_vehicle(_Cv2Canvas(frame), x, y, scale, color)
        return frame

    def _paint_frame_with_vehicles(self, cv):
        """One frame of the stream through ``cv`` (host image or recorded list); advances ``frame_count``."""
        w, h = self.width, self.height
        self._paint_road(cv)
        # The reference reseeds NumPy's legacy global RNG every frame; a private RandomState
        # with the same seed yields the same draws without clobbering global state.
        rs = np.random.RandomState(self.frame_count % 100)
        for i in range(rs.randint(2, 5)):
            t = rs.uniform(0.2, 0.9)
            y = int(h // 2 + (h // 2) * t)
            lane = rs.choice([-80, 0, 80])
            x = w // 2 + int(lane * t) + rs.randint(-20, 20)
            x += int(30 * np.sin(self.frame_count * 0.05 + i))
            self._paint_vehicle(cv, x, y, 0.3 + 0.7 * t, _VEHICLE_COLORS[i % 4])
        self.frame_count += 1

    def generate_frame_with_vehicles(self) -> np.ndarray:
        frame = np.zeros((self.height, self.width, 3), dtype=np.uint8)
        self._paint_frame_with_vehicles(_Cv2Canvas(frame))
        return frame

    def generate_video_stream(self, num_frames: int = 300) -> Iterator[np.ndarray]:
        self.frame_count = 0
        for _ in range(num_frames):
            yield self.generate_frame_with_vehicles()

    def reset(self):
        self.frame_count = 0

    # ------------------------------------------------------------------ batched forms (new)
    def generate_batch(self, num_frames: int, start_frame: Optional[int] = None,
                       out: Optional[np.ndarray] = None) -> np.ndarray:
        """``uint8[num_frames,H,W,3]`` of consecutive frames (optionally from ``start_frame``)."""
        if start_frame is not None:
            self.frame_count = start_frame
        if out is None:
            out = np.empty((num_frames, self.height, self.width, 3), np.uint8)
        for i in range(num_frames):
            out[i] = self.generate_frame_with_vehicles()
        return out


    def generate_batch_device(self, num_frames: int, start_frame: Optional[int] = None, device=None, out=None,
                              return_ms: bool = False, recorded: bool = False):
        """The same ``num_frames`` consecutive frames as :meth:`generate_batch`, rasterised ON THE GPU into a
        ``uint8[num_frames, H, W, 3]`` CUDA tensor, bit-identical to the host frames (SURVEY.md 8f rank 4: no CPU
        rasterisation and no 6 MB-per-frame upload in a benchmark's set-up).  ``lane_generate_frames`` lays the scene out
        in the library's C++ host code (NumPy's legacy ``RandomState`` draws included) and ``k7_draw`` draws it;
        ``recorded=True`` records the scene with this class's own Python code into a ``DrawList`` instead (the two must
        agree; tests compare both with the cv2 generator).  There is no CPU fallback."""
        import ctypes as C
        import torch
        from .. import _native
        if start_frame is not None:
            self.frame_count = start_frame
        dev = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
        if out is None:
            out = torch.empty((num_frames, self.height, self.width, 3), dtype=torch.uint8, device=dev)
        elif tuple(out.shape) != (num_frames, self.height, self.width, 3) or out.dtype != torch.uint8 or not out.is_cuda \
                or not out.is_contiguous():
            raise ValueError("out must be a contiguous CUDA uint8 tensor [num_frames, H, W, 3]")
        if recorded:
            from ..visualization.draw_list import DrawList
            out.zero_()
            dl = DrawList(num_frames)
            for i in range(num_frames):
                self._paint_frame_with_vehicles(_ListCanvas(dl, i))
            with torch.cuda.device(out.device):
                return dl.execute(out, return_ms=return_ms)
        lib = _native.lib()
        ms = C.c_float(0.0)
        with torch.cuda.device(out.device):
            stream = torch.cuda.current_stream(out.device).cuda_stream
            rc = lib.lane_generate_frames(C.c_void_p(out.data_ptr()), 1, num_frames, self.height, self.width,
                                          int(self.frame_count), out.device.index, C.c_void_p(stream), C.byref(ms))
        _native.check_global(rc)
        self.frame_count += num_frames
        return (out, ms.value) if return_ms else out


def multi_camera_batch(num_streams: int, frames_per_stream: int, width: int = 1920, height: int = 1080,
                       phase: int = 1000, period: Optional[int] = None) -> np.ndarray:
    """``uint8[S,T,H,W,3]``: camera ``s`` is the scene generator started at ``frame_count = s*phase``.

    ``period`` (optional) generates only that many distinct frames per stream and tiles them in
    time -- for benchmarks whose input only has to be synthetic and larger than L2, not unique.
    """
    out = np.empty((num_streams, frames_per_stream, height, width, 3), np.uint8)
    distinct = frames_per_stream if period is None else min(period, frames_per_stream)
    for s in range(num_streams):
        gen = SyntheticDataGenerator(width, height)
        gen.generate_batch(distinct, start_frame=s * phase, out=out[s, :distinct])
        for t in range(distinct, frames_per_stream):
            out[s, t] = out[s, t % distinct]
    return out
