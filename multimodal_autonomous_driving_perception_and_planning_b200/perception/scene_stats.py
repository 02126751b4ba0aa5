"""Image statistics of the reference's SceneClassifier, batched on the GPU (SURVEY.md section 8f, rank 2).

Mirror of the pixel work in ``/root/reference/src/tagging/scene_classifier.py``:

* ``_analyze_conditions`` (:237-257): ``avg_brightness = np.mean(cvtColor(frame, BGR2GRAY))`` and
  ``laplacian_var = cv2.Laplacian(gray, cv2.CV_64F).var()``;
* ``_classify_road_type`` (:183-186): ``green_ratio`` of ``cv2.inRange(cvtColor(frame, BGR2HSV), (35,40,40), (85,255,255))``.

The device (kernel K6, ``lane_frame_stats``) returns exact integer sums per frame; the float64 quantities are formed
here from those integers, so ``avg_brightness`` and ``green_ratio`` are bit-identical to the reference expressions and
``laplacian_var`` agrees with numpy's two-pass variance to rounding (1e-12 relative in the tests).
There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import List, Optional

import numpy as np

from .. import _native


class _FrameStat(C.Structure):          # mirrors lane_frame_stat in include/lane_b200.h
    _fields_ = [("sum_gray", C.c_uint64), ("sum_laplacian", C.c_int64), ("sum_laplacian_sq", C.c_uint64),
                ("green_pixels", C.c_uint64)]


@dataclass
class SceneStats:
    avg_brightness: float        # scene_classifier.py:238
    laplacian_var: float         # :254
    green_ratio: float           # :186
    sum_gray: int
    sum_laplacian: int
    sum_laplacian_sq: int
    green_pixels: int

    @property
    def is_night(self) -> bool:                 # :240
        return self.avg_brightness < 60

    @property
    def is_day(self) -> bool:                   # :242
        return self.avg_brightness > 120

    @property
    def low_contrast(self) -> bool:             # :255  (fog / rain hint)
        return self.laplacian_var < 100

    @property
    def looks_residential(self) -> bool:        # :187
        return self.green_ratio > 0.15


class SceneStatsAnalyzer:
    def __init__(self, *, device: Optional[int] = None):
        self._device = device

    def analyze_batch(self, frames) -> List[SceneStats]:
        """frames: uint8 ``[N,H,W,3]`` BGR, numpy (host) or a CUDA torch tensor.  One entry per frame."""
        shape = tuple(frames.shape)
        if len(shape) != 4 or shape[-1] != 3 or str(frames.dtype).replace("torch.", "") != "uint8":
            raise ValueError("frames must be uint8 [N,H,W,3]")
        n, h, w = shape[:3]
        out = (_FrameStat * n)()
        lib = _native.lib()
        if isinstance(frames, np.ndarray):
            src = np.ascontiguousarray(frames)
            dev = self._device
            if dev is None:
                import torch
                dev = torch.cuda.current_device()
            rc = lib.lane_frame_stats(src.ctypes.data_as(C.c_void_p), 0, n, h, w, out, int(dev), None)
        else:
            import torch
            src = frames.contiguous()
            stream = torch.cuda.current_stream(src.device).cuda_stream
            rc = lib.lane_frame_stats(C.c_void_p(src.data_ptr()), 1, n, h, w, out, src.device.index, C.c_void_p(stream))
        _native.check_global(rc)
        px = h * w
        res = []
        for s in out:
            sg, s1, s2, gp = int(s.sum_gray), int(s.sum_laplacian), int(s.sum_laplacian_sq), int(s.green_pixels)
            res.append(SceneStats(sg / px, (s2 * px - s1 * s1) / (px * px), gp / px, sg, s1, s2, gp))
        return res
