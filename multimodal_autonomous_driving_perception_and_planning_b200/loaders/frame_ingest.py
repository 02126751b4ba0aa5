"""Batched frame ingest on the GPU: the resize step of the reference's ``VideoDataLoader``.

``VideoDataLoader.read_frame`` / ``read_frame_at`` (/root/reference/data/loaders/video_loader.py:96-131) decode a
frame with ``cv2.VideoCapture`` and, when ``target_size`` is set, run ``cv2.resize(frame, self.target_size)``
(:108, :128).  Decoding stays where it is (codec I/O is out of scope); ``FrameIngest`` takes the decoded frames of a
batch and produces exactly what those ``cv2.resize`` calls produce, on the device, so the result can go straight
into ``LaneDetector.detect_batch`` as a CUDA tensor without a second trip over PCIe.

There is no CPU fallback: without the CUDA library / a GPU the calls raise.
"""
import ctypes as C
from typing import Optional, Tuple

import cv2
import numpy as np

from .. import _native


class FrameIngest:
    """``target_size`` = (width, height) as in ``VideoDataLoader(video_path, target_size=...)``; ``None`` = no resize."""

    def __init__(self, target_size: Optional[Tuple[int, int]] = None, *, device: Optional[int] = None):
        self.target_size = None if target_size is None else (int(target_size[0]), int(target_size[1]))
        self._device = device

    def _device_index(self) -> int:
        if self._device is not None:
            return int(self._device)
        import torch
        return int(torch.cuda.current_device())

    @staticmethod
    def _check(frames):
        shape = tuple(frames.shape)
        if len(shape) not in (3, 4) or (len(shape) == 4 and shape[-1] not in (1, 3)):
            raise cv2.error(f"FrameIngest: expected uint8 frames [N,H,W,3], [N,H,W,1] or [N,H,W], got {shape}")
        if str(frames.dtype).replace("torch.", "") != "uint8":
            raise cv2.error(f"FrameIngest: expected uint8 frames, got {frames.dtype}")

    def resize_batch(self, frames):
        """frames: uint8 ``[N,H,W,C]`` (C = 1 or 3) or ``[N,H,W]``, numpy (host) or a CUDA torch tensor.
        numpy in -> numpy out (copies inside the call); CUDA tensor in -> CUDA tensor out, enqueued on torch's
        current stream without synchronising.  Equal to ``np.stack([cv2.resize(f, target_size) for f in frames])``."""
        self._check(frames)
        if self.target_size is None:
            return frames
        dw, dh = self.target_size
        n, sh, sw = int(frames.shape[0]), int(frames.shape[1]), int(frames.shape[2])
        cn = int(frames.shape[3]) if len(frames.shape) == 4 else 1
        out_shape = (n, dh, dw) + ((cn,) if len(frames.shape) == 4 else ())
        lib = _native.lib()
        if isinstance(frames, np.ndarray):
            src = np.ascontiguousarray(frames)
            dst = np.empty(out_shape, np.uint8)
            rc = lib.lane_resize_batch(src.ctypes.data_as(C.c_void_p), n, sh, sw, cn, dst.ctypes.data_as(C.c_void_p), dh, dw,
                                       0, self._device_index(), None)
            _native.check_global(rc)
            return dst
        import torch
        if not frames.is_cuda:
            raise cv2.error("FrameIngest: torch input must be a CUDA tensor (pass numpy for host frames)")
        src = frames.contiguous()
        dst = torch.empty(out_shape, dtype=torch.uint8, device=src.device)
        stream = torch.cuda.current_stream(src.device).cuda_stream
        rc = lib.lane_resize_batch(C.c_void_p(src.data_ptr()), n, sh, sw, cn, C.c_void_p(dst.data_ptr()), dh, dw, 1,
                                   src.device.index, C.c_void_p(stream))
        _native.check_global(rc)
        return dst

    def from_nv12(self, frames):
        """Decoder output -> BGR: ``frames`` uint8 ``[N, H*3/2, W]`` in NV12 layout (numpy or CUDA tensor) becomes
        ``[N, H, W, 3]``, equal to ``cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12)`` per frame, followed by the resize when
        ``target_size`` is set (what ``VideoDataLoader.read_frame`` returns for that frame).  With ``target_size`` the
        conversion and the resize are one kernel: the full-resolution BGR frame is never stored."""
        return self._from_yuv420(frames, _native.INPUT_NV12)

    def from_i420(self, frames):
        """``from_nv12`` for the planar layout software decoders hand out (FFmpeg / PyAV ``yuv420p``): uint8
        ``[N, H*3/2, W]`` = Y plane, then the U plane, then the V plane (each ``H/2 x W/2``); equal to
        ``cv2.cvtColor(f, cv2.COLOR_YUV2BGR_I420)`` per frame, resized when ``target_size`` is set."""
        return self._from_yuv420(frames, _native.INPUT_I420)

    def _from_yuv420(self, frames, fmt):
        check_yuv420(frames, "FrameIngest")
        n, h, w = int(frames.shape[0]), int(frames.shape[1]) * 2 // 3, int(frames.shape[2])
        dw, dh = (w, h) if self.target_size is None else self.target_size
        lib = _native.lib()
        if isinstance(frames, np.ndarray):
            src = np.ascontiguousarray(frames)
            dst = np.empty((n, dh, dw, 3), np.uint8)
            rc = lib.lane_yuv420_to_bgr_batch(src.ctypes.data_as(C.c_void_p), fmt, n, h, w, dst.ctypes.data_as(C.c_void_p),
                                              dh, dw, 0, self._device_index(), None)
        else:
            import torch
            if not frames.is_cuda:
                raise cv2.error("FrameIngest: torch input must be a CUDA tensor (pass numpy for host frames)")
            src = frames.contiguous()
            dst = torch.empty((n, dh, dw, 3), dtype=torch.uint8, device=src.device)
            stream = torch.cuda.current_stream(src.device).cuda_stream
            rc = lib.lane_yuv420_to_bgr_batch(C.c_void_p(src.data_ptr()), fmt, n, h, w, C.c_void_p(dst.data_ptr()), dh, dw,
                                              1, src.device.index, C.c_void_p(stream))
        _native.check_global(rc)
        return dst

    def resize(self, frame: np.ndarray) -> np.ndarray:
        """One frame, as ``read_frame`` does it."""
        return self.resize_batch(frame[None])[0]


def check_yuv420(frames, who: str):
    """uint8 ``[N, H*3/2, W]`` with even H and W (NV12 / I420), else ``cv2.error`` (what cv2.cvtColor raises)."""
    shape = tuple(frames.shape)
    if len(shape) != 3 or shape[1] % 3 or shape[2] % 2 or (shape[1] * 2 // 3) % 2:
        raise cv2.error(f"{who}: expected NV12 / I420 frames [N, H*3/2, W] with even H and W, got {shape}")
    if str(frames.dtype).replace("torch.", "") != "uint8":
        raise cv2.error(f"{who}: expected uint8 frames, got {frames.dtype}")


def check_target_size(target_size) -> Tuple[int, int]:
    """``target_size`` as ``cv2.resize`` takes ``dsize``: (width, height), two positive integers, else ``cv2.error``."""
    try:
        w, h = target_size
    except (TypeError, ValueError):
        raise cv2.error(f"target_size must be (width, height), got {target_size!r}") from None
    if not all(isinstance(v, (int, np.integer)) and not isinstance(v, (bool, np.bool_)) for v in (w, h)) or w < 1 or h < 1:
        raise cv2.error(f"target_size must be two positive integers (width, height), got {target_size!r}")
    return int(w), int(h)
