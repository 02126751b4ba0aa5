"""Annotated frames -> a video encoder's input: batched BGR -> I420 / NV12, bit-exact with
``cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420)``.

Every encoder takes 4:2:0 input: libx264 through an FFmpeg pipe with ``-pix_fmt yuv420p`` (I420), PyAV, or a hardware
encoder's NV12 surface.  Frames annotated on the device (``LaneDetector.draw_lanes_batch``,
``OverlayRenderer.draw_lane_offset_indicator_batch``) are converted where they are, by the K8 kernel, and only the
1.5 B/px result leaves HBM -- half the bytes of the BGR frame.  Encoding itself stays with the encoder.

NV12 here is cv2's I420 with U and V interleaved (cv2 has no BGR -> NV12 code).

There is no CPU fallback for CUDA tensors: without the CUDA library / a GPU the calls raise.  Host (numpy) frames are
converted by cv2 on the host, as before.
"""
import ctypes as C

import cv2
import numpy as np

from .. import _native


def bgr_to_i420(frames, out=None):
    """``uint8[N,H,W,3]`` BGR frames -> ``uint8[N,H*3/2,W]`` I420 (Y plane, then U, then V, each chroma plane
    ``H/2 x W/2``), equal to ``cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420)`` per frame; H and W must be even.

    numpy (or CPU tensor) in: converted on the host with cv2, ``ValueError`` for odd sizes; ``out`` (optional) is a
    numpy array of the output shape.
    CUDA tensor in: converted on the device, enqueued on torch's current stream.  Without ``out`` it returns a CUDA
    tensor (no synchronisation).  ``out`` may be a CUDA tensor, a host numpy array or a CPU tensor (pinned or not) of
    the output shape; it is filled and returned, and for host memory the call returns when the bytes are there.  Bad
    shapes, dtypes and odd sizes raise ``cv2.error`` before any native call."""
    return _convert(frames, out, _native.INPUT_I420, "bgr_to_i420")


def bgr_to_nv12(frames, out=None):
    """``uint8[N,H,W,3]`` BGR frames -> ``uint8[N,H*3/2,W]`` in the NV12 layout (Y plane followed by the interleaved
    half-resolution UV plane): the samples of :func:`bgr_to_i420`.  Also makes decoder-shaped inputs for
    ``LaneDetector.detect_batch_nv12`` / ``FrameIngest.from_nv12`` out of the synthetic frames.  Inputs, ``out`` and
    errors as for :func:`bgr_to_i420`."""
    return _convert(frames, out, _native.INPUT_NV12, "bgr_to_nv12")


def _is_torch(x) -> bool:
    return type(x).__module__.split(".")[0] == "torch"


def _convert(frames, out, fmt, who):
    if _is_torch(frames) and frames.device.type != "cpu":
        return _device(frames, out, fmt, who)
    return _host(frames, out, fmt)


def _host(frames, out, fmt):
    frames = np.asarray(frames)
    n, h, w = frames.shape[:3]
    if h % 2 or w % 2:
        raise ValueError(("NV12" if fmt == _native.INPUT_NV12 else "I420") + " needs even width and height")
    shape = (n, h * 3 // 2, w)
    if out is None:
        out = np.empty(shape, np.uint8)
    elif not isinstance(out, np.ndarray) or out.shape != shape or out.dtype != np.uint8:
        raise ValueError(f"out must be a uint8 numpy array of shape {shape}")
    for i in range(n):
        i420 = cv2.cvtColor(frames[i], cv2.COLOR_BGR2YUV_I420)
        if fmt == _native.INPUT_I420:
            out[i] = i420
            continue
        out[i, :h] = i420[:h]
        u = i420[h:h + h // 4].reshape(h // 2, w // 2)
        v = i420[h + h // 4:].reshape(h // 2, w // 2)
        out[i, h:] = np.stack([u, v], axis=-1).reshape(h // 2, w)
    return out


def check_bgr(frames, who: str):
    """uint8 ``[N, H, W, 3]`` with even, positive H and W, else ``cv2.error`` (what cv2.cvtColor raises)."""
    shape = tuple(frames.shape)
    if len(shape) != 4 or shape[3] != 3:
        raise cv2.error(f"{who}: expected BGR frames [N, H, W, 3], got {shape}")
    if str(frames.dtype).replace("torch.", "") != "uint8":
        raise cv2.error(f"{who}: expected uint8 frames, got {frames.dtype}")
    if shape[1] < 2 or shape[2] < 2 or shape[1] % 2 or shape[2] % 2:
        raise cv2.error(f"{who}: YUV 4:2:0 needs even, positive width and height, got {shape}")


def _check_out(out, shape, frames, who):
    if isinstance(out, np.ndarray):
        ok = out.shape == shape and out.dtype == np.uint8 and out.flags.c_contiguous and out.flags.writeable
    elif _is_torch(out):
        import torch
        ok = (tuple(out.shape) == shape and out.dtype == torch.uint8 and out.is_contiguous()
              and out.device.type in ("cpu", frames.device.type) and (out.device.type == "cpu" or out.device == frames.device))
    else:
        ok = False
    if not ok:
        raise cv2.error(f"{who}: out must be a contiguous uint8 array / tensor of shape {shape} in host memory or on "
                        f"the frames' device")


def _device(frames, out, fmt, who):
    import torch
    check_bgr(frames, who)
    n, h, w = (int(s) for s in frames.shape[:3])
    shape = (n, h * 3 // 2, w)
    if out is not None:
        _check_out(out, shape, frames, who)
    if not frames.is_cuda:
        raise cv2.error(f"{who}: torch input must be a CUDA tensor (pass numpy for host frames)")
    src = frames.contiguous()
    if out is None:
        out = torch.empty(shape, dtype=torch.uint8, device=src.device)
    if n == 0:
        return out
    on_device = _is_torch(out) and out.is_cuda
    dst = out.ctypes.data if isinstance(out, np.ndarray) else out.data_ptr()
    lib = _native.lib()
    stream = torch.cuda.current_stream(src.device).cuda_stream
    rc = lib.lane_bgr_to_yuv420_batch(C.c_void_p(src.data_ptr()), fmt, n, h, w, C.c_void_p(dst), int(on_device),
                                      src.device.index, C.c_void_p(stream))
    _native.check_global(rc)
    return out
