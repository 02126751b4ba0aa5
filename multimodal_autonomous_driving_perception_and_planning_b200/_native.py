"""ctypes binding of ``csrc/liblane_b200.so`` (the C ABI declared in ``include/lane_b200.h``).

There is no CPU fallback: if the shared library is missing or no sm_100 device is visible the
calls raise.  Build the library with ``python __graft_entry__.py`` / ``make -C .../csrc``.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
# LANE_B200_LIB: an alternative build of the same library (A/B timing of kernel variants); never a CPU path
LIB_PATH = os.environ.get("LANE_B200_LIB") or os.path.join(CSRC, "liblane_b200.so")

NUM_POINTS = 50
NUM_STAGES = 7
STAGE_NAMES = ("h2d", "blur_hist", "canny", "compact", "ppht", "fit", "d2h")
TAP_BLUR, TAP_HIST, TAP_CLASS, TAP_EDGES, TAP_POINTS, TAP_SEGMENTS, TAP_GRAY, TAP_FRAME = 1, 2, 3, 4, 5, 6, 7, 8
FLAG_SEGMENTS_TRUNCATED, FLAG_POINTS_TRUNCATED = 1, 2
PATH_FUSED_EDGE, PATH_CLUSTER_CANNY, PATH_PPHT_DSMEM = 1, 2, 4
PATH_ALL_FAST = 7
INPUT_BGR, INPUT_NV12, INPUT_I420 = 0, 1, 2          # LANE_INPUT_*: frame layouts the detect / ingest calls accept
#                                                     (and NV12 / I420: what lane_bgr_to_yuv420_batch writes)
# raw 8-bit Bayer mosaics [n][h][w], named by the sensor's top-left 2x2 (cv2.COLOR_Bayer<P>2BGR)
INPUT_BAYER_RGGB, INPUT_BAYER_BGGR, INPUT_BAYER_GRBG, INPUT_BAYER_GBRG = 16, 17, 18, 19
BAYER = {"rggb": INPUT_BAYER_RGGB, "bggr": INPUT_BAYER_BGGR, "grbg": INPUT_BAYER_GRBG, "gbrg": INPUT_BAYER_GBRG}
# packed YUV 4:2:2 camera frames [n][h][w][2], w even: UYVY (U Y0 V Y1, GMSL / FPD-Link) and YUYV (Y0 U Y1 V, V4L2)
INPUT_UYVY, INPUT_YUYV = 8, 9
YUV422 = {"uyvy": INPUT_UYVY, "yuyv": INPUT_YUYV}


class LaneSide(C.Structure):
    _fields_ = [("valid", C.c_int32), ("n_lines", C.c_int32), ("raw", C.c_double * 3),
                ("coeffs", C.c_double * 3), ("confidence", C.c_double),
                ("points", (C.c_int32 * 2) * NUM_POINTS)]


class LaneRecord(C.Structure):
    _fields_ = [("side", LaneSide * 2), ("offset", C.c_double), ("offset_valid", C.c_int32),
                ("median_x2", C.c_int32), ("low", C.c_int32), ("high", C.c_int32), ("n_edges", C.c_int32),
                ("n_roi_points", C.c_int32), ("n_segments", C.c_int32), ("hysteresis_rounds", C.c_int32),
                ("flags", C.c_int32), ("n_segments_found", C.c_int32)]


class LaneRigSource(C.Structure):
    """lane_rig_source: one camera of a lane_detect_rig call."""
    _fields_ = [("frames", C.c_void_p), ("format", C.c_int32), ("src_h", C.c_int32), ("src_w", C.c_int32),
                ("n", C.c_int32), ("stream_id", C.c_int32)]


# numpy view of lane_record (same layout) so batches decode without a Python loop per field
SIDE_DTYPE = np.dtype([("valid", "<i4"), ("n_lines", "<i4"), ("raw", "<f8", (3,)), ("coeffs", "<f8", (3,)),
                       ("confidence", "<f8"), ("points", "<i4", (NUM_POINTS, 2))], align=True)
RECORD_DTYPE = np.dtype([("side", SIDE_DTYPE, (2,)), ("offset", "<f8"), ("offset_valid", "<i4"),
                         ("median_x2", "<i4"), ("low", "<i4"), ("high", "<i4"), ("n_edges", "<i4"),
                         ("n_roi_points", "<i4"), ("n_segments", "<i4"), ("hysteresis_rounds", "<i4"),
                         ("flags", "<i4"), ("n_segments_found", "<i4")], align=True)
assert RECORD_DTYPE.itemsize == C.sizeof(LaneRecord), (RECORD_DTYPE.itemsize, C.sizeof(LaneRecord))


class LaneError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"lane_b200 error {code}: {msg}")
        self.code = code


def check_global(rc: int) -> None:
    """Raise LaneError for a non-zero code from a call that reports through lane_last_error(NULL): context creation
    and the context-free entry points."""
    if rc:
        raise LaneError(rc, (lib().lane_last_error(None) or b"").decode())


def build(verbose: bool = False) -> str:
    """Compile the CUDA sources for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    out = subprocess.run(["make", "-C", CSRC, "-j8"], capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("building liblane_b200.so failed:\n" + out.stdout[-4000:] + out.stderr[-4000:])
    if verbose:
        print(out.stdout[-2000:])
    return LIB_PATH


_lib = None

_PROTOS = {
    "lane_frame_stats": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "lane_resize_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_void_p]),
    "lane_abi_version": (C.c_int, []),
    "lane_last_error": (C.c_char_p, [C.c_void_p]),
    "lane_ctx_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "lane_ctx_destroy": (None, [C.c_void_p]),
    "lane_set_roi_mask": (C.c_int, [C.c_void_p, C.c_void_p]),
    "lane_set_roi_masks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "lane_set_threshold_lut": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "lane_set_hough_params": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "lane_set_smoothing": (C.c_int, [C.c_void_p, C.c_double, C.c_double]),
    "lane_set_debug": (C.c_int, [C.c_void_p, C.c_int]),
    "lane_set_preprocess": (C.c_int, [C.c_void_p, C.c_int]),
    "lane_detect_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                    C.c_void_p, C.c_void_p]),
    "lane_detect_batch_nv12": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    "lane_detect_batch_ingest": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                           C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lane_detect_rig": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lane_nv12_to_bgr_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "lane_yuv420_to_bgr_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                           C.c_int, C.c_int, C.c_void_p]),
    "lane_bayer_to_bgr_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                          C.c_int, C.c_int, C.c_void_p]),
    "lane_yuv422_to_bgr_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                           C.c_int, C.c_int, C.c_void_p]),
    "lane_bgr_to_yuv420_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                           C.c_void_p]),
    "lane_detect_enqueue": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "lane_detect_collect": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "lane_rig_enqueue": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "lane_ctx_stream": (C.c_void_p, [C.c_void_p]),
    "lane_ctx_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "lane_ctx_records_device": (C.c_void_p, [C.c_void_p]),
    "lane_ctx_fence_records": (C.c_int, [C.c_void_p, C.c_void_p]),
    "lane_ctx_last_paths": (C.c_int, [C.c_void_p]),
    "lane_set_profiling": (C.c_int, [C.c_void_p, C.c_int]),
    "lane_get_stage_ms": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "lane_debug_tap": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "lane_edge_count_rect": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "lane_hough_lines_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.POINTER(C.c_float)]),
    "lane_draw_commands": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                     C.c_void_p, C.POINTER(C.c_float)]),
    "lane_generate_frames": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p,
                                       C.POINTER(C.c_float)]),
    "lane_draw_lanes_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_float)]),
    "lane_draw_lanes_records": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "lane_hough_accumulator": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                         C.POINTER(C.c_int)]),
}


def lib() -> C.CDLL:
    """Load the shared library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: the CUDA extension must be built first "
                "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def exported_symbols():
    return sorted(_PROTOS)


def threshold_lut():
    """low/high for every 2*median in 0..510, evaluated with the reference's own expressions
    (/root/reference/src/perception/lane_detector.py:80-81) in Python float64."""
    low = np.empty(511, np.uint8)
    high = np.empty(511, np.uint8)
    for k in range(511):
        median = np.float64(k) / 2.0
        low[k] = int(max(0, 0.7 * median))
        high[k] = int(min(255, 1.3 * median))
    return low, high


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _rig_sources(sources, on_device: bool):
    """The lane_rig_source array of ``LaneContext.detect_rig``'s ``sources``, and their total frame count."""
    arr = (LaneRigSource * max(len(sources), 1))()
    total = 0
    for i, (frames, fmt, (h, w), n, sid) in enumerate(sources):
        fp = frames if on_device else (frames.ctypes.data if n else None)
        arr[i] = LaneRigSource(fp, int(fmt), int(h), int(w), int(n), int(sid))
        total += int(n)
    return arr, total


class LaneContext:
    """One native context: fixed (H, W), up to max_batch frames per call, one CUDA stream.

    ``roi_mask`` is uint8 ``(H, W)``, or ``(R, H, W)`` for one mask per camera stream: mask r is stream r's, and every
    call then takes at most R streams (see lane_set_roi_masks)."""

    def __init__(self, height: int, width: int, max_batch: int, roi_mask: np.ndarray, device: int = 0,
                 max_segments: int = 256, debug: bool = False):
        self._h = None
        L = lib()
        h = C.c_void_p()
        check_global(L.lane_ctx_create(device, height, width, max_batch, max_segments, C.byref(h)))
        self._h = h
        self.height, self.width, self.max_batch, self.device = height, width, max_batch, device
        self.max_segments = max_segments
        if debug:
            self._check(L.lane_set_debug(self._h, 1))
        self.debug = debug
        mask = np.ascontiguousarray(roi_mask, dtype=np.uint8)
        if mask.ndim == 3 and mask.shape[0] >= 1 and mask.shape[1:] == (height, width):
            self._check(L.lane_set_roi_masks(self._h, _ptr(mask), mask.shape[0]))
        elif mask.shape == (height, width):
            self._check(L.lane_set_roi_mask(self._h, _ptr(mask)))
        else:
            raise ValueError(f"roi mask shape {mask.shape} is neither {(height, width)} nor (R, {height}, {width})")
        self.n_roi = mask.shape[0] if mask.ndim == 3 else 1
        low, high = threshold_lut()
        self._check(L.lane_set_threshold_lut(self._h, _ptr(low), _ptr(high)))
        self.settings = {"hough": (50, 50, 150), "lut": (low, high), "blur": True}   # what copy_settings_to replays
        self._records = np.zeros(max_batch, RECORD_DTYPE)
        self._inflight = []                       # sizes of the batches in flight, oldest first

    def _check(self, rc):
        if rc != 0:
            raise LaneError(rc, (lib().lane_last_error(self._h) or b"").decode())

    def close(self):
        if self._h is not None and _lib is not None:
            _lib.lane_ctx_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- configuration
    def set_hough_params(self, threshold=50, min_line_length=50, max_line_gap=150):
        self._check(lib().lane_set_hough_params(self._h, int(threshold), int(round(min_line_length)),
                                                int(round(max_line_gap))))
        self.settings["hough"] = (int(threshold), int(round(min_line_length)), int(round(max_line_gap)))

    def set_preprocess(self, gaussian_blur: bool):
        """False: skip the 5x5 blur, Canny runs on the plain grayscale plane (scene_classifier.py:145-146)."""
        self._check(lib().lane_set_preprocess(self._h, int(gaussian_blur)))
        self.settings["blur"] = bool(gaussian_blur)

    def set_threshold_lut(self, low511: np.ndarray, high511: np.ndarray):
        low = np.ascontiguousarray(low511, dtype=np.uint8)
        high = np.ascontiguousarray(high511, dtype=np.uint8)
        if low.shape != (511,) or high.shape != (511,):
            raise ValueError("threshold LUTs must have 511 entries (one per 2*median)")
        self._check(lib().lane_set_threshold_lut(self._h, _ptr(low), _ptr(high)))
        self.settings["lut"] = (low, high)

    def copy_settings_to(self, other: "LaneContext"):
        """Replay this context's Hough literals, threshold LUT and preprocess mode on another context."""
        other.set_hough_params(*self.settings["hough"])
        other.set_threshold_lut(*self.settings["lut"])
        other.set_preprocess(self.settings["blur"])

    def set_profiling(self, on: bool):
        self._check(lib().lane_set_profiling(self._h, int(on)))

    def stream(self) -> int:
        return int(lib().lane_ctx_stream(self._h) or 0)

    def last_paths(self) -> int:
        """PATH_* bits of the kernels the last batch ran on (PATH_ALL_FAST when nothing fell back)."""
        return int(lib().lane_ctx_last_paths(self._h))

    def records_device_ptr(self) -> int:
        """Device address of the records of the batch enqueued last (see lane_ctx_records_device)."""
        return int(lib().lane_ctx_records_device(self._h) or 0)

    def fence_records(self, reader_stream: int):
        """Work already enqueued on ``reader_stream`` (a cudaStream_t value) reads ``records_device_ptr()`` of the batch
        collected last; the kernel that next writes that result slot waits for it (see lane_ctx_fence_records)."""
        self._check(lib().lane_ctx_fence_records(self._h, C.c_void_p(reader_stream)))

    # ---- hot path
    def detect(self, frames, n: int, on_device: bool, stream_id, n_streams: int, prev_fit: np.ndarray,
               prev_valid: np.ndarray, smoothing: float, one_minus: float, fmt: int = INPUT_BGR,
               src_hw=None) -> np.ndarray:
        """frames: int device pointer (on_device) or C-contiguous uint8 ndarray in layout ``fmt`` (INPUT_*) at size
        ``src_hw`` = (h, w) (None: the context's) -- BGR [n,h,w,3], the decoder layouts [n,h*3/2,w], Bayer [n,h,w] or
        YUV 4:2:2 [n,h,w,2].  Frames of another layout or size become the context's BGR frames on the device first
        (lane_detect_batch_ingest).
        prev_fit float64[S,2,3] and prev_valid uint8[S,2] are updated in place.  Returns a RECORD_DTYPE array of n
        records (a copy)."""
        L = lib()
        self._check(L.lane_set_smoothing(self._h, float(smoothing), float(one_minus)))
        fp = C.c_void_p(frames) if on_device else _ptr(frames)
        sid = None if stream_id is None else np.ascontiguousarray(stream_id, dtype=np.int32)
        sh, sw = (self.height, self.width) if src_hw is None else (int(src_hw[0]), int(src_hw[1]))
        self._check(L.lane_detect_batch_ingest(self._h, fp, int(on_device), n, int(fmt), sh, sw, _ptr(sid), n_streams,
                                               _ptr(prev_fit), _ptr(prev_valid), _ptr(self._records)))
        return self._records[:n].copy()

    def detect_rig(self, sources, on_device: bool, n_streams: int, prev_fit: np.ndarray, prev_valid: np.ndarray,
                   smoothing: float, one_minus: float) -> np.ndarray:
        """One call for cameras of different sizes and layouts (lane_detect_rig).  ``sources``: one tuple
        ``(frames, fmt, (h, w), n, stream_id)`` per camera, ``frames`` an int device pointer (on_device) or a C-contiguous
        uint8 ndarray of ``n`` frames in layout ``fmt`` (INPUT_*) at size (h, w).  State arrays as for ``detect``.
        Returns the records of all frames in source order (a copy)."""
        L = lib()
        self._check(L.lane_set_smoothing(self._h, float(smoothing), float(one_minus)))
        arr, total = _rig_sources(sources, on_device)
        self._check(L.lane_detect_rig(self._h, arr, len(sources), int(on_device), n_streams, _ptr(prev_fit),
                                      _ptr(prev_valid), _ptr(self._records)))
        return self._records[:total].copy()

    def enqueue_rig(self, sources, on_device: bool, n_streams: int, prev_fit, prev_valid, smoothing, one_minus):
        """Asynchronous ``detect_rig`` (lane_rig_enqueue): ``sources`` as there, host frames in page-locked memory, and
        the state rules of ``enqueue``.  ``collect`` returns the tick's records in source order.  The frames must stay
        alive and unchanged until then."""
        L = lib()
        self._check(L.lane_set_smoothing(self._h, float(smoothing), float(one_minus)))
        arr, total = _rig_sources(sources, on_device)
        self._check(L.lane_rig_enqueue(self._h, arr, len(sources), int(on_device), n_streams, _ptr(prev_fit),
                                       _ptr(prev_valid)))
        self._inflight.append(total)

    def enqueue(self, frames_ptr: int, n: int, stream_id, n_streams, prev_fit, prev_valid, smoothing, one_minus):
        """Asynchronous form for device-resident frames.  With ``prev_fit`` / ``prev_valid`` the batch starts from that
        state (one batch in flight).  With both ``None`` it continues from the state the previous batch left on the
        device, and a second batch may be queued behind the first (enqueue, enqueue, collect, enqueue, collect, ...):
        the device then never waits for the host between batches."""
        L = lib()
        self._check(L.lane_set_smoothing(self._h, float(smoothing), float(one_minus)))
        sid = None if stream_id is None else np.ascontiguousarray(stream_id, dtype=np.int32)
        self._check(L.lane_detect_enqueue(self._h, C.c_void_p(frames_ptr), n, _ptr(sid), n_streams,
                                          _ptr(prev_fit), _ptr(prev_valid)))
        self._inflight.append(n)

    def collect(self, prev_fit, prev_valid) -> np.ndarray:
        """Waits for the oldest batch in flight; ``prev_fit`` / ``prev_valid`` receive the state after it."""
        self._check(lib().lane_detect_collect(self._h, _ptr(prev_fit), _ptr(prev_valid), _ptr(self._records)))
        return self._records[:self._inflight.pop(0)].copy()

    def stage_ms(self):
        ms = np.zeros(NUM_STAGES, np.float32)
        launches = np.zeros(NUM_STAGES, np.int32)
        self._check(lib().lane_get_stage_ms(self._h, _ptr(ms), _ptr(launches)))
        return dict(zip(STAGE_NAMES, ms.tolist())), dict(zip(STAGE_NAMES, launches.tolist()))

    # ---- verification taps
    def tap(self, what: int, frame_index: int) -> np.ndarray:
        h, w = self.height, self.width
        if what in (TAP_BLUR, TAP_CLASS, TAP_EDGES, TAP_GRAY):
            out = np.empty((h, w), np.uint8)
        elif what == TAP_FRAME:
            out = np.empty((h, w, 3), np.uint8)
        elif what == TAP_HIST:
            out = np.empty(256, np.uint32)
        elif what == TAP_POINTS:
            out = np.empty((max(int(self._records[frame_index]["n_roi_points"]), 1), 2), np.int32)
        elif what == TAP_SEGMENTS:
            out = np.empty((self.max_segments, 4), np.int32)
        else:
            raise ValueError(what)
        written = C.c_size_t(0)
        self._check(lib().lane_debug_tap(self._h, what, frame_index, _ptr(out), out.nbytes, C.byref(written)))
        if what in (TAP_POINTS, TAP_SEGMENTS):
            rows = written.value // (out.shape[1] * 4)
            return out[:rows].copy()
        return out

    def edge_count_rect(self, n: int, x0: int, y0: int, x1: int, y1: int) -> np.ndarray:
        """Edge pixels inside [x0,x1) x [y0,y1) of each of the ``n`` frames of the last batch (device popcount)."""
        out = np.zeros(n, np.int32)
        self._check(lib().lane_edge_count_rect(self._h, int(x0), int(y0), int(x1), int(y1), _ptr(out)))
        return out

    def hough_lines_batch(self, n: int, threshold: int = 50, max_peaks: int = 256, with_accum: bool = False):
        """Standard Hough transform (what ``cv2.HoughLines(masked, 1, pi/180, threshold)`` computes) of all ``n`` frames
        of the last batch.  Returns ``(peaks, counts, accum, ms)``: ``peaks[i]`` = int32 rows (rho_index, angle_index,
        votes) of frame i in cv2 order, ``counts[i]`` = peaks found, ``accum`` = int32 [n, 182, 2(W+H)+3] or None,
        ``ms`` = device time of the batch."""
        numrho = 2 * (self.width + self.height) + 1
        peaks = np.zeros((n, max_peaks, 3), np.int32)
        counts = np.zeros(n, np.int32)
        acc = np.empty((n, 182, numrho + 2), np.int32) if with_accum else None
        ms = C.c_float(0)
        self._check(lib().lane_hough_lines_batch(self._h, int(threshold), int(max_peaks), _ptr(peaks), _ptr(counts),
                                                 _ptr(acc), C.byref(ms)))
        return [peaks[i, :min(int(counts[i]), max_peaks)].copy() for i in range(n)], counts, acc, float(ms.value)

    def hough_accumulator(self, frame_index: int, threshold: int = 0, max_peaks: int = 0):
        """Standard-Hough accumulator int32[182][2(W+H)+3] of the ROI-masked edges of one frame of the
        last batch, plus (optionally) its peaks as rows (rho_index, angle_index, votes) in cv2 order."""
        numrho = 2 * (self.width + self.height) + 1
        acc = np.empty((182, numrho + 2), np.int32)
        peaks = np.empty((max(max_peaks, 1), 3), np.int32)
        found = C.c_int(0)
        self._check(lib().lane_hough_accumulator(self._h, frame_index, _ptr(acc), threshold,
                                                 _ptr(peaks) if max_peaks else None, max_peaks, C.byref(found)))
        return acc, peaks[:min(found.value, max_peaks)].copy(), found.value
