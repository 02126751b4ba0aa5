"""Lane detection behind the reference's ``LaneDetector`` API, computed on a B200.

Mirror of ``/root/reference/src/perception/lane_detector.py``: the same public names, argument
meaning and return types (``LaneLine``, ``LaneDetector.detect / draw_lanes /
get_lane_center_offset / reset``, attributes ``roi_vertices``, ``prev_left_fit``,
``prev_right_fit``, ``smoothing_factor``), plus the new ``detect_batch`` / ``detect_streams``.
Every pixel stage runs in hand-written CUDA (``csrc/``) through the C ABI in
``include/lane_b200.h``; there is no OpenCV on the detection path and no CPU fallback.  cv2 is
used only where the reference's result *is* cv2's rasteriser and does not depend on the frame:
the ROI polygon mask (``cv2.fillPoly``, built once per frame size) and ``draw_lanes``.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import cv2
import numpy as np

from .. import _native
from ..loaders.frame_ingest import check_target_size, check_yuv420


@dataclass
class LaneLine:
    """Represents a detected lane line (reference: lane_detector.py:13-19)."""
    points: np.ndarray  # int32 [50, 2] (x, y)
    side: str  # "left" or "right"
    confidence: float
    polynomial: Optional[np.ndarray] = None  # float64 [3], highest power first


LanePair = Tuple[Optional[LaneLine], Optional[LaneLine]]
_SIDES = ("left", "right")


def _is_torch_cuda(x) -> bool:
    return type(x).__module__.startswith("torch") and hasattr(x, "is_cuda") and bool(x.is_cuda)


class LaneDetector:
    """Edge + Hough lane detector with temporal smoothing (reference: lane_detector.py:22-277).

    ``LaneDetector(roi_vertices=None)`` is the reference signature; the keyword-only extras pick the
    GPU and the largest batch one native call processes (larger batches are chunked).
    """

    def __init__(self, roi_vertices: Optional[np.ndarray] = None, *, device: Optional[int] = None,
                 max_batch: int = 64, max_segments: int = 256, debug: bool = False):
        self.roi_vertices = roi_vertices
        self.prev_left_fit = None
        self.prev_right_fit = None
        self.smoothing_factor = 0.7
        self._device = device
        self._max_batch = int(max_batch)
        self._max_segments = int(max_segments)
        self._debug = bool(debug)
        self._ctx: Optional[_native.LaneContext] = None
        self._ctx_key = None
        self._dense_ctx: Optional[_native.LaneContext] = None   # larger max_segments, for frames the default truncated
        self._dense_key = None
        self._roi_cache = {}        # (h, w, vertex key) -> rasterised ROI mask
        self.dense_reruns = 0       # chunks re-run because HoughLinesP found more segments than max_segments
        self._stream_fit = None     # float64 [S,2,3] for detect_streams
        self._stream_valid = None   # uint8  [S,2]
        self.last_records = None    # RECORD_DTYPE array of the last call (diagnostics)

    # ------------------------------------------------------------------ static inputs
    def _get_roi_mask(self, shape: Tuple[int, int], vertices=None) -> np.ndarray:
        """ROI mask exactly as the reference rasterises it (lane_detector.py:47-64), of ``vertices`` when given, else
        of ``roi_vertices`` or the default trapezoid."""
        h, w = shape[:2]
        if vertices is None:
            vertices = self.roi_vertices
        if vertices is None:
            vertices = np.array([[(int(w * 0.1), h), (int(w * 0.4), int(h * 0.6)),
                                  (int(w * 0.6), int(h * 0.6)), (int(w * 0.9), h)]], dtype=np.int32)
        mask = np.zeros((h, w), dtype=np.uint8)
        cv2.fillPoly(mask, vertices, 255)
        return mask

    @staticmethod
    def _vertex_key(vertices):
        if vertices is None:
            return None
        a = np.asarray(vertices)
        return a.shape, a.dtype.str, a.tobytes()

    def _roi_key(self, stream_rois, n_masks: int):
        """Key of the context's mask set: one ROI (``stream_rois`` None), or ``n_masks`` masks, one per stream, where an
        entry of None is the detector's own ROI and streams past the end of ``stream_rois`` get an empty mask (no frame
        of the call belongs to them; they only make room for the streams whose smoothing state the detector holds)."""
        own = self._vertex_key(self.roi_vertices)
        if stream_rois is None:
            return (own,)
        keys = [own if v is None else self._vertex_key(v) for v in stream_rois]
        return tuple(keys) + ("empty",) * (n_masks - len(keys))

    def _roi_masks(self, h: int, w: int, roi_key, stream_rois) -> np.ndarray:
        """The masks of ``roi_key``: ``(H, W)`` for one ROI, else ``(R, H, W)``.  Rasterised masks are cached by their
        vertices, so a rig's masks are drawn once."""
        if len(self._roi_cache) > 256:
            self._roi_cache.clear()
        masks = []
        for i, k in enumerate(roi_key):
            ck = (h, w, k)
            m = self._roi_cache.get(ck)
            if m is None:
                if k == "empty":
                    m = np.zeros((h, w), np.uint8)
                else:
                    v = None if stream_rois is None or stream_rois[i] is None else stream_rois[i]
                    m = self._get_roi_mask((h, w), v)
                self._roi_cache[ck] = m
            masks.append(m)
        return masks[0] if stream_rois is None else np.stack(masks)

    def _device_index(self, frames=None) -> int:
        """GPU the context lives on: the device of a CUDA tensor input, else ``device=``, else torch's current one."""
        if frames is not None and _is_torch_cuda(frames):
            idx = frames.device.index
            idx = 0 if idx is None else int(idx)
            if self._device is not None and int(self._device) != idx:
                raise ValueError(f"frames are on cuda:{idx} but this LaneDetector was created with device={self._device}")
            return idx
        if self._device is not None:
            return int(self._device)
        try:
            import torch
            if torch.cuda.is_available():
                return int(torch.cuda.current_device())
        except Exception:
            pass
        return 0

    def _context(self, h: int, w: int, n: int, frames=None, stream_rois=None, n_masks: int = 1) -> _native.LaneContext:
        roi_key = self._roi_key(stream_rois, n_masks)
        key = (h, w, roi_key, self._device_index(frames))
        if self._ctx is None or self._ctx_key != key or self._ctx.max_batch < min(n, self._max_batch):
            if self._ctx is not None:
                self._ctx.close()
            cap = max(min(n, self._max_batch), 1)
            self._ctx = _native.LaneContext(h, w, cap, self._roi_masks(h, w, roi_key, stream_rois), device=key[3],
                                            max_segments=self._max_segments, debug=self._debug)
            self._ctx_key = key
        return self._ctx

    # ------------------------------------------------------------------ input checking
    @staticmethod
    def _check_frames(frames, batched: bool):
        nd = 4 if batched else 3
        shape = tuple(frames.shape)
        if len(shape) != nd or shape[-1] != 3:
            # the reference fails inside cv2.cvtColor for anything but 3-channel input
            raise cv2.error(f"LaneDetector: expected uint8 BGR frame(s) of shape "
                            f"{'[N,H,W,3]' if batched else '[H,W,3]'}, got {shape}")
        dt = str(frames.dtype).replace("torch.", "")
        if dt != "uint8":
            # the reference fails inside cv2.Canny (depth assertion) for non-8-bit input
            raise cv2.error(f"LaneDetector: frames must be uint8, got {dt}")

    # ------------------------------------------------------------------ record decoding
    def _lanes_from_records(self, recs: np.ndarray) -> List[LanePair]:
        """Records -> (left, right) pairs.  The point and coefficient arrays of a batch are copied out of the record
        buffer once; every LaneLine then holds its own rows of those copies (host time matters here: at 8 000 frames/s
        end to end, two array copies per lane were 7 % of the call)."""
        sides = recs["side"]
        valid = sides["valid"].astype(bool)
        points = np.ascontiguousarray(sides["points"], dtype=np.int32)          # [n, 2, 50, 2]
        coeffs = np.ascontiguousarray(sides["coeffs"], dtype=np.float64)        # [n, 2, 3]
        conf = sides["confidence"].tolist()
        out: List[LanePair] = []
        for i in range(len(recs)):
            v = valid[i]
            left = LaneLine(points[i, 0], "left", conf[i][0], coeffs[i, 0]) if v[0] else None
            right = LaneLine(points[i, 1], "right", conf[i][1], coeffs[i, 1]) if v[1] else None
            out.append((left, right))
        return out

    def _run(self, frames, stream_id, n_streams, prev_fit, prev_valid, fmt: int = _native.INPUT_BGR,
             target_size: Optional[Tuple[int, int]] = None, stream_rois=None) -> np.ndarray:
        """Chunked native calls over frames [N,H,W,3] (numpy or CUDA torch; [N,H*3/2,W] for the YUV 4:2:0 layouts of
        ``fmt``), detected at ``target_size`` = (width, height) when given (the device resizes every frame to it first);
        state arrays updated in place.  ``stream_rois``: one ROI per stream (see ``detect_streams``)."""
        n, sh, sw = int(frames.shape[0]), int(frames.shape[1]), int(frames.shape[2])
        if fmt != _native.INPUT_BGR:
            sh = sh * 2 // 3
        fbytes = sh * sw * 3 if fmt == _native.INPUT_BGR else sh * sw * 3 // 2
        h, w = (sh, sw) if target_size is None else (target_size[1], target_size[0])
        n_masks = 1 if stream_rois is None else max(len(stream_rois), n_streams)
        ctx = self._context(h, w, n, frames, stream_rois, n_masks)
        s, oms = self.smoothing_factor, 1 - self.smoothing_factor
        chunks = []
        on_device = _is_torch_cuda(frames)
        if on_device:
            import torch
            frames = frames.contiguous()
            torch.cuda.current_stream(frames.device).synchronize()
        else:
            frames = np.ascontiguousarray(frames)

        def call(c, a, b):
            sid = None if stream_id is None else stream_id[a:b]
            src = frames.data_ptr() + a * fbytes if on_device else frames[a:b]
            return c.detect(src, b - a, on_device, sid, n_streams, prev_fit, prev_valid, s, oms, fmt=fmt, src_hw=(sh, sw))

        for a in range(0, n, ctx.max_batch):
            b = min(a + ctx.max_batch, n)
            fit0, valid0 = prev_fit.copy(), prev_valid.copy()
            recs = call(ctx, a, b)
            if recs["flags"].any():
                # cv2.HoughLinesP has no cap on the number of segments: a frame that found more than max_segments would
                # otherwise be fitted on a truncated list.  Re-run the chunk, from the state it started with, on a context
                # sized for what was found (the reference result, just slower), never return a truncated fit silently.
                prev_fit[...], prev_valid[...] = fit0, valid0
                dense = self._dense_context(h, w, int(recs["n_segments_found"].max()), ctx.device, stream_rois, n_masks)
                recs = np.concatenate([call(dense, i, min(i + dense.max_batch, b)) for i in range(a, b, dense.max_batch)])
                if recs["flags"].any():
                    raise _native.LaneError(-5, "segment list still truncated after the dense re-run")
                self.dense_reruns += 1
            chunks.append(recs)
        recs = chunks[0] if len(chunks) == 1 else np.concatenate(chunks)
        self.last_records = recs
        return recs

    def _dense_context(self, h: int, w: int, need: int, device: int, stream_rois=None,
                       n_masks: int = 1) -> _native.LaneContext:
        cap = 1 << max(int(need) - 1, 1).bit_length()
        roi_key = self._roi_key(stream_rois, n_masks)
        key = (h, w, roi_key, device)
        if self._dense_ctx is None or self._dense_key != key or self._dense_ctx.max_segments < need:
            if self._dense_ctx is not None:
                self._dense_ctx.close()
            self._dense_ctx = _native.LaneContext(h, w, 8, self._roi_masks(h, w, roi_key, stream_rois), device=device,
                                                  max_segments=cap, debug=self._debug)
            self._dense_key = key
        self._ctx.copy_settings_to(self._dense_ctx)
        return self._dense_ctx

    def _state_arrays(self):
        fit = np.zeros((1, 2, 3), np.float64)
        valid = np.zeros((1, 2), np.uint8)
        for s, p in enumerate((self.prev_left_fit, self.prev_right_fit)):
            if p is not None:
                fit[0, s] = np.asarray(p, dtype=np.float64)
                valid[0, s] = 1
        return fit, valid

    # ------------------------------------------------------------------ public API
    def detect(self, frame: np.ndarray) -> LanePair:
        """Detect lane lines in one BGR frame (reference: lane_detector.py:178-218)."""
        self._check_frames(frame, batched=False)
        return self.detect_batch(frame[None])[0]

    def detect_batch(self, frames, *, target_size: Optional[Tuple[int, int]] = None) -> List[LanePair]:
        """``frames`` uint8 [N,H,W,3] (numpy, or a CUDA torch tensor already on the device).

        Semantics: identical to calling ``detect`` on ``frames[0..N-1]`` in order on this instance --
        the temporal smoothing is carried through the batch and left in ``prev_*_fit``.

        ``target_size`` = (width, height), as ``VideoDataLoader(..., target_size=...)`` and ``cv2.resize`` take it: every
        frame is first resized to it on the device, so the call equals ``detect_batch`` of
        ``np.stack([cv2.resize(f, target_size) for f in frames])`` (``roi_vertices`` are in target coordinates).
        """
        self._check_frames(frames, batched=True)
        if target_size is not None:
            target_size = check_target_size(target_size)
        if frames.shape[0] == 0:
            return []
        fit, valid = self._state_arrays()
        recs = self._run(frames, None, 1, fit, valid, target_size=target_size)
        lanes = self._lanes_from_records(recs)
        self._adopt_state(lanes)
        return lanes

    def detect_batches(self, batches):
        """Pipelined ``detect_batch`` over a sequence of device-resident batches: a generator that yields, for every CUDA
        tensor ``[N,H,W,3]`` of ``batches`` in order, what ``detect_batch`` would return for it.

        Two batches are kept in flight on the native context with the temporal-smoothing state carried on the device (the
        streaming form of the C ABI: ``lane_detect_enqueue`` twice, then collect / enqueue alternately), so the GPU never
        waits for the host between batches and the Hough half of batch i runs under the edge kernels of batch i+1.
        Results, state chain and ``prev_*_fit`` are exactly those of calling ``detect_batch`` batch after batch; a batch whose
        segment lists overflow is re-run on the dense context like there (the queue is drained and restarted around it).
        Batches that are not CUDA tensors of one common shape on one device simply go through ``detect_batch``."""
        import torch
        it = iter(batches)
        queue = []                                   # [tensor, state_before (fit, valid)] of the batches in flight
        ctx = None
        fit, valid = self._state_arrays()
        s, oms = self.smoothing_factor, 1 - self.smoothing_factor

        def streamable(fr):
            return (_is_torch_cuda(fr) and len(fr.shape) == 4 and fr.shape[0] > 0 and ctx is not None and
                    fr.shape[0] <= ctx.max_batch and (int(fr.shape[1]), int(fr.shape[2])) == (ctx.height, ctx.width) and
                    fr.device.index == ctx.device)

        def enqueue(fr, explicit):
            fr = fr.contiguous()
            torch.cuda.ExternalStream(ctx.stream(), device=fr.device).wait_stream(torch.cuda.current_stream(fr.device))
            if explicit:
                ctx.enqueue(fr.data_ptr(), int(fr.shape[0]), None, 1, fit, valid, s, oms)
            else:
                ctx.enqueue(fr.data_ptr(), int(fr.shape[0]), None, 1, None, None, s, oms)
            queue.append([fr, None])

        def drain():
            while ctx is not None and ctx._inflight:
                ctx.collect(np.zeros((1, 2, 3)), np.zeros((1, 2), np.uint8))
            queue.clear()

        try:
            nxt = next(it, None)
            while nxt is not None or queue:
                if not queue:                        # (re)start the pipeline with the detector's current state
                    cur = nxt
                    nxt = next(it, None)
                    self._check_frames(cur, batched=True)
                    if _is_torch_cuda(cur) and cur.shape[0] > 0:
                        ctx = self._context(int(cur.shape[1]), int(cur.shape[2]), int(cur.shape[0]), cur)
                    if not streamable(cur):
                        yield self.detect_batch(cur)
                        continue
                    fit, valid = self._state_arrays()
                    enqueue(cur, explicit=True)
                if nxt is not None and len(queue) < 2:
                    self._check_frames(nxt, batched=True)
                    if streamable(nxt):
                        enqueue(nxt, explicit=False)
                        nxt = next(it, None)
                head = queue[0][0]
                state_before = (fit.copy(), valid.copy())
                recs = ctx.collect(fit, valid)       # fit / valid now hold the state after `head`
                queue.pop(0)
                if recs["flags"].any():
                    # truncated segment lists: the batches behind it started from a wrong state; drain, redo this batch
                    # the blocking way (dense context) from the state it started with, and restart the pipeline
                    requeue = [q[0] for q in queue]
                    drain()
                    for side, p in enumerate(("prev_left_fit", "prev_right_fit")):
                        setattr(self, p, state_before[0][0, side].copy() if state_before[1][0, side] else None)
                    lanes = self.detect_batch(head)
                    yield lanes
                    fit, valid = self._state_arrays()
                    for k, fr in enumerate(requeue):
                        enqueue(fr, explicit=(k == 0))
                    continue
                self.last_records = recs
                lanes = self._lanes_from_records(recs)
                self._adopt_state(lanes)
                yield lanes
        finally:
            drain()

    def _adopt_state(self, lanes: List[LanePair]):
        """Like the reference (:210-216), prev_*_fit aliases the last returned polynomial of that side."""
        for left, _ in reversed(lanes):
            if left is not None:
                self.prev_left_fit = left.polynomial
                break
        for _, right in reversed(lanes):
            if right is not None:
                self.prev_right_fit = right.polynomial
                break

    def detect_batch_nv12(self, frames, *, target_size: Optional[Tuple[int, int]] = None) -> List[LanePair]:
        """``detect_batch`` for frames still in a video decoder's NV12 layout: uint8 ``[N, H*3/2, W]`` (Y plane, then
        the interleaved half-resolution UV plane), numpy or CUDA tensor.  Equal to ``detect_batch`` on
        ``cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12)`` of every frame -- the conversion runs on the device, so a host batch
        moves 1.5 B/px over PCIe instead of 3.

        ``target_size`` = (width, height): the decoder's frames at camera resolution are detected at that size, equal to
        ``detect_batch`` of ``cv2.resize(cv2.cvtColor(f, COLOR_YUV2BGR_NV12), target_size)`` (``VideoDataLoader`` with
        ``target_size``); conversion and resize are one kernel and only the NV12 bytes cross PCIe."""
        return self._detect_yuv420(frames, _native.INPUT_NV12, target_size)

    def detect_batch_i420(self, frames, *, target_size: Optional[Tuple[int, int]] = None) -> List[LanePair]:
        """``detect_batch_nv12`` for the planar layout software decoders hand out (FFmpeg / PyAV ``yuv420p``): uint8
        ``[N, H*3/2, W]`` = Y plane, U plane, V plane; equal to ``detect_batch`` on
        ``cv2.cvtColor(f, cv2.COLOR_YUV2BGR_I420)`` of every frame, resized to ``target_size`` when given."""
        return self._detect_yuv420(frames, _native.INPUT_I420, target_size)

    def _detect_yuv420(self, frames, fmt: int, target_size) -> List[LanePair]:
        check_yuv420(frames, "LaneDetector")
        if target_size is not None:
            target_size = check_target_size(target_size)
        if frames.shape[0] == 0:
            return []
        fit, valid = self._state_arrays()
        recs = self._run(frames, None, 1, fit, valid, fmt=fmt, target_size=target_size)
        lanes = self._lanes_from_records(recs)
        self._adopt_state(lanes)
        return lanes

    def detect_streams(self, frames, stream_ids: Optional[Sequence[int]] = None, *,
                       stream_rois: Optional[Sequence[Optional[np.ndarray]]] = None) -> List[LanePair]:
        """Multi-camera form: ``frames`` is [S,T,H,W,3] (stream-major) or [N,H,W,3] with ``stream_ids[N]``.

        Every stream keeps its own smoothing state inside this detector (``reset`` clears all of them);
        frames of one stream must be in temporal order.  Returns one pair per frame, in input order.

        ``stream_rois`` gives every camera its own ROI: entry s is stream s's polygon in ``roi_vertices`` form (int32
        [1,K,2], rasterised with ``cv2.fillPoly`` as the reference does), or None for this detector's own ROI.  It needs
        an entry for every stream id of the call (``ValueError`` otherwise).  Stream s's results then equal those of
        ``LaneDetector(roi_vertices=stream_rois[s])`` run on that stream's frames in order, and the whole rig still runs
        as one batched call.  Without it, every stream uses this detector's ROI.
        """
        if len(frames.shape) == 5:
            s_, t_ = int(frames.shape[0]), int(frames.shape[1])
            stream_ids = np.repeat(np.arange(s_, dtype=np.int32), t_)
            frames = frames.reshape((s_ * t_,) + tuple(frames.shape[2:]))
        if stream_ids is None:
            raise ValueError("stream_ids is required for [N,H,W,3] input")
        self._check_frames(frames, batched=True)
        stream_ids = np.asarray(stream_ids, dtype=np.int32)
        if stream_ids.shape != (frames.shape[0],) or (len(stream_ids) and stream_ids.min() < 0):
            raise ValueError("stream_ids must be non-negative int32[N]")
        if frames.shape[0] == 0:
            return []
        n_streams = int(stream_ids.max()) + 1
        if stream_rois is not None:
            stream_rois = list(stream_rois)
            if len(stream_rois) < n_streams:
                raise ValueError(f"stream_rois has {len(stream_rois)} entries; stream id {n_streams - 1} needs {n_streams}")
        if self._stream_fit is None or self._stream_fit.shape[0] < n_streams:
            fit = np.zeros((n_streams, 2, 3), np.float64)
            valid = np.zeros((n_streams, 2), np.uint8)
            if self._stream_fit is not None:
                k = self._stream_fit.shape[0]
                fit[:k], valid[:k] = self._stream_fit, self._stream_valid
            self._stream_fit, self._stream_valid = fit, valid
        recs = self._run(frames, stream_ids, self._stream_fit.shape[0], self._stream_fit, self._stream_valid,
                         stream_rois=stream_rois)
        return self._lanes_from_records(recs)

    def draw_lanes(self, frame: np.ndarray, left_lane: Optional[LaneLine], right_lane: Optional[LaneLine],
                   fill_lane: bool = True) -> np.ndarray:
        """Overlay rendering of ONE host frame with cv2, as in the reference (lane_detector.py:220-251): translucent fill
        between the lanes, then the two polylines (blue left, red right).  ``draw_lanes_batch`` is the device form."""
        if fill_lane and left_lane is not None and right_lane is not None:
            filled = frame.copy()
            outline = np.vstack([left_lane.points, right_lane.points[::-1]])
            cv2.fillPoly(filled, [outline], (0, 255, 100))
            frame = cv2.addWeighted(frame, 0.7, filled, 0.3, 0)
        for lane, colour in ((left_lane, (255, 0, 0)), (right_lane, (0, 0, 255))):
            if lane is not None:
                cv2.polylines(frame, [lane.points], False, colour, 3)
        return frame

    def draw_lanes_batch(self, frames, lanes: Sequence[LanePair], fill_lane: bool = True):
        """``draw_lanes`` for a whole batch on the GPU, IN PLACE: ``frames`` uint8 ``[N,H,W,3]`` (CUDA tensor: stays in
        HBM; numpy: round trip inside the call), ``lanes`` as ``detect_batch`` returned them.  Pixels equal the
        reference's ``draw_lanes(frame, left, right, fill_lane)`` (csrc/k7_draw.cu restates cv2's fillPoly / addWeighted
        / thick polylines bit for bit).  No CPU fallback."""
        from ..visualization.overlays import draw_lanes_batch
        return draw_lanes_batch(frames, lanes, fill_lane, self._device if not _is_torch_cuda(frames) else None)

    def get_lane_center_offset(self, frame_width: int, left_lane: Optional[LaneLine],
                               right_lane: Optional[LaneLine]) -> Optional[float]:
        """Vehicle offset from the lane centre in px, None unless both lanes exist
        (reference: lane_detector.py:253-272; the x positions are the last sample points)."""
        if left_lane is None or right_lane is None:
            return None
        lane_center = (left_lane.points[-1, 0] + right_lane.points[-1, 0]) / 2
        return frame_width / 2 - lane_center

    def reset(self):
        """Reset lane tracking state (reference: lane_detector.py:274-277)."""
        self.prev_left_fit = None
        self.prev_right_fit = None
        self._stream_fit = None
        self._stream_valid = None

    def close(self):
        for name in ("_ctx", "_dense_ctx"):
            c = getattr(self, name)
            if c is not None:
                c.close()
                setattr(self, name, None)
