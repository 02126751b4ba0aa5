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

import os
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import cv2
import numpy as np

from .. import _native
from ..loaders.frame_ingest import check_target_size
from ..loaders.frame_layout import BY_FORMAT, LAYOUTS, Layout, check_frames, named


@dataclass
class LaneLine:
    """Represents a detected lane line (reference: lane_detector.py:13-19)."""
    points: np.ndarray  # int32 [50, 2] (x, y)
    side: str  # "left" or "right"
    confidence: float
    polynomial: Optional[np.ndarray] = None  # float64 [3], highest power first


LanePair = Tuple[Optional[LaneLine], Optional[LaneLine]]
_SIDES = ("left", "right")
_COPY_PIECE = 4 << 20         # bytes per host thread task when detect_rig_stream copies a numpy tick into pinned memory


def _is_torch_cuda(x) -> bool:
    return type(x).__module__.startswith("torch") and hasattr(x, "is_cuda") and bool(x.is_cuda)


def _is_pinned_tensor(x) -> bool:
    """A contiguous CPU torch tensor in page-locked memory (the copy engine reads it where it is); an empty one has no
    memory to lock."""
    return (type(x).__module__.startswith("torch") and hasattr(x, "is_pinned") and not x.is_cuda and x.is_contiguous()
            and (x.numel() == 0 or bool(x.is_pinned())))


def _frame_bytes(fmt: int, h: int, w: int) -> int:
    """Bytes of one h x w frame in layout ``fmt`` (INPUT_*), from the layout table."""
    return BY_FORMAT[fmt].frame_bytes(h, w)


def _two_deep(items, plan, start, joins, enqueue, blocking, restore, adopt):
    """The queue of ``detect_batches`` and ``detect_rig_stream``: yields one result per item, in order, with up to two
    items in flight on a native context.  ``plan(item)`` checks an item when its turn comes (raising its argument errors
    after the items before it are out) and returns ``p``.  ``start(p)`` takes the detector's state for a first item in
    flight, ``(ctx, fit, valid)`` (the arrays ``ctx.collect`` fills), or None to run it through ``blocking(item, p)``.
    An item queues behind the one in flight if ``joins(p)``.  ``enqueue(item, p, explicit)`` starts it from ``fit`` /
    ``valid`` or from the device state, returning what must live until it is collected.  ``restore(fit, valid)`` and
    ``adopt(recs, p)`` make the state before / after an item the detector's; ``adopt`` returns its result.  An item whose
    segment lists overflow started the items behind it from a wrong state: the queue is drained, the item redone through
    ``blocking`` from the state before it, and the items behind it planned again."""
    it, pending, queue = iter(items), [], []     # queue: (item, plan, what enqueue keeps alive), oldest first
    end = object()
    ctx = fit = valid = None

    def take():
        return pending.pop(0) if pending else next(it, end)

    def drain():
        while ctx is not None and ctx._inflight:
            ctx.collect(fit.copy(), valid.copy())
        queue.clear()

    try:
        nxt = take()
        while nxt is not end or queue:
            if not queue:                            # (re)start with the detector's current state
                cur, nxt = nxt, take()
                p = plan(cur)
                started = start(p)
                if started is None:
                    yield blocking(cur, p)
                    continue
                ctx, fit, valid = started
                queue.append((cur, p, enqueue(cur, p, True)))
            if nxt is not end and len(queue) < 2:
                try:
                    p = plan(nxt)
                except Exception:
                    p = end                          # planned again, and raised, when its turn comes
                if p is not end and joins(p):
                    queue.append((nxt, p, enqueue(nxt, p, False)))
                    nxt = take()
            before = (fit.copy(), valid.copy())
            recs = ctx.collect(fit, valid)           # fit / valid now hold the state after the oldest item
            item, p, _ = queue.pop(0)
            if recs["flags"].any():
                # truncated segment lists: redo the item the blocking way (dense context) and restart with the rest
                pending[:0] = [q[0] for q in queue] + ([] if nxt is end else [nxt])
                drain()
                restore(*before)
                yield blocking(item, p)
                nxt = take()
                continue
            yield adopt(recs, p)
    finally:
        drain()


@dataclass
class _Plan:
    """One detect call's batch as its argument checks found it: source s has ``counts[s]`` frames ``cams[s]`` in layout
    ``fmts[s]`` (INPUT_*) at ``sizes[s]`` = (h, w); every source with frames is of one ``kind`` (``("cuda", index)``,
    ``"host"`` for numpy, ``"pinned"``; None when the batch has no frame), detected at ``h`` x ``w``.

    ``rig``: the batch takes the rig entries (``lane_detect_rig`` / ``lane_rig_enqueue``), source s being stream s.
    Otherwise it is one source through ``lane_detect_batch_ingest`` / ``lane_detect_enqueue``, which read BGR frames at
    the detection size in place, with per-frame stream ids ``frame_sids`` (None: every frame is stream 0)."""
    cams: list
    fmts: list
    sizes: list
    counts: list
    kind: object
    h: Optional[int]
    w: Optional[int]
    stream_rois: Optional[list]
    rig: bool = True
    frame_sids: Optional[np.ndarray] = None

    def __post_init__(self):
        self.base = [0]                              # source s's frames are [base[s], base[s+1]) of the concatenation
        for t in self.counts:
            self.base.append(self.base[-1] + t)
        self.n = self.base[-1]
        self.live = [s for s, t in enumerate(self.counts) if t]
        if self.rig:
            self.n_streams = len(self.cams)
        else:
            self.n_streams = 1 if self.frame_sids is None or not self.n else int(self.frame_sids.max()) + 1

    @classmethod
    def of_frames(cls, frames, fmt: int, target_size=None, frame_sids=None, stream_rois=None) -> "_Plan":
        """One checked array of frames in layout ``fmt`` (INPUT_*), detected at ``target_size`` = (width, height) when
        given."""
        n, (sh, sw) = int(frames.shape[0]), BY_FORMAT[fmt].hw(frames.shape)
        h, w = (sh, sw) if target_size is None else (target_size[1], target_size[0])
        kind = ("cuda", frames.device.index) if _is_torch_cuda(frames) else "host"
        return cls([frames], [fmt], [(sh, sw)], [n], kind, h, w, stream_rois, rig=False, frame_sids=frame_sids)

    def n_masks(self, n_streams: int) -> int:
        return 1 if self.stream_rois is None else max(len(self.stream_rois), n_streams)

    def per_camera(self, items):
        return [items[self.base[s]:self.base[s + 1]] for s in range(len(self.cams))]

    def sources(self, data, a: int, b: int, on_device: bool) -> list:
        """``(frames, fmt, (h, w), n, stream id)`` of every source's share of frames [a, b): a device pointer into
        ``data[s]`` (on_device) or a view of it."""
        out = []
        for s in self.live:
            lo, hi = max(a, self.base[s]), min(b, self.base[s + 1])
            if lo < hi:
                i, j = lo - self.base[s], hi - self.base[s]
                src = data[s].data_ptr() + i * _frame_bytes(self.fmts[s], *self.sizes[s]) if on_device else data[s][i:j]
                out.append((src, self.fmts[s], self.sizes[s], j - i, s))
        return out


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

    def _run(self, p: _Plan, prev_fit: np.ndarray, prev_valid: np.ndarray) -> np.ndarray:
        """Plan ``p`` through its blocking entry in chunks of the context's max_batch, from the state ``prev_fit`` /
        ``prev_valid`` (one row per stream, updated in place); each chunk is re-run on the dense context when its segment
        lists overflow."""
        on_device = p.kind not in ("host", "pinned")
        if on_device:
            import torch
            data = {s: p.cams[s].contiguous() for s in p.live}
            torch.cuda.current_stream(data[p.live[0]].device).synchronize()
        else:
            data = {s: np.ascontiguousarray(p.cams[s]) for s in p.live}
        n_streams = prev_fit.shape[0]
        n_masks = p.n_masks(n_streams)
        ctx = self._context(p.h, p.w, p.n, data[p.live[0]], p.stream_rois, n_masks)
        sm, oms = self.smoothing_factor, 1 - self.smoothing_factor

        def call(c, a, b):
            sources = p.sources(data, a, b, on_device)
            if p.rig:
                return c.detect_rig(sources, on_device, n_streams, prev_fit, prev_valid, sm, oms)
            (src, fmt, hw, k, _), = sources
            sid = None if p.frame_sids is None else p.frame_sids[a:b]
            return c.detect(src, k, on_device, sid, n_streams, prev_fit, prev_valid, sm, oms, fmt=fmt, src_hw=hw)

        chunks = []
        for a in range(0, p.n, ctx.max_batch):
            b = min(a + ctx.max_batch, p.n)
            fit0, valid0 = prev_fit.copy(), prev_valid.copy()
            recs = call(ctx, a, b)
            if recs["flags"].any():
                # cv2.HoughLinesP has no cap on the number of segments: a frame that found more than max_segments would
                # otherwise be fitted on a truncated list.  Re-run the chunk, from the state it started with, on a context
                # sized for what was found (the reference result, just slower), never return a truncated fit silently.
                prev_fit[...], prev_valid[...] = fit0, valid0
                dense = self._dense_context(p.h, p.w, int(recs["n_segments_found"].max()), ctx.device, p.stream_rois,
                                            n_masks)
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
        return self._detect_frames(frames, _native.INPUT_BGR, target_size)

    def _detect_frames(self, frames, fmt: int, target_size) -> List[LanePair]:
        """``detect_batch`` and its decoder-layout forms, on frames checked for layout ``fmt`` (INPUT_*)."""
        if target_size is not None:
            target_size = check_target_size(target_size)
        if frames.shape[0] == 0:
            return []
        fit, valid = self._state_arrays()
        lanes = self._lanes_from_records(self._run(_Plan.of_frames(frames, fmt, target_size), fit, valid))
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
        Batches that are not CUDA tensors of one common shape on one device simply go through ``detect_batch``.  A
        malformed batch raises ``detect_batch``'s error when its turn comes, after the batches before it are yielded."""
        def plan(fr):
            self._check_frames(fr, batched=True)
            return _Plan.of_frames(fr, _native.INPUT_BGR)

        def restore(fit0, valid0):
            for side, p in enumerate(("prev_left_fit", "prev_right_fit")):
                setattr(self, p, fit0[0, side].copy() if valid0[0, side] else None)

        def adopt(lanes, p, fit, valid):
            self._adopt_state(lanes)
            return lanes

        yield from self._stream(batches, plan, lambda p: self._state_arrays(), lambda fr, p: self.detect_batch(fr),
                                restore, adopt)

    def _stream(self, items, plan, state, blocking, restore, adopt, cap: Optional[int] = None, stage=None):
        """``_two_deep`` over plans, the queue of ``detect_batches`` and ``detect_rig_stream``.  ``plan(item)`` checks an
        item and returns its ``_Plan``; ``state(p)`` returns ``(fit, valid)``, the detector's state for a first item in
        flight as arrays ``collect`` may fill; ``blocking`` and ``restore`` are ``_two_deep``'s; ``adopt(lanes, p, fit,
        valid)`` makes the state after an item (its pairs ``lanes``) the detector's and returns the item's result.  The
        context is sized for ``cap`` frames (None: the first item's).  CUDA frames are read in place once the work on the
        caller's stream is done, pinned ones in place, and host (numpy) frames only through ``stage(p, explicit)``, which
        copies them into page-locked memory and returns them per source; without it host items run blocking."""
        import torch
        ctx = fit = valid = None

        def streams(p) -> bool:
            return bool(p.n) and (p.kind != "host" or stage is not None)

        def start(p):
            nonlocal ctx, fit, valid
            if not streams(p):
                return None
            fit, valid = state(p)
            ctx = self._context(p.h, p.w, cap or p.n, p.cams[p.live[0]], p.stream_rois, p.n_masks(len(fit)))
            return (ctx, fit, valid) if joins(p) else None

        def joins(p) -> bool:
            """Whether p can queue behind the item in flight: same context and streams, and it fits."""
            if not streams(p) or p.n_streams > len(fit) or p.n > ctx.max_batch or self._ctx is not ctx:
                return False
            try:
                dev = self._device_index(p.cams[p.live[0]])
            except ValueError:
                return False
            return self._ctx_key == (p.h, p.w, self._roi_key(p.stream_rois, p.n_masks(len(fit))), dev)

        def enqueue(item, p, explicit: bool):
            on_device = p.kind not in ("host", "pinned")
            if p.kind == "host":
                data = stage(p, explicit)
            elif p.kind == "pinned":
                data = {s: p.cams[s].numpy() for s in p.live}
            else:
                data = {s: p.cams[s].contiguous() for s in p.live}
                dev = data[p.live[0]].device
                torch.cuda.ExternalStream(ctx.stream(), device=dev).wait_stream(torch.cuda.current_stream(dev))
            sources = p.sources(data, 0, p.n, on_device)
            fit0, valid0 = (fit, valid) if explicit else (None, None)
            sm, oms = self.smoothing_factor, 1 - self.smoothing_factor
            if p.rig:
                ctx.enqueue_rig(sources, on_device, len(fit), fit0, valid0, sm, oms)
            else:
                (src, _, _, k, _), = sources
                ctx.enqueue(src, k, p.frame_sids, len(fit), fit0, valid0, sm, oms)
            return data

        def adopt_records(recs, p):
            self.last_records = recs
            return adopt(self._lanes_from_records(recs), p, fit, valid)

        yield from _two_deep(items, plan, start, joins, enqueue, blocking, restore, adopt_records)

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
        return self._detect_camera(frames, LAYOUTS["nv12"], target_size)

    def detect_batch_i420(self, frames, *, target_size: Optional[Tuple[int, int]] = None) -> List[LanePair]:
        """``detect_batch_nv12`` for the planar layout software decoders hand out (FFmpeg / PyAV ``yuv420p``): uint8
        ``[N, H*3/2, W]`` = Y plane, U plane, V plane; equal to ``detect_batch`` on
        ``cv2.cvtColor(f, cv2.COLOR_YUV2BGR_I420)`` of every frame, resized to ``target_size`` when given."""
        return self._detect_camera(frames, LAYOUTS["i420"], target_size)

    def detect_batch_bayer(self, frames, pattern: str, *, target_size: Optional[Tuple[int, int]] = None) -> List[LanePair]:
        """``detect_batch`` for raw camera frames: uint8 ``[N, H, W]`` 8-bit Bayer mosaics (numpy or CUDA tensor, H and W
        at least 3) whose top-left 2x2 is ``pattern`` ("rggb", "bggr", "grbg" or "gbrg"; no default).  Equal to
        ``detect_batch`` of ``cv2.cvtColor(f, cv2.COLOR_Bayer<P>2BGR)`` of every frame, resized to ``target_size`` =
        (width, height) when given, with the same ``prev_*_fit`` after it.  Demosaic and resize are one kernel on the
        device, so a host batch moves 1 B/px over PCIe."""
        return self._detect_camera(frames, named(pattern, _native.BAYER, "Bayer pattern"), target_size)

    def detect_batch_yuv422(self, frames, order: str, *, target_size: Optional[Tuple[int, int]] = None) -> List[LanePair]:
        """``detect_batch`` for packed YUV 4:2:2 camera frames: uint8 ``[N, H, W, 2]`` (numpy or CUDA tensor, W even) in
        byte order ``order`` ("uyvy": U Y0 V Y1, GMSL / FPD-Link cameras; "yuyv": Y0 U Y1 V, V4L2 USB cameras; no
        default).  Equal to ``detect_batch`` of ``cv2.cvtColor(f, cv2.COLOR_YUV2BGR_UYVY | COLOR_YUV2BGR_YUY2)`` of every
        frame, resized to ``target_size`` = (width, height) when given, with the same ``prev_*_fit`` after it.
        Conversion and resize are one kernel on the device, so a host batch moves 2 B/px over PCIe instead of 3."""
        return self._detect_camera(frames, named(order, _native.YUV422, "YUV 4:2:2 order"), target_size)

    def _detect_camera(self, frames, layout: Layout, target_size) -> List[LanePair]:
        """``detect_batch`` of frames in a camera ``layout``, checked against it."""
        check_frames(frames, layout, "LaneDetector")
        return self._detect_frames(frames, layout.fmt, target_size)

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
        p = _Plan.of_frames(frames, _native.INPUT_BGR, frame_sids=stream_ids,
                            stream_rois=None if stream_rois is None else list(stream_rois))
        if p.stream_rois is not None and len(p.stream_rois) < p.n_streams:
            raise ValueError(f"stream_rois has {len(p.stream_rois)} entries; stream id {p.n_streams - 1} needs "
                             f"{p.n_streams}")
        self._grow_stream_state(p.n_streams)
        return self._lanes_from_records(self._run(p, self._stream_fit, self._stream_valid))

    def _grow_stream_state(self, n_streams: int):
        """Per-stream smoothing state of ``detect_streams`` / ``detect_rig`` for at least ``n_streams`` streams."""
        if self._stream_fit is None or self._stream_fit.shape[0] < n_streams:
            fit = np.zeros((n_streams, 2, 3), np.float64)
            valid = np.zeros((n_streams, 2), np.uint8)
            if self._stream_fit is not None:
                k = self._stream_fit.shape[0]
                fit[:k], valid[:k] = self._stream_fit, self._stream_valid
            self._stream_fit, self._stream_valid = fit, valid

    def detect_rig(self, frames: Sequence, layouts: Optional[Sequence[str]] = None, *,
                   target_size: Optional[Tuple[int, int]] = None,
                   stream_rois: Optional[Sequence[Optional[np.ndarray]]] = None) -> List[List[LanePair]]:
        """A rig of cameras that differ in resolution and decoder layout, in one batched call.

        ``frames[s]`` is camera s (= stream s of ``detect_streams``): uint8 ``[T_s, H_s, W_s, 3]`` BGR,
        ``[T_s, H_s*3/2, W_s]`` NV12 / I420, ``[T_s, H_s, W_s]`` raw Bayer or ``[T_s, H_s, W_s, 2]`` packed YUV 4:2:2, as
        ``layouts[s]`` ("bgr", "nv12", "i420", "bayer_rggb", "bayer_bggr", "bayer_grbg", "bayer_gbrg", "uyvy", "yuyv";
        default all "bgr") says, its frames in temporal order.  ``T_s`` may differ between cameras and may be 0, or the entry None: no frame this tick.  Every
        camera is a numpy array, or every camera is a CUDA tensor on one device.  Every frame is detected at
        ``target_size`` = (width, height), which may be left out only when all cameras share one size; the device converts
        and resizes all frames in one kernel (only the source bytes of host frames cross PCIe) and runs the rest of the
        path once for the rig.  ``stream_rois`` as in ``detect_streams``, polygons in target coordinates.

        Returns one list of pairs per camera.  Camera s's pairs equal those of a fresh
        ``LaneDetector(roi_vertices=stream_rois[s])`` given its frames through ``detect_batch`` / ``detect_batch_nv12`` /
        ``detect_batch_i420(frames[s], target_size=target_size)`` / ``detect_batch_bayer`` / ``detect_batch_yuv422``; its
        smoothing state is stream s's of ``detect_streams``, so it carries across calls of either kind (``reset`` clears
        it).
        """
        return self._detect_rig(self._rig_plan(frames, layouts, target_size, stream_rois))

    def _detect_rig(self, p: _Plan) -> List[List[LanePair]]:
        if not p.n:
            return [[] for _ in p.cams]
        self._grow_stream_state(p.n_streams)
        return p.per_camera(self._lanes_from_records(self._run(p, self._stream_fit, self._stream_valid)))

    def detect_rig_stream(self, ticks, layouts: Optional[Sequence[str]] = None, *,
                          target_size: Optional[Tuple[int, int]] = None,
                          stream_rois: Optional[Sequence[Optional[np.ndarray]]] = None):
        """Generator: for every tick of ``ticks`` (a per-camera sequence, as ``detect_rig``'s ``frames``) yield what
        ``detect_rig`` would return for it, with two ticks in flight on the native context.

        The form for a recorded multi-camera drive: the Hough half of tick i runs under the edge kernels of tick i+1, and
        the host copies of tick i+1 under the compute of tick i (``lane_rig_enqueue``).  Results, the per-camera smoothing
        state and ``last_records`` are exactly those of calling ``detect_rig`` tick after tick with the same ``layouts`` /
        ``target_size`` / ``stream_rois``; the state is adopted after every tick, so it carries into later ``detect_rig``
        / ``detect_streams`` calls.  Ticks may differ in frame counts, and a camera may be None or have 0 frames.

        A tick is every camera a CUDA tensor on one device, every camera a contiguous CPU tensor in pinned memory (read
        in place), or every camera a numpy array (copied into one of two pinned buffers the generator owns).  Every tick
        is referenced until it has been yielded; pinned tensors must not change until then.  A tick the pipeline cannot
        take (more frames than ``max_batch``, another device, a tick without frames) drains it and goes through
        ``detect_rig``; so do ticks whose segment lists overflow, from the state they started with.  Argument errors are
        ``detect_rig``'s, raised when the tick's turn comes.
        """
        import torch
        pinned = [None, None]         # pinned host copies of numpy ticks, one per tick in flight
        last_buf = 1                  # the pinned buffer of the numpy tick enqueued last
        copier = None                 # the host threads of those copies, made by the first tick that needs them

        def stage(p, explicit: bool):
            nonlocal last_buf, copier
            # a tick that joins takes the pinned buffer the numpy tick enqueued last does not use (only that one can still
            # be in flight)
            k = last_buf = 0 if explicit else 1 - last_buf
            need = sum(p.cams[s].nbytes for s in p.live)
            if pinned[k] is None or pinned[k].numel() < need:
                pinned[k] = torch.empty(need, dtype=torch.uint8, pin_memory=True)
            flat, off, src, pieces = pinned[k].numpy(), 0, {}, []
            for s in p.live:
                cam = np.ascontiguousarray(p.cams[s]).reshape(-1)
                src[s] = flat[off:off + cam.nbytes].reshape(p.cams[s].shape)
                cuts = list(range(0, cam.nbytes, _COPY_PIECE)) + [cam.nbytes]
                pieces += [(flat[off + a:off + b], cam[a:b]) for a, b in zip(cuts, cuts[1:])]
                off += cam.nbytes
            if len(pieces) > 1 and copier is None:
                copier = ThreadPoolExecutor(max(1, min(8, (os.cpu_count() or 2) // 2)))
            # one host thread copies ~10 GB/s: a tick of an 8-camera rig (35 MB) would take longer than its compute
            list(copier.map(lambda ds: np.copyto(*ds), pieces) if len(pieces) > 1 else
                 (np.copyto(*ds) for ds in pieces))
            return src

        def state(p):
            self._grow_stream_state(p.n_streams)
            return self._stream_fit.copy(), self._stream_valid.copy()

        def restore(fit0, valid0):
            self._stream_fit, self._stream_valid = fit0, valid0

        def adopt(lanes, p, fit, valid):
            self._stream_fit, self._stream_valid = fit.copy(), valid.copy()
            return p.per_camera(lanes)

        try:
            yield from self._stream(ticks, lambda t: self._rig_plan(t, layouts, target_size, stream_rois, pinned=True),
                                    state, lambda t, p: self._detect_rig(p), restore, adopt, cap=self._max_batch,
                                    stage=stage)
        finally:
            if copier is not None:
                copier.shutdown()

    def _rig_plan(self, frames, layouts, target_size, stream_rois, pinned: bool = False) -> _Plan:
        """``detect_rig``'s argument checks on one tick, and what they found.  ``pinned``: page-locked contiguous CPU
        torch tensors are a kind of their own (``detect_rig_stream`` reads them in place)."""
        cams = list(frames)
        layouts = ["bgr"] * len(cams) if layouts is None else list(layouts)
        if len(layouts) != len(cams):
            raise ValueError(f"{len(cams)} cameras but {len(layouts)} layouts")
        if target_size is not None:
            target_size = check_target_size(target_size)
        if stream_rois is not None:
            stream_rois = list(stream_rois)
            if len(stream_rois) < len(cams):
                raise ValueError(f"stream_rois has {len(stream_rois)} entries for {len(cams)} cameras")
        fmts, sizes, counts, kinds = [], [], [], set()
        for s, (f, lay) in enumerate(zip(cams, layouts)):
            if lay not in LAYOUTS:
                raise ValueError(f"camera {s}: layout {lay!r} is not one of {sorted(LAYOUTS)}")
            fmts.append(LAYOUTS[lay].fmt)
            if f is None:
                sizes.append(None)
                counts.append(0)
                continue
            kinds.add(("cuda", f.device.index) if _is_torch_cuda(f) else "host" if isinstance(f, np.ndarray) else
                      "pinned" if pinned and _is_pinned_tensor(f) else "other")
            if len(kinds) > 1 or "other" in kinds:
                raise ValueError("rig cameras must all be numpy arrays or all CUDA tensors on one device" +
                                 (", or all pinned contiguous CPU tensors" if pinned else ""))
            sizes.append(self._rig_frame_size(f, lay, s))
            counts.append(int(f.shape[0]))
        used = {sz for sz, t in zip(sizes, counts) if t}
        if target_size is None and len(used) > 1:
            raise ValueError(f"cameras of sizes {sorted(used)} need a target_size")
        hw = (None, None) if not used else next(iter(used)) if target_size is None else (target_size[1], target_size[0])
        return _Plan(cams, fmts, sizes, counts, next(iter(kinds)) if used else None, *hw, stream_rois)

    @staticmethod
    def _rig_frame_size(f, layout: str, s: int) -> Tuple[int, int]:
        """(H, W) of camera s's frames in ``layout``; ``ValueError`` when the shape or size is not that layout's,
        ``cv2.error`` for a BGR camera's channel count or any dtype (what cv2.cvtColor raises)."""
        lay, shape = LAYOUTS[layout], tuple(f.shape)
        hw = lay.hw(shape)
        if hw is None and layout == "bgr" and len(shape) == 4:
            raise cv2.error(f"LaneDetector: camera {s}: expected 3-channel BGR frames, got {shape}")
        if hw is None:
            raise ValueError(f"camera {s}: layout {layout!r} needs frames [T,{lay.dims}], got {shape}")
        if lay.refuses(*hw):
            raise ValueError(f"camera {s}: {layout} needs {lay.rule}, got {hw[1]}x{hw[0]}")
        if str(f.dtype).replace("torch.", "") != "uint8":
            raise cv2.error(f"LaneDetector: camera {s}: frames must be uint8, got {f.dtype}")
        return hw

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
