"""Which native calls every public ``LaneDetector`` call makes, driven with a fake ``_native.LaneContext`` so it holds
without a GPU or the library: the entry point, each source's layout, size, frames and stream id, the per-frame stream
ids, ``n_streams``, whether explicit state was passed and which, the chunk bounds, the contexts made, the dense re-run
of a chunk whose segment lists overflow, and the detector's state after each call.

Every frame carries a tag in its first byte.  The fake's records and state updates are a function of the tag, the
stream and the state the frame starts from, so a wrong chunk, stream id or state chain shows in the results."""
import numpy as np
import pytest

from multimodal_autonomous_driving_perception_and_planning_b200 import LaneDetector, _native

BGR, NV12, I420 = _native.INPUT_BGR, _native.INPUT_NV12, _native.INPUT_I420
H, W = 48, 64
INGEST, RIG = "lane_detect_batch_ingest", "lane_detect_rig"
RIG_ENQUEUE, COLLECT = "lane_rig_enqueue", "lane_detect_collect"


def bgr(tags, h=H, w=W):
    f = np.zeros((len(tags), h, w, 3), np.uint8)
    f[:, 0, 0, 0] = tags
    return f


def yuv(tags, h=H, w=W):
    f = np.zeros((len(tags), h * 3 // 2, w), np.uint8)
    f[:, 0, 0] = tags
    return f


def tags_of(frames, fmt):
    return tuple(int(t) for t in (frames[:, 0, 0, 0] if fmt == BGR else frames[:, 0, 0]))


def step(fit, valid, tag, sid, overflow):
    """The fake's record of frame ``tag`` on stream ``sid``; updates state row ``sid`` in place.  A side whose
    ``(tag + side) % 5 == 4`` finds no lane and keeps its state."""
    rec = np.zeros((), _native.RECORD_DTYPE)
    for side in (0, 1):
        if (tag + side) % 5 == 4:
            continue
        prev = fit[sid, side, 2] if valid[sid, side] else 0.0
        c = np.array([float(tag), float(sid + 10 * side), 0.5 * prev + tag + 1])
        rec["side"][side]["valid"] = 1
        rec["side"][side]["coeffs"] = c
        rec["side"][side]["confidence"] = tag / 256
        rec["side"][side]["points"] = tag + side
        fit[sid, side], valid[sid, side] = c, 1
    if overflow:
        rec["flags"], rec["n_segments_found"] = _native.FLAG_SEGMENTS_TRUNCATED, 300
        fit[sid, :, 2] += 1000.0                     # a truncated chunk leaves a wrong state behind
    return rec


class Recorder:
    def __init__(self):
        self.made, self.calls, self.overflow, self._seen = [], [], set(), 0

    def take(self):
        """Calls since the last take."""
        out, self._seen = self.calls[self._seen:], len(self.calls)
        return out


class Call:
    def __init__(self, entry, ctx, sources, frame_sids, n_streams, explicit, state_in):
        self.entry, self.ctx, self.sources, self.frame_sids = entry, ctx, tuple(sources), frame_sids
        self.n_streams, self.explicit, self.state_in = n_streams, explicit, state_in
        self.state_out = self.recs = None

    @property
    def key(self):
        return self.entry, self.ctx, self.sources, self.frame_sids, self.n_streams, self.explicit

    @property
    def flagged(self):
        return bool(self.recs["flags"].any())


class FakeContext:
    rec: Recorder = None

    def __init__(self, height, width, max_batch, roi_mask, device=0, max_segments=256, debug=False):
        mask = np.asarray(roi_mask)
        assert mask.dtype == np.uint8 and mask.shape[-2:] == (height, width) and mask.ndim in (2, 3)
        self.height, self.width, self.max_batch, self.device = height, width, max_batch, device
        self.max_segments, self.n_roi = max_segments, (mask.shape[0] if mask.ndim == 3 else 1)
        self.no = len(self.rec.made)
        self.rec.made.append((self.no, height, width, max_batch, max_segments, self.n_roi))
        self._inflight, self._dev = [], None
        self.closed = False

    def close(self):
        self.closed = True

    def copy_settings_to(self, other):
        pass

    def stream(self):
        return 0

    def _run(self, call, frames, fit, valid):
        """Records of ``frames`` = [(tag, sid)] from state fit / valid (updated in place)."""
        assert not self.closed and len(frames) <= self.max_batch and call.n_streams <= fit.shape[0]
        assert all(s < call.n_streams for _, s in frames) and (self.n_roi == 1 or call.n_streams <= self.n_roi)
        over = self.max_segments < 512
        recs = np.stack([step(fit, valid, t, s, over and t in self.rec.overflow) for t, s in frames])
        call.state_out, call.recs = (fit.copy(), valid.copy()), recs
        self.rec.calls.append(call)
        return recs

    @staticmethod
    def _state(fit, valid):
        return None if fit is None else (fit.copy(), valid.copy())

    def _rig(self, entry, sources, on_device, n_streams, fit, valid, smoothing, one_minus):
        assert not on_device and (smoothing, one_minus) == (0.7, 1 - 0.7)
        srcs = [(fmt, tuple(hw), tags_of(f, fmt)[:n] if n else (), sid) for f, fmt, hw, n, sid in sources]
        assert all(len(t) == n for (_, _, t, _), (_, _, _, n, _) in zip(srcs, sources))
        call = Call(entry, self.no, srcs, None, n_streams, fit is not None, self._state(fit, valid))
        return call, [(t, sid) for _, _, tags, sid in srcs for t in tags]

    def detect(self, frames, n, on_device, stream_id, n_streams, prev_fit, prev_valid, smoothing, one_minus,
               fmt=BGR, src_hw=None):
        assert not on_device and (smoothing, one_minus) == (0.7, 1 - 0.7) and len(frames) == n
        hw = (self.height, self.width) if src_hw is None else tuple(int(x) for x in src_hw)
        sids = None if stream_id is None else tuple(int(s) for s in stream_id)
        tags = tags_of(frames, fmt)
        call = Call(INGEST, self.no, [(fmt, hw, tags, None)], sids, n_streams, True, self._state(prev_fit, prev_valid))
        return self._run(call, list(zip(tags, sids or (0,) * n)), prev_fit, prev_valid).copy()

    def detect_rig(self, sources, on_device, n_streams, prev_fit, prev_valid, smoothing, one_minus):
        call, frames = self._rig(RIG, sources, on_device, n_streams, prev_fit, prev_valid, smoothing, one_minus)
        return self._run(call, frames, prev_fit, prev_valid).copy()

    def enqueue_rig(self, sources, on_device, n_streams, prev_fit, prev_valid, smoothing, one_minus):
        call, frames = self._rig(RIG_ENQUEUE, sources, on_device, n_streams, prev_fit, prev_valid, smoothing,
                                 one_minus)
        assert len(self._inflight) < 2 and (prev_fit is not None or self._dev is not None)
        if prev_fit is not None:
            self._dev = (prev_fit.copy(), prev_valid.copy())
        call.state_in = (self._dev[0].copy(), self._dev[1].copy())
        self._run(call, frames, *self._dev)
        self._inflight.append(call)

    def enqueue(self, *args):
        raise AssertionError("host frames never take lane_detect_enqueue")

    def collect(self, prev_fit, prev_valid):
        self.rec.calls.append(Call(COLLECT, self.no, (), None, None, False, None))
        done = self._inflight.pop(0)
        prev_fit[...], prev_valid[...] = done.state_out
        return done.recs.copy()


@pytest.fixture
def rec(monkeypatch):
    r = Recorder()
    monkeypatch.setattr(FakeContext, "rec", r)
    monkeypatch.setattr(_native, "LaneContext", FakeContext)
    return r


def zeros(s=1):
    return np.zeros((s, 2, 3)), np.zeros((s, 2), np.uint8)


def padded(state, s):
    fit, valid = zeros(s)
    fit[:len(state[0])], valid[:len(state[1])] = state
    return fit, valid


def chain(calls, state):
    """Every call starts from the state the un-truncated call before it left (a dense re-run: from the state the
    truncated call started from).  Returns the records of the un-truncated calls and the state after the last."""
    recs = []
    for c in calls:
        assert c.explicit
        want = padded(state, len(c.state_in[0]))
        np.testing.assert_array_equal(c.state_in[0], want[0])
        np.testing.assert_array_equal(c.state_in[1], want[1])
        if not c.flagged:
            state = c.state_out
            recs.append(c.recs)
    return (np.concatenate(recs) if recs else np.zeros(0, _native.RECORD_DTYPE)), state


def pairs(lanes):
    return [tuple(None if l is None else (l.side, l.confidence, l.polynomial.tolist(), l.points.tolist()) for l in p)
            for p in lanes]


def rec_pairs(recs):
    out = []
    for r in recs:
        out.append(tuple((side, float(r["side"][k]["confidence"]), r["side"][k]["coeffs"].tolist(),
                          r["side"][k]["points"].tolist()) if r["side"][k]["valid"] else None
                         for k, side in enumerate(("left", "right"))))
    return out


def single_state(det):
    """The detector's ``prev_*_fit`` as state arrays."""
    fit, valid = zeros()
    for k, p in enumerate((det.prev_left_fit, det.prev_right_fit)):
        if p is not None:
            fit[0, k], valid[0, k] = p, 1
    return fit, valid


def check_single(det, lanes, calls, before):
    """A detect_batch-like call: results are the un-truncated records, prev_*_fit aliases the last returned polynomial
    of its side and equals the state the calls left."""
    recs, after = chain(calls, before)
    assert pairs(lanes) == rec_pairs(recs)
    for k, name in enumerate(("prev_left_fit", "prev_right_fit")):
        last = [p[k] for p in lanes if p[k] is not None]
        if last:
            assert getattr(det, name) is last[-1].polynomial
    got = single_state(det)
    np.testing.assert_array_equal(got[0], after[0])
    np.testing.assert_array_equal(got[1], after[1])
    return after


def check_streams(det, calls, before):
    """A per-stream call: the detector's stream state is the state the calls left."""
    recs, after = chain(calls, before)
    np.testing.assert_array_equal(det._stream_fit, after[0])
    np.testing.assert_array_equal(det._stream_valid, after[1])
    return recs


def keys(calls):
    return [c.key for c in calls]


# ------------------------------------------------------------------ single-stream calls
def test_detect(rec):
    det = LaneDetector(max_batch=4)
    state = zeros()
    for t in (7, 9, 3):
        lanes = [det.detect(bgr([t])[0])]
        calls = rec.take()
        assert keys(calls) == [(INGEST, 0, ((BGR, (H, W), (t,), None),), None, 1, True)]
        state = check_single(det, lanes, calls, state)
    assert rec.made == [(0, H, W, 1, 256, 1)]
    assert det.last_records is not None and len(det.last_records) == 1


def test_detect_batch_chunked_over_max_batch(rec):
    det = LaneDetector(max_batch=4)
    lanes = det.detect_batch(bgr(range(10)))
    calls = rec.take()
    assert keys(calls) == [(INGEST, 0, ((BGR, (H, W), tuple(range(a, b)), None),), None, 1, True)
                           for a, b in ((0, 4), (4, 8), (8, 10))]
    state = check_single(det, lanes, calls, zeros())
    assert rec.made == [(0, H, W, 4, 256, 1)] and det.dense_reruns == 0
    assert det.detect_batch(bgr([]).reshape(0, H, W, 3)) == [] and rec.take() == []
    lanes = det.detect_batch(bgr([20, 21]))             # carries the state on, on the same context
    calls = rec.take()
    assert keys(calls) == [(INGEST, 0, ((BGR, (H, W), (20, 21), None),), None, 1, True)]
    check_single(det, lanes, calls, state)
    assert len(det.last_records) == 2


def test_detect_batch_target_size(rec):
    det = LaneDetector(max_batch=4)
    lanes = det.detect_batch(bgr(range(5)), target_size=(32, 24))
    calls = rec.take()
    assert keys(calls) == [(INGEST, 0, ((BGR, (H, W), (0, 1, 2, 3), None),), None, 1, True),
                           (INGEST, 0, ((BGR, (H, W), (4,), None),), None, 1, True)]
    check_single(det, lanes, calls, zeros())
    assert rec.made == [(0, 24, 32, 4, 256, 1)]


def test_detect_batch_overflow_reruns_the_chunk_on_the_dense_context(rec):
    rec.overflow = {5}
    det = LaneDetector(max_batch=4)
    lanes = det.detect_batch(bgr(range(10)))
    calls = rec.take()
    src = lambda a, b: ((BGR, (H, W), tuple(range(a, b)), None),)   # noqa: E731
    assert keys(calls) == [(INGEST, 0, src(0, 4), None, 1, True), (INGEST, 0, src(4, 8), None, 1, True),
                           (INGEST, 1, src(4, 8), None, 1, True), (INGEST, 0, src(8, 10), None, 1, True)]
    assert [c.flagged for c in calls] == [False, True, False, False]
    check_single(det, lanes, calls, zeros())
    assert rec.made == [(0, H, W, 4, 256, 1), (1, H, W, 8, 512, 1)]
    assert det.dense_reruns == 1 and len(det.last_records) == 10


@pytest.mark.parametrize("fmt", [NV12, I420])
@pytest.mark.parametrize("target", [None, (32, 24)])
def test_detect_batch_yuv420(rec, fmt, target):
    det = LaneDetector(max_batch=4)
    call = det.detect_batch_nv12 if fmt == NV12 else det.detect_batch_i420
    lanes = call(yuv(range(6)), target_size=target)
    calls = rec.take()
    assert keys(calls) == [(INGEST, 0, ((fmt, (H, W), (0, 1, 2, 3), None),), None, 1, True),
                           (INGEST, 0, ((fmt, (H, W), (4, 5), None),), None, 1, True)]
    check_single(det, lanes, calls, zeros())
    assert rec.made == [(0, H, W, 4, 256, 1) if target is None else (0, 24, 32, 4, 256, 1)]
    assert call(yuv([]), target_size=target) == [] and rec.take() == []


def test_detect_batches_on_host_batches_are_blocking_calls(rec):
    det = LaneDetector(max_batch=4)
    batches = [bgr(range(3)), bgr(range(10, 15)), bgr([20])]
    state = zeros()
    for b, ctx, lanes in zip(batches, (0, 1, 1), det.detect_batches(batches)):
        calls = rec.take()
        tags = tuple(int(t) for t in b[:, 0, 0, 0])
        assert keys(calls) == [(INGEST, ctx, ((BGR, (H, W), tags[a:a + 4], None),), None, 1, True)
                               for a in range(0, len(tags), 4)]
        state = check_single(det, lanes, calls, state)
    assert rec.made == [(0, H, W, 3, 256, 1), (1, H, W, 4, 256, 1)]      # a larger batch grows the context


# ------------------------------------------------------------------ per-stream calls
ROI = np.array([[(0, 47), (0, 20), (63, 20), (63, 47)]], np.int32)


@pytest.mark.parametrize("rois", [None, [None, ROI]])
def test_detect_streams_5d(rec, rois):
    rec.overflow = {11}
    det = LaneDetector(max_batch=4)
    frames = bgr([10 * s + t for s in range(2) for t in range(3)]).reshape(2, 3, H, W, 3)
    lanes = det.detect_streams(frames, stream_rois=rois)
    calls = rec.take()
    assert keys(calls) == [(INGEST, 0, ((BGR, (H, W), (0, 1, 2, 10), None),), (0, 0, 0, 1), 2, True),
                           (INGEST, 0, ((BGR, (H, W), (11, 12), None),), (1, 1), 2, True),
                           (INGEST, 1, ((BGR, (H, W), (11, 12), None),), (1, 1), 2, True)]
    assert [c.flagged for c in calls] == [False, True, False]
    recs = check_streams(det, calls, zeros(0))
    assert pairs(lanes) == rec_pairs(recs)
    n_roi = 1 if rois is None else 2
    assert rec.made == [(0, H, W, 4, 256, n_roi), (1, H, W, 8, 512, n_roi)]
    assert det.prev_left_fit is None and det.prev_right_fit is None and det.dense_reruns == 1


@pytest.mark.parametrize("rois", [None, [ROI, None, ROI, None]])
def test_detect_streams_with_stream_ids(rec, rois):
    det = LaneDetector(max_batch=4)
    lanes = det.detect_streams(bgr([1, 2, 3, 4, 5]), stream_ids=[2, 0, 2, 1, 0], stream_rois=rois)
    calls = rec.take()
    assert keys(calls) == [(INGEST, 0, ((BGR, (H, W), (1, 2, 3, 4), None),), (2, 0, 2, 1), 3, True),
                           (INGEST, 0, ((BGR, (H, W), (5,), None),), (0,), 3, True)]
    recs = check_streams(det, calls, zeros(0))
    assert pairs(lanes) == rec_pairs(recs)
    state = det._stream_fit.copy(), det._stream_valid.copy()
    # fewer streams: the call still passes every stream the detector holds state for
    lanes = det.detect_streams(bgr([6, 7]), stream_ids=[1, 1], stream_rois=rois)
    calls = rec.take()
    assert keys(calls) == [(INGEST, 0, ((BGR, (H, W), (6, 7), None),), (1, 1), 3, True)]
    assert pairs(lanes) == rec_pairs(check_streams(det, calls, state))
    assert rec.made == [(0, H, W, 4, 256, 1 if rois is None else 4)]
    assert det.detect_streams(bgr([]), stream_ids=[]) == [] and rec.take() == []


# ------------------------------------------------------------------ rigs
RIG_LAYOUTS = ["bgr", "bgr", "nv12", "i420", "i420"]


def rig_tick(base):
    """Cameras of mixed sizes and layouts, one absent and one without frames; 8 frames in all."""
    return [bgr([base, base + 1, base + 2]), None, yuv([base + 10, base + 11], 32, 64), yuv([], 24, 32),
            yuv([base + 20, base + 21, base + 22], 24, 32)]


def rig_calls(base, entry, ctx, explicit=True):
    s = ((BGR, (H, W), (base, base + 1, base + 2), 0), (NV12, (32, 64), (base + 10,), 2))
    t = ((NV12, (32, 64), (base + 11,), 2), (I420, (24, 32), (base + 20, base + 21, base + 22), 4))
    return [(entry, ctx, s, None, 5, explicit), (entry, ctx, t, None, 5, explicit)]


def test_detect_rig_chunks_straddle_cameras(rec):
    det = LaneDetector(max_batch=4)
    out = det.detect_rig(rig_tick(0), RIG_LAYOUTS, target_size=(W, H))
    calls = rec.take()
    assert keys(calls) == rig_calls(0, RIG, 0)
    recs, state = chain(calls, zeros(5))
    lanes = rec_pairs(recs)
    assert [pairs(c) for c in out] == [lanes[0:3], [], lanes[3:5], [], lanes[5:8]]
    np.testing.assert_array_equal(det._stream_fit, state[0])
    out = det.detect_rig(rig_tick(100), RIG_LAYOUTS, target_size=(W, H), stream_rois=[ROI, None, None, ROI, None])
    calls = rec.take()
    assert keys(calls) == rig_calls(100, RIG, 1)
    recs, state = chain(calls, state)
    lanes = rec_pairs(recs)
    assert [pairs(c) for c in out] == [lanes[0:3], [], lanes[3:5], [], lanes[5:8]]
    np.testing.assert_array_equal(det._stream_fit, state[0])
    np.testing.assert_array_equal(det._stream_valid, state[1])
    assert rec.made == [(0, H, W, 4, 256, 1), (1, H, W, 4, 256, 5)]
    assert len(det.last_records) == 8 and det.prev_left_fit is None


def test_detect_rig_one_camera_and_overflow(rec):
    rec.overflow = {11}
    det = LaneDetector(max_batch=4)
    out = det.detect_rig([bgr([1])])
    calls = rec.take()
    assert keys(calls) == [(RIG, 0, ((BGR, (H, W), (1,), 0),), None, 1, True)]
    recs, state = chain(calls, zeros(1))
    assert [pairs(c) for c in out] == [rec_pairs(recs)]
    out = det.detect_rig(rig_tick(0), RIG_LAYOUTS, target_size=(W, H))
    calls = rec.take()
    first, second = rig_calls(0, RIG, 1)
    assert keys(calls) == [first, second, second[:1] + (2,) + second[2:]]
    assert [c.flagged for c in calls] == [False, True, False]
    recs, state = chain(calls, state)
    lanes = rec_pairs(recs)
    assert [pairs(c) for c in out] == [lanes[0:3], [], lanes[3:5], [], lanes[5:8]]
    np.testing.assert_array_equal(det._stream_fit, state[0])
    assert rec.made == [(0, H, W, 1, 256, 1), (1, H, W, 4, 256, 1), (2, H, W, 8, 512, 1)]
    assert det.dense_reruns == 1


def test_detect_rig_stream_ticks_that_cannot_stream_run_blocking(rec):
    """Ticks larger than max_batch and ticks without frames never reach the queue, so this runs without CUDA."""
    det = LaneDetector(max_batch=4)
    ticks = [rig_tick(0), [None, None, None, yuv([], 24, 32), None], rig_tick(100)]
    out = list(det.detect_rig_stream(ticks, RIG_LAYOUTS, target_size=(W, H)))
    calls = rec.take()
    assert keys(calls) == rig_calls(0, RIG, 0) + rig_calls(100, RIG, 0)
    recs, state = chain(calls, zeros(5))
    lanes = rec_pairs(recs)
    assert [[pairs(c) for c in t] for t in out] == [[lanes[0:3], [], lanes[3:5], [], lanes[5:8]], [[]] * 5,
                                                   [lanes[8:11], [], lanes[11:13], [], lanes[13:16]]]
    np.testing.assert_array_equal(det._stream_fit, state[0])
    assert rec.made == [(0, H, W, 4, 256, 1)]


@pytest.mark.gpu
@pytest.mark.skipif(not __import__("torch").cuda.is_available(), reason="pinned staging needs CUDA")
def test_detect_rig_stream_numpy_ticks(rec):
    """Numpy ticks are staged in pinned memory and queued two deep; a tick that overflows is redone blocking."""
    rec.overflow = {41}
    det = LaneDetector(max_batch=8)
    small = lambda b: [bgr([b, b + 1]), None, yuv([b + 10, b + 11], 32, 64)]   # noqa: E731
    big = [bgr(range(90, 99)), None, yuv([100], 32, 64)]                        # 10 frames > max_batch
    ticks, layouts = [small(0), small(30), small(60), big, small(120)], ["bgr", "bgr", "nv12"]
    out = list(det.detect_rig_stream(ticks, layouts, target_size=(W, H)))
    calls = rec.take()
    src = lambda b: ((BGR, (H, W), (b, b + 1), 0), (NV12, (32, 64), (b + 10, b + 11), 2))   # noqa: E731
    chunks = [((BGR, (H, W), tuple(range(90, 98)), 0),), ((BGR, (H, W), (98,), 0), (NV12, (32, 64), (100,), 2))]
    assert keys(calls) == [
        (RIG_ENQUEUE, 0, src(0), None, 3, True), (RIG_ENQUEUE, 0, src(30), None, 3, False),
        (COLLECT, 0, (), None, None, False),                                  # tick 0
        (RIG_ENQUEUE, 0, src(60), None, 3, False), (COLLECT, 0, (), None, None, False),   # tick 1 overflowed
        (COLLECT, 0, (), None, None, False),                                  # drained: tick 2
        (RIG, 0, src(30), None, 3, True), (RIG, 1, src(30), None, 3, True),  # tick 1 redone, then dense
        (RIG_ENQUEUE, 0, src(60), None, 3, True), (COLLECT, 0, (), None, None, False),   # tick 2; tick 3 cannot join
        (RIG, 0, chunks[0], None, 3, True), (RIG, 0, chunks[1], None, 3, True),   # tick 3, blocking
        (RIG_ENQUEUE, 0, src(120), None, 3, True), (COLLECT, 0, (), None, None, False),
    ]
    # the same ticks through detect_rig, one after another
    ref = LaneDetector(max_batch=8)
    want = [ref.detect_rig(t, layouts, target_size=(W, H)) for t in ticks]
    assert [[pairs(c) for c in t] for t in out] == [[pairs(c) for c in t] for t in want]
    np.testing.assert_array_equal(det._stream_fit, ref._stream_fit)
    np.testing.assert_array_equal(det._stream_valid, ref._stream_valid)
    np.testing.assert_array_equal(det.last_records, ref.last_records)
