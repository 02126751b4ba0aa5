"""The two-deep queue that ``LaneDetector.detect_batches`` and ``detect_rig_stream`` share, driven with a fake context
and fake callables, so its protocol (order, depth, explicit state, overflow restarts, errors, early close) is checked
without a GPU.

An item is ``(kind, v)``: its result is the state after it, the state before plus ``v``.  ``"dev"`` items stream,
``"host"`` items can neither start nor join the queue (they run blocking), ``"over"`` items overflow their segment lists
in the queue (their device state is then wrong on purpose, so the items behind them must be redone), and ``"bad"``
is a malformed item that ``plan`` rejects."""
import numpy as np
import pytest

from multimodal_autonomous_driving_perception_and_planning_b200.perception.lane_detector import _two_deep

REC = np.dtype([("flags", np.int32)])


class FakeContext:
    def __init__(self):
        self._inflight = []           # (state after, overflowed) of the items in flight, oldest first
        self.device_state = None
        self.deepest = 0

    def enqueue(self, v, overflow, explicit_state):
        if explicit_state is not None:
            self.device_state = explicit_state
        assert self.device_state is not None, "an item without explicit state needs one on the device"
        self.device_state += 1000.0 if overflow else v
        self._inflight.append((self.device_state, overflow))
        self.deepest = max(self.deepest, len(self._inflight))

    def collect(self, fit, valid):
        state, overflow = self._inflight.pop(0)
        fit[0] = state
        valid[0] = 1
        return np.array([(int(overflow),)], REC)


class Detector:
    """The callables a user of the driver supplies, over a detector whose state is one number."""

    def __init__(self):
        self.state = 0.0
        self.ctx = FakeContext()
        self.fit = self.valid = None
        self.planned, self.enqueued, self.blocked = [], [], []

    def plan(self, item):
        self.planned.append(item)
        if item[0] == "bad":
            raise ValueError(f"malformed item {item}")
        return item

    def joins(self, p):
        return p[0] in ("dev", "over")

    def start(self, p):
        if not self.joins(p):
            return None
        self.fit, self.valid = np.array([self.state]), np.zeros(1, np.uint8)
        return self.ctx, self.fit, self.valid

    def enqueue(self, item, p, explicit):
        self.enqueued.append((item, explicit))
        self.ctx.enqueue(item[1], item[0] == "over", self.fit[0] if explicit else None)
        return item

    def blocking(self, item, p):
        self.blocked.append(item)
        self.state += item[1]
        return item, self.state

    def restore(self, fit, valid):
        self.state = float(fit[0])

    def adopt(self, recs, p):
        self.state = float(self.fit[0])
        return p, self.state

    def run(self, items):
        return _two_deep(items, self.plan, self.start, self.joins, self.enqueue, self.blocking, self.restore, self.adopt)


def expected(items):
    out, state = [], 0.0
    for it in items:
        state += it[1]
        out.append((it, state))
    return out


def test_items_come_out_in_order_two_in_flight_explicit_state_only_at_start():
    items = [("dev", v) for v in (1, 2, 3, 4, 5, 6)]
    det = Detector()
    assert list(det.run(items)) == expected(items)
    assert det.ctx.deepest == 2
    assert det.enqueued == [(it, k == 0) for k, it in enumerate(items)]
    assert det.blocked == [] and not det.ctx._inflight
    assert det.planned == items            # each item planned once when nothing restarts


def test_overflowing_item_is_redone_blocking_and_the_rest_replanned_in_order():
    items = [("dev", 1), ("dev", 2), ("over", 4), ("dev", 8), ("dev", 16), ("dev", 32)]
    det = Detector()
    assert list(det.run(items)) == expected(items)
    assert det.blocked == [("over", 4)]    # from the state before it: 1 + 2
    assert det.ctx.deepest == 2
    # the item behind the overflowing one was planned for the queue, then again after the restart, which starts
    # with explicit state
    assert det.planned.count(("dev", 8)) == 2
    explicit = [it for it, e in det.enqueued if e]
    assert explicit == [("dev", 1), ("dev", 8)]


def test_overflow_at_the_end_and_back_to_back():
    items = [("dev", 1), ("over", 2), ("over", 4), ("dev", 8)]
    det = Detector()
    assert list(det.run(items)) == expected(items)
    assert det.blocked == [("over", 2), ("over", 4)]
    assert not det.ctx._inflight
    items = [("dev", 1), ("over", 2)]
    det = Detector()
    assert list(det.run(items)) == expected(items)


def test_item_that_cannot_join_runs_blocking_between_streamed_items():
    items = [("dev", 1), ("dev", 2), ("host", 4), ("dev", 8), ("host", 16), ("host", 32), ("dev", 64)]
    det = Detector()
    assert list(det.run(items)) == expected(items)
    assert det.blocked == [("host", 4), ("host", 16), ("host", 32)]
    assert [it for it, e in det.enqueued if e] == [("dev", 1), ("dev", 8), ("dev", 64)]
    assert det.ctx.deepest <= 2


@pytest.mark.parametrize("where", [0, 1, 2, 4])
def test_malformed_item_raises_after_the_items_before_it_are_yielded(where):
    items = [("dev", 1), ("dev", 2), ("host", 4), ("dev", 8), ("dev", 16)]
    items.insert(where, ("bad", 0))
    det = Detector()
    got = []
    with pytest.raises(ValueError, match="malformed"):
        for r in det.run(items):
            got.append(r)
    assert got == expected(items[:where])
    assert not det.ctx._inflight           # the queue was drained on the way out


def test_closing_early_leaves_nothing_in_flight():
    items = [("dev", v) for v in range(1, 7)]
    det = Detector()
    g = det.run(items)
    assert next(g) == expected(items)[0]
    assert det.ctx._inflight               # the next item is queued
    g.close()
    assert not det.ctx._inflight
    assert list(det.run([])) == []
