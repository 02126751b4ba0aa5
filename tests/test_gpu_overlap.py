"""Two batches in flight with the back half of the path (PPHT, fit, record copies) on the context's second stream: the
edge kernels of batch i+1 run while batch i is still in its Hough transform, on buffers kept per result slot.  Records must
equal those of running the batches one after the other, byte for byte, at a size where the kernels really overlap."""
import numpy as np
import pytest

from multimodal_autonomous_driving_perception_and_planning_b200 import LaneDetector, SyntheticDataGenerator, _native

pytestmark = pytest.mark.gpu


def _batches(w, h, n, count):
    import torch
    gen = SyntheticDataGenerator(w, h)
    out = []
    for b in range(count):               # different content per batch: distinct stretches of the stream, one with noise
        fr = gen.generate_batch_device(n, start_frame=37 * b)
        if b == 2:
            g = torch.Generator(device="cuda").manual_seed(5)
            noise = torch.randint(0, 256, fr[: n // 4].shape, dtype=torch.uint8, device="cuda", generator=g)
            fr[: n // 4] = noise          # dense frames: thousands of ROI points, PPHT falls to the global-memory kernel
        out.append(fr)
    return out


@pytest.mark.parametrize("w,h,n", [(1920, 1080, 96), (640, 480, 150)])
def test_streaming_with_overlap_equals_batch_after_batch(w, h, n):
    import torch
    batches = _batches(w, h, n, 6)
    det = LaneDetector(max_batch=n, max_segments=4096)
    want = []
    for fr in batches:
        det.detect_batch(fr)
        want.append(det.last_records.copy())
    det.close()

    det = LaneDetector(max_batch=n, max_segments=4096)
    ctx = det._context(h, w, n)
    pf, pv = np.zeros((1, 2, 3)), np.zeros((1, 2), np.uint8)
    for rep in range(3):                 # repeated: a race would not show every time
        pf[:] = 0
        pv[:] = 0
        ctx.enqueue(batches[0].data_ptr(), n, None, 1, pf, pv, 0.7, 1 - 0.7)
        got = []
        for i in range(len(batches)):
            if i + 1 < len(batches):
                ctx.enqueue(batches[i + 1].data_ptr(), n, None, 1, None, None, 0.7, 1 - 0.7)
            got.append(ctx.collect(pf, pv).copy())
        for i, (a, b) in enumerate(zip(got, want)):
            assert a.tobytes() == b.tobytes(), (rep, i)
    assert ctx.last_paths() & _native.PATH_FUSED_EDGE
    # profiling mode (one stream, stage events) interleaved with the two-stream mode gives the same records
    ctx.set_profiling(True)
    pf[:] = 0
    pv[:] = 0
    ctx.enqueue(batches[0].data_ptr(), n, None, 1, pf, pv, 0.7, 1 - 0.7)
    ctx.enqueue(batches[1].data_ptr(), n, None, 1, None, None, 0.7, 1 - 0.7)
    a = ctx.collect(pf, pv).copy()
    ctx.set_profiling(False)
    ctx.enqueue(batches[2].data_ptr(), n, None, 1, None, None, 0.7, 1 - 0.7)     # mode changes with a batch in flight
    b = ctx.collect(pf, pv).copy()
    c = ctx.collect(pf, pv).copy()
    assert [x.tobytes() for x in (a, b, c)] == [x.tobytes() for x in want[:3]]
    ms, _ = ctx.stage_ms()
    assert ms["ppht"] > 0
    det.close()


def test_detect_batches_generator_equals_detect_batch_batch_after_batch():
    """The public pipelined form: same lanes, same state chain, dense batches re-run, odd batches passed through."""
    import torch
    w, h, n = 1920, 1080, 48
    batches = _batches(w, h, n, 6)
    batches.insert(3, batches[1][:17].contiguous())                    # a shorter batch in the middle
    host_batch = batches[0][:5].cpu().numpy()                          # a host batch: goes through detect_batch
    seq = batches[:5] + [host_batch] + batches[5:]
    ref_det = LaneDetector(max_batch=n, max_segments=256)              # small cap: the noise batch overflows it
    want = [ref_det.detect_batch(b) for b in seq]
    assert ref_det.dense_reruns >= 1
    det = LaneDetector(max_batch=n, max_segments=256)
    got = list(det.detect_batches(seq))
    assert len(got) == len(want)
    for k, (a, b) in enumerate(zip(got, want)):
        assert len(a) == len(b)
        for (la, ra), (lb, rb) in zip(a, b):
            for x, y in ((la, lb), (ra, rb)):
                assert (x is None) == (y is None), k
                if x is not None:
                    assert np.array_equal(x.points, y.points) and np.array_equal(x.polynomial, y.polynomial), k
                    assert x.confidence == y.confidence and x.side == y.side
    assert np.array_equal(det.prev_left_fit, ref_det.prev_left_fit) and np.array_equal(det.prev_right_fit, ref_det.prev_right_fit)
    assert det.dense_reruns == ref_det.dense_reruns
    # stopping early leaves nothing in flight
    g = det.detect_batches(batches)
    next(g)
    g.close()
    assert not det._ctx._inflight
    det.detect_batch(batches[0])
    det.close()
    ref_det.close()


def test_detect_batches_yields_the_batches_before_a_malformed_one_then_raises():
    """A malformed batch raises detect_batch's error when its turn comes: the batches before it are yielded first, and
    nothing is left in flight."""
    import cv2
    batches = _batches(640, 480, 8, 2)
    ref = LaneDetector(max_batch=8)
    want = [ref.detect_batch(b) for b in batches]
    det = LaneDetector(max_batch=8)
    got = []
    with pytest.raises(cv2.error):
        for lanes in det.detect_batches(batches + [batches[0][..., :2], batches[0]]):
            got.append(lanes)
    assert len(got) == len(want)
    for a, b in zip(got, want):
        for pa, pb in zip(a, b):
            for x, y in zip(pa, pb):
                assert (x is None) == (y is None)
                assert x is None or (np.array_equal(x.points, y.points) and np.array_equal(x.polynomial, y.polynomial))
    assert np.array_equal(det.prev_left_fit, ref.prev_left_fit) and np.array_equal(det.prev_right_fit, ref.prev_right_fit)
    assert not det._ctx._inflight
    det.close()
    ref.close()
