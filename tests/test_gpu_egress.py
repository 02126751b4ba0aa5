"""Annotated frames out to an encoder's layout on the device (K8, csrc/k8_egress.cu): bgr_to_i420 / bgr_to_nv12 of CUDA
tensors byte-equal to cv2.cvtColor(f, COLOR_BGR2YUV_I420) and the oracle for every destination (device tensor, host
numpy, pinned CPU tensor, a pageable batch that takes the staging ring over several chunks), misaligned pointers and
widths that are not a multiple of 8; stream ordering; the whole annotate chain; a round trip into the project's own
I420 ingest; and the raw entry's device-side argument checks.

Run on the B200 box: python -m pytest tests -m gpu.
"""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

import cv2  # noqa: E402

from multimodal_autonomous_driving_perception_and_planning_b200 import (LaneDetector, OverlayRenderer,  # noqa: E402
                                                                        SyntheticDataGenerator, _native, bgr_to_i420,
                                                                        bgr_to_nv12)
from draw_util import cv2_draw_lanes, cv2_offset_indicator  # noqa: E402
import bgr_yuv420 as egress  # noqa: E402
from test_oracle_egress import SIZES, random_bgr, random_sizes  # noqa: E402
from util import gen_frames  # noqa: E402
from yuv420 import i420_to_nv12  # noqa: E402

FNS = {"i420": bgr_to_i420, "nv12": bgr_to_nv12}
ORACLE = {"i420": egress.bgr_to_i420, "nv12": egress.bgr_to_nv12}
ODD_WIDTHS = [(4, 6), (10, 66), (8, 1924), (480, 644)]          # W % 8 != 0: the scalar kernel


def cv2_yuv(frames, layout):
    out = np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420) for f in frames])
    return out if layout == "i420" else np.stack([i420_to_nv12(f) for f in out])


def _pinned(shape):
    import torch
    return torch.empty(shape, dtype=torch.uint8).pin_memory()


@pytest.mark.parametrize("layout", ["i420", "nv12"])
@pytest.mark.parametrize("hw", SIZES + ODD_WIDTHS)
def test_kernel_equals_cv2_and_oracle_for_every_destination(layout, hw):
    import torch
    frames = np.stack([random_bgr(hw, 31 * k + hw[0] + hw[1]) for k in range(2)])
    want = cv2_yuv(frames, layout)
    assert np.array_equal(want[1], ORACLE[layout](frames[1]))
    fn = FNS[layout]
    src = torch.from_numpy(frames).cuda()
    got = fn(src)
    assert got.is_cuda and tuple(got.shape) == want.shape
    assert np.array_equal(got.cpu().numpy(), want)
    host = np.zeros(want.shape, np.uint8)
    assert fn(src, out=host) is host and np.array_equal(host, want)
    pinned = _pinned(want.shape)
    assert fn(src, out=pinned) is pinned and np.array_equal(pinned.numpy(), want)
    dev = torch.zeros(want.shape, dtype=torch.uint8, device="cuda")
    assert fn(src, out=dev) is dev and np.array_equal(dev.cpu().numpy(), want)


@pytest.mark.parametrize("layout", ["i420", "nv12"])
def test_random_even_sizes(layout):
    import torch
    for k, hw in enumerate(random_sizes(k=40, seed=11)):
        frames = np.stack([random_bgr(hw, 500 + k), random_bgr(hw, 600 + k)])
        got = FNS[layout](torch.from_numpy(frames).cuda()).cpu().numpy()
        assert np.array_equal(got, cv2_yuv(frames, layout)), hw


@pytest.mark.parametrize("layout", ["i420", "nv12"])
@pytest.mark.parametrize("where", ["pageable", "pinned"])
def test_large_host_batch_over_several_chunks(layout, where):
    """16 x 1080p = 50 MB of output: two conversion chunks; a pageable destination of this size takes the staging
    ring, a pinned one the DMA."""
    import torch
    frames = np.stack([random_bgr((1080, 1920), 900 + k) for k in range(16)])
    want = cv2_yuv(frames, layout)
    assert want.nbytes >= 24 << 20
    out = np.zeros(want.shape, np.uint8) if where == "pageable" else _pinned(want.shape)
    got = FNS[layout](torch.from_numpy(frames).cuda(), out=out)
    assert got is out
    assert np.array_equal(np.asarray(got), want)


@pytest.mark.parametrize("layout", ["i420", "nv12"])
@pytest.mark.parametrize("hw", [(480, 640), (6, 10)])
def test_misaligned_source_and_destination(layout, hw):
    import torch
    frames = np.stack([random_bgr(hw, 77 + k) for k in range(3)])
    want = cv2_yuv(frames, layout)
    flat = torch.zeros(frames.size + 1, dtype=torch.uint8, device="cuda")
    flat[1:] = torch.from_numpy(frames.reshape(-1)).cuda()
    src_odd = flat[1:].view(frames.shape)
    assert np.array_equal(FNS[layout](src_odd).cpu().numpy(), want)
    dflat = torch.zeros(want.size + 1, dtype=torch.uint8, device="cuda")
    dst_odd = dflat[1:].view(want.shape)
    FNS[layout](torch.from_numpy(frames).cuda(), out=dst_odd)
    assert np.array_equal(dst_odd.cpu().numpy(), want)
    hflat = np.zeros(want.size + 1, np.uint8)
    host_odd = hflat[1:].reshape(want.shape)
    FNS[layout](src_odd, out=host_odd)
    assert np.array_equal(host_odd, want)


def test_empty_batch():
    import torch
    got = bgr_to_i420(torch.zeros((0, 4, 6, 3), dtype=torch.uint8, device="cuda"))
    assert got.is_cuda and tuple(got.shape) == (0, 6, 6)
    out = np.zeros((0, 6, 6), np.uint8)
    assert bgr_to_nv12(torch.zeros((0, 4, 6, 3), dtype=torch.uint8, device="cuda"), out=out) is out
    a = torch.zeros(72, dtype=torch.uint8, device="cuda")
    assert _native.lib().lane_bgr_to_yuv420_batch(ctypes.c_void_p(a.data_ptr()), _native.INPUT_I420, 0, 4, 6,
                                                  ctypes.c_void_p(a.data_ptr()), 1, 0, None) == 0


@pytest.mark.parametrize("layout", ["i420", "nv12"])
def test_frames_written_on_the_current_stream_convert_without_a_sync(layout):
    """The frames are rasterised by a kernel on a side stream made current; the conversion follows it on that stream
    without an explicit synchronisation, into device and host memory."""
    import torch
    gen = SyntheticDataGenerator(1920, 1080)
    want = cv2_yuv(gen.generate_batch(8, start_frame=40), layout)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        frames = gen.generate_batch_device(8, start_frame=40)
        dev = FNS[layout](frames)
        host = FNS[layout](gen.generate_batch_device(8, start_frame=40), out=np.zeros(want.shape, np.uint8))
    s.synchronize()
    assert np.array_equal(host, want)
    assert np.array_equal(dev.cpu().numpy(), want)


def test_annotate_chain_to_i420_equals_cv2():
    """generator frames -> detect_batches -> draw_lanes_batch -> offset indicator -> bgr_to_i420(out=host), against
    cv2's calls on the host frames."""
    import torch
    n, w, h = 32, 1920, 1080
    gen = SyntheticDataGenerator(w, h)
    batches = [gen.generate_batch_device(n, start_frame=k * n) for k in range(2)]
    clean = [b.cpu().numpy() for b in batches]
    det, ov = LaneDetector(max_batch=n), OverlayRenderer()
    out = _pinned((n, h * 3 // 2, w))
    for i, lanes in enumerate(det.detect_batches(batches)):
        view = batches[i]
        det.draw_lanes_batch(view, lanes)
        offs = [det.get_lane_center_offset(w, l, r) for l, r in lanes]
        ov.draw_lane_offset_indicator_batch(view, offs)
        got = bgr_to_i420(view, out=out).numpy()
        for k in range(0, n, 5):
            l, r = lanes[k]
            drawn = cv2_offset_indicator(cv2_draw_lanes(clean[i][k].copy(), None if l is None else l.points,
                                                        None if r is None else r.points), offs[k])
            assert np.array_equal(got[k], cv2.cvtColor(drawn, cv2.COLOR_BGR2YUV_I420)), (i, k)
    torch.cuda.synchronize()
    det.close()


def test_round_trip_into_the_i420_ingest():
    """detect_batch_i420(bgr_to_i420(frames)) equals detect_batch of cv2's I420 round trip of the same frames."""
    import torch
    bgr = np.stack(gen_frames(1920, 1080, 12))
    i420 = bgr_to_i420(torch.from_numpy(bgr).cuda())
    prepared = np.stack([cv2.cvtColor(cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420), cv2.COLOR_YUV2BGR_I420) for f in bgr])
    a, b = LaneDetector(max_batch=12), LaneDetector(max_batch=12)
    got = a.detect_batch_i420(i420)
    want = b.detect_batch(prepared)
    assert a.last_records.tobytes() == b.last_records.tobytes()
    for p, q in ((a.prev_left_fit, b.prev_left_fit), (a.prev_right_fit, b.prev_right_fit)):
        assert (p is None) == (q is None) and (p is None or np.asarray(p).tobytes() == np.asarray(q).tobytes())
    assert len(got) == len(want)
    a.close()
    b.close()


def test_raw_entry_rejects_host_sources_and_bad_device_arguments():
    import torch
    lib = _native.lib()
    host = np.zeros(4 * 6 * 3, np.uint8)
    hp = host.ctypes.data_as(ctypes.c_void_p)
    d = torch.zeros(4 * 6 * 3, dtype=torch.uint8, device="cuda")
    dp = ctypes.c_void_p(d.data_ptr())
    I420 = _native.INPUT_I420
    assert lib.lane_bgr_to_yuv420_batch(hp, I420, 1, 4, 6, dp, 1, 0, None) == -1        # host source
    assert b"device memory" in lib.lane_last_error(None)
    assert lib.lane_bgr_to_yuv420_batch(dp, I420, 1, 4, 6, hp, 1, 0, None) == -1        # host dst flagged as device
    assert lib.lane_bgr_to_yuv420_batch(dp, I420, 1, 4, 6, dp, 1, 4096, None) == -1     # device out of range
    assert lib.lane_bgr_to_yuv420_batch(dp, I420, 1, 4, 6, dp, 1, -1, None) == -1
    assert lib.lane_bgr_to_yuv420_batch(dp, 3, 1, 4, 6, dp, 1, 0, None) == -1           # unknown format
    assert lib.lane_bgr_to_yuv420_batch(dp, I420, 1, 4, 5, dp, 1, 0, None) == -1        # odd width
    assert lib.lane_bgr_to_yuv420_batch(dp, I420, 1, 4, 6, hp, 0, 0, None) == 0         # and valid calls still work
    torch.cuda.synchronize()
    assert np.array_equal(host[:36].reshape(6, 6), cv2.cvtColor(np.zeros((4, 6, 3), np.uint8), cv2.COLOR_BGR2YUV_I420))
