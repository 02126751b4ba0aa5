"""The host/device boundary shared by the context-free entry points (csrc/host_stage.h): each of the nine reports a
failure under its own name, answers a missing GPU with LANE_ERR_NO_DEVICE and a device index out of range with
LANE_ERR_INVALID, and host batches large enough to take the staging ring (pageable, 24 MB or more) come out byte-equal
to the same batch as a CUDA tensor."""
import ctypes as C

import numpy as np
import pytest

from multimodal_autonomous_driving_perception_and_planning_b200 import FrameIngest, _native, draw_lanes_batch
from multimodal_autonomous_driving_perception_and_planning_b200.perception.scene_stats import SceneStatsAnalyzer

N, H, W = 2, 4, 6
NO_DEVICE, INVALID = -3, -1


def _calls():
    """One valid call per entry point, `device` left open; the buffers stay alive with the returned closures."""
    bgr = np.zeros((N, H, W, 3), np.uint8)
    yuv = np.zeros((N, H * 3 // 2, W), np.uint8)
    pts = np.zeros((N, 50, 2), np.int32)
    valid = np.zeros(N, np.uint8)
    commands = np.zeros(1, np.int32)
    begin = np.zeros(N + 1, np.int64)
    stats = (C.c_uint64 * (4 * N))()
    keep = (bgr, yuv, pts, valid, commands, begin, stats)
    p = lambda a: a.ctypes.data_as(C.c_void_p)      # noqa: E731
    lib = _native.lib()
    calls = {
        "lane_resize_batch": lambda d: lib.lane_resize_batch(p(bgr), N, H, W, 3, p(bgr), H, W, 0, d, None),
        "lane_nv12_to_bgr_batch": lambda d: lib.lane_nv12_to_bgr_batch(p(yuv), N, H, W, p(bgr), 0, d, None),
        "lane_yuv420_to_bgr_batch": lambda d: lib.lane_yuv420_to_bgr_batch(p(yuv), _native.INPUT_I420, N, H, W, p(bgr), H, W,
                                                                           0, d, None),
        "lane_bgr_to_yuv420_batch": lambda d: lib.lane_bgr_to_yuv420_batch(p(bgr), _native.INPUT_I420, N, H, W, p(yuv), 1, d,
                                                                           None),
        "lane_frame_stats": lambda d: lib.lane_frame_stats(p(bgr), 0, N, H, W, stats, d, None),
        "lane_draw_commands": lambda d: lib.lane_draw_commands(p(bgr), 0, N, H, W, p(commands), p(begin), d, None, None),
        "lane_generate_frames": lambda d: lib.lane_generate_frames(p(bgr), 0, N, H, W, 0, d, None, None),
        "lane_draw_lanes_batch": lambda d: lib.lane_draw_lanes_batch(p(bgr), 0, N, H, W, p(pts), p(valid), p(pts), p(valid),
                                                                     1, d, None, None),
        "lane_draw_lanes_records": lambda d: lib.lane_draw_lanes_records(p(bgr), N, H, W, p(bgr), 1, d, None),
    }
    return calls, keep


def test_nine_entry_points_name_themselves_without_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    calls, _keep = _calls()
    assert len(calls) == 9
    for name, call in calls.items():
        assert call(0) == NO_DEVICE, name
        msg = _native.lib().lane_last_error(None)
        assert msg.startswith(name.encode() + b": ") and b"no CPU fallback" in msg, (name, msg)


@pytest.mark.gpu
@pytest.mark.parametrize("device", [4096, -1])
def test_device_out_of_range_is_an_invalid_argument(device):
    calls, _keep = _calls()
    for name, call in calls.items():
        assert call(device) == INVALID, name
        msg = _native.lib().lane_last_error(None)
        assert msg.startswith(name.encode() + b": ") and b"device out of range" in msg, (name, msg)


def _rng_frames(shape, seed):
    return np.random.default_rng(seed).integers(0, 256, shape, dtype=np.uint8)


@pytest.mark.gpu
def test_pageable_host_batches_through_the_ring_equal_the_device_path():
    import torch
    # 32 x 480 x 640 BGR = 29 MB in, upscaled to 88 MB out: the ring in both directions
    frames = _rng_frames((32, 480, 640, 3), 1)
    assert frames.nbytes >= 24 << 20
    ing = FrameIngest((1280, 720))
    host = ing.resize_batch(frames)
    assert host.nbytes >= 24 << 20
    assert np.array_equal(host, ing.resize_batch(torch.from_numpy(frames).cuda()).cpu().numpy())

    # 12 NV12 frames at 1080p = 37 MB, converted and resized in one pass
    nv12 = _rng_frames((12, 1080 * 3 // 2, 1920), 2)
    ing = FrameIngest((640, 360))
    assert np.array_equal(ing.from_nv12(nv12), ing.from_nv12(torch.from_numpy(nv12).cuda()).cpu().numpy())

    # frame statistics of 29 MB of host frames: input only
    stats = SceneStatsAnalyzer()
    assert stats.analyze_batch(frames) == stats.analyze_batch(torch.from_numpy(frames).cuda())

    # lanes drawn in place on 29 MB of host frames: the ring both ways
    t = np.linspace(0.0, 1.0, 50)
    left = np.stack([100 + 180 * t, 479 - 180 * t], -1).round().astype(np.int32)
    right = np.stack([540 - 180 * t, 479 - 180 * t], -1).round().astype(np.int32)
    lanes = [(left if i % 3 != 1 else None, right if i % 4 != 2 else None) for i in range(frames.shape[0])]
    on_host = draw_lanes_batch(frames.copy(), lanes)
    on_device = draw_lanes_batch(torch.from_numpy(frames).cuda(), lanes).cpu().numpy()
    assert not np.array_equal(on_host, frames)
    assert np.array_equal(on_host, on_device)
