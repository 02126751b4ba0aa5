"""The camera frame layouts ``LaneDetector`` and ``FrameIngest`` take: one row per layout name of ``detect_rig``.

Every shape check, size rule and byte count of the Python side asks this table (the native side's is the
``lane_input_*`` set in ``csrc/k0_common.cuh``, which refuses the same sizes).  A row gives the ``INPUT_*`` code, how an
array of frames ``[N, ...]`` holds an H x W frame, the sizes the conversion takes and the context-free entry that
converts the layout on its own.
"""
from typing import NamedTuple, Optional, Tuple

import cv2

from .. import _native


class Layout(NamedTuple):
    fmt: int                  # LANE_INPUT_*
    family: str               # what messages call the layout
    dims: str                 # the array's shape after its frame count, as messages print it
    planar: bool              # 4:2:0: the array has H*3/2 rows (Y, then the chroma planes)
    channels: int             # the array's last dimension; 0 for [N, rows, W]
    h_step: int               # H a multiple of h_step, W of w_step, both at least min_side
    w_step: int
    min_side: int
    rule: str                 # the size rule in words ("" when every size is taken)
    entry: Optional[str]      # the context-free conversion entry (BGR has none)

    def frame_shape(self, h: int, w: int) -> Tuple[int, ...]:
        """The shape of one h x w frame of this layout in an array."""
        return (h * 3 // 2 if self.planar else h, w) + ((self.channels,) if self.channels else ())

    def frame_bytes(self, h: int, w: int) -> int:
        """Bytes of one dense h x w frame: 3 B/px BGR, 1.5 B/px YUV 4:2:0, 1 B/px Bayer, 2 B/px YUV 4:2:2."""
        rows, w, *c = self.frame_shape(h, w)
        return rows * w * (c[0] if c else 1)

    def hw(self, shape) -> Optional[Tuple[int, int]]:
        """(H, W) of the frames of an array of ``shape`` ``[N, ...]``, or None when its rank or last dimension is not
        this layout's."""
        shape = tuple(int(x) for x in shape)
        if len(shape) != (4 if self.channels else 3) or (self.channels and shape[3] != self.channels):
            return None
        if self.planar:
            return None if shape[1] % 3 else (shape[1] * 2 // 3, shape[2])
        return shape[1], shape[2]

    def refuses(self, h: int, w: int) -> bool:
        """Whether the conversion refuses h x w frames (``rule`` says why)."""
        return bool(h % self.h_step or w % self.w_step or min(h, w) < self.min_side)


_YUV420 = dict(family="YUV 4:2:0", dims="H*3/2,W", planar=True, channels=0, h_step=2, w_step=2, min_side=1,
               rule="even width and height", entry="lane_yuv420_to_bgr_batch")
_BAYER = dict(family="Bayer", dims="H,W", planar=False, channels=0, h_step=1, w_step=1, min_side=3,
              rule="at least 3 rows and 3 columns", entry="lane_bayer_to_bgr_batch")
_YUV422 = dict(family="YUV 4:2:2", dims="H,W,2", planar=False, channels=2, h_step=1, w_step=2, min_side=1,
               rule="an even width", entry="lane_yuv422_to_bgr_batch")

LAYOUTS = {
    "bgr": Layout(_native.INPUT_BGR, "BGR", "H,W,3", False, 3, 1, 1, 1, "", None),
    "nv12": Layout(_native.INPUT_NV12, **_YUV420),
    "i420": Layout(_native.INPUT_I420, **_YUV420),
    **{"bayer_" + p: Layout(fmt, **_BAYER) for p, fmt in _native.BAYER.items()},
    **{o: Layout(fmt, **_YUV422) for o, fmt in _native.YUV422.items()},
}
BY_FORMAT = {lay.fmt: lay for lay in LAYOUTS.values()}


def named(name, names: dict, what: str) -> Layout:
    """The layout ``names[name]`` names (``_native.BAYER`` by pattern, ``_native.YUV422`` by byte order), else
    ``ValueError``."""
    if not isinstance(name, str) or name not in names:
        raise ValueError(f"{what} {name!r} is not one of {sorted(names)}")
    return BY_FORMAT[names[name]]


def check_frames(frames, layout: Layout, who: str) -> Tuple[int, int]:
    """(H, W) of uint8 frames ``[N, ...]`` in ``layout`` at a size it takes, else ``cv2.error`` (what cv2.cvtColor
    raises)."""
    shape = tuple(frames.shape)
    hw = layout.hw(shape)
    if hw is None or layout.refuses(*hw):
        raise cv2.error(f"{who}: expected {layout.family} frames [N,{layout.dims}]"
                        f"{' with ' + layout.rule if layout.rule else ''}, got {shape}")
    if str(frames.dtype).replace("torch.", "") != "uint8":
        raise cv2.error(f"{who}: expected uint8 frames, got {frames.dtype}")
    return hw
