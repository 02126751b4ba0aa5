"""TEST INFRASTRUCTURE ONLY -- CPU restatement of ``cv2.cvtColor(raw, cv2.COLOR_Bayer{RGGB,BGGR,GRBG,GBRG}2BGR)``
(uint8).

A camera that skips the ISP records the sensor's raw 8-bit Bayer mosaic: 1 B/px, one colour sample per pixel.  A cv2
user turns it into the BGR frame ``LaneDetector`` takes with ``cv2.cvtColor(raw, cv2.COLOR_BayerRGGB2BGR)`` (the
bilinear demosaic), then ``cv2.resize`` to the loader's ``target_size``.  The four pattern names give the sensor's
top-left 2x2: RGGB means row 0 is R G and row 1 is G B.  They are cv2's newer aliases:
``COLOR_BayerRGGB2BGR == COLOR_BayerBG2BGR``, ``BGGR == RG``, ``GRBG == GB``, ``GBRG == GR``.

The four patterns are one RGGB mosaic read at a phase (py, px): RGGB (0, 0), GRBG (0, 1), GBRG (1, 0), BGGR (1, 1).
For H >= 3 and W >= 3, output pixel (y, x) is the interior formula evaluated at (clamp(y, 1, H-2), clamp(x, 1, W-2)):

    own colour                         the raw value
    at an R or B site:  G            = (up + down + left + right + 2) >> 2
                        other chroma = (four diagonals + 2) >> 2
    at a G site:        colour of the horizontal neighbours = (left + right + 1) >> 1
                        colour of the vertical neighbours   = (up + down + 1) >> 1

Below 3 rows or 3 columns cv2 returns an all-zero frame; that case is refused here (ValueError) as it is on the device.
Pinned against cv2 by tests/test_bayer_host.py; csrc/k0_common.cuh (k0_bayer_resize_px) computes the same.

Only tests/, __graft_entry__.smoke() and the probes under tools/ may import this module.
"""
import numpy as np

PHASE = {"rggb": (0, 0), "grbg": (0, 1), "gbrg": (1, 0), "bggr": (1, 1)}


def bayer_to_bgr(raw: np.ndarray, pattern: str) -> np.ndarray:
    """uint8 [H, W] mosaic (H, W >= 3) in ``pattern`` ("rggb", "bggr", "grbg", "gbrg") -> uint8 [H, W, 3] BGR."""
    raw = np.asarray(raw, dtype=np.uint8)
    if raw.ndim != 2 or raw.shape[0] < 3 or raw.shape[1] < 3:
        raise ValueError(f"a Bayer frame needs shape [H, W] with H, W >= 3, got {raw.shape}")
    py, px = PHASE[pattern]
    h, w = raw.shape
    r = raw.astype(np.int32)
    cy = np.clip(np.arange(h), 1, h - 2)[:, None]
    cx = np.clip(np.arange(w), 1, w - 2)[None, :]

    def at(dy, dx):
        return r[cy + dy, cx + dx]

    own = at(0, 0)
    hsum, vsum = at(0, -1) + at(0, 1), at(-1, 0) + at(1, 0)
    diag = at(-1, -1) + at(-1, 1) + at(1, -1) + at(1, 1)
    red_row = ((cy + py) & 1) == 0                  # the site's row of the RGGB mosaic holds R (and G)
    chroma_site = ((cy + py) & 1) == ((cx + px) & 1)  # an R or B site (else G)
    g = np.where(chroma_site, (hsum + vsum + 2) >> 2, own)
    near = np.where(chroma_site, own, (hsum + 1) >> 1)      # R on a red row, B on a blue row
    far = np.where(chroma_site, (diag + 2) >> 2, (vsum + 1) >> 1)
    red = np.where(red_row, near, far)
    blue = np.where(red_row, far, near)
    return np.stack([blue, g, red], axis=-1).astype(np.uint8)


def mosaic_of_bgr(bgr: np.ndarray, pattern: str) -> np.ndarray:
    """The raw frame a sensor with ``pattern`` would record of a BGR scene: every site keeps its own channel.  Used
    to make test and probe inputs that look like camera output."""
    py, px = PHASE[pattern]
    h, w = bgr.shape[:2]
    y = (np.arange(h)[:, None] + py) & 1
    x = (np.arange(w)[None, :] + px) & 1
    channel = np.where((y == 0) & (x == 0), 2, np.where((y == 1) & (x == 1), 0, 1))   # R = 2, G = 1, B = 0
    return np.take_along_axis(bgr, channel[..., None], axis=2)[..., 0].copy()
