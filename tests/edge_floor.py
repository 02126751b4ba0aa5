"""The fused edge kernel's magnitude floor, restated on the host (shared by test_edge_floor_host.py and
test_gpu_edge_floor.py).

k1_fused only evaluates non-maximum suppression for pixels whose gradient magnitude is above a per-frame floor `pre`,
which k1_probe estimates from a 64 x 64 lattice of unblurred gray samples.  The first pass is exact only when the
frame's true Canny `low` is at least `pre`; otherwise the frame is listed and rebuilt by the redo pass with pre = low.
``probe_floor`` predicts the floor bit for bit, ``trap_frame`` builds frames whose floor is far too high, and
``lost_edges`` names the final edge pixels a skipped or wrong redo would lose.
"""
import cv2
import numpy as np

from oracle import stages as S

_LOW_LUT = S.threshold_lut()[0]


def lattice(h, w):
    """Rows and columns k1_probe samples: the 64 x 64 lattice at the centres of its cells, or every row / column of a
    side shorter than 64 (then both sides use the general formula)."""
    ny, nx = min(h, 64), min(w, 64)
    iy, ix = np.arange(ny, dtype=np.int64), np.arange(nx, dtype=np.int64)
    if ny == 64 and nx == 64:
        return ((2 * iy + 1) * h) >> 7, ((2 * ix + 1) * w) >> 7
    return ((2 * iy + 1) * h) // (2 * ny), ((2 * ix + 1) * w) // (2 * nx)


def probe_floor(frame):
    """k1_probe's floor for one BGR frame: Q15 gray of the lattice samples, the first value whose running count
    exceeds half the samples, low = lut_low[2 * median], pre = max(0, low - max(4, low // 8))."""
    ys, xs = lattice(*frame.shape[:2])
    px = frame[ys][:, xs].astype(np.int64)
    g = (3735 * px[..., 0] + 19235 * px[..., 1] + 9798 * px[..., 2] + (1 << 14)) >> 15
    run = np.cumsum(np.bincount(g.ravel(), minlength=256))
    med = int(np.argmax(run > g.size // 2))
    low = int(_LOW_LUT[2 * med])
    return max(0, low - max(4, low // 8))


def true_low(frame):
    """The frame's Canny low threshold (median of the blurred gray plane through the reference LUT)."""
    return S.thresholds(S.blur5(S.gray(frame)))[0]


def redone(frame, forced=None):
    """Whether the first pass lists the frame for the redo pass: its true low is below the floor it ran with."""
    pre = probe_floor(frame) if forced is None else forced
    return true_low(frame) < pre


def trap_frame(h, w, seed, lattice_value=240):
    """A dark textured scene (background 40, +-3 noise) with faint lines (+25), every probe-lattice pixel painted
    `lattice_value`: the probe then sees a bright frame while the blurred frame's median stays near 40."""
    rng = np.random.default_rng(seed)
    lines = np.zeros((h, w), np.uint8)
    for _ in range(max(6, (h * w) // 20000)):
        x0, x1 = (int(v) for v in rng.integers(-w // 4, w + w // 4, 2))
        y0, y1 = (int(v) for v in rng.integers(-h // 4, h + h // 4, 2))
        cv2.line(lines, (x0, y0), (x1, y1), 25, int(rng.integers(1, 4)))
    img = 40 + lines[..., None].astype(np.int16) + rng.integers(-3, 4, (h, w, 3))
    img = np.clip(img, 0, 255).astype(np.uint8)
    ys, xs = lattice(h, w)
    img[np.ix_(ys, xs)] = lattice_value
    return img


def lost_edges(frame, pre):
    """Final Canny edge pixels of the frame with magnitude <= pre: what the first pass alone, with floor `pre`, cannot
    produce.  Returns (mask, low)."""
    b = S.blur5(S.gray(frame))
    low, high, _ = S.thresholds(b)
    t = S.canny(b, low, high)
    return (t.edges != 0) & (t.mag <= pre), low


def boundary_lattice_values(h, w, seed):
    """Lattice values v whose trap frame gets pre == low and pre == low + 1 (the two sides of the redo decision), the
    frame's true low unchanged by the paint: {pre - low: v} for 0 and 1, smallest v first."""
    low = true_low(trap_frame(h, w, seed, 40))
    out = {}
    for v in range(256):
        f = trap_frame(h, w, seed, v)
        d = probe_floor(f) - low
        if d in (0, 1) and d not in out and true_low(f) == low:
            out[d] = v
        if len(out) == 2 or d > 1:
            break
    return out
