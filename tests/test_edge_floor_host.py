"""Host-side guards for test_gpu_edge_floor.py: the restated probe (edge_floor.probe_floor) must keep predicting a redo
for the trap frames and none for the generator frames, and the boundary frames must exist.  Without these the GPU tests
could silently stop reaching the fused edge kernel's redo pass when the probe, the generator or the oracle changes."""
import numpy as np
import pytest

from edge_floor import boundary_lattice_values, lattice, lost_edges, probe_floor, redone, trap_frame, true_low
from oracle import stages as S
from util import gen_frames

TRAP_SHAPES = [(480, 640), (1080, 1920), (135, 480), (32, 640)]
# generator frames with final edge pixels at exactly mag == low + 1: (width, height, n, start, frames, their low)
BOUNDARY_GEN = [(640, 480, 4, 7, (2, 3), 99), (1920, 1080, 4, 7, (0,), 97)]


def test_lattice_matches_k1_probe_branches():
    ys, xs = lattice(480, 640)
    assert len(ys) == len(xs) == 64 and ys[0] == 3 and xs[-1] == ((127 * 640) >> 7)
    ys, xs = lattice(32, 640)                    # fewer than 64 rows: every row, 64 columns by the general formula
    assert list(ys) == list(range(32)) and len(xs) == 64 and xs[0] == 640 // 128
    ys, xs = lattice(7, 9)
    assert list(ys) == list(range(7)) and list(xs) == list(range(9))


def test_probe_floor_of_flat_frames():
    lo = S.threshold_lut()[0]
    for v in (0, 5, 40, 128, 255):
        low = int(lo[2 * v])
        assert probe_floor(np.full((64, 96, 3), v, np.uint8)) == max(0, low - max(4, low // 8))
    # Q15 gray: pure blue 255 is (3735 * 255 + 2^14) >> 15 = 29
    assert probe_floor(np.dstack([np.full((70, 70), 255, np.uint8), np.zeros((70, 70, 2), np.uint8)])) == \
        max(0, int(lo[58]) - 4)


@pytest.mark.parametrize("shape", TRAP_SHAPES)
def test_trap_frames_are_redone_and_lose_edges(shape):
    for seed in range(2):
        f = trap_frame(*shape, seed)
        pre = probe_floor(f)
        lost, low = lost_edges(f, pre)
        assert low < pre and redone(f), (shape, seed, low, pre)
        assert lost.any(), (shape, seed)
    if shape != (32, 640):                       # the lattice is a tenth of that frame and makes its own strong edges
        assert lost.sum() > 0.9 * (S.canny(S.blur5(S.gray(f)), *S.thresholds(S.blur5(S.gray(f)))[:2]).edges != 0).sum()


@pytest.mark.parametrize("shape", TRAP_SHAPES)
def test_generator_frames_are_not_redone(shape):
    h, w = shape
    for f in gen_frames(w, h, 8):
        assert not redone(f)


def test_lattice_value_reaches_both_sides_of_the_redo_decision():
    vals = boundary_lattice_values(480, 640, 0)
    assert set(vals) == {0, 1}, vals
    low = true_low(trap_frame(480, 640, 0, 40))
    assert probe_floor(trap_frame(480, 640, 0, vals[0])) == low and not redone(trap_frame(480, 640, 0, vals[0]))
    assert probe_floor(trap_frame(480, 640, 0, vals[1])) == low + 1 and redone(trap_frame(480, 640, 0, vals[1]))


@pytest.mark.parametrize("w,h,n,start,idx,low", BOUNDARY_GEN)
def test_generator_boundary_frames_have_edges_at_low_plus_one(w, h, n, start, idx, low):
    frames = gen_frames(w, h, n, start)
    for i in idx:
        b = S.blur5(S.gray(frames[i]))
        lo, hi, _ = S.thresholds(b)
        t = S.canny(b, lo, hi)
        assert lo == low and ((t.edges != 0) & (t.mag == low + 1)).any(), (w, i)
        assert not redone(frames[i], forced=low) and redone(frames[i], forced=low + 1)
