"""CPU: the outer-contour oracle (oracle/contours_ref.py) equals cv2.findContours(RETR_EXTERNAL, CHAIN_APPROX_NONE |
CHAIN_APPROX_SIMPLE) bit for bit, in cv2's order."""
import cv2
import numpy as np
import pytest

from oracle import contours_ref as R
from test_gpu_components import _blobby, _diagonals, _serpentine, _spiral

MODES = {"none": cv2.CHAIN_APPROX_NONE, "simple": cv2.CHAIN_APPROX_SIMPLE}


def _same(w, approx):
    want = [c.reshape(-1, 2) for c in cv2.findContours(w.astype(np.uint8), cv2.RETR_EXTERNAL, MODES[approx])[0]]
    got = R.find_contours(w, approx)
    assert len(got) == len(want)
    for k, (a, b) in enumerate(zip(got, want)):
        assert a.dtype == np.int32 and np.array_equal(a, b), (k, a[:8], b[:8])


def _nested(H, W):
    """Concentric rings two pixels apart, an island in every lake, and a single pixel in the innermost."""
    m = np.zeros((H, W), bool)
    for r in range(0, min(H, W) // 2, 2):
        m[r, r:W - r] = m[H - 1 - r, r:W - r] = m[r:H - r, r] = m[r:H - r, W - 1 - r] = True
    return m


@pytest.mark.parametrize("approx", ["none", "simple"])
@pytest.mark.parametrize("H,W", [(1, 1), (1, 2), (2, 1), (1, 4096), (4096, 1), (3, 3), (4, 5), (31, 45), (64, 64)])
def test_shapes_and_structured_masks(H, W, approx):
    y, x = np.indices((H, W))
    masks = [np.zeros((H, W), bool), np.ones((H, W), bool), (x + y) % 2 == 0, x % 3 == 0, y % 3 == 1,
             _spiral(H, W), _serpentine(H, W), _diagonals(H, W), _nested(H, W), (x == y) | (x == W - 1 - y),
             (x * 7 + y * 3) % 11 == 0]
    for w in masks:
        _same(w, approx)


def test_all_ones_4x5_is_the_14_point_frame():
    got = R.find_contours(np.ones((4, 5), bool), "none")
    assert len(got) == 1 and len(got[0]) == 14
    assert R.find_contours(np.ones((4, 5), bool), "simple")[0].tolist() == [[0, 0], [0, 3], [4, 3], [4, 0]]


@pytest.mark.parametrize("approx", ["none", "simple"])
def test_random_masks_near_both_percolation_thresholds(approx):
    rng = np.random.default_rng(1 if approx == "none" else 2)
    for _ in range(150):
        H, W = (int(v) for v in rng.integers(1, 60, 2))
        _same(rng.random((H, W)) < rng.choice([0.2, 0.3, 0.407, 0.41, 0.5, 0.59, 0.593, 0.7, 0.8]), approx)
    for d in (0.41, 0.59):
        _same(rng.random((300, 400)) < d, approx)


def test_edges_corners_single_pixels_and_islands_in_lakes():
    for H, W in ((7, 9), (12, 5)):
        for y, x in ((0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1), (0, 3), (H - 1, 2), (3, 0), (2, W - 1), (3, 3)):
            w = np.zeros((H, W), bool)
            w[y, x] = True
            for approx in MODES:
                _same(w, approx)
                _same(~w, approx)
    w = _nested(41, 41)
    assert len(R.find_contours(w)) == 1                               # only the outer ring: islands in lakes are not traced
    w[20, :] = True                                                    # a bridge across every ring: one component
    _same(w, "simple")
    _same(w, "none")


@pytest.mark.parametrize("approx", ["none", "simple"])
def test_blobby_scene(approx):
    n = 10980
    w = _blobby(n, n, 5, 0.5, 12.0) ^ (np.random.default_rng(5).random((n, n)) < 1e-3)
    _same(w, approx)
