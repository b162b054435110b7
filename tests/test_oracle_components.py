"""CPU: the connected-component oracle (oracle/components_ref.py) against a brute-force flood fill and OpenCV."""
from collections import deque

import cv2
import numpy as np
import pytest

from oracle import components_ref as R


def _flood(w, connectivity):
    """Labels by breadth-first flood fill from each unlabelled water pixel in raster order."""
    H, W = w.shape
    steps = [(-1, 0), (1, 0), (0, -1), (0, 1)]
    if connectivity == 8:
        steps += [(-1, -1), (-1, 1), (1, -1), (1, 1)]
    lab = np.zeros((H, W), np.int32)
    n = 0
    for y in range(H):
        for x in range(W):
            if not w[y, x] or lab[y, x]:
                continue
            n += 1
            lab[y, x] = n
            q = deque([(y, x)])
            while q:
                cy, cx = q.popleft()
                for dy, dx in steps:
                    v, u = cy + dy, cx + dx
                    if 0 <= v < H and 0 <= u < W and w[v, u] and not lab[v, u]:
                        lab[v, u] = n
                        q.append((v, u))
    return lab, n


def _brute_stats(lab, n):
    out = []
    for k in range(1, n + 1):
        ys, xs = np.nonzero(lab == k)
        out.append([xs.min(), ys.min(), xs.max(), ys.max(), len(xs), xs.sum(), ys.sum()])
    return np.array(out, np.int64).reshape(n, 7)


def _masks(H, W, seed):
    rng = np.random.default_rng(seed)
    checker = (np.indices((H, W)).sum(0) % 2).astype(bool)
    return [np.zeros((H, W), bool), np.ones((H, W), bool), checker] + \
        [rng.random((H, W)) < p for p in (0.3, 0.41, 0.59, 0.9)]


@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("H,W", [(1, 1), (1, 23), (19, 1), (17, 29), (40, 33)])
def test_labels_and_stats_equal_a_flood_fill(conn, H, W):
    for i, w in enumerate(_masks(H, W, H * 31 + W)):
        lab, n = R.label(w, conn)
        want, wn = _flood(w, conn)
        assert n == wn and np.array_equal(lab, want), (i, conn)
        assert np.array_equal(R.stats(lab, n), _brute_stats(want, wn)), i


def test_checkerboard_counts():
    w = (np.indices((10, 13)).sum(0) % 2 == 0)
    assert R.label(w, 4)[1] == int(w.sum()) and R.label(w, 8)[1] == 1


def _cv(w, conn):
    n, lab, st, cen = cv2.connectedComponentsWithStats(w.astype(np.uint8), connectivity=conn, ltype=cv2.CV_32S)
    return n - 1, lab, st[1:].astype(np.int64), cen[1:]


@pytest.mark.parametrize("seed", range(6))
def test_opencv_is_bit_exact_at_connectivity_4(seed):
    rng = np.random.default_rng(seed)
    H, W = 37 + seed, 53 + 3 * seed
    for w in [rng.random((H, W)) < p for p in (0.3, 0.59, 0.8)]:
        lab, n = R.label(w, 4)
        cn, clab, cst, ccen = _cv(w, 4)
        assert cn == n and np.array_equal(clab, lab)
        st, cen = R.opencv_stats(R.stats(lab, n))
        assert np.array_equal(st, cst)
        assert np.array_equal(cen.view(np.int64), ccen.view(np.int64))


@pytest.mark.parametrize("seed", range(6))
def test_opencv_has_the_same_partition_and_statistics_at_connectivity_8(seed):
    rng = np.random.default_rng(100 + seed)
    H, W = 37 + seed, 53 + 3 * seed
    for w in [rng.random((H, W)) < p for p in (0.3, 0.41, 0.8)]:
        lab, n = R.label(w, 8)
        cn, clab, cst, ccen = _cv(w, 8)
        assert cn == n
        # a bijection between the two numberings
        pairs = np.unique(np.stack([lab.ravel(), clab.ravel()], 1), axis=0)
        assert len(pairs) == n + 1 and len(np.unique(pairs[:, 0])) == n + 1 and len(np.unique(pairs[:, 1])) == n + 1
        to_ours = np.zeros(n + 1, np.int64)
        to_ours[pairs[:, 1]] = pairs[:, 0]
        order = np.argsort(to_ours[1:])                      # OpenCV row k (label k + 1) -> our label order
        st, cen = R.opencv_stats(R.stats(lab, n))
        assert np.array_equal(st, cst[order])
        assert np.array_equal(cen.view(np.int64), ccen[order].view(np.int64))


@pytest.mark.parametrize("conn", [4, 8])
def test_remove_small_follows_the_two_steps(conn):
    rng = np.random.default_rng(conn)
    w = rng.random((30, 41)) < 0.55
    for mw, ml in ((0, 0), (1, 1), (3, 0), (0, 4), (5, 7), (10 ** 6, 0)):
        got = R.remove_small(w, mw, ml, conn)
        lab, n = _flood(w, conn)
        size = np.bincount(lab.ravel(), minlength=n + 1)
        step1 = w & (size[lab] >= mw)
        lab2, n2 = _flood(~step1, conn)
        size2 = np.bincount(lab2.ravel(), minlength=n2 + 1)
        want = step1 | ((lab2 > 0) & (size2[lab2] < ml))
        assert got.dtype == np.uint8 and np.array_equal(got, want.astype(np.uint8)), (mw, ml)
    assert np.array_equal(R.remove_small(w, 1, 1, conn), w.astype(np.uint8))


def test_step_one_can_merge_land_so_step_two_keeps_it():
    # a 1-pixel water ring splits a 3x3 land square from the outer land; removing the ring (step 1) joins them, so the
    # square is no longer a small land component in step 2
    w = np.zeros((9, 9), bool)
    w[2:7, 2:7] = True
    w[3:6, 3:6] = False
    out = R.remove_small(w, 17, 10, 4)
    assert not out.any()
    out_no_step1 = R.remove_small(w, 0, 10, 4)
    assert out_no_step1[3:6, 3:6].all()


def test_water_rule():
    p = np.array([[0.5, 0.50001, 0.0, 1.0]], np.float32)
    assert R.water(p).tolist() == [[False, True, False, True]]
    assert R.water(np.array([[0, 1, 255]], np.uint8)).tolist() == [[False, True, True]]
