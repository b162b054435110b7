"""CPU: the patch sampler's oracle (oracle/patch_ref.py) -- the eight dihedral ops, the k-th focus pixel and its clamped
window -- and the package's host-side job draw (rbunet.patches.draw_jobs) against the oracle's restatement."""
import itertools

import numpy as np
import pytest
import torch

from oracle import patch_ref as P


def _index_form(win: np.ndarray, op: int, h: int, w: int) -> np.ndarray:
    """out[i][j] = win[a][b], i' = fh ? h-1-i : i, j' = fw ? w-1-j : j, (a, b) = t ? (j', i') : (i', j')."""
    out = np.empty((h, w), dtype=win.dtype)
    for i in range(h):
        for j in range(w):
            ii = h - 1 - i if op & 2 else i
            jj = w - 1 - j if op & 1 else j
            out[i, j] = win[jj, ii] if op & 4 else win[ii, jj]
    return out


@pytest.mark.parametrize("h,w", [(5, 5), (3, 7)])
def test_the_eight_ops_are_the_dihedral_group(h, w):
    a = np.arange(h * w).reshape(h, w) * 7 % 101                        # no symmetry
    imgs = {}
    for op in range(8):
        win = a.T.copy() if (op & 4) else a                             # the window the op reads: w x h for ops 4-7
        got = P.apply_op(torch.from_numpy(win), op).numpy()
        assert got.shape == (h, w)
        assert np.array_equal(got, _index_form(win, op, h, w)), op
        if h == w:
            imgs[op] = P.apply_op(torch.from_numpy(a), op).numpy()
    if h == w:
        group = [np.rot90(a, k) for k in range(4)] + [np.rot90(np.flip(a, 1), k) for k in range(4)]
        assert len({g.tobytes() for g in imgs.values()}) == 8
        assert {g.tobytes() for g in imgs.values()} == {np.ascontiguousarray(g).tobytes() for g in group}
        assert np.array_equal(imgs[0], a) and np.array_equal(imgs[4], a.T)
        assert np.array_equal(imgs[3], np.rot90(a, 2)) and np.array_equal(imgs[6], np.rot90(a, 1))


def _focus_cases():
    rng = np.random.RandomState(0)
    one = np.zeros((6, 9), np.uint8)
    one[3, 4] = 1
    rows = np.zeros((7, 5), np.uint8)                                   # empty rows between populated ones
    rows[0, 0] = rows[0, 4] = rows[3, 2] = rows[6, 4] = 9
    corners = np.zeros((5, 8), np.uint8)
    corners[0, 0] = corners[0, 7] = corners[4, 0] = corners[4, 7] = 255
    last_row = np.zeros((4, 6), np.uint8)
    last_row[3, 1:] = 1
    last_col = np.zeros((6, 4), np.uint8)
    last_col[:, 3] = 1
    return [one, rows, corners, last_row, last_col, (rng.rand(11, 13) < 0.3).astype(np.uint8),
            np.ones((3, 4), np.uint8)]


@pytest.mark.parametrize("idx", range(7))
def test_kth_focus_equals_a_brute_force_scan(idx):
    f = _focus_cases()[idx]
    scan = [(y, x) for y in range(f.shape[0]) for x in range(f.shape[1]) if f[y, x]]
    assert [P.kth_focus(f, k) for k in range(len(scan))] == scan


@pytest.mark.parametrize("H,W", [(1, 1), (4, 7), (9, 5)])
def test_the_clamped_window_holds_its_focus_pixel(H, W):
    for py, px in itertools.product(range(H), range(W)):
        f = np.zeros((H, W), np.uint8)
        f[py, px] = 1
        for ph, pw, op in itertools.product(range(1, H + 1), range(1, W + 1), range(8)):
            wh, ww = (pw, ph) if op & 4 else (ph, pw)
            if wh > H or ww > W:
                continue
            y, x = P.origin((0, op, 0, 0, 1, 12345), H, W, ph, pw, f)
            assert 0 <= y <= H - wh and 0 <= x <= W - ww
            assert y <= py < y + wh and x <= px < x + ww


def test_origin_falls_back_to_the_drawn_one_without_focus_pixels():
    f = np.zeros((8, 8), np.uint8)
    assert P.origin((0, 5, 2, 3, 1, 7), 8, 8, 4, 4, f) == (2, 3)
    assert P.origin((0, 5, 2, 3, 1, 7), 8, 8, 4, 4, None) == (2, 3)
    f[7, 7] = 1
    assert P.origin((0, 5, 2, 3, 0, 7), 8, 8, 4, 4, f) == (2, 3)       # not a focus job
    assert P.origin((0, 5, 2, 3, 1, 7), 8, 8, 4, 4, f) == (4, 4)


@pytest.mark.parametrize("dihedral", [True, False])
@pytest.mark.parametrize("B,fraction", [(1, 0.0), (7, 0.33), (64, 0.33), (10, 0.25), (5, 1.0)])
def test_draw_jobs_equals_the_oracle(B, fraction, dihedral):
    from rbunet.patches import draw_jobs
    sizes = [(300, 200), (64, 64), (97, 81)]
    ph, pw = (64, 48) if not dihedral else (48, 64)
    n_focus = round(fraction * B)
    got = draw_jobs(B, sizes, ph, pw, n_focus, dihedral, torch.Generator().manual_seed(B))
    want = P.draw_jobs(B, sizes, ph, pw, n_focus, dihedral, torch.Generator().manual_seed(B))
    assert got.dtype.itemsize == 32
    cols = np.stack([got[k].astype(np.int64) for k in ("scene", "op", "y0", "x0", "focus", "r")], 1)
    assert np.array_equal(cols, want)
    assert int(got["focus"].sum()) == n_focus and got["focus"][:n_focus].all()
    assert ((got["scene"] >= 0) & (got["scene"] < len(sizes))).all()
    assert ((got["op"] >= 0) & (got["op"] < 8)).all() and (dihedral or (got["op"] == 0).all())
    assert ((got["r"] >= 0) & (got["r"] < 2 ** 62)).all()
    for j in got:
        wh, ww = (pw, ph) if j["op"] & 4 else (ph, pw)
        H, W = sizes[j["scene"]]
        assert 0 <= j["y0"] <= H - wh and 0 <= j["x0"] <= W - ww


def test_draw_jobs_uses_the_default_generator_and_every_op():
    from rbunet.patches import draw_jobs
    torch.manual_seed(3)
    a = draw_jobs(256, [(64, 64)], 16, 16, 0, True)
    torch.manual_seed(3)
    assert np.array_equal(a, draw_jobs(256, [(64, 64)], 16, 16, 0, True))
    assert set(a["op"].tolist()) == set(range(8))
    assert not np.array_equal(a, draw_jobs(256, [(64, 64)], 16, 16, 0, True))
