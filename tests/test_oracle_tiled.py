"""CPU: the sliding-window oracle (oracle/tiled_ref.py) -- plans, reflection, blend -- and the package's host-side plan
against it (rbunet.predict_tiled copies exactly these tables to the device)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import tiled_ref as T

# (H, W, tile, overlap): H = tile, H < tile with H not a multiple of 16, H >> tile, overlap 0 and overlap = tile - 16
PLANS = [(64, 64, 64, 16), (17, 530, 64, 16), (1000, 777, 64, 16), (200, 328, 64, 0), (200, 328, 64, 48),
         (16, 16, 512, 64), (513, 1100, 512, 496), (333, 95, (96, 32), (0, 16))]


def _pair(v):
    return v if isinstance(v, tuple) else (v, v)


@pytest.mark.parametrize("H,W,tile,overlap", PLANS)
def test_plan_covers_every_pixel_with_tiles_inside_the_scene(H, W, tile, overlap):
    tile, overlap = _pair(tile), _pair(overlap)
    p = T.plan(H, W, tile, overlap)
    for n, o, ext, t, ov, first, count in ((H, p["oy"], p["th"], tile[0], overlap[0], p["row_first"], p["row_count"]),
                                           (W, p["ox"], p["tw"], tile[1], overlap[1], p["col_first"], p["col_count"])):
        if n >= t:
            assert ext == t and o[0] == 0 and o[-1] == n - t and (o >= 0).all() and (o + t <= n).all()
            assert len(o) == -(-(n - t) // (t - ov)) + 1 and (np.diff(o) > 0).all() and (np.diff(o) <= t - ov).all()
        else:
            assert len(o) == 1 and o[0] == 0 and ext % 16 == 0 and n <= ext < n + 16
        assert (count >= 1).all()
        canvas = np.zeros(n, dtype=np.int64)          # coverage from the origins alone
        for oi in o:
            canvas[oi:oi + ext] += 1
        assert (canvas == count).all()
        for y in range(n):
            for i in range(first[y], first[y] + count[y]):
                assert o[i] <= y < o[i] + ext


@pytest.mark.parametrize("H,W,tile,overlap", PLANS)
def test_package_plan_equals_the_oracle(H, W, tile, overlap):
    from rbunet import tiled
    tile, overlap = _pair(tile), _pair(overlap)
    for sigma in (0.125, 0.3):
        p = T.plan(H, W, tile, overlap, sigma)
        q = tiled.plan_tiles(H, W, tile, overlap, sigma)
        assert (q.th, q.tw, q.ny, q.nx) == (p["th"], p["tw"], p["ny"], p["nx"])
        for k in ("oy", "ox", "row_first", "row_count", "col_first", "col_count"):
            assert np.array_equal(getattr(q, k), p[k]), k
        assert q.wy.dtype == np.float32 and np.array_equal(q.wy.view(np.uint32), p["wy"].view(np.uint32))
        assert np.array_equal(q.wx.view(np.uint32), p["wx"].view(np.uint32))


def test_gaussian_window():
    w = T.gaussian(64, 0.125)
    assert w.dtype == np.float32 and w.max() == 1.0 and np.array_equal(w, w[::-1])
    d = np.arange(64)
    assert np.allclose(w, np.exp(-0.5 * ((d + 0.5 - 32) / 8.0) ** 2) / np.exp(-0.5 * (0.5 / 8.0) ** 2), rtol=1e-7)


@pytest.mark.parametrize("H,W", [(16, 16), (17, 530), (200, 328), (31, 47), (1000, 777)])
def test_gather_reflects_like_f_pad(H, W):
    g = torch.Generator().manual_seed(H * W)
    x = torch.rand((3, H, W), generator=g)
    p = T.plan(H, W, (64, 64), (16, 16))
    ph, pw = p["th"] - H if H < 64 else 0, p["tw"] - W if W < 64 else 0
    padded = F.pad(x[None], (0, pw, 0, ph), mode="reflect")[0]
    tiles = T.gather(x, p, 0, p["ny"] * p["nx"])
    for t in range(p["ny"] * p["nx"]):
        iy, ix = divmod(t, p["nx"])
        oy, ox = p["oy"][iy], p["ox"][ix]
        assert torch.equal(tiles[t], padded[:, oy:oy + p["th"], ox:ox + p["tw"]]), t


def _brute_force_f64(tiles, p):
    """Every tile placed on the whole scene with its coverage mask, summed in float64."""
    K = tiles.shape[1]
    num = np.zeros((K, p["H"], p["W"]))
    den = np.zeros((p["H"], p["W"]))
    w2 = p["wy"].astype(np.float64)[:, None] * p["wx"].astype(np.float64)[None, :]
    for t in range(tiles.shape[0]):
        iy, ix = divmod(t, p["nx"])
        oy, ox = p["oy"][iy], p["ox"][ix]
        h, w = min(p["th"], p["H"] - oy), min(p["tw"], p["W"] - ox)
        num[:, oy:oy + h, ox:ox + w] += w2[:h, :w] * tiles[t, :, :h, :w].double().numpy()
        den[oy:oy + h, ox:ox + w] += w2[:h, :w]
    return num / den


@pytest.mark.parametrize("H,W,tile,overlap,K", [(200, 328, 64, 16, 1), (200, 328, 64, 48, 3), (17, 530, 64, 16, 2),
                                                (130, 97, 32, 0, 1), (64, 64, 64, 16, 5)])
def test_blend_matches_a_float64_brute_force(H, W, tile, overlap, K):
    p = T.plan(H, W, (tile, tile), (overlap, overlap))
    g = torch.Generator().manual_seed(K * 1000 + H)
    tiles = torch.rand((p["ny"] * p["nx"], K, p["th"], p["tw"]), generator=g) * 4 - 2
    got = T.blend(tiles, p)
    want = _brute_force_f64(tiles, p)
    assert got.dtype == torch.float32 and got.shape == (K, H, W)
    assert np.abs(got.double().numpy() - want).max() <= 2e-6 * max(1.0, np.abs(want).max())


def test_blend_of_identical_tiles_is_the_value_and_labels_follow_the_rules():
    p = T.plan(96, 80, (32, 32), (8, 8))
    v = torch.tensor([0.25, 0.75, 0.75])[None, :, None, None].expand(p["ny"] * p["nx"], 3, 32, 32).contiguous()
    out = T.blend(v, p)
    assert torch.allclose(out, v[0, :, :1, :1].expand(3, 96, 80), rtol=1e-6)
    assert (T.labels(out, "RobustUNet") == 1).all()                          # tie between classes 1 and 2 -> 1
    half = torch.full((1, 4, 4), 0.5)
    assert (T.labels(half, "RobustUNet") == 0).all() and (T.labels(torch.zeros(1, 4, 4), "UNet") == 0).all()
    assert (T.labels(torch.full((1, 4, 4), 1e-30), "UNet") == 1).all()
