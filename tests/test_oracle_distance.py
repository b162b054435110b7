"""CPU: the NumPy restatement of the distance transform and the coastline metrics (oracle/distance_ref.py) against the
definitions: brute-force minima, scipy.ndimage.distance_transform_edt, the OpenCV coastline band, pairwise distances with
np.percentile; and the host metric rule of rbunet.coastline_metrics against the oracle's."""
import math

import numpy as np
import pytest
from scipy import ndimage

from oracle import distance_ref as R
from oracle import imageops_ref


def _blobby(H, W, seed, p=0.5):
    rng = np.random.default_rng(seed)
    f = ndimage.gaussian_filter(rng.standard_normal((H, W)), 3.0)
    return f > np.quantile(f, p)


def test_edt_equals_brute_force_minimum():
    rng = np.random.default_rng(0)
    for i in range(40):
        H, W = rng.integers(1, 41, size=2)
        F = rng.random((H, W)) < rng.choice([0.002, 0.02, 0.2, 0.7])
        if i == 0:
            F[:] = False
        assert np.array_equal(R.edt(F), R.edt_brute(F)), (H, W)


@pytest.mark.parametrize("kind", ["sparse", "dense", "blobby", "corner"])
def test_edt_equals_scipy(kind):
    rng = np.random.default_rng(1)
    H, W = 500, 700
    if kind == "sparse":
        F = rng.random((H, W)) < 2e-4
    elif kind == "dense":
        F = rng.random((H, W)) < 0.6
    elif kind == "blobby":
        F = _blobby(H, W, 2)
    else:
        F = np.zeros((H, W), bool)
        F[H - 1, W - 1] = True
    want = np.rint(ndimage.distance_transform_edt(~F) ** 2).astype(np.int64)
    assert np.array_equal(R.edt(F), want)


def test_edt_of_an_empty_image_is_minus_one_and_zero_on_features():
    assert (R.edt(np.zeros((3, 5), bool)) == -1).all()
    assert (R.edt(np.ones((3, 5), bool)) == 0).all()


def test_coastline_is_the_3x3_opencv_band():
    rng = np.random.default_rng(3)
    for seed in range(6):
        w = _blobby(60 + seed, 80 - seed, seed) if seed % 2 else rng.random((37, 51)) < 0.4
        band = imageops_ref.coastline_mask(w.astype(np.uint8), 3) != 0
        assert np.array_equal(R.coastline(w), band)
    w = np.ones((4, 4), bool)                          # all water: no coastline, the border included
    assert not R.coastline(w).any()


def test_water_rules():
    p = np.array([0.5, 0.5000001, 0.0, 1.0], np.float32)
    assert R.water(p, 0.5).tolist() == [False, True, False, True]
    assert R.water(p, 0.5, is_target=True).tolist() == [True, True, False, True]
    assert R.water(np.array([0, 2, 255], np.uint8)).tolist() == [False, True, True]


def _brute_metrics(pred, target, threshold, taus, s):
    """The metrics from all pairwise distances between the two coastlines."""
    P = np.argwhere(R.coastline(R.water(pred, threshold)))
    G = np.argwhere(R.coastline(R.water(target, threshold, True)))
    d2 = ((P[:, None, :] - G[None, :, :]) ** 2).sum(-1)
    a2, b2 = d2.min(1), d2.min(0)
    a, b = np.sqrt(a2.astype(np.float64)) * s, np.sqrt(b2.astype(np.float64)) * s
    out = {"n_pred": len(P), "n_target": len(G), "pred_to_target": a.mean(), "target_to_pred": b.mean(),
           "mean_distance": (a.sum() + b.sum()) / (len(a) + len(b)), "hausdorff": max(a.max(), b.max()),
           "hausdorff95": max(np.percentile(np.sqrt(a2.astype(np.float64)), 95) * s,
                              np.percentile(np.sqrt(b2.astype(np.float64)), 95) * s)}
    for tau in taus:
        lim = math.floor((tau / s) ** 2)
        c0, c1 = int((a2 <= lim).sum()), int((b2 <= lim).sum())
        p, r = c0 / (len(P) + 1e-8), c1 / (len(G) + 1e-8)
        out[f"precision@{tau:g}"], out[f"recall@{tau:g}"] = p, r
        out[f"f1@{tau:g}"] = 2 * p * r / (p + r + 1e-8)
        out[f"surface_dice@{tau:g}"] = (c0 + c1) / (len(P) + len(G))
    return out, a2, b2


def _compare(got, want):
    assert list(got) == list(want)
    for k, v in want.items():
        if k.startswith(("n_", "hausdorff")) or "@" in k:
            assert got[k] == v, (k, got[k], v)
        else:
            assert abs(got[k] - v) <= 1e-12 * abs(v), (k, got[k], v)


@pytest.mark.parametrize("seed", range(4))
def test_metrics_equal_pairwise_distances(seed):
    rng = np.random.default_rng(seed)
    H, W = 48 + seed, 64 - seed
    pred = _blobby(H, W, seed).astype(np.float32) * rng.random((H, W)).astype(np.float32)
    pred[0, :5] = 0.5                                                     # exactly at the threshold: not water
    target = _blobby(H, W, seed + 10).astype(np.uint8)
    taus, s = (1.0, 2.0, 3.5), (1.0, 10.0, 0.5, 3.0)[seed]
    taus = tuple(t * s for t in taus)
    st = R.coastline_stats(pred, target, 0.5, [R.tolerance_d2(t, s) for t in taus])
    want, a2, b2 = _brute_metrics(pred, target, 0.5, taus, s)
    assert st[0, 0] == len(a2) and st[1, 0] == len(b2)
    assert st[0, 2] == a2.max() and st[1, 2] == b2.max()
    _compare(R.metrics_from_stats(st, taus, s), want)
    import rbunet
    _compare(rbunet.distance.metrics_from_stats(st.tolist(), taus, s), want)


def test_empty_and_one_sided_coastlines():
    water = np.zeros((20, 30), np.uint8)
    water[5:12, 8:20] = 1
    none = np.zeros_like(water)
    full = np.ones_like(water)                                           # all water: no coastline either
    import rbunet
    for pred, target, kind in ((none, none, "both"), (full, none, "both"), (water, none, "target"),
                               (none, water, "pred")):
        st = R.coastline_stats(pred, target, 0.5, [4])
        for m in (R.metrics_from_stats(st, (2.0,)), rbunet.distance.metrics_from_stats(st.tolist(), (2.0,))):
            if kind == "both":
                assert m["n_pred"] == m["n_target"] == 0
                assert all(math.isnan(m[k]) for k in ("mean_distance", "hausdorff", "hausdorff95", "surface_dice@2"))
                assert m["precision@2"] == m["recall@2"] == m["f1@2"] == 0
            else:
                assert all(math.isinf(m[k]) for k in ("pred_to_target", "mean_distance", "hausdorff", "hausdorff95"))
                assert m["precision@2"] == m["recall@2"] == m["f1@2"] == m["surface_dice@2"] == 0
        assert (st[:, 1:5] == -1).all() and (st[:, 5:] == 0).all()
        if kind == "target":
            assert st[0, 0] > 0 and st[1, 0] == 0


def test_host_tolerance_threshold_at_integer_ratios():
    assert R.tolerance_d2(10, 10.0) == 1
    assert R.tolerance_d2(30, 10.0) == 9
    assert R.tolerance_d2(20, 10.0) == 4
    assert R.tolerance_d2(5, 1.0) == 25
    assert R.tolerance_d2(0.3, 0.1) == 8                # 0.3 / 0.1 = 2.9999999999999996 in floats
    assert R.tolerance_d2(1e9, 1.0) == 2 ** 31 - 1
    import rbunet
    assert rbunet.distance._tolerances((10, 30, 0.3, 1e9), 10.0, "x")[1] == [1, 9, 0, 2 ** 31 - 1]
    assert rbunet.distance._tolerances((0.3,), 0.1, "x")[1] == [8]
