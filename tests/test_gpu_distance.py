"""GPU: the exact distance transform (rbu_edt, rbunet.distance_transform) and the coastline statistics and metrics
(rbu_coastline_stats, rbunet.coastline_stats / coastline_metrics) against the CPU oracle (oracle/distance_ref.py)."""
import math

import numpy as np
import pytest
import torch
from scipy import ndimage

import rbunet
from rbunet import _lib
from rbunet.ops import _p
from oracle import distance_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _blobby(H, W, seed, p=0.5, sigma=3.0):
    rng = np.random.default_rng(seed)
    f = ndimage.gaussian_filter(rng.standard_normal((H, W)), sigma)
    return f > np.quantile(f, p)


def _masks(H, W, seed):
    """empty, full, one corner pixel, sparse, blobby."""
    rng = np.random.default_rng(seed)
    corner = np.zeros((H, W), bool)
    corner[H - 1, 0] = True
    sparse = rng.random((H, W)) < 3e-3
    sparse[rng.integers(H), rng.integers(W)] = True
    return [np.zeros((H, W), bool), np.ones((H, W), bool), corner, sparse, _blobby(H, W, seed, 0.7, 2.0)]


def _edt_ref(F):
    """The oracle's separable EDT; at larger sizes scipy's, which tests/test_oracle_distance.py pins to it."""
    if F.size <= 40000 or F.shape[0] == 1:
        return R.edt(F)
    if not F.any():
        return np.full(F.shape, -1, np.int64)
    return np.rint(ndimage.distance_transform_edt(~F) ** 2).astype(np.int64)


@pytest.mark.parametrize("H,W", [(1, 1), (1, 300), (300, 1), (17, 530), (1000, 777), (1, 32768)])
def test_edt_is_bit_exact(H, W):
    masks = _masks(H, W, H * 7 + W)
    batch = torch.from_numpy(np.stack(masks).astype(np.uint8)).to(DEV)
    got = rbunet.distance_transform(batch).cpu().numpy()
    assert got.dtype == np.int32 and got.shape == (len(masks), H, W)
    for i, F in enumerate(masks):
        assert np.array_equal(got[i], _edt_ref(F)), (H, W, i)
        alone = rbunet.distance_transform(torch.from_numpy(F).to(DEV)).cpu().numpy()       # bool [H,W]
        assert np.array_equal(alone, got[i])


def test_edt_writes_inside_sentinel_filled_buffers():
    B, H, W = 3, 70, 131
    masks = np.stack(_masks(H, W, 5)[2:])
    feats = torch.from_numpy(masks.astype(np.uint8)).to(DEV)
    nbytes = int(_lib.lib().rbu_edt_workspace_bytes(B, H, W))
    ws = torch.full((nbytes + 4096,), 0xA5, dtype=torch.uint8, device=DEV)
    out = torch.full((B * H * W + 2048,), -777, dtype=torch.int32, device=DEV)
    body = out[1024:1024 + B * H * W]
    _lib.call("rbu_edt", _p(feats), B, H, W, _p(body), _p(ws), nbytes, _lib.stream_ptr())
    o = out.cpu().numpy()
    assert (o[:1024] == -777).all() and (o[1024 + B * H * W:] == -777).all()
    assert (ws[nbytes:].cpu().numpy() == 0xA5).all()
    got = o[1024:1024 + B * H * W].reshape(B, H, W)
    for i in range(B):
        assert np.array_equal(got[i], R.edt(masks[i]))


def test_edt_of_a_30000_by_24000_scene_equals_closed_forms():
    H, W = 30000, 24000
    n = min(H, W)
    f = torch.zeros((3, H, W), dtype=torch.uint8, device=DEV)
    f[0, H - 1, W - 1] = 1                                     # one corner pixel
    c = 12345
    f[1, :, c:] = 1                                            # a vertical half-plane
    k = torch.arange(n, device=DEV)
    f[2, k, k] = 1                                             # the diagonal y = x
    D = rbunet.distance_transform(f)
    assert D.shape == (3, H, W) and D.dtype == torch.int32
    xs = torch.arange(W, device=DEV, dtype=torch.int64)
    for y0 in range(0, H, 2000):
        ys = torch.arange(y0, min(y0 + 2000, H), device=DEV, dtype=torch.int64)[:, None]
        corner = (H - 1 - ys) ** 2 + (W - 1 - xs) ** 2
        half = ((c - xs).clamp(min=0) ** 2).expand(len(ys), W)
        kk = ((ys + xs) // 2).clamp(max=n - 1)
        diag = (ys - kk) ** 2 + (xs - kk) ** 2
        for i, want in enumerate((corner, half, diag)):
            assert torch.equal(D[i, y0:y0 + len(ys)].long(), want), (i, y0)
    assert int(D[0, 0, 0]) == (H - 1) ** 2 + (W - 1) ** 2


def _pair(H, W, seed, pred_dtype, target_dtype):
    """A probability map (or its labels) and a target mask with nearby, different coastlines."""
    rng = np.random.default_rng(seed)
    base = _blobby(H, W, seed)
    shifted = np.roll(_blobby(H, W, seed), (rng.integers(-4, 5), rng.integers(-4, 5)), axis=(0, 1)) | \
        (_blobby(H, W, seed + 100, 0.9) & (rng.random((H, W)) < 0.5))
    prob = np.where(shifted, 0.5 + 0.5 * rng.random((H, W)), 0.5 * rng.random((H, W))).astype(np.float32)
    prob[rng.random((H, W)) < 0.05] = 0.5                     # exactly at the threshold: not water
    pred = {"f32": prob, "u8": (prob > 0.5).astype(np.uint8) * 3, "bool": prob > 0.5}[pred_dtype]
    target = {"f32": base.astype(np.float32) * rng.choice([1.0, 0.25], (H, W)).astype(np.float32),
              "u8": base.astype(np.uint8), "bool": base}[target_dtype]
    return pred, target


def _same_metrics(got, want):
    """Equal keys; the means within 1e-12 relative, everything else equal (NaN matching NaN)."""
    assert list(got) == list(want)
    for k, v in want.items():
        if math.isnan(v):
            assert math.isnan(got[k]), k
        elif k in ("pred_to_target", "target_to_pred", "mean_distance") and math.isfinite(v):
            assert abs(got[k] - v) <= 1e-12 * abs(v), (k, got[k], v)
        else:
            assert got[k] == v, (k, got[k], v)


def _oracle_stats(pred, target, tol_d2, threshold=0.5):
    return np.stack([R.coastline_stats(p, t, threshold, tol_d2) for p, t in zip(pred, target)])


def _check_stats(got, want):
    assert got.shape == want.shape
    ints = [0, 2, 3, 4] + list(range(5, want.shape[-1]))
    bad = np.argwhere(got[..., ints] != want[..., ints])
    assert not len(bad), [(tuple(i), got[..., ints][tuple(i)], want[..., ints][tuple(i)]) for i in bad[:10]]
    ok = np.abs(got[..., 1] - want[..., 1]) <= 1e-12 * np.abs(want[..., 1])
    assert ok.all(), (got[..., 1], want[..., 1])


@pytest.mark.parametrize("pd,td", [("f32", "u8"), ("u8", "bool"), ("bool", "f32"), ("f32", "f32")])
def test_coastline_stats_equal_the_oracle(pd, td):
    B, H, W = 3, 96, 131
    pairs = [_pair(H, W, 10 * i + len(pd + td), pd, td) for i in range(B)]
    pred = np.stack([p for p, _ in pairs])
    target = np.stack([t for _, t in pairs])
    pred[2] = 0                                                                # no predicted coastline in image 2
    taus, s = (1.0, 2.0, 3.0, 5.0), 1.0
    tol = [R.tolerance_d2(t, s) for t in taus]
    want = _oracle_stats(pred, target, tol)
    got = rbunet.coastline_stats(torch.from_numpy(pred).to(DEV), torch.from_numpy(target).to(DEV), tolerances=taus,
                                 pixel_size=s)
    assert got.dtype == torch.float64 and got.shape == (B, 2, 5 + len(taus))
    _check_stats(got.cpu().numpy(), want)
    assert want[2, 0, 0] == 0 and (want[2, :, 1:5] == -1).all()
    # [B,1,H,W] (the RobustUNet K = 1 output) gives the same; metrics equal the oracle's rule
    got4 = rbunet.coastline_stats(torch.from_numpy(pred).to(DEV)[:, None], torch.from_numpy(target).to(DEV)[:, None],
                                  tolerances=taus, pixel_size=s)
    assert torch.equal(got4, got)
    mets = rbunet.coastline_metrics(torch.from_numpy(pred).to(DEV), torch.from_numpy(target).to(DEV), tolerances=taus)
    for b in range(B):
        _same_metrics(mets[b], R.metrics_from_stats(want[b], taus, s))
    assert mets[2]["n_pred"] == 0 and mets[2]["surface_dice@1"] == 0 and math.isinf(mets[2]["mean_distance"])


def test_a_larger_image_with_pixel_size_and_many_tolerances():
    H, W = 300, 257
    pred, target = _pair(H, W, 77, "f32", "u8")
    taus, s = (10, 20, 30, 50, 70, 100, 150, 400), 10.0                 # tau / s integer: distances exactly at tau count
    tol = [R.tolerance_d2(t, s) for t in taus]
    want = _oracle_stats(pred[None], target[None], tol)
    got = rbunet.coastline_stats(torch.from_numpy(pred).to(DEV), torch.from_numpy(target).to(DEV), tolerances=taus,
                                 pixel_size=s)
    _check_stats(got.cpu().numpy(), want)


def test_batch_members_and_repeated_runs_are_bit_identical():
    B, H, W = 4, 150, 211
    pairs = [_pair(H, W, 300 + i, "f32", "u8") for i in range(B)]
    pred = torch.from_numpy(np.stack([p for p, _ in pairs])).to(DEV)
    target = torch.from_numpy(np.stack([t for _, t in pairs])).to(DEV)
    a = rbunet.coastline_stats(pred, target)
    b = rbunet.coastline_stats(pred, target)
    assert torch.equal(a.view(torch.int64), b.view(torch.int64))
    for i in range(B):
        alone = rbunet.coastline_stats(pred[i], target[i])
        assert torch.equal(alone[0].view(torch.int64), a[i].view(torch.int64)), i


def test_predict_tiled_labels_end_to_end():
    torch.manual_seed(0)
    model = rbunet.RobustUNet(3, 1, 16).to(DEV).eval()
    H, W = 1000, 777
    g = torch.Generator().manual_seed(4)
    x = torch.randn((3, H, W), generator=g).to(DEV)
    labels = rbunet.predict_tiled(model, x, tile=256, overlap=32)
    mask = torch.from_numpy(_blobby(H, W, 9).astype(np.uint8)).to(DEV)
    taus, s = (10, 20, 50), 10.0
    got = rbunet.coastline_metrics(labels, mask, tolerances=taus, pixel_size=s)[0]
    st = R.coastline_stats(labels.cpu().numpy(), mask.cpu().numpy(), 0.5, [R.tolerance_d2(t, s) for t in taus])
    want = R.metrics_from_stats(st, taus, s)
    assert want["n_pred"] > 0 and want["n_target"] > 0
    _same_metrics(got, want)


def test_launch_count_is_fixed_and_nothing_synchronises():
    counts = set()
    for B, H, W in ((1, 40, 50), (3, 40, 50), (1, 333, 517), (5, 333, 517)):
        p = torch.rand((B, H, W), device=DEV)
        t = (torch.rand((B, H, W), device=DEV) > 0.5).to(torch.uint8)
        rbunet.coastline_stats(p, t)
        n0 = _lib.launch_count()
        rbunet.coastline_stats(p, t)
        counts.add(_lib.launch_count() - n0)
    assert counts == {9}
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        st = rbunet.coastline_stats(p, t)
        d = rbunet.distance_transform(t)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert st.shape == (5, 2, 8) and d.shape == t.shape


def test_coastline_metrics_makes_one_copy():
    p = torch.rand((3, 64, 80), device=DEV)
    t = (torch.rand((3, 64, 80), device=DEV) > 0.5).to(torch.uint8)
    rbunet.coastline_metrics(p, t)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        rbunet.coastline_metrics(p, t)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    copies = [n for n in names if n.startswith("Memcpy ")]
    assert len(copies) == 1 and copies[0].startswith("Memcpy DtoH"), copies


def test_argument_errors_raise_before_any_launch():
    p = torch.rand((2, 32, 40), device=DEV)
    t = (torch.rand((2, 32, 40), device=DEV) > 0.5).to(torch.uint8)
    rbunet.coastline_stats(p, t)
    cs, cm, dt = rbunet.coastline_stats, rbunet.coastline_metrics, rbunet.distance_transform
    cases = [
        (RuntimeError, "coastline_stats", lambda: cs(p.cpu(), t)),
        (RuntimeError, "coastline_metrics", lambda: cm(p, t.cpu())),
        (RuntimeError, "distance_transform", lambda: dt(t.cpu())),
        (TypeError, "coastline_stats", lambda: cs(p.double(), t)),
        (TypeError, "coastline_stats", lambda: cs(p, t.to(torch.int64))),
        (TypeError, "coastline_metrics", lambda: cm(p.numpy(force=True), t)),
        (TypeError, "distance_transform", lambda: dt(p)),
        (ValueError, "coastline_stats", lambda: cs(p, t[:1])),
        (ValueError, "coastline_stats", lambda: cs(p[:, :, :39], t[:, :, :39].transpose(1, 2))),
        (ValueError, "coastline_stats", lambda: cs(p[:, None].expand(2, 2, 32, 40), t[:, None].expand(2, 2, 32, 40))),
        (ValueError, "coastline_stats", lambda: cs(p[:, :0], t[:, :0])),
        (ValueError, "coastline_stats", lambda: cs(torch.zeros((1, 1, 32769), device=DEV),
                                                    torch.zeros((1, 1, 32769), device=DEV))),
        (ValueError, "coastline_stats", lambda: cs(p, t, tolerances=tuple(range(1, 10)))),
        (ValueError, "coastline_stats", lambda: cs(p, t, tolerances=(1.0, 0.0))),
        (ValueError, "coastline_stats", lambda: cs(p, t, tolerances=(float("inf"),))),
        (ValueError, "coastline_metrics", lambda: cm(p, t, tolerances=(-1,))),
        (ValueError, "coastline_metrics", lambda: cm(p, t, pixel_size=0)),
        (ValueError, "coastline_metrics", lambda: cm(p, t, pixel_size=float("nan"))),
        (ValueError, "coastline_stats", lambda: cs(p, t, threshold=float("nan"))),
        (ValueError, "distance_transform", lambda: dt(t[0, 0])),
        (ValueError, "distance_transform", lambda: dt(t[None])),
        (ValueError, "distance_transform", lambda: dt(torch.zeros((1, 32769), dtype=torch.uint8, device=DEV))),
    ]
    if torch.cuda.device_count() > 1:
        cases.append((ValueError, "coastline_stats", lambda: cs(p, t.to("cuda:1"))))
    for exc, who, fn in cases:
        n0 = _lib.launch_count()
        with pytest.raises(exc, match=f"rbunet.{who}"):
            fn()
        assert _lib.launch_count() == n0, who
    torch.cuda.synchronize()
