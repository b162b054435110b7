"""GPU: connected-component labelling (rbu_label_components, rbunet.label_components), component statistics
(rbu_component_stats, rbunet.component_stats) and small-region removal (rbu_remove_small_regions,
rbunet.remove_small_regions) bit for bit against the CPU oracle (oracle/components_ref.py)."""
import ctypes

import cv2
import numpy as np
import pytest
import torch
from scipy import ndimage

import rbunet
from rbunet import _lib
from rbunet.ops import _p
from oracle import components_ref as R
from oracle import distance_ref as D

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _blobby(H, W, seed, p=0.5, sigma=3.0):
    rng = np.random.default_rng(seed)
    f = ndimage.gaussian_filter(rng.standard_normal((H, W)), sigma)
    return f > np.quantile(f, p)


def _spiral(H, W):
    """A one-pixel path winding inwards, rings two pixels apart."""
    m = np.zeros((H, W), bool)
    t, l, b, r = 0, 0, H - 1, W - 1
    while t <= b and l <= r:
        m[t, l:r + 1] = True
        m[t:b + 1, r] = True
        m[b, l:r + 1] = True
        m[t + 2:b + 1, l] = True
        if t + 2 <= b and l + 1 <= r:
            m[t + 2, l:l + 2] = True
        t, l, b, r = t + 2, l + 2, b - 2, r - 2
    return m


def _serpentine(H, W):
    """Every other row is water, joined alternately at the right and the left end: one component."""
    m = np.zeros((H, W), bool)
    m[0::2] = True
    for y in range(1, H, 2):
        m[y, W - 1 if (y // 2) % 2 == 0 else 0] = True
    return m


def _diagonals(H, W):
    """Diagonal and anti-diagonal one-pixel chains every 37 columns: joined at 8, single pixels at 4."""
    y, x = np.indices((H, W))
    return ((x - y) % 37 == 0) | ((x + y) % 37 == 5)


def _masks(H, W, seed):
    rng = np.random.default_rng(seed)
    y, x = np.indices((H, W))
    return {
        "empty": np.zeros((H, W), bool), "full": np.ones((H, W), bool),
        "p0.3": rng.random((H, W)) < 0.3, "p0.9": rng.random((H, W)) < 0.9,
        "p0.41": rng.random((H, W)) < 0.41, "p0.59": rng.random((H, W)) < 0.59,
        "blobby": _blobby(H, W, seed), "checker": (x + y) % 2 == 0, "spiral": _spiral(H, W),
        "serpentine": _serpentine(H, W), "diagonals": _diagonals(H, W),
        "rows": y % 3 == 0, "cols": x % 3 == 1,
    }


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


SHAPES = [(1, 1), (1, 300), (300, 1), (1, 32768), (17, 530), (1000, 777), (512, 512)]


@pytest.mark.parametrize("conn", [4, 8])
@pytest.mark.parametrize("H,W", SHAPES)
def test_labels_are_bit_exact(H, W, conn):
    masks = _masks(H, W, H * 13 + W)
    batch = _t(np.stack(list(masks.values())).astype(np.uint8))
    labels, counts = rbunet.label_components(batch, conn)
    assert labels.dtype == torch.int32 and labels.shape == batch.shape and counts.shape == (len(masks),)
    got, cnt = labels.cpu().numpy(), counts.cpu().numpy()
    for i, (name, w) in enumerate(masks.items()):
        want, n = R.label(w, conn)
        assert cnt[i] == n, (name, cnt[i], n)
        assert np.array_equal(got[i], want), name
    names = list(masks)
    assert cnt[names.index("checker")] == (1 if conn == 8 and H > 1 and W > 1 else (H * W + 1) // 2)
    if H > 2 and W > 2:
        assert cnt[names.index("serpentine")] == 1
    for name in ("blobby", "spiral"):                                # an image alone equals its batch member
        alone, c1 = rbunet.label_components(_t(masks[name]), conn)
        assert torch.equal(alone, labels[names.index(name)]) and int(c1[0]) == cnt[names.index(name)]


@pytest.mark.parametrize("conn", [4, 8])
def test_input_dtypes_threshold_and_views(conn):
    H, W = 70, 91
    rng = np.random.default_rng(conn)
    prob = rng.random((H, W)).astype(np.float32)
    prob[rng.random((H, W)) < 0.2] = 0.5                              # exactly at the threshold: land
    w = R.water(prob)
    want, n = R.label(w, conn)
    for m in (_t(prob), _t(prob)[None, None], _t(w), _t(w.astype(np.uint8) * rng.choice([1, 255], (H, W)).astype(np.uint8))):
        lab, c = rbunet.label_components(m, conn)
        assert lab.shape == m.shape and int(c[0]) == n
        assert np.array_equal(lab.reshape(H, W).cpu().numpy(), want)
    lab, _ = rbunet.label_components(_t(prob), conn, threshold=0.25)
    assert np.array_equal(lab.cpu().numpy(), R.label(R.water(prob, 0.25), conn)[0])
    big = _t(np.ascontiguousarray(prob.T))                            # a transposed (non-contiguous) view
    lab, c = rbunet.label_components(big.t(), conn)
    assert np.array_equal(lab.cpu().numpy(), want)
    out = rbunet.remove_small_regions(big.t(), 3, 3, conn)
    assert np.array_equal(out.cpu().numpy(), R.remove_small(w, 3, 3, conn))


def test_repeated_runs_and_batches_are_identical():
    masks = [_blobby(300, 411, s, 0.45, 1.5) | (np.random.default_rng(s).random((300, 411)) < 0.05) for s in range(4)]
    batch = _t(np.stack(masks))
    for conn in (4, 8):
        a, ca = rbunet.label_components(batch, conn)
        b, cb = rbunet.label_components(batch, conn)
        assert torch.equal(a, b) and torch.equal(ca, cb)
        ra = rbunet.remove_small_regions(batch, 20, 30, conn)
        assert torch.equal(ra, rbunet.remove_small_regions(batch, 20, 30, conn))
        for i in range(len(masks)):
            assert torch.equal(rbunet.remove_small_regions(batch[i], 20, 30, conn), ra[i])
            assert torch.equal(rbunet.label_components(batch[i], conn)[0], a[i])


def test_a_30000_by_24000_scene_equals_closed_forms():
    H, W, k = 30000, 24000, 5
    m = torch.zeros((3, H, W), dtype=torch.uint8, device=DEV)
    m[0, :, ::k] = 1                                                   # one-pixel stripes every k columns
    m[1].view(H // 3, 3, W // 3, 3)[:, :2, :, :2] = 1                  # 2x2 blocks with one-pixel gaps
    m[2] = 1
    nbx = W // 3
    for conn in (4, 8):
        labels, counts = rbunet.label_components(m, conn)
        assert counts.tolist() == [(W + k - 1) // k, (H // 3) * nbx, 1]
        xs = torch.arange(W, device=DEV)
        for y0 in range(0, H, 3000):
            ys = torch.arange(y0, y0 + 3000, device=DEV)[:, None]
            stripes = torch.where(xs % k == 0, xs // k + 1, 0).expand(3000, W)
            block = ((ys % 3 < 2) & (xs % 3 < 2))
            blocks = torch.where(block, (ys // 3) * nbx + xs // 3 + 1, 0)
            assert torch.equal(labels[0, y0:y0 + 3000].long(), stripes), (conn, y0)
            assert torch.equal(labels[1, y0:y0 + 3000].long(), blocks), (conn, y0)
            assert bool((labels[2, y0:y0 + 3000] == 1).all())
        del labels
    out = rbunet.remove_small_regions(m, 5, 0, 8)                      # the 2x2 blocks go, the stripes stay
    assert torch.equal(out[0], m[0]) and not bool(out[1].any()) and bool(out[2].all())


def test_outputs_stay_inside_sentinel_filled_buffers():
    B, H, W = 3, 70, 131
    masks = np.stack([_masks(H, W, 9)[k] for k in ("p0.59", "spiral", "blobby")])
    m = _t(masks.astype(np.uint8))
    n = B * H * W
    nbytes = int(_lib.lib().rbu_label_workspace_bytes(B, H, W))
    ws = torch.full((nbytes + 4096,), 0xA5, dtype=torch.uint8, device=DEV)
    lab = torch.full((n + 2048,), -777, dtype=torch.int32, device=DEV)
    cnt = torch.full((B + 8,), -777, dtype=torch.int32, device=DEV)
    _lib.call("rbu_label_components", _p(m), 1, 0.5, B, H, W, 8, _p(lab[1024:]), _p(cnt[4:]), _p(ws), nbytes,
              _lib.stream_ptr())
    lo, co = lab.cpu().numpy(), cnt.cpu().numpy()
    assert (lo[:1024] == -777).all() and (lo[1024 + n:] == -777).all()
    assert (co[:4] == -777).all() and (co[4 + B:] == -777).all()
    assert (ws[nbytes:].cpu().numpy() == 0xA5).all()
    for i in range(B):
        want, k = R.label(masks[i], 8)
        assert co[4 + i] == k and np.array_equal(lo[1024 + i * H * W:1024 + (i + 1) * H * W].reshape(H, W), want)
    # statistics: rows before and after the offsets' range keep their sentinels
    counts = co[4:4 + B].astype(np.int64)
    offs = torch.tensor(np.concatenate([[5], 5 + np.cumsum(counts)]), dtype=torch.int64, device=DEV)
    rows = int(counts.sum())
    st = torch.full((rows + 10, 7), -555, dtype=torch.int64, device=DEV)
    _lib.call("rbu_component_stats", _p(lab[1024:]), B, H, W, _p(offs), _p(st), _lib.stream_ptr())
    so = st.cpu().numpy()
    assert (so[:5] == -555).all() and (so[5 + rows:] == -555).all()
    r0 = 5
    for i in range(B):
        want, k = R.label(masks[i], 8)
        assert np.array_equal(so[r0:r0 + k], R.stats(want, k))
        r0 += k
    # removal
    nb2 = int(_lib.lib().rbu_remove_small_regions_workspace_bytes(B, H, W))
    ws2 = torch.full((nb2 + 4096,), 0x5A, dtype=torch.uint8, device=DEV)
    out = torch.full((n + 2048,), 77, dtype=torch.uint8, device=DEV)
    _lib.call("rbu_remove_small_regions", _p(m), 1, 0.5, B, H, W, 4, 6, 9, _p(out[1024:]), _p(ws2), nb2,
              _lib.stream_ptr())
    oo = out.cpu().numpy()
    assert (oo[:1024] == 77).all() and (oo[1024 + n:] == 77).all() and (ws2[nb2:].cpu().numpy() == 0x5A).all()
    for i in range(B):
        assert np.array_equal(oo[1024 + i * H * W:1024 + (i + 1) * H * W].reshape(H, W), R.remove_small(masks[i], 6, 9, 4))


@pytest.mark.parametrize("conn", [4, 8])
def test_component_stats_equal_the_oracle_and_opencv(conn):
    H, W = 333, 517
    ms = _masks(H, W, 21)
    names = ["p0.3", "p0.59", "blobby", "spiral", "diagonals", "full", "empty"]
    batch = _t(np.stack([ms[k] for k in names]))
    labels, counts = rbunet.label_components(batch, conn)
    res = rbunet.component_stats(labels, counts)
    assert len(res) == len(names)
    for i, k in enumerate(names):
        st, cen = res[i]
        assert st.is_cuda and cen.is_cuda and st.dtype == torch.int64 and cen.dtype == torch.float64
        lab, n = R.label(ms[k], conn)
        want_st, want_cen = R.opencv_stats(R.stats(lab, n))
        assert st.shape == (n, 5) and cen.shape == (n, 2)
        assert np.array_equal(st.cpu().numpy(), want_st), k
        assert np.array_equal(cen.cpu().numpy().view(np.int64), want_cen.view(np.int64)), k
        if conn == 4:
            _, _, cst, ccen = cv2.connectedComponentsWithStats(ms[k].astype(np.uint8), connectivity=4, ltype=cv2.CV_32S)
            assert np.array_equal(st.cpu().numpy(), cst[1:].astype(np.int64)), k
            assert np.array_equal(cen.cpu().numpy().view(np.int64), ccen[1:].view(np.int64)), k
    one = rbunet.component_stats(labels[2], counts[2:3])                # an [H,W] label image
    assert torch.equal(one[0][0], res[2][0]) and torch.equal(one[0][1], res[2][1])


@pytest.mark.parametrize("conn", [4, 8])
def test_remove_small_regions_equals_the_oracle(conn):
    H, W = 257, 300
    ms = _masks(H, W, 5)
    rng = np.random.default_rng(conn)
    speckled = _blobby(H, W, 3) ^ (rng.random((H, W)) < 1e-2)
    masks = [speckled, ms["p0.41"], ms["p0.59"], ms["checker"], ms["spiral"], ms["full"], ms["empty"]]
    batch = _t(np.stack(masks))
    for mw, ml in ((0, 0), (1, 1), (0, 1), (4, 0), (0, 6), (12, 40), (2 ** 40, 3)):
        out = rbunet.remove_small_regions(batch, mw, ml, conn)
        assert out.dtype == torch.uint8 and out.shape == batch.shape
        got = out.cpu().numpy()
        for i, w in enumerate(masks):
            assert np.array_equal(got[i], R.remove_small(w, mw, ml, conn)), (mw, ml, i)
        if max(mw, ml) <= 1:
            assert np.array_equal(got, np.stack(masks).astype(np.uint8))
    # step 1 removes a water ring, which joins the land it enclosed to the outer land: step 2 no longer fills it
    w = np.zeros((40, 40), bool)
    w[10:25, 10:25] = True
    w[11:24, 11:24] = False
    out = rbunet.remove_small_regions(_t(w), 57, 200, conn).cpu().numpy()
    assert not out.any() and R.remove_small(w, 57, 200, conn).sum() == 0
    assert rbunet.remove_small_regions(_t(w), 0, 200, conn).cpu().numpy()[11:24, 11:24].all()


def test_predict_tiled_then_cleaning_then_coastline_metrics():
    torch.manual_seed(0)
    model = rbunet.RobustUNet(3, 1, 16).to(DEV).eval()
    H, W = 1000, 777
    g = torch.Generator().manual_seed(4)
    x = torch.randn((3, H, W), generator=g).to(DEV)
    labels = rbunet.predict_tiled(model, x, tile=256, overlap=32)
    target = torch.from_numpy(_blobby(H, W, 9).astype(np.uint8)).to(DEV)
    clean = rbunet.remove_small_regions(labels, 30, 30, 8)
    taus, s = (10, 20, 50), 10.0
    got = rbunet.coastline_metrics(clean, target, tolerances=taus, pixel_size=s)[0]
    want_clean = R.remove_small(labels.cpu().numpy() != 0, 30, 30, 8)
    assert np.array_equal(clean.cpu().numpy(), want_clean)
    st = D.coastline_stats(want_clean, target.cpu().numpy(), 0.5, [D.tolerance_d2(t, s) for t in taus])
    want = D.metrics_from_stats(st, taus, s)
    assert list(got) == list(want)
    for k, v in want.items():
        assert got[k] == v or (v != v and got[k] != got[k]) or abs(got[k] - v) <= 1e-12 * abs(v), k


def test_launch_counts_are_fixed_and_nothing_synchronises():
    lab_n, rem_n, st_n = set(), set(), set()
    for B, H, W in ((1, 40, 50), (3, 40, 50), (1, 333, 517), (5, 333, 517)):
        for dens in (0.0, 0.5, 1.0):
            m = (torch.rand((B, H, W), device=DEV) < dens)
            lab, cnt = rbunet.label_components(m, 8)
            n0 = _lib.launch_count()
            lab, cnt = rbunet.label_components(m, 4)
            lab_n.add(_lib.launch_count() - n0)
            n0 = _lib.launch_count()
            rbunet.remove_small_regions(m, 5, 5, 8)
            rem_n.add(_lib.launch_count() - n0)
            n0 = _lib.launch_count()
            rbunet.component_stats(lab, cnt)
            st_n.add(_lib.launch_count() - n0)
    assert lab_n == {6} and rem_n == {8} and st_n == {2}
    p = torch.rand((2, 200, 300), device=DEV)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        lab, cnt = rbunet.label_components(p, 8)
        out = rbunet.remove_small_regions(p, 10, 10)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert lab.shape == p.shape and out.shape == p.shape
    rbunet.component_stats(lab, cnt)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        rbunet.component_stats(lab, cnt)
        torch.cuda.synchronize()
    copies = [e.name for e in prof.events() if e.name.startswith("Memcpy ")]
    assert len(copies) == 1 and copies[0].startswith("Memcpy DtoH"), copies


def test_argument_errors_raise_before_any_launch():
    p = torch.rand((2, 32, 40), device=DEV)
    m = (p > 0.5).to(torch.uint8)
    lab, cnt = rbunet.label_components(p)
    lc, cs, rs = rbunet.label_components, rbunet.component_stats, rbunet.remove_small_regions
    cases = [
        (RuntimeError, "label_components", lambda: lc(p.cpu())),
        (RuntimeError, "remove_small_regions", lambda: rs(m.cpu(), 1, 1)),
        (RuntimeError, "component_stats", lambda: cs(lab.cpu(), cnt)),
        (TypeError, "label_components", lambda: lc(p.double())),
        (TypeError, "label_components", lambda: lc(p.numpy(force=True))),
        (TypeError, "remove_small_regions", lambda: rs(m.to(torch.int64), 1, 1)),
        (TypeError, "component_stats", lambda: cs(lab.long(), cnt)),
        (TypeError, "component_stats", lambda: cs(lab, cnt.long())),
        (ValueError, "component_stats", lambda: cs(lab, cnt[:1])),
        (ValueError, "label_components", lambda: lc(p[:, None].expand(2, 2, 32, 40))),
        (ValueError, "label_components", lambda: lc(p[0, 0])),
        (ValueError, "label_components", lambda: lc(p[:, :0])),
        (ValueError, "label_components", lambda: lc(torch.zeros((1, 32769), device=DEV))),
        (ValueError, "label_components", lambda: lc(p, 6)),
        (ValueError, "label_components", lambda: lc(p, True)),
        (ValueError, "label_components", lambda: lc(p, 4.0)),
        (ValueError, "label_components", lambda: lc(p, threshold=float("nan"))),
        (ValueError, "remove_small_regions", lambda: rs(p, 1, 1, connectivity=0)),
        (ValueError, "remove_small_regions", lambda: rs(p, -1, 1)),
        (ValueError, "remove_small_regions", lambda: rs(p, 1, -5)),
        (TypeError, "remove_small_regions", lambda: rs(p, 1.5, 1)),
        (TypeError, "remove_small_regions", lambda: rs(p, 1, True)),
        (ValueError, "remove_small_regions", lambda: rs(p, 1, 1, threshold=float("inf"))),
    ]
    if torch.cuda.device_count() > 1:
        cases.append((ValueError, "component_stats", lambda: cs(lab, cnt.to("cuda:1"))))
    for exc, who, fn in cases:
        n0 = _lib.launch_count()
        with pytest.raises(exc, match=f"rbunet.{who}"):
            fn()
        assert _lib.launch_count() == n0, who
    # the C ABI checks every argument before it launches
    nb = int(_lib.lib().rbu_label_workspace_bytes(2, 32, 40))
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    out = torch.empty((2, 32, 40), dtype=torch.int32, device=DEV)
    c = torch.empty(2, dtype=torch.int32, device=DEV)
    for args in ((_p(m), 1, 0.5, 2, 32, 40, 6, _p(out), _p(c), _p(ws), nb),
                 (_p(m), 2, 0.5, 2, 32, 40, 4, _p(out), _p(c), _p(ws), nb),
                 (_p(m), 1, 0.5, 2, 32, 40, 4, _p(out), _p(c), _p(ws), nb - 1),
                 (_p(m), 1, 0.5, 0, 32, 40, 4, _p(out), _p(c), _p(ws), nb),
                 (_p(m), 1, 0.5, 2, 32, 40, 4, _p(out), ctypes.c_void_p(0), _p(ws), nb)):
        n0 = _lib.launch_count()
        assert _lib.lib().rbu_label_components(*args, _lib.stream_ptr()) != 0
        assert _lib.launch_count() == n0
    torch.cuda.synchronize()
