"""GPU: outer-contour tracing (rbu_trace_contours / rbu_write_contours, rbunet.find_contours) bit for bit against the CPU
oracle (oracle/contours_ref.py) and cv2.findContours(RETR_EXTERNAL, CHAIN_APPROX_NONE | SIMPLE)."""
import ctypes

import cv2
import numpy as np
import pytest
import torch

import rbunet
from rbunet import _lib
from rbunet.ops import _p
from oracle import components_ref as C
from oracle import contours_ref as R
from test_gpu_components import _blobby, _masks, _t
from tools.components_bench import blobby

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MODES = {"none": cv2.CHAIN_APPROX_NONE, "simple": cv2.CHAIN_APPROX_SIMPLE}


def _cv(w, approx):
    cs = cv2.findContours(np.ascontiguousarray(w).astype(np.uint8), cv2.RETR_EXTERNAL, MODES[approx])[0]
    return [c.reshape(-1, 2) for c in cs]


def _check(pair, want, what):
    pts, offs = pair
    assert pts.is_cuda and offs.is_cuda and pts.dtype == torch.int32 and offs.dtype == torch.int64, what
    p, o = pts.cpu().numpy(), offs.cpu().numpy()
    assert o.shape == (len(want) + 1,) and o[0] == 0 and o[-1] == p.shape[0], (what, o[:3], o[-3:], p.shape)
    for k, w in enumerate(want):
        assert np.array_equal(p[o[k]:o[k + 1]], w), (what, k, len(want))


def _rings(H, W):
    """Nested square rings with islands in the lakes, a ring touching each edge, and corner pixels."""
    m = np.zeros((H, W), bool)
    for i, r in enumerate(range(2, min(H, W) // 2 - 2, 3)):
        m[r, r:W - r] = m[H - 1 - r, r:W - r] = m[r:H - r, r] = m[r:H - r, W - 1 - r] = True
    m[0, :] = m[:, 0] = True
    m[H - 1, W // 3:] = True
    m[[0, 0, H - 1, H - 1], [0, W - 1, 0, W - 1]] = True
    return m


def _lines(H, W):
    m = np.zeros((H, W), bool)
    y, x = np.indices((H, W))
    m |= (y == x) | (y == W - 1 - x)
    m[H // 2, ::2] = True
    m[::5, W // 3] = True
    return m


SHAPES = [(1, 1), (1, 4096), (4096, 1), (2, 3), (17, 530), (333, 517), (512, 512)]


@pytest.mark.parametrize("approx", ["none", "simple"])
@pytest.mark.parametrize("H,W", SHAPES)
def test_contours_are_bit_exact(H, W, approx):
    masks = _masks(H, W, H * 7 + W)
    masks.update({"rings": _rings(H, W), "lines": _lines(H, W),
                  "p0.2": np.random.default_rng(H).random((H, W)) < 0.2,
                  "p0.8": np.random.default_rng(W).random((H, W)) < 0.8})
    names = list(masks)
    batch = _t(np.stack([masks[k] for k in names]).astype(np.uint8))
    res = rbunet.find_contours(batch, approx)
    assert len(res) == len(names)
    for i, k in enumerate(names):
        want = R.find_contours(masks[k], approx)
        _check(res[i], want, (k, H, W))
        if H * W <= 512 * 512:
            _check(res[i], _cv(masks[k], approx), ("cv2", k, H, W))
    for k in ("blobby", "spiral", "rings"):                          # an image alone equals its batch member
        one = rbunet.find_contours(_t(masks[k]), approx)[0]
        i = names.index(k)
        assert torch.equal(one[0], res[i][0]) and torch.equal(one[1], res[i][1])


def test_random_small_masks_equal_opencv():
    rng = np.random.default_rng(11)
    for it in range(40):
        H, W = (int(v) for v in rng.integers(1, 60, 2))
        ws = [rng.random((H, W)) < d for d in (0.2, 0.41, 0.5, 0.59, 0.8)]
        for approx in ("none", "simple"):
            res = rbunet.find_contours(_t(np.stack(ws)), approx)
            for w, r in zip(ws, res):
                _check(r, _cv(w, approx), (it, H, W, approx))


def test_blobby_scene_equals_opencv():
    m = blobby(1, 10980, 10980, 1, 1e-3)[0]                           # the scene of tools/contours_bench.py
    w = m.cpu().numpy()
    for approx in ("simple", "none"):
        _check(rbunet.find_contours(m, approx)[0], _cv(w, approx), approx)


def test_input_dtypes_threshold_and_views():
    H, W = 70, 91
    rng = np.random.default_rng(3)
    prob = rng.random((H, W)).astype(np.float32)
    prob[rng.random((H, W)) < 0.2] = 0.5                              # exactly at the threshold: land
    w = C.water(prob)
    want = R.find_contours(w, "simple")
    for m in (_t(prob), _t(prob)[None, None], _t(w), _t(w.astype(np.uint8) * rng.choice([1, 255], (H, W)).astype(np.uint8))):
        res = rbunet.find_contours(m)
        assert len(res) == 1
        _check(res[0], want, str(m.dtype))
    _check(rbunet.find_contours(_t(prob), threshold=0.25)[0], R.find_contours(C.water(prob, 0.25), "simple"), "thr")
    big = _t(np.ascontiguousarray(prob.T))                            # a transposed (non-contiguous) view
    _check(rbunet.find_contours(big.t(), "none")[0], R.find_contours(w, "none"), "view")


def test_repeated_runs_and_batches_are_identical():
    masks = [_blobby(300, 411, s, 0.45, 1.5) | (np.random.default_rng(s).random((300, 411)) < 0.05) for s in range(4)]
    batch = _t(np.stack(masks))
    for approx in ("none", "simple"):
        a = rbunet.find_contours(batch, approx)
        b = rbunet.find_contours(batch, approx)
        for i in range(len(masks)):
            assert torch.equal(a[i][0], b[i][0]) and torch.equal(a[i][1], b[i][1])
            one = rbunet.find_contours(batch[i], approx)[0]
            assert torch.equal(one[0], a[i][0]) and torch.equal(one[1], a[i][1])


def test_a_30000_by_24000_scene_equals_closed_forms():
    H, W = 30000, 24000
    m = torch.zeros((H, W), dtype=torch.uint8, device=DEV)
    m.view(H // 50, 50, W // 40, 40)[:, 1:48, :, 2:37] = 1            # 47 x 35 rectangles, 600 x 600 of them
    ny, nx = H // 50, W // 40
    y0 = torch.arange(ny, device=DEV).repeat_interleave(nx) * 50 + 1
    x0 = torch.arange(nx, device=DEV).repeat(ny) * 40 + 2
    order = torch.arange(ny * nx - 1, -1, -1, device=DEV)            # decreasing raster order of the top-left corners
    y0, x0 = y0[order], x0[order]
    x1, y1 = x0 + 34, y0 + 46
    pts, offs = rbunet.find_contours(m, "simple")[0]
    assert offs.shape == (ny * nx + 1,) and pts.shape == (4 * ny * nx, 2)
    assert torch.equal(offs, torch.arange(ny * nx + 1, device=DEV) * 4)
    want = torch.stack([torch.stack([x0, y0], 1), torch.stack([x0, y1], 1), torch.stack([x1, y1], 1),
                        torch.stack([x1, y0], 1)], 1).reshape(-1, 2).int()
    assert torch.equal(pts, want)
    pts, offs = rbunet.find_contours(m, "none")[0]
    per = 2 * (47 + 35) - 4
    assert torch.equal(offs, torch.arange(ny * nx + 1, device=DEV) * per)
    first = pts.view(ny * nx, per, 2)
    assert torch.equal(first[:, 0], torch.stack([x0, y0], 1).int())  # each contour starts at its corner
    assert torch.equal(first[:, 46], torch.stack([x0, y1], 1).int())  # down the left side first
    del pts, offs, first
    pts, offs = rbunet.find_contours(torch.ones((H, W), dtype=torch.bool, device=DEV))[0]
    assert pts.tolist() == [[0, 0], [0, H - 1], [W - 1, H - 1], [W - 1, 0]] and offs.tolist() == [0, 4]


def test_outputs_stay_inside_sentinel_filled_buffers():
    B, H, W = 3, 70, 131
    masks = np.stack([_masks(H, W, 9)[k] for k in ("p0.59", "spiral", "blobby")])
    m = _t(masks.astype(np.uint8))
    nbytes = int(_lib.lib().rbu_contours_workspace_bytes(B, H, W))
    ws = torch.full((nbytes + 4096,), 0xA5, dtype=torch.uint8, device=DEV)
    cnt = torch.full((B + 8, 2), -777, dtype=torch.int64, device=DEV)
    _lib.call("rbu_trace_contours", _p(m), 1, 0.5, B, H, W, 2, _p(cnt[4:]), _p(ws), nbytes, _lib.stream_ptr())
    co = cnt.cpu().numpy()
    assert (co[:4] == -777).all() and (co[4 + B:] == -777).all()
    want = [R.find_contours(w, "simple") for w in masks]
    assert co[4:4 + B].tolist() == [[len(c), sum(len(x) for x in c)] for c in want]
    n_offs, n_pts = int((co[4:4 + B, 0] + 1).sum()), int(co[4:4 + B, 1].sum())
    coff = torch.tensor(np.concatenate([[0], np.cumsum(co[4:4 + B, 0] + 1)[:-1]]) + 5, dtype=torch.int64, device=DEV)
    poff = torch.tensor(np.concatenate([[0], np.cumsum(co[4:4 + B, 1])[:-1]]) + 7, dtype=torch.int64, device=DEV)
    offs = torch.full((n_offs + 20,), -555, dtype=torch.int64, device=DEV)
    pts = torch.full((n_pts + 20, 2), -999, dtype=torch.int32, device=DEV)
    _lib.call("rbu_write_contours", _p(ws), nbytes, B, H, W, _p(coff), _p(poff), _p(offs), _p(pts), _lib.stream_ptr())
    oo, po = offs.cpu().numpy(), pts.cpu().numpy()
    offs.fill_(-555)                                                   # the write call can be repeated
    pts[7:7 + n_pts].fill_(-999)
    _lib.call("rbu_write_contours", _p(ws), nbytes, B, H, W, _p(coff), _p(poff), _p(offs), _p(pts), _lib.stream_ptr())
    assert np.array_equal(offs.cpu().numpy(), oo) and np.array_equal(pts.cpu().numpy(), po)
    assert (oo[:5] == -555).all() and (oo[5 + n_offs:] == -555).all()
    assert (po[:7] == -999).all() and (po[7 + n_pts:] == -999).all()
    assert (ws[nbytes:].cpu().numpy() == 0xA5).all()
    c0, p0 = 5, 7
    for i in range(B):
        n = len(want[i])
        o = oo[c0:c0 + n + 1]
        for k in range(n):
            assert np.array_equal(po[p0 + o[k]:p0 + o[k + 1]], want[i][k])
        c0, p0 = c0 + n + 1, p0 + o[-1]


def test_predict_tiled_then_cleaning_then_contours():
    torch.manual_seed(0)
    model = rbunet.RobustUNet(3, 1, 16).to(DEV).eval()
    H, W = 1000, 777
    g = torch.Generator().manual_seed(4)
    x = torch.randn((3, H, W), generator=g).to(DEV)
    labels = rbunet.predict_tiled(model, x, tile=256, overlap=32)
    clean = rbunet.remove_small_regions(labels, 30, 30, 8)
    band = rbunet.coastline_mask(clean * 255, 5)
    for approx in ("simple", "none"):
        _check(rbunet.find_contours(band, approx)[0], _cv(band.cpu().numpy(), approx), approx)


def test_launch_counts_are_fixed_and_one_copy():
    seen = {}
    for B, H, W in ((1, 40, 50), (3, 40, 50), (1, 333, 517)):
        for dens in (0.0, 0.5, 1.0):
            m = torch.rand((B, H, W), device=DEV) < dens
            m[:, ::2, ::2] |= dens == 0.5                              # a checkerboard-like mix
            for approx in ("none", "simple"):
                n0 = _lib.launch_count()
                rbunet.find_contours(m, approx)
                seen.setdefault((B, H, W), set()).add(_lib.launch_count() - n0)
    for (B, H, W), n in seen.items():
        cap = min(4 * H * W, 8 * (H * W + 2 * H + 2 * W + 4) // 3)
        assert n == {15 + (cap - 1).bit_length()}, ((B, H, W), n)
    p = torch.rand((2, 200, 300), device=DEV)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        from rbunet.contours import _trace
        _trace(p, "simple", 0.5, "rbunet.find_contours")
    finally:
        torch.cuda.set_sync_debug_mode(0)
    rbunet.find_contours(p)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        rbunet.find_contours(p)
        torch.cuda.synchronize()
    copies = [e.name for e in prof.events() if e.name.startswith("Memcpy ")]
    assert len(copies) == 1 and copies[0].startswith("Memcpy DtoH"), copies


def test_argument_errors_raise_before_any_launch():
    p = torch.rand((2, 32, 40), device=DEV)
    fc = rbunet.find_contours
    cases = [
        (RuntimeError, lambda: fc(p.cpu())),
        (TypeError, lambda: fc(p.double())),
        (TypeError, lambda: fc(p.numpy(force=True))),
        (TypeError, lambda: fc(p, 2)),
        (ValueError, lambda: fc(p, "tc89")),
        (ValueError, lambda: fc(p[:, None].expand(2, 2, 32, 40))),
        (ValueError, lambda: fc(p[0, 0])),
        (ValueError, lambda: fc(p[:, :0])),
        (ValueError, lambda: fc(torch.zeros((1, 32769), device=DEV))),
        (ValueError, lambda: fc(p, threshold=float("nan"))),
        (ValueError, lambda: fc(p, threshold="0.5")),
    ]
    for exc, fn in cases:
        n0 = _lib.launch_count()
        with pytest.raises(exc, match="rbunet.find_contours"):
            fn()
        assert _lib.launch_count() == n0
    m = (p > 0.5).to(torch.uint8)
    nb = int(_lib.lib().rbu_contours_workspace_bytes(2, 32, 40))
    assert int(_lib.lib().rbu_contours_workspace_bytes(0, 32, 40)) == 0
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    c = torch.empty((2, 2), dtype=torch.int64, device=DEV)
    for args in ((_p(m), 1, 0.5, 2, 32, 40, 3, _p(c), _p(ws), nb),
                 (_p(m), 2, 0.5, 2, 32, 40, 2, _p(c), _p(ws), nb),
                 (_p(m), 1, 0.5, 2, 32, 40, 2, _p(c), _p(ws), nb - 1),
                 (_p(m), 1, 0.5, 0, 32, 40, 2, _p(c), _p(ws), nb),
                 (_p(m), 1, 0.5, 2, 32, 40, 2, ctypes.c_void_p(0), _p(ws), nb)):
        n0 = _lib.launch_count()
        assert _lib.lib().rbu_trace_contours(*args, _lib.stream_ptr()) != 0
        assert _lib.launch_count() == n0
    o = torch.empty(8, dtype=torch.int64, device=DEV)
    n0 = _lib.launch_count()
    assert _lib.lib().rbu_write_contours(_p(ws), nb - 1, 2, 32, 40, _p(c), _p(c), _p(o), _p(o), _lib.stream_ptr()) != 0
    assert _lib.lib().rbu_write_contours(_p(ws), nb, 2, 32, 40, ctypes.c_void_p(0), _p(c), _p(o), _p(o),
                                         _lib.stream_ptr()) != 0
    assert _lib.launch_count() == n0
    torch.cuda.synchronize()

