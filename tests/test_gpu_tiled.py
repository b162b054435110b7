"""GPU: sliding-window prediction of whole scenes (rbu_tile_gather, rbu_tile_blend, rbunet.predict_tiled) against the
CPU oracle (oracle/tiled_ref.py), bit for bit."""
import numpy as np
import pytest
import torch

import rbunet
from rbunet import _lib, tiled
from rbunet.ops import _p
from oracle import tiled_ref as T
from gpu_util import rel_l2

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _tables(p):
    """The plan's device tables as predict_tiled builds them: pointers (oy, ox, rf, rc, cf, cc, wy, wx) and the buffer."""
    table = torch.from_numpy(p.table()).to(DEV)
    return [_p(table[o:]) for o in p.offsets()], table


def _scene(nc, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randn((nc, H, W), generator=g)


@pytest.mark.parametrize("H,W", [(16, 16), (17, 530), (200, 328), (1000, 777)])
@pytest.mark.parametrize("nc", [3, 4])
def test_gather_is_bit_exact(H, W, nc):
    x = _scene(nc, H, W, H + W + nc)
    p = tiled.plan_tiles(H, W, (64, 64), (16, 16), 0.125)
    po = T.plan(H, W, (64, 64), (16, 16))
    ptrs, keep = _tables(p)
    n = p.ny * p.nx
    xd = x.to(DEV)
    for t0, Tb in ((0, min(5, n)), (max(0, n - 7), min(7, n))):            # first batch and a batch ending at the last tile
        out = torch.full((Tb, nc, p.th, p.tw), float("nan"), device=DEV)
        _lib.call("rbu_tile_gather", _p(xd), nc, H, W, ptrs[0], ptrs[1], p.ny, p.nx, p.th, p.tw, t0, Tb, _p(out),
                  _lib.stream_ptr())
        want = T.gather(x, po, t0, Tb)
        assert torch.equal(out.cpu(), want), (t0, Tb)


def _blend(tiles_d, p, K, thr, with_out):
    ptrs, keep = _tables(p)
    labels = torch.full((p.H, p.W), 255, dtype=torch.uint8, device=DEV)
    out = torch.full((K, p.H, p.W), float("nan"), device=DEV) if with_out else None
    _lib.call("rbu_tile_blend", _p(tiles_d), K, p.H, p.W, ptrs[0], ptrs[1], p.ny, p.nx, p.th, p.tw, *ptrs[2:], thr,
              _p(out), _p(labels), _lib.stream_ptr())
    return labels.cpu(), (out.cpu() if with_out else None)


@pytest.mark.parametrize("K,network", [(1, "RobustUNet"), (1, "UNet"), (2, "UNet"), (5, "RobustUNet"), (32, "UNet")])
@pytest.mark.parametrize("with_out", [True, False])
@pytest.mark.parametrize("H,W,tile,overlap", [(200, 328, 64, 16), (17, 530, 64, 48), (333, 95, 32, 0)])
def test_blend_is_bit_exact(K, network, with_out, H, W, tile, overlap):
    p = tiled.plan_tiles(H, W, (tile, tile), (overlap, overlap), 0.125)
    po = T.plan(H, W, (tile, tile), (overlap, overlap))
    thr = 0.5 if network == "RobustUNet" else 0.0
    g = torch.Generator().manual_seed(K * 7 + H)
    n = p.ny * p.nx
    tiles = torch.rand((n, K, p.th, p.tw), generator=g) * 2 - (0.5 if thr else 1.0)
    tiles[::2, :, : p.th // 2, : p.tw // 2] = thr          # blended values exactly at the threshold where one tile covers
    if K > 1:
        tiles[:, K - 1] = tiles[:, 0]                      # exact arg-max ties between the first and the last class
    labels, out = _blend(tiles.to(DEV), p, K, thr, with_out)
    want = T.blend(tiles, po)
    want_labels = T.labels(want, network)
    if with_out:
        assert torch.equal(out.view(torch.int32), want.view(torch.int32))
    assert torch.equal(labels, want_labels)
    if K == 1:
        assert (want == thr).any()
    else:
        assert ((want[0] == want[K - 1]) & (want_labels == 0) & (want[0] == want.max(0).values)).any()


MODELS = [("RobustUNet", lambda: rbunet.RobustUNet(3, 1, 16)), ("RobustUNet", lambda: rbunet.RobustUNet(3, 4, 16)),
          ("UNet", lambda: rbunet.UNet(3, 2))]


def _model(make, seed=0):
    torch.manual_seed(seed)
    m = make().to(DEV).eval()
    with torch.no_grad():                 # move the BatchNorm running statistics away from the identity
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.running_mean.uniform_(-0.1, 0.1)
                mod.running_var.uniform_(0.5, 1.5)
    return m


def _oracle_predict(model, x, p, batch_size, network):
    """The oracle's tiles through model() in predict_tiled's batches, then the oracle blend."""
    n = p["ny"] * p["nx"]
    outs = []
    with torch.no_grad():
        for t0 in range(0, n, batch_size):
            Tb = min(batch_size, n - t0)
            outs.append(model(T.gather(x, p, t0, Tb).to(DEV)).cpu())
    want = T.blend(torch.cat(outs), p)
    return T.labels(want, network), want


@pytest.mark.parametrize("idx", range(len(MODELS)))
def test_predict_tiled_equals_the_oracle_blend_of_the_model(idx):
    network, make = MODELS[idx]
    model = _model(make)
    for (H, W), bs in (((40, 200), 3), ((200, 328), 8)):              # the 200x328 results are reused below
        x = _scene(3, H, W, H)
        labels, out = rbunet.predict_tiled(model, x.to(DEV), tile=64, overlap=16, batch_size=bs, return_outputs=True)
        p = T.plan(H, W, (64, 64), (16, 16))
        want_labels, want = _oracle_predict(model, x, p, bs, network)
        K = want.shape[0]
        assert labels.dtype == torch.uint8 and labels.shape == (H, W) and out.shape == (K, H, W)
        assert torch.equal(out.cpu().view(torch.int32), want.view(torch.int32)), (H, W)
        assert torch.equal(labels.cpu(), want_labels), (H, W)
        only = rbunet.predict_tiled(model, x.to(DEV)[None], tile=64, overlap=16, batch_size=bs)
        assert torch.equal(only.cpu(), want_labels)                           # [1,nc,H,W] input, labels only
    x = _scene(3, 200, 328, 200).to(DEV)
    _, other = rbunet.predict_tiled(model, x, tile=64, overlap=16, batch_size=5, return_outputs=True)
    assert rel_l2(other, out) < 1e-5
    l2, again = rbunet.predict_tiled(model, x, tile=64, overlap=16, batch_size=8, return_outputs=True)
    assert torch.equal(again.view(torch.int32), out.view(torch.int32)) and torch.equal(l2, labels)


@pytest.mark.parametrize("idx", range(len(MODELS)))
def test_a_scene_of_one_tile_is_the_model_output(idx):
    network, make = MODELS[idx]
    model = _model(make, 1)
    x = _scene(3, 64, 96, 5).to(DEV)
    labels, out = rbunet.predict_tiled(model, x, tile=(64, 96), overlap=16, return_outputs=True)
    with torch.no_grad():
        ref = model(x[None])[0]
    out, ref, labels = out.cpu().double(), ref.cpu().double(), labels.cpu()
    ulp = torch.from_numpy(np.spacing(np.abs(ref.float().numpy()))).double()
    assert ((out - ref).abs() <= 2 * ulp).all()
    if ref.shape[0] == 1:
        thr = 0.5 if network == "RobustUNet" else 0.0
        clear = (ref[0] - thr).abs() > 1e-6
        assert torch.equal(labels[clear], (ref[0] > thr).to(torch.uint8)[clear])
    else:
        top2 = ref.topk(2, dim=0).values
        clear = (top2[0] - top2[1]) > 1e-6
        assert torch.equal(labels[clear], ref.argmax(0).to(torch.uint8)[clear])


def test_launches_are_one_gather_per_batch_the_network_and_one_blend():
    model = _model(MODELS[0][1])
    x = _scene(3, 200, 328, 9).to(DEV)
    p = tiled.plan_tiles(200, 328, (64, 64), (16, 16), 0.125)
    n = p.ny * p.nx
    assert n % 8                                                # a last batch smaller than the others
    rbunet.predict_tiled(model, x, tile=64, overlap=16, batch_size=8)         # packs the weights once
    net = {}
    with torch.no_grad():
        for Tb in (8, n % 8):
            n0 = _lib.launch_count()
            model(torch.zeros((Tb, 3, 64, 64), device=DEV))
            net[Tb] = _lib.launch_count() - n0
    n0 = _lib.launch_count()
    rbunet.predict_tiled(model, x, tile=64, overlap=16, batch_size=8)
    batches = -(-n // 8)
    assert _lib.launch_count() - n0 == batches + (batches - 1) * net[8] + net[n % 8] + 1


def test_never_synchronises():
    model = _model(MODELS[0][1])
    x = _scene(3, 200, 328, 10).to(DEV)
    rbunet.predict_tiled(model, x, tile=64, overlap=16)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        labels = rbunet.predict_tiled(model, x, tile=64, overlap=16)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert labels.shape == (200, 328)


def test_argument_errors_raise_before_any_launch():
    model = _model(MODELS[0][1])
    x = _scene(3, 64, 64, 11).to(DEV)
    rbunet.predict_tiled(model, x, tile=32, overlap=8)
    cases = [
        (RuntimeError, lambda: rbunet.predict_tiled(model, x.cpu())),
        (TypeError, lambda: rbunet.predict_tiled(model, x.half())),
        (TypeError, lambda: rbunet.predict_tiled(model, x.cpu().numpy())),
        (ValueError, lambda: rbunet.predict_tiled(model, x[:2])),                              # wrong nc
        (ValueError, lambda: rbunet.predict_tiled(model, torch.cat([x, x])[None].reshape(2, 3, 64, 64))),   # batch 2
        (ValueError, lambda: rbunet.predict_tiled(model, x[:, :15])),                          # H < 16
        (ValueError, lambda: rbunet.predict_tiled(model, x[:, :, :15])),                       # W < 16
        (ValueError, lambda: rbunet.predict_tiled(model, x, tile=40)),
        (ValueError, lambda: rbunet.predict_tiled(model, x, tile=0)),
        (ValueError, lambda: rbunet.predict_tiled(model, x, tile=(64, 8))),
        (TypeError, lambda: rbunet.predict_tiled(model, x, tile=64.0)),
        (ValueError, lambda: rbunet.predict_tiled(model, x, tile=32, overlap=32)),
        (ValueError, lambda: rbunet.predict_tiled(model, x, tile=32, overlap=-1)),
        (ValueError, lambda: rbunet.predict_tiled(model, x, batch_size=0)),
        (ValueError, lambda: rbunet.predict_tiled(model, x, sigma_scale=0.0)),
        (ValueError, lambda: rbunet.predict_tiled(model, x, sigma_scale=float("nan"))),
        (ValueError, lambda: rbunet.predict_tiled(model, x, tile=512, sigma_scale=0.01)),      # window underflows
        (TypeError, lambda: rbunet.predict_tiled(torch.nn.DataParallel(model), x)),
        (TypeError, lambda: rbunet.predict_tiled(torch.nn.Conv2d(3, 1, 1).to(DEV).eval(), x)),
    ]
    for exc, fn in cases:
        n0 = _lib.launch_count()
        with pytest.raises(exc, match="rbunet.predict_tiled"):
            fn()
        assert _lib.launch_count() == n0
    model.train()
    with pytest.raises(ValueError, match="rbunet.predict_tiled.*eval"):
        rbunet.predict_tiled(model, x)
    cpu_model = rbunet.RobustUNet(3, 1, 16).eval()
    with pytest.raises(ValueError, match="rbunet.predict_tiled"):
        rbunet.predict_tiled(cpu_model, x)
    torch.cuda.synchronize()
