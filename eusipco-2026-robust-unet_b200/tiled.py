"""Whole-scene prediction at full resolution: sliding-window (tiled) inference with Gaussian blending on the GPU.

The reference's prediction path (predict_coastline.py:386-392,583-602) resizes a scene to 512², predicts, and scales the
mask back up, which quantises the coastline to scene/512 pixels.  `predict_tiled` instead cuts the normalised scene into
overlapping tiles, runs them through the network in batches and blends the outputs back with a separable Gaussian window
(the sliding-window inference of nnU-Net and MONAI), with no host round trip.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np
import torch

from ._lib import call, stream_ptr
from .model import RobustUNet
from .ops import _p
from .unet import UNet

_WHO = "rbunet.predict_tiled"


def _axis(n: int, tile: int, overlap: int):
    """(tile origins, tile extent) along one axis.  n >= tile: ceil((n - tile) / s) + 1 tiles, s = tile - overlap, at
    min(i*s, n - tile), so the last tile ends at the scene edge.  n < tile: one tile shrunk to ceil16(n) (the network
    needs multiples of 16), whose < 16 rows past the scene are reflected."""
    if n < tile:
        return np.zeros(1, dtype=np.int64), -(-n // 16) * 16
    s = tile - overlap
    count = -(-(n - tile) // s) + 1
    return np.minimum(np.arange(count, dtype=np.int64) * s, n - tile), tile


def _cover(origins, extent: int, n: int):
    """Per index 0..n-1: the first tile covering it and the number of covering tiles (origins are increasing)."""
    idx = np.arange(n)
    first = np.searchsorted(origins + extent, idx, side="right")
    return first, np.searchsorted(origins, idx, side="right") - first


def _gaussian(extent: int, sigma_scale: float):
    """exp(-0.5 ((d + 0.5 - extent/2) / (sigma_scale * extent))^2) in float64, divided by its maximum, rounded to fp32."""
    d = np.arange(extent, dtype=np.float64)
    w = np.exp(-0.5 * ((d + 0.5 - extent / 2) / (sigma_scale * extent)) ** 2)
    return (w / w.max()).astype(np.float32)


@dataclass
class TilePlan:
    H: int
    W: int
    th: int
    tw: int
    oy: np.ndarray          # tile origins per axis; tile t = iy * nx + ix
    ox: np.ndarray
    row_first: np.ndarray   # per output row / column: first covering tile, number of covering tiles
    row_count: np.ndarray
    col_first: np.ndarray
    col_count: np.ndarray
    wy: np.ndarray          # fp32 window tables [th] / [tw]
    wx: np.ndarray

    @property
    def ny(self):
        return len(self.oy)

    @property
    def nx(self):
        return len(self.ox)

    def table(self) -> np.ndarray:
        """All tables in one int32 array (the weights as their bits), in the order of `offsets`."""
        parts = [self.oy, self.ox, self.row_first, self.row_count, self.col_first, self.col_count]
        return np.concatenate([a.astype(np.int32) for a in parts] + [self.wy.view(np.int32), self.wx.view(np.int32)])

    def offsets(self):
        sizes = [self.ny, self.nx, self.H, self.H, self.W, self.W, self.th, self.tw]
        return np.concatenate([[0], np.cumsum(sizes)[:-1]]).tolist()


def plan_tiles(H: int, W: int, tile, overlap, sigma_scale: float) -> TilePlan:
    oy, th = _axis(H, tile[0], overlap[0])
    ox, tw = _axis(W, tile[1], overlap[1])
    rf, rc = _cover(oy, th, H)
    cf, cc = _cover(ox, tw, W)
    return TilePlan(H, W, th, tw, oy, ox, rf, rc, cf, cc, _gaussian(th, sigma_scale), _gaussian(tw, sigma_scale))


def _pair(v, name):
    a, b = v if isinstance(v, (tuple, list)) and len(v) == 2 else (v, v)
    for u in (a, b):
        if isinstance(u, bool) or not isinstance(u, (int, np.integer)):
            raise TypeError(f"{_WHO}: {name} must be an int or a pair of ints, got {v!r}")
    return int(a), int(b)


def _network(model):
    """(input channels, classes, threshold of the K = 1 label rule) of a RobustUNet or UNet in eval mode."""
    if isinstance(model, RobustUNet):
        nc, K, thr = model.inc.conv1.in_channels, model.outc[0].out_channels, 0.5      # probabilities
    elif isinstance(model, UNet):
        nc, K, thr = model.enc1[0].in_channels, model.final.out_channels, 0.0          # logits
    else:
        raise TypeError(f"{_WHO}: model must be an rbunet.RobustUNet or rbunet.UNet, got {type(model).__name__}")
    if model.training:
        raise ValueError(f"{_WHO}: the model must be in eval mode (model.eval()): train-mode BatchNorm would make each "
                         "tile depend on the rest of its batch")
    return nc, K, thr


def _scene(x, nc):
    if not isinstance(x, torch.Tensor):
        raise TypeError(f"{_WHO}: x must be a torch.Tensor, got {type(x).__name__}")
    if not x.is_cuda:
        raise RuntimeError(f"{_WHO} runs on CUDA tensors only (no CPU fallback)")
    if x.dtype != torch.float32:
        raise TypeError(f"{_WHO}: x must be float32, got {x.dtype}")
    if x.dim() == 4 and x.shape[0] == 1:
        x = x[0]
    if x.dim() != 3:
        raise ValueError(f"{_WHO}: x must be [nc,H,W] or [1,nc,H,W], got {tuple(x.shape)}")
    if x.shape[0] != nc:
        raise ValueError(f"{_WHO}: the model expects {nc} input channels, x has {x.shape[0]}")
    if x.shape[1] < 16 or x.shape[2] < 16:
        raise ValueError(f"{_WHO}: H and W must be >= 16, got {x.shape[1]}x{x.shape[2]}")
    return x.contiguous()


def predict_tiled(model, x, tile=512, overlap=64, batch_size: int = 16, sigma_scale: float = 0.125,
                  return_outputs: bool = False):
    """Predict a whole scene at full resolution by sliding-window inference.

    model        rbunet.RobustUNet or rbunet.UNet in eval mode.
    x            fp32 CUDA scene [nc,H,W] or [1,nc,H,W], already normalised (e.g. rbunet.preprocess(scene_u8[None], nc));
                 any H, W >= 16.
    tile         int or (th, tw), multiples of 16.  An axis shorter than its tile gets one tile of ceil16(size), the
                 missing (< 16) rows or columns filled by reflection (F.pad(mode="reflect")).
    overlap      int or pair, 0 <= overlap < tile.  Per axis: ceil((H - th) / s) + 1 tiles at min(i*s, H - th), s = th -
                 overlap, row-major (t = iy*nx + ix).
    batch_size   tiles per network call.
    sigma_scale  the window w[d] = exp(-0.5 ((d + 0.5 - th/2) / (sigma_scale*th))^2), normalised to a maximum of 1.

    Returns labels, uint8 [H,W]: blended > 0.5 (RobustUNet, K = 1), blended > 0 (UNet logits, K = 1), the arg-max over
    the classes with ties to the lowest index (K >= 2).  With return_outputs=True, (labels, out): out is the blended fp32
    [K,H,W] of the model's outputs as they come (probabilities for RobustUNet, logits for UNet).

    Each output pixel is sum_t w_t v_t / sum_t w_t over the tiles covering it, with w_t the outer product of the window
    tables: one deterministic gather kernel, no atomics.  Runs under torch.no_grad() and never synchronises: one
    non-blocking copy of the plan tables, one gather launch and one network call per batch, one blend launch.
    Peak extra memory: the fp32 tile outputs, about (th*tw / s^2) * H*W*K*4 bytes, plus one batch's activations."""
    nc, K, thr = _network(model)
    x = _scene(x, nc)
    tile, overlap = _pair(tile, "tile"), _pair(overlap, "overlap")
    if any(t < 16 or t % 16 for t in tile):
        raise ValueError(f"{_WHO}: tile must be a multiple of 16 and >= 16, got {tile}")
    if any(not 0 <= o < t for o, t in zip(overlap, tile)):
        raise ValueError(f"{_WHO}: overlap must satisfy 0 <= overlap < tile, got overlap {overlap}, tile {tile}")
    if isinstance(batch_size, bool) or not isinstance(batch_size, (int, np.integer)) or batch_size < 1:
        raise ValueError(f"{_WHO}: batch_size must be a positive int, got {batch_size!r}")
    if not (isinstance(sigma_scale, (int, float)) and math.isfinite(sigma_scale) and sigma_scale > 0):
        raise ValueError(f"{_WHO}: sigma_scale must be a positive number, got {sigma_scale!r}")
    dev = x.device
    if any(p.device != dev for p in model.parameters()):
        raise ValueError(f"{_WHO}: the model's parameters are not all on {dev}, where x is")
    _, H, W = x.shape
    p = plan_tiles(H, W, tile, overlap, float(sigma_scale))
    if np.float32(p.wy.min()) * np.float32(p.wx.min()) == 0:
        raise ValueError(f"{_WHO}: sigma_scale {sigma_scale} is too small for a {p.th}x{p.tw} tile: the window's corner "
                         "weights underflow to 0 in fp32")
    T, th, tw = p.ny * p.nx, p.th, p.tw
    Tb_max = min(int(batch_size), T)

    with torch.no_grad(), torch.cuda.device(dev):
        tab = p.table()
        host = torch.empty(tab.size, dtype=torch.int32, pin_memory=True)
        host.numpy()[:] = tab
        table = host.to(dev, non_blocking=True)
        oy, ox, rf, rc, cf, cc, wy, wx = (_p(table[o:]) for o in p.offsets())
        tiles = torch.empty((T, K, th, tw), dtype=torch.float32, device=dev)
        batch = torch.empty((Tb_max, nc, th, tw), dtype=torch.float32, device=dev)
        for t0 in range(0, T, Tb_max):
            Tb = min(Tb_max, T - t0)
            call("rbu_tile_gather", _p(x), nc, H, W, oy, ox, p.ny, p.nx, th, tw, t0, Tb, _p(batch), stream_ptr(),
                 nbytes=2.0 * Tb * nc * th * tw * 4)
            tiles[t0:t0 + Tb] = model(batch[:Tb])
        labels = torch.empty((H, W), dtype=torch.uint8, device=dev)
        out = torch.empty((K, H, W), dtype=torch.float32, device=dev) if return_outputs else None
        call("rbu_tile_blend", _p(tiles), K, H, W, oy, ox, p.ny, p.nx, th, tw, rf, rc, cf, cc, wy, wx, thr, _p(out),
             _p(labels), stream_ptr(), nbytes=float(tiles.numel() * 4 + H * W * (1 + (K * 4 if return_outputs else 0))))
    return (labels, out) if return_outputs else labels
