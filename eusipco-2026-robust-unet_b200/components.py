"""Cleaning predicted water masks on the GPU: connected-component labelling, per-component statistics and small-region
removal (csrc/components.cu; DESIGN.md §8 item 9).

A whole-scene prediction carries speckle: small false water blobs inland and land specks at sea.  Each one adds its own
ring of coastline, so one blob far inland sets the Hausdorff distance of `coastline_metrics`, and every blob becomes a
polygon of its own when the coastline band is traced.  `remove_small_regions` is the usual cure (skimage's
remove_small_objects / remove_small_holes); `label_components` and `component_stats` are the building blocks
(scipy.ndimage.label, cv2.connectedComponentsWithStats), e.g. to keep only the largest water body.

Definitions:
  water         the rules of coastline_stats' pred: float32 p > threshold (strict); uint8 / bool nonzero.  Masks are
                [H,W], [B,H,W] or [B,1,H,W], 1 <= H, W <= 32768, B <= 65535.
  connectivity  4 (edge neighbours) or 8 (edge and corner neighbours).
  labels        int32, 0 on land, components numbered 1..n in raster order of their first pixel (minimum y*W + x):
                exactly scipy.ndimage.label(water, generate_binary_structure(2, 1 if connectivity == 4 else 2)).
"""
from __future__ import annotations

import math

import torch

from . import _lib
from ._lib import call, stream_ptr
from .distance import _KIND, _check_hw, _mask
from .ops import _p

MAX_IMAGES = 65535


def _connectivity(connectivity, who):
    if isinstance(connectivity, bool) or not isinstance(connectivity, int) or connectivity not in (4, 8):
        raise ValueError(f"{who}: connectivity must be 4 or 8, got {connectivity!r}")
    return int(connectivity)


def _water(mask, threshold, connectivity, who):
    m = _mask(mask, "mask", who)
    B, H, W = m.shape
    _check_hw(who, H, W)
    if not 1 <= B <= MAX_IMAGES:
        raise ValueError(f"{who}: 1 to {MAX_IMAGES} images per call, got {B}")
    if not (isinstance(threshold, (int, float)) and not isinstance(threshold, bool) and math.isfinite(threshold)):
        raise ValueError(f"{who}: threshold must be a finite number, got {threshold!r}")
    conn = _connectivity(connectivity, who)
    m = m.detach().contiguous()
    return (m.view(torch.uint8) if m.dtype == torch.bool else m), conn


def label_components(mask: torch.Tensor, connectivity: int = 4, threshold: float = 0.5):
    """Connected components of the water of `mask` (a CUDA tensor [H,W], [B,H,W] or [B,1,H,W]; float32, uint8 or bool).

    Returns (labels, counts): labels int32 with the mask's shape, 0 on land and 1..n_b on the components of image b in
    raster order of their first pixel (= scipy.ndimage.label with the 4- or 8-neighbour structure); counts int32 [B]
    holds n_b (B = 1 for an [H,W] mask).  Both stay on the device: six launches whatever the content, never
    synchronises."""
    who = "rbunet.label_components"
    m, conn = _water(mask, threshold, connectivity, who)
    B, H, W = m.shape
    dev = m.device
    with torch.cuda.device(dev):
        nbytes = int(_lib.lib().rbu_label_workspace_bytes(B, H, W))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        labels = torch.empty((B, H, W), dtype=torch.int32, device=dev)
        counts = torch.empty((B,), dtype=torch.int32, device=dev)
        call("rbu_label_components", _p(m), _KIND[m.dtype], float(threshold), B, H, W, conn, _p(labels), _p(counts),
             _p(ws), nbytes, stream_ptr(), nbytes=float(m.numel() * m.element_size() + 4 * B * H * W))
    return labels.reshape(mask.shape), counts


def component_stats(labels: torch.Tensor, counts: torch.Tensor) -> list:
    """Per image, (stats, centroids) of the components of `labels` (as label_components returns them, [H,W], [B,H,W] or
    [B,1,H,W] int32) with counts int32 [B]:
      stats      int64 [n_b, 5] in OpenCV's layout: CC_STAT_LEFT, TOP, WIDTH, HEIGHT, AREA;
      centroids  float64 [n_b, 2]: (sum of x / area, sum of y / area) from exact integer sums.
    Row k describes label k + 1.  Equal to cv2.connectedComponentsWithStats(...)[2][1:] and [3][1:] for the same labels.
    Both are CUDA tensors.  Makes exactly one device-to-host copy (the counts, to size the output); two launches."""
    who = "rbunet.component_stats"
    for name, t in (("labels", labels), ("counts", counts)):
        if not isinstance(t, torch.Tensor):
            raise TypeError(f"{who}: {name} must be a torch.Tensor, got {type(t).__name__}")
        if not t.is_cuda:
            raise RuntimeError(f"{who} runs on CUDA tensors only (no CPU fallback): {name} is on {t.device}")
        if t.dtype != torch.int32:
            raise TypeError(f"{who}: {name} must be int32, got {t.dtype}")
    lab = labels
    if lab.dim() == 4:
        if lab.shape[1] != 1:
            raise ValueError(f"{who}: labels must be [H,W], [B,H,W] or [B,1,H,W], got {tuple(labels.shape)}")
        lab = lab[:, 0]
    if lab.dim() == 2:
        lab = lab[None]
    if lab.dim() != 3:
        raise ValueError(f"{who}: labels must be [H,W], [B,H,W] or [B,1,H,W], got {tuple(labels.shape)}")
    B, H, W = lab.shape
    _check_hw(who, H, W)
    if not 1 <= B <= MAX_IMAGES:
        raise ValueError(f"{who}: 1 to {MAX_IMAGES} images per call, got {B}")
    if counts.shape != (B,):
        raise ValueError(f"{who}: counts must be [{B}], got {tuple(counts.shape)}")
    if counts.device != lab.device:
        raise ValueError(f"{who}: labels are on {lab.device}, counts on {counts.device}")
    lab = lab.contiguous()
    dev = lab.device
    with torch.cuda.device(dev):
        n = [int(c) for c in counts.cpu().tolist()]            # the one device-to-host copy
        if min(n) < 0:
            raise ValueError(f"{who}: counts must be non-negative, got {n}")
        offsets = torch.cat([torch.zeros((1,), dtype=torch.int64, device=dev), counts.cumsum(0, dtype=torch.int64)])
        rows = sum(n)
        raw = torch.empty((max(rows, 1), 7), dtype=torch.int64, device=dev)
        call("rbu_component_stats", _p(lab), B, H, W, _p(offsets), _p(raw), stream_ptr(),
             nbytes=float(4 * B * H * W + 56 * rows))
        raw = raw[:rows]
        left, top = raw[:, 0], raw[:, 1]
        stats = torch.stack([left, top, raw[:, 2] - left + 1, raw[:, 3] - top + 1, raw[:, 4]], dim=1)
        area = raw[:, 4].to(torch.float64)
        centroids = torch.stack([raw[:, 5].to(torch.float64) / area, raw[:, 6].to(torch.float64) / area], dim=1)
    out, r0 = [], 0
    for k in n:
        out.append((stats[r0:r0 + k], centroids[r0:r0 + k]))
        r0 += k
    return out


def _min_size(v, name, who):
    if isinstance(v, bool) or not isinstance(v, int):
        raise TypeError(f"{who}: {name} must be a non-negative int, got {v!r}")
    if v < 0:
        raise ValueError(f"{who}: {name} must be a non-negative int, got {v}")
    return min(v, 2 ** 31 - 1)            # no component has more than 2^30 pixels


def remove_small_regions(mask: torch.Tensor, min_water: int, min_land: int, connectivity: int = 4,
                         threshold: float = 0.5) -> torch.Tensor:
    """The cleaned water mask, uint8 0/1 with the mask's shape, in two steps at the same connectivity:
      1. every water component with fewer than min_water pixels becomes land;
      2. on the result of step 1, every land component with fewer than min_land pixels becomes water.
    Regions touching the image border get no special treatment; 0 or 1 makes its step the identity.  mask as for
    label_components.  Eight launches whatever the content; never synchronises."""
    who = "rbunet.remove_small_regions"
    mw, ml = _min_size(min_water, "min_water", who), _min_size(min_land, "min_land", who)
    m, conn = _water(mask, threshold, connectivity, who)
    B, H, W = m.shape
    dev = m.device
    with torch.cuda.device(dev):
        nbytes = int(_lib.lib().rbu_remove_small_regions_workspace_bytes(B, H, W))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        out = torch.empty((B, H, W), dtype=torch.uint8, device=dev)
        call("rbu_remove_small_regions", _p(m), _KIND[m.dtype], float(threshold), B, H, W, conn, mw, ml, _p(out),
             _p(ws), nbytes, stream_ptr(), nbytes=float(m.numel() * m.element_size() + B * H * W))
    return out.reshape(mask.shape)
