"""How far the predicted coastline is from the true one: the exact Euclidean distance transform and coastline distance
metrics on the GPU (csrc/distance.cu; DESIGN.md §8 item 8).

The area metrics (`calculate_metrics`, `batch_metrics`, `class_metrics`) are dominated by open water and inland pixels on
a whole scene; a coastline 30 pixels off can still score an IoU above 0.99.  `coastline_metrics` reports the position
errors of coastline and calving-front work and of MONAI / `surface-distance`: the directed and symmetric mean distances,
the Hausdorff distance and its 95th percentile, and per tolerance the share of each line within it (precision, recall,
F1, surface Dice).

Definitions:
  water       float32 pred: p > threshold (strict); float32 target: t != 0; uint8 / bool: nonzero.
  coastline   the non-water pixels with a water pixel among their four in-image neighbours (= coastline_mask(water, 3)
              != 0).  P is the coastline of pred, G that of target.
  samples     direction 0 (pred -> target): the distances from each pixel of P to the nearest pixel of G; direction 1
              (target -> pred): from each pixel of G to the nearest pixel of P.  Distances are Euclidean, in pixels,
              times pixel_size.
"""
from __future__ import annotations

import ctypes
import math

import torch

from . import _lib
from ._lib import call, stream_ptr
from .ops import _p

MAX_SIDE = 32768
MAX_TOLERANCES = 8
_KIND = {torch.float32: 0, torch.uint8: 1, torch.bool: 1}      # RBU_KIND_F32, RBU_KIND_U8
_DIST_KEYS = ("pred_to_target", "target_to_pred", "mean_distance", "hausdorff", "hausdorff95")


def _check_hw(who, H, W):
    if not (1 <= H <= MAX_SIDE and 1 <= W <= MAX_SIDE):
        raise ValueError(f"{who}: H and W must be in [1, {MAX_SIDE}], got {H}x{W}")


def distance_transform(features: torch.Tensor) -> torch.Tensor:
    """Exact squared Euclidean distance transform of a uint8 / bool CUDA tensor [H,W] or [B,H,W] (nonzero = feature):
    int32 of the same shape, D(y,x) = min over feature pixels (v,u) of (y-v)^2 + (x-u)^2, 0 on the features and -1
    everywhere in an image without a feature pixel.  Equal to rint(scipy.ndimage.distance_transform_edt(F == 0) ** 2).
    Four launches whatever the size; never synchronises."""
    who = "rbunet.distance_transform"
    if not isinstance(features, torch.Tensor):
        raise TypeError(f"{who}: features must be a torch.Tensor, got {type(features).__name__}")
    if not features.is_cuda:
        raise RuntimeError(f"{who} runs on CUDA tensors only (no CPU fallback)")
    if features.dtype not in (torch.uint8, torch.bool):
        raise TypeError(f"{who}: features must be uint8 or bool, got {features.dtype}")
    if features.dim() not in (2, 3):
        raise ValueError(f"{who}: features must be [H,W] or [B,H,W], got {tuple(features.shape)}")
    f = features if features.dim() == 3 else features[None]
    B, H, W = f.shape
    _check_hw(who, H, W)
    if not 1 <= B <= 65535:
        raise ValueError(f"{who}: 1 to 65535 images per call, got {B}")
    f = f.contiguous().view(torch.uint8)
    dev = f.device
    with torch.cuda.device(dev):
        nbytes = int(_lib.lib().rbu_edt_workspace_bytes(B, H, W))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        out = torch.empty((B, H, W), dtype=torch.int32, device=dev)
        call("rbu_edt", _p(f), B, H, W, _p(out), _p(ws), nbytes, stream_ptr(), nbytes=5.0 * B * H * W)
    return out.reshape(features.shape)


def _mask(x, name, who):
    if not isinstance(x, torch.Tensor):
        raise TypeError(f"{who}: {name} must be a torch.Tensor, got {type(x).__name__}")
    if not x.is_cuda:
        raise RuntimeError(f"{who} runs on CUDA tensors only (no CPU fallback): {name} is on {x.device}")
    if x.dtype not in _KIND:
        raise TypeError(f"{who}: {name} must be float32, uint8 or bool, got {x.dtype}")
    if x.dim() == 4:
        if x.shape[1] != 1:
            raise ValueError(f"{who}: {name} has {x.shape[1]} channels; multi-class outputs are not supported -- take "
                             "the per-pixel labels of rbunet.predict_tiled and compare one class mask at a time")
        x = x[:, 0]
    if x.dim() == 2:
        x = x[None]
    if x.dim() != 3:
        raise ValueError(f"{who}: {name} must be [H,W], [B,H,W] or [B,1,H,W], got {tuple(x.shape)}")
    return x


def _tolerances(tolerances, pixel_size, who):
    if not (isinstance(pixel_size, (int, float)) and not isinstance(pixel_size, bool) and math.isfinite(pixel_size)
            and pixel_size > 0):
        raise ValueError(f"{who}: pixel_size must be a positive finite number, got {pixel_size!r}")
    taus = tuple(tolerances)
    if len(taus) > MAX_TOLERANCES:
        raise ValueError(f"{who}: at most {MAX_TOLERANCES} tolerances, got {len(taus)}")
    for t in taus:
        if not (isinstance(t, (int, float)) and not isinstance(t, bool) and math.isfinite(t) and t > 0):
            raise ValueError(f"{who}: tolerances must be positive finite numbers, got {t!r}")
    # floor((tau / s)^2) in Python floats; every d^2 is below 2^31 - 1, so larger thresholds are clamped there
    d2 = [min(math.floor((float(t) / float(pixel_size)) ** 2), 2 ** 31 - 1) for t in taus]
    return taus, d2


def _stats(pred, target, threshold, tolerances, pixel_size, who):
    p, t = _mask(pred, "pred", who), _mask(target, "target", who)
    if p.shape != t.shape:
        raise ValueError(f"{who}: pred {tuple(pred.shape)} and target {tuple(target.shape)} differ")
    if p.device != t.device:
        raise ValueError(f"{who}: pred is on {p.device}, target on {t.device}")
    B, H, W = p.shape
    _check_hw(who, H, W)
    if B > 32767:
        raise ValueError(f"{who}: at most 32767 images per call, got {B}")
    if not (isinstance(threshold, (int, float)) and not isinstance(threshold, bool) and math.isfinite(threshold)):
        raise ValueError(f"{who}: threshold must be a finite number, got {threshold!r}")
    taus, d2 = _tolerances(tolerances, pixel_size, who)
    T = len(taus)
    p = p.detach().contiguous()
    t = t.detach().contiguous()
    p = p.view(torch.uint8) if p.dtype == torch.bool else p
    t = t.view(torch.uint8) if t.dtype == torch.bool else t
    dev = p.device
    tol = (ctypes.c_int * max(T, 1))(*d2)
    with torch.cuda.device(dev):
        nbytes = int(_lib.lib().rbu_coastline_stats_workspace_bytes(B, H, W))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        out = torch.empty((B, 2, 5 + T), dtype=torch.float64, device=dev)
        call("rbu_coastline_stats", _p(p), _KIND[p.dtype], _p(t), _KIND[t.dtype], float(threshold), B, H, W,
             ctypes.cast(tol, ctypes.c_void_p), T, _p(out), _p(ws), nbytes, stream_ptr(),
             nbytes=float(p.numel() * p.element_size() + t.numel() * t.element_size()))
    return out, taus


def coastline_stats(pred: torch.Tensor, target: torch.Tensor, threshold: float = 0.5, tolerances=(1.0, 2.0, 5.0),
                    pixel_size: float = 1.0) -> torch.Tensor:
    """The raw per-image, per-direction coastline statistics, a float64 CUDA tensor [B, 2, 5 + T] (the counterpart of
    confusion_counts): per direction (0: pred -> target, 1: target -> pred) the sample count n, the sum of the
    distances in pixels, the maximum squared distance, the two squared-distance order statistics that numpy's linear
    95th percentile interpolates between, and per tolerance tau_k the count of samples with d^2 <= floor((tau_k /
    pixel_size)^2).  Without a distance (n = 0, or the opposite coastline is empty) entries 1-4 are -1 and the counts 0.

    pred, target   CUDA tensors of equal shape [H,W], [B,H,W] or [B,1,H,W]; float32, uint8 or bool, dtypes may differ.
    threshold      water in a float32 pred is p > threshold; a float32 target is water where t != 0.
    tolerances     up to 8 positive distances, in the units of pixel_size.
    Nine launches and one memset whatever the shape; never synchronises, so a validation loop can accumulate without waiting."""
    return _stats(pred, target, threshold, tolerances, pixel_size, "rbunet.coastline_stats")[0]


def metrics_from_stats(st, tolerances, pixel_size: float = 1.0) -> dict:
    """The metric dict of one image from its [2, 5 + T] row of coastline_stats (host values):
      n_pred, n_target                 coastline pixels of pred and target;
      pred_to_target, target_to_pred   the directed mean distances;
      mean_distance                    the average symmetric surface distance (sum_0 + sum_1) / (n_0 + n_1);
      hausdorff                        the larger of the two directed maxima;
      hausdorff95                      the larger of the two directed np.percentile(d, 95) (MONAI, directed=False);
      precision@tau, recall@tau        the share of P within tau of G, of G within tau of P (c / (n + 1e-8));
      f1@tau                           2PR / (P + R + 1e-8);
      surface_dice@tau                 (c_0 + c_1) / (n_0 + n_1).
    Distances are in the units of pixel_size.  Both coastlines empty: distances and surface Dice NaN, precision, recall
    and F1 0.  Exactly one empty: distances inf."""
    s = float(pixel_size)
    n0, n1 = int(st[0][0]), int(st[1][0])
    out = {"n_pred": n0, "n_target": n1}
    if n0 == 0 or n1 == 0:
        out.update(dict.fromkeys(_DIST_KEYS, math.nan if n0 == n1 else math.inf))
    else:
        p95 = []
        for d in range(2):
            virtual = (int(st[d][0]) - 1) * 0.95            # numpy's linear method: gamma = virtual - floor(virtual)
            g = virtual - math.floor(virtual)
            a, b = math.sqrt(st[d][3]), math.sqrt(st[d][4])
            p95.append((b - (b - a) * (1 - g) if g >= 0.5 else a + (b - a) * g) * s)    # numpy's _lerp
        out.update({"pred_to_target": st[0][1] / n0 * s, "target_to_pred": st[1][1] / n1 * s,
                    "mean_distance": (st[0][1] + st[1][1]) / (n0 + n1) * s,
                    "hausdorff": math.sqrt(max(st[0][2], st[1][2])) * s, "hausdorff95": max(p95)})
    for k, tau in enumerate(tolerances):
        c0, c1 = float(st[0][5 + k]), float(st[1][5 + k])
        p, r = c0 / (n0 + 1e-8), c1 / (n1 + 1e-8)
        out[f"precision@{tau:g}"] = p
        out[f"recall@{tau:g}"] = r
        out[f"f1@{tau:g}"] = 2 * p * r / (p + r + 1e-8)
        out[f"surface_dice@{tau:g}"] = (c0 + c1) / (n0 + n1) if n0 + n1 else math.nan
    return out


def coastline_metrics(pred: torch.Tensor, target: torch.Tensor, threshold: float = 0.5, tolerances=(1.0, 2.0, 5.0),
                      pixel_size: float = 1.0) -> list:
    """One metric dict per image (keys in metrics_from_stats) from ONE device->host copy of coastline_stats (the
    counterpart of batch_metrics).  Same arguments as coastline_stats."""
    out, taus = _stats(pred, target, threshold, tolerances, pixel_size, "rbunet.coastline_metrics")
    return [metrics_from_stats(st, taus, pixel_size) for st in out.cpu().tolist()]
