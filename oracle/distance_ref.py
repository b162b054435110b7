"""TEST INFRASTRUCTURE — CPU restatement (NumPy, integer arithmetic) of the exact Euclidean distance transform and the
coastline distance metrics of csrc/distance.cu (include/rbunet.h: rbu_edt, rbu_coastline_stats; DESIGN.md §8 item 8).
Only tests/ and tools/ may import this file; the product package never does.

Functions
---------
water                 the water rules: float32 pred p > threshold, float32 target t != 0, uint8 / bool nonzero.
coastline             the non-water pixels with a water pixel among their four in-image neighbours
                      (= imageops_ref.coastline_mask(water_u8, 3) != 0).
edt                   D_F(y,x) = min over feature pixels of (y-v)^2 + (x-u)^2, int64, -1 without features: the separable
                      form of Meijster et al. (2000) with integer intersections.
coastline_stats       the [2, 5+T] per-direction quantities of one image, as rbu_coastline_stats lays them out.
tolerance_d2          floor((tau / pixel_size)^2) in Python floats, the host threshold of each tolerance.
metrics_from_stats    the metric dict of one image from its [2, 5+T] row (what rbunet.coastline_metrics returns).
"""
import math

import numpy as np

from oracle.imageops_ref import percentile_indices


def water(a: np.ndarray, threshold: float = 0.5, is_target: bool = False) -> np.ndarray:
    """include/rbunet.h rbu_coastline_stats, 'water': float32 pred p > threshold (strict, the pred rule of
    confusion_counts), float32 target t != 0 (counts_kernel's target rule), uint8 / bool nonzero."""
    if a.dtype == np.float32:
        return a != 0 if is_target else a > np.float32(threshold)
    return a != 0


def coastline(w: np.ndarray) -> np.ndarray:
    """'coastline of a water mask': not water, with water among the four in-image neighbours; the scene border is never
    coastline by itself (outside pixels are not water)."""
    n = np.zeros_like(w, dtype=bool)
    n[1:, :] |= w[:-1, :]
    n[:-1, :] |= w[1:, :]
    n[:, 1:] |= w[:, :-1]
    n[:, :-1] |= w[:, 1:]
    return n & ~w


def _column_pass(f: np.ndarray) -> np.ndarray:
    """g(y,x): distance to the nearest feature row of column x (int64), -1 where the column has none."""
    H, W = f.shape
    big = 1 << 40
    rows = np.arange(H, dtype=np.int64)[:, None]
    above = np.where(f, rows, -big)
    above = np.maximum.accumulate(above, axis=0)
    below = np.where(f, rows, big)
    below = np.minimum.accumulate(below[::-1], axis=0)[::-1]
    g = np.minimum(rows - above, below - rows)
    return np.where(g >= big // 2, -1, g)


def _row_pass(g: np.ndarray) -> np.ndarray:
    """Per row: D(x) = min over columns u with g(u) >= 0 of (x-u)^2 + g(u)^2 by Meijster's lower envelope; the
    intersection of the parabolas of s < u is Sep = (u^2 - s^2 + g(u)^2 - g(s)^2) // (2(u - s)), exact integers."""
    H, W = g.shape
    out = np.full((H, W), -1, dtype=np.int64)
    for y in range(H):
        gy = g[y].tolist()
        ss, gg, tt = [], [], []
        for u in range(W):
            gu = gy[u]
            if gu < 0:
                continue
            fu = gu * gu
            while ss and (tt[-1] - ss[-1]) ** 2 + gg[-1] ** 2 > (tt[-1] - u) ** 2 + fu:
                ss.pop(); gg.pop(); tt.pop()
            w = 0
            if ss:
                w = 1 + (u * u - ss[-1] ** 2 + fu - gg[-1] ** 2) // (2 * (u - ss[-1]))
                if w >= W:
                    continue
            ss.append(u); gg.append(gu); tt.append(w)
        if not ss:
            continue
        row = out[y]
        q = len(ss) - 1
        for x in range(W - 1, -1, -1):
            row[x] = (x - ss[q]) ** 2 + gg[q] ** 2
            if x == tt[q]:
                q -= 1
    return out


def edt(features: np.ndarray) -> np.ndarray:
    """include/rbunet.h rbu_edt on one [H,W] image (nonzero = feature): exact squared distances, int64; 0 on the features;
    -1 everywhere when there is no feature pixel."""
    f = np.asarray(features) != 0
    if not f.any():
        return np.full(f.shape, -1, dtype=np.int64)
    return _row_pass(_column_pass(f))


def edt_brute(features: np.ndarray) -> np.ndarray:
    """The definition itself: the minimum over all feature pixels (small images only)."""
    f = np.asarray(features) != 0
    H, W = f.shape
    if not f.any():
        return np.full((H, W), -1, dtype=np.int64)
    v, u = np.nonzero(f)
    yy, xx = np.mgrid[0:H, 0:W]
    d = (yy[..., None] - v) ** 2 + (xx[..., None] - u) ** 2
    return d.min(-1).astype(np.int64)


def tolerance_d2(tau: float, pixel_size: float) -> int:
    """'for each tolerance tau_k, the count of samples with d^2 <= floor((tau_k / pixel_size)^2)', in Python floats.
    Clamped to 2^31 - 1, above every possible d^2, so that it fits the int32 of the C ABI."""
    return min(math.floor((float(tau) / float(pixel_size)) ** 2), 2 ** 31 - 1)


def coastline_stats(pred: np.ndarray, target: np.ndarray, threshold: float = 0.5, tol_d2=()) -> np.ndarray:
    """[2, 5 + T] float64 of one image: per direction (0: pred -> target, samples D_G at P; 1: target -> pred, samples
    D_P at G) n, sum of sqrt(d2), max d2, the d2 order statistics at numpy's 95th-percentile ranks, tolerance counts.
    Without a distance (n = 0, or an empty opposite coastline) entries 1-4 are -1 and the counts 0."""
    P = coastline(water(pred, threshold, False))
    G = coastline(water(target, threshold, True))
    DP, DG = edt(P), edt(G)
    out = np.zeros((2, 5 + len(tol_d2)), dtype=np.float64)
    for d, (src, dist) in enumerate(((P, DG), (G, DP))):
        s = dist[src]
        out[d, 0] = s.size
        if s.size == 0 or (s < 0).any():         # no distance: no samples, or no opposite coastline
            out[d, 1:5] = -1
            continue
        srt = np.sort(s)
        prev, nxt, _ = percentile_indices(s.size, 95)
        out[d, 1] = float(np.sqrt(s.astype(np.float64)).sum())
        out[d, 2] = srt[-1]
        out[d, 3], out[d, 4] = srt[prev], srt[nxt]
        for k, t in enumerate(tol_d2):
            out[d, 5 + k] = int((s <= t).sum())
    return out


def _lerp(a: float, b: float, t: float) -> float:
    """numpy's _lerp (numpy/lib/_function_base_impl.py): a + (b-a)*t, and b - (b-a)*(1-t) where t >= 0.5."""
    diff = b - a
    return b - diff * (1 - t) if t >= 0.5 else a + diff * t


def metrics_from_stats(st: np.ndarray, tolerances, pixel_size: float = 1.0) -> dict:
    """DESIGN.md §8 item 8 'Metrics': distances times pixel_size in float64; ratios as metrics_from_counts.  Both
    coastlines empty: distances and surface Dice NaN, precision / recall / F1 0; exactly one empty: distances inf."""
    s = float(pixel_size)
    n0, n1 = int(st[0, 0]), int(st[1, 0])
    out = {"n_pred": n0, "n_target": n1}
    if n0 == 0 and n1 == 0:
        dist = dict.fromkeys(("pred_to_target", "target_to_pred", "mean_distance", "hausdorff", "hausdorff95"), math.nan)
    elif n0 == 0 or n1 == 0:
        dist = dict.fromkeys(("pred_to_target", "target_to_pred", "mean_distance", "hausdorff", "hausdorff95"), math.inf)
    else:
        p95 = []
        for d in range(2):
            _, _, gamma = percentile_indices(int(st[d, 0]), 95)
            p95.append(_lerp(math.sqrt(st[d, 3]), math.sqrt(st[d, 4]), gamma) * s)
        dist = {"pred_to_target": st[0, 1] / n0 * s, "target_to_pred": st[1, 1] / n1 * s,
                "mean_distance": (st[0, 1] + st[1, 1]) / (n0 + n1) * s,
                "hausdorff": math.sqrt(max(st[0, 2], st[1, 2])) * s, "hausdorff95": max(p95)}
    out.update(dist)
    for k, tau in enumerate(tolerances):
        c0, c1 = float(st[0, 5 + k]), float(st[1, 5 + k])
        p = c0 / (n0 + 1e-8)
        r = c1 / (n1 + 1e-8)
        out[f"precision@{tau:g}"] = p
        out[f"recall@{tau:g}"] = r
        out[f"f1@{tau:g}"] = 2 * p * r / (p + r + 1e-8)
        out[f"surface_dice@{tau:g}"] = (c0 + c1) / (n0 + n1) if n0 + n1 else math.nan
    return out
