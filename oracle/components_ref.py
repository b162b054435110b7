"""TEST INFRASTRUCTURE — CPU restatement (NumPy / SciPy) of the connected-component labelling, component statistics and
small-region removal of csrc/components.cu (include/rbunet.h: rbu_label_components, rbu_component_stats,
rbu_remove_small_regions; DESIGN.md §8 item 9).  Only tests/ and tools/ may import this file; the product package never
does.

Functions
---------
water           the water rule: float32 p > threshold (strict), uint8 / bool nonzero (distance_ref.water of a pred).
label           int32 labels, 0 background, components 1..n in raster order of their first pixel, and n:
                scipy.ndimage.label with generate_binary_structure(2, 1) (connectivity 4) or (2, 2) (connectivity 8).
stats           int64 [n, 7] (left, top, right, bottom, area, sum x, sum y) of labels 1..n.
opencv_stats    stats [n, 5] in OpenCV's CC_STAT layout and float64 centroids [n, 2] = (sum x / area, sum y / area).
remove_small    the two-step removal: water components below min_water become land, then land components of that
                result below min_land become water; uint8 0/1.
"""
import numpy as np
from scipy import ndimage

from oracle.distance_ref import water as _water


def water(a: np.ndarray, threshold: float = 0.5) -> np.ndarray:
    return _water(a, threshold, is_target=False)


def structure(connectivity: int) -> np.ndarray:
    return ndimage.generate_binary_structure(2, {4: 1, 8: 2}[connectivity])


def label(w: np.ndarray, connectivity: int):
    """(labels int32, n) of a boolean [H, W] mask; scipy numbers components in raster order of their first pixel."""
    lab, n = ndimage.label(w, structure(connectivity))
    return lab.astype(np.int32), int(n)


def stats(lab: np.ndarray, n: int) -> np.ndarray:
    """int64 [n, 7]: left, top, right, bottom (inclusive), area, sum of x, sum of y of labels 1..n."""
    H, W = lab.shape
    ys, xs = np.indices((H, W), dtype=np.int64)
    l, x, y = lab.ravel(), xs.ravel(), ys.ravel()
    out = np.zeros((n + 1, 7), np.int64)
    out[:, 0] = out[:, 1] = np.iinfo(np.int64).max
    out[:, 2] = out[:, 3] = -1
    np.minimum.at(out[:, 0], l, x)
    np.minimum.at(out[:, 1], l, y)
    np.maximum.at(out[:, 2], l, x)
    np.maximum.at(out[:, 3], l, y)
    out[:, 4] = np.bincount(l, minlength=n + 1)
    out[:, 5] = _int_bincount(l, x, n + 1)
    out[:, 6] = _int_bincount(l, y, n + 1)
    return out[1:]


def _int_bincount(l, v, size):
    """Exact int64 sums of v per label (np.bincount's weights are float64)."""
    s = np.zeros(size, np.int64)
    np.add.at(s, l, v)
    return s


def opencv_stats(st: np.ndarray):
    """(stats int64 [n, 5] = left, top, width, height, area; centroids float64 [n, 2]) from stats() rows."""
    cc = np.stack([st[:, 0], st[:, 1], st[:, 2] - st[:, 0] + 1, st[:, 3] - st[:, 1] + 1, st[:, 4]], axis=1)
    area = st[:, 4].astype(np.float64)
    cen = np.stack([st[:, 5].astype(np.float64) / area, st[:, 6].astype(np.float64) / area], axis=1)
    return cc, cen


def remove_small(w: np.ndarray, min_water: int, min_land: int, connectivity: int) -> np.ndarray:
    """Step 1: water components with fewer than min_water pixels become land.  Step 2, on that result: land components
    with fewer than min_land pixels become water.  uint8 0/1."""
    out = w.astype(bool).copy()
    lab, n = label(out, connectivity)
    area = np.bincount(lab.ravel(), minlength=n + 1)
    out &= area[lab] >= min_water
    lab, n = label(~out, connectivity)
    area = np.bincount(lab.ravel(), minlength=n + 1)
    out |= (lab > 0) & (area[lab] < min_land)
    return out.astype(np.uint8)
