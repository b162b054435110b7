"""TEST INFRASTRUCTURE — CPU restatement (NumPy / SciPy / Python) of the outer-contour tracing of csrc/contours.cu
(include/rbunet.h: rbu_trace_contours, rbu_write_contours; DESIGN.md §8 item 10), which equals
cv2.findContours(mask, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_NONE | CHAIN_APPROX_SIMPLE).  Only tests/ and tools/ may
import this file; the product package never does.

Definition
----------
foreground  8-connected components of the mask; the image is framed by background.
external    a component is traced iff the 4-connected background component (the frame included) that holds the pixel
            above its raster-first pixel p0 touches the frame (p0 on the top row: that pixel is the frame itself).
order       contours in decreasing raster order of p0.
stepping    chain codes 0 = (+1,0), 1 = (+1,-1), 2 = (0,-1), ... 7 = (+1,+1), y pointing down.  From p0 the first
            foreground neighbour i1 among codes 4, 3, 2, 1, 0, 7, 6, 5; none: the contour is the single point p0.  A state
            (p, c) has c pointing at the previous pixel; its successor scans c+1, c+2, ... (mod 8) around p for the first
            foreground neighbour q at code d and is (q, (d+4) mod 8).  The contour is the cycle of states from
            (p0, code of i1); it emits each state's pixel.
simple      CHAIN_APPROX_SIMPLE keeps a state's pixel iff its outgoing code differs from the previous state's (cyclically;
            the start's predecessor is the last state, whose outgoing code is (code of i1) ^ 4).

Functions
---------
external_starts  raster-first pixels (flat y*W + x) of the traced components, in raster order.
trace            one contour: int32 [n, 2] (x, y) points from a start pixel.
find_contours    list of int32 [n_k, 2] arrays in cv2's order.
"""
import numpy as np
from scipy import ndimage

_CODES = ((1, 0), (1, -1), (0, -1), (-1, -1), (-1, 0), (-1, 1), (0, 1), (1, 1))


def external_starts(w: np.ndarray) -> np.ndarray:
    w = np.asarray(w, bool)
    H, W = w.shape
    fg, n = ndimage.label(w, np.ones((3, 3), bool))
    if n == 0:
        return np.zeros((0,), np.int64)
    _, first = np.unique(fg.ravel(), return_index=True)
    first = first[1:] if fg.ravel()[first[0]] == 0 else first          # drop the background label
    bg, _ = ndimage.label(np.pad(~w, 1, constant_values=True))          # 4-connected, the frame included
    y0, x0 = first // W, first % W
    keep = bg[y0, x0 + 1] == bg[0, 0]                                    # padded (y0 - 1 + 1, x0 + 1): the pixel above
    return np.sort(first[keep]).astype(np.int64)


def trace(w: np.ndarray, p0: int, approx: str = "simple") -> np.ndarray:
    w = np.asarray(w, bool)
    return _trace(np.pad(w, 1).ravel().tolist(), w.shape[1], p0, approx == "none")


def _trace(P: list, W: int, p0: int, none: bool) -> np.ndarray:
    """P: the frame-padded mask as a flat list."""
    Wp = W + 2
    D = [dx + dy * Wp for dx, dy in _CODES]
    s = (p0 // W + 1) * Wp + p0 % W + 1
    for c1 in (4, 3, 2, 1, 0, 7, 6, 5):
        if P[s + D[c1]]:
            break
    else:
        return np.array([[p0 % W, p0 // W]], np.int32)
    p, c, prev_d, pts = s, c1, c1 ^ 4, []
    while True:
        for k in range(1, 9):
            d = (c + k) & 7
            if P[p + D[d]]:
                break
        if none or d != prev_d:
            pts.append(p)
        prev_d = d
        p, c = p + D[d], (d + 4) & 7
        if p == s and c == c1:
            break
    a = np.array(pts, np.int64)
    return np.stack([a % Wp - 1, a // Wp - 1], axis=1).astype(np.int32)


def find_contours(w: np.ndarray, approx: str = "simple") -> list:
    w = np.asarray(w, bool)
    P = np.pad(w, 1).ravel().tolist()
    return [_trace(P, w.shape[1], int(p0), approx == "none") for p0 in external_starts(w)[::-1]]
