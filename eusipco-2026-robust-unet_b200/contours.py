"""Outer contours of water masks on the GPU, bit for bit with cv2.findContours(mask, RETR_EXTERNAL, CHAIN_APPROX_NONE
or CHAIN_APPROX_SIMPLE) (csrc/contours.cu; DESIGN.md §8 item 10).

The coastline polygons of predict_coastline.py:605-616 come from tracing the coastline band: with this module the band
never leaves the device, only its points do (`find_contours(coastline_mask(clean * 255, 5))`); cv2.approxPolyDP then
runs on the host copy of those points.

Definitions:
  mask        the rules of label_components: float32 p > threshold (strict); uint8 / bool nonzero.  [H,W], [B,H,W] or
              [B,1,H,W], 1 <= H, W <= 32768, B <= 65535.
  traced      foreground components are 8-connected and the image is framed by background.  A component is traced iff
              the 4-connected background component (the frame included) holding the pixel above its raster-first pixel
              p0 touches the frame: islands in lakes are not traced.
  order       contours in decreasing raster order of p0 (the last component found comes first).
  stepping    chain codes 0 = (+1,0), 1 = (+1,-1), 2 = (0,-1) ... 7 = (+1,+1), y pointing down.  From p0 the first
              foreground neighbour i1 among codes 4, 3, 2, 1, 0, 7, 6, 5; without one the contour is the single point
              p0.  A state (p, c) has c pointing at the previous pixel; its successor scans c+1, c+2, ... (mod 8) around
              p for the first foreground neighbour q at code d and is (q, (d+4) mod 8).  The contour is the cycle of
              states from (p0, code of i1); it emits each state's pixel (a pixel may appear up to 4 times).
  simple      CHAIN_APPROX_SIMPLE keeps the points where the chain code changes, as cv2 does.
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import call, stream_ptr
from .components import _water
from .distance import _KIND
from .ops import _p

APPROX = {"none": 1, "simple": 2}          # RBU_APPROX_NONE, RBU_APPROX_SIMPLE (= cv2.CHAIN_APPROX_NONE, SIMPLE)


def _trace(mask, approx, threshold, who):
    """Checks the arguments and enqueues the trace: (m [B,H,W], counts int64 [B, 2] = contours, points; workspace).
    Never synchronises."""
    if not isinstance(approx, str):
        raise TypeError(f"{who}: approx must be 'simple' or 'none', got {approx!r}")
    if approx not in APPROX:
        raise ValueError(f"{who}: approx must be 'simple' or 'none', got {approx!r}")
    m, _ = _water(mask, threshold, 8, who)
    B, H, W = m.shape
    dev = m.device
    with torch.cuda.device(dev):
        nbytes = int(_lib.lib().rbu_contours_workspace_bytes(B, H, W))
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        counts = torch.empty((B, 2), dtype=torch.int64, device=dev)
        call("rbu_trace_contours", _p(m), _KIND[m.dtype], float(threshold), B, H, W, APPROX[approx], _p(counts), _p(ws),
             nbytes, stream_ptr(), nbytes=float(m.numel() * m.element_size() + 14 * B * H * W))
    return m, counts, ws


def find_contours(mask: torch.Tensor, approx: str = "simple", threshold: float = 0.5) -> list:
    """The outer contours of the water of `mask` (a CUDA tensor [H,W], [B,H,W] or [B,1,H,W]; float32, uint8 or bool),
    one (points, offsets) pair per image, both CUDA tensors:
      points   int32 [N_b, 2], (x, y);
      offsets  int64 [n_b + 1]; contour k is points[offsets[k]:offsets[k + 1]].
    Contour k equals cv2.findContours(m_b, cv2.RETR_EXTERNAL, mode)[0][k].reshape(-1, 2) bit for bit, in the same order,
    with mode CHAIN_APPROX_SIMPLE for approx="simple" and CHAIN_APPROX_NONE for "none".  Makes exactly one device-to-host
    copy (the per-image contour and point counts, to size the output)."""
    who = "rbunet.find_contours"
    m, counts, ws = _trace(mask, approx, threshold, who)
    B, H, W = m.shape
    dev = m.device
    with torch.cuda.device(dev):
        n = counts.cpu().tolist()                                # the one device-to-host copy
        n_pts = sum(p for _, p in n)
        n_offs = sum(c + 1 for c, _ in n)
        zero = torch.zeros((1,), dtype=torch.int64, device=dev)
        coff = torch.cat([zero, (counts[:, 0] + 1).cumsum(0)])[:B]
        poff = torch.cat([zero, counts[:, 1].cumsum(0)])[:B]
        points = torch.empty((max(n_pts, 1), 2), dtype=torch.int32, device=dev)
        offsets = torch.empty((n_offs,), dtype=torch.int64, device=dev)
        call("rbu_write_contours", _p(ws), ws.numel(), B, H, W, _p(coff), _p(poff), _p(offsets), _p(points),
             stream_ptr(), nbytes=float(8 * n_pts + 8 * n_offs + 14 * B * H * W))
    out, c0, p0 = [], 0, 0
    for c, p in n:
        out.append((points[p0:p0 + p], offsets[c0:c0 + c + 1]))
        c0, p0 = c0 + c + 1, p0 + p
    return out
