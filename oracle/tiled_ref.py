"""TEST INFRASTRUCTURE — CPU restatement (numpy / torch fp32) of `rbunet.predict_tiled`, the sliding-window prediction of
a whole scene: the tiling plan, the Gaussian window tables, the reflecting tile gather, the blend in the kernel's
documented fp32 order, and the label rules.  Only tests/ and tools/ may import this file; the product package never does.

Functions
---------
plan_axis      tile origins and tile extent along one axis
cover          per output index: the first covering tile and the number of covering tiles
gaussian       the 1-D window table (float64, divided by its maximum, rounded to fp32), as nnU-Net builds it
plan           the whole plan of an H x W scene
gather         the [Tb, nc, th, tw] tiles t0 .. t0+Tb-1 of an [nc, H, W] scene, reflecting beyond the scene
blend          the blended [K, H, W] in rbu_tile_blend's order: i ascending outer, j ascending inner, every step one
               separately rounded fp32 operation (torch's CPU fp32 mul / add / div are IEEE round-to-nearest)
labels         blended > 0.5 (RobustUNet, K = 1), blended > 0 (UNet, K = 1), arg-max with ties to the lowest index (K >= 2)
"""
import numpy as np
import torch


def plan_axis(n: int, tile: int, overlap: int):
    """(origins, extent).  n >= tile: ceil((n - tile) / s) + 1 tiles of `tile` with s = tile - overlap, origin
    min(i*s, n - tile), so the last one ends at the scene edge.  n < tile: one tile of ceil16(n), reflected past n."""
    if n < tile:
        return np.zeros(1, dtype=np.int64), -(-n // 16) * 16
    s = tile - overlap
    count = -(-(n - tile) // s) + 1
    return np.array([min(i * s, n - tile) for i in range(count)], dtype=np.int64), tile


def cover(origins, extent: int, n: int):
    """Per index 0..n-1: the first tile whose [origin, origin + extent) holds it and how many do (contiguous: origins
    are increasing)."""
    first = np.zeros(n, dtype=np.int64)
    count = np.zeros(n, dtype=np.int64)
    for y in range(n):
        hits = [i for i, o in enumerate(origins) if o <= y < o + extent]
        first[y], count[y] = hits[0], len(hits)
        assert hits == list(range(hits[0], hits[0] + len(hits)))
    return first, count


def gaussian(extent: int, sigma_scale: float):
    d = np.arange(extent, dtype=np.float64)
    w = np.exp(-0.5 * ((d + 0.5 - extent / 2) / (sigma_scale * extent)) ** 2)
    return (w / w.max()).astype(np.float32)


def plan(H: int, W: int, tile=(512, 512), overlap=(64, 64), sigma_scale: float = 0.125):
    oy, th = plan_axis(H, tile[0], overlap[0])
    ox, tw = plan_axis(W, tile[1], overlap[1])
    rf, rc = cover(oy, th, H)
    cf, cc = cover(ox, tw, W)
    return {"H": H, "W": W, "oy": oy, "ox": ox, "th": th, "tw": tw, "ny": len(oy), "nx": len(ox),
            "row_first": rf, "row_count": rc, "col_first": cf, "col_count": cc,
            "wy": gaussian(th, sigma_scale), "wx": gaussian(tw, sigma_scale)}


def _reflect(idx, n):
    idx = np.abs(idx)
    return np.where(idx >= n, 2 * (n - 1) - idx, idx)


def gather(x: torch.Tensor, p, t0: int, Tb: int) -> torch.Tensor:
    """x: fp32 [nc, H, W] -> fp32 [Tb, nc, th, tw]."""
    out = []
    for t in range(t0, t0 + Tb):
        iy, ix = divmod(t, p["nx"])
        rows = torch.from_numpy(_reflect(p["oy"][iy] + np.arange(p["th"]), p["H"]))
        cols = torch.from_numpy(_reflect(p["ox"][ix] + np.arange(p["tw"]), p["W"]))
        out.append(x[:, rows][:, :, cols])
    return torch.stack(out)


def blend(tiles: torch.Tensor, p) -> torch.Tensor:
    """tiles: fp32 [ny*nx, K, th, tw] -> fp32 [K, H, W], bit for bit what rbu_tile_blend computes."""
    H, W, nx = p["H"], p["W"], p["nx"]
    K = tiles.shape[1]
    ys, xs = np.arange(H), np.arange(W)
    wy, wx = torch.from_numpy(p["wy"]), torch.from_numpy(p["wx"])
    num = torch.zeros((K, H, W), dtype=torch.float32)
    den = torch.zeros((H, W), dtype=torch.float32)
    for a in range(int(p["row_count"].max())):
        vy = a < p["row_count"]
        i = np.where(vy, p["row_first"] + a, p["row_first"])
        dy = ys - p["oy"][i]
        for b in range(int(p["col_count"].max())):
            vx = b < p["col_count"]
            j = np.where(vx, p["col_first"] + b, p["col_first"])
            dx = xs - p["ox"][j]
            valid = torch.from_numpy(vy[:, None] & vx[None, :])
            w = wy[dy][:, None] * wx[dx][None, :]                                  # one fp32 multiply per pixel
            t = torch.from_numpy(i[:, None] * nx + j[None, :])
            v = tiles[t, :, torch.from_numpy(dy)[:, None], torch.from_numpy(dx)[None, :]].permute(2, 0, 1)
            num = torch.where(valid, num + w * v, num)                              # mul, then add: no fused op
            den = torch.where(valid, den + w, den)
    return num / den


def labels(out: torch.Tensor, network: str) -> torch.Tensor:
    """uint8 [H, W] from the blended [K, H, W]; network is "RobustUNet" (probabilities) or "UNet" (logits)."""
    if out.shape[0] == 1:
        return (out[0] > (0.5 if network == "RobustUNet" else 0.0)).to(torch.uint8)
    return torch.argmax(out, dim=0).to(torch.uint8)
