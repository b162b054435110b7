"""Distance transform and coastline metrics on the GPU: rbunet.distance_transform (rbu_edt) and rbunet.coastline_metrics
(rbu_coastline_stats + one copy) on one 10 980^2 scene with a synthetic blobby coastline and on 64 x 512^2 patches.
Reports:
  - rbu_edt and rbu_coastline_stats alone: CUDA events, a 256 MiB L2 flush before every repetition, median ms, and
    algorithmic GB/s against the device-to-device copy peak measured in the same run.  The EDT counts 1 byte read and
    4 bytes written per pixel; the statistics count the two inputs read once;
  - the whole rbunet.coastline_metrics call (device work, one copy, the host dicts);
  - the per-kernel times of one rbu_coastline_stats call on the scene (torch.profiler, a separate run);
  - for context, scipy.ndimage.distance_transform_edt plus NumPy on one host core for the 10 980^2 case (host time);
  - the GPU's name and power limit, read in the same run.
Usage: python tools/coastline_bench.py [--reps N] [--out profiles/r09_coastline_metrics.txt] [--no-host]"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rbunet  # noqa: E402
from rbunet import _lib  # noqa: E402
from rbunet.ops import _p  # noqa: E402

DEV = "cuda:0"
FLUSH = None
LINES = []
TAUS, PIXEL = (10.0, 20.0, 50.0), 10.0


def emit(s=""):
    print(s, flush=True)
    LINES.append(s)


def timed(fn, reps, flush=True):
    """Median ms of fn() over `reps` repetitions after two warm-up calls."""
    global FLUSH
    if FLUSH is None:
        FLUSH = torch.empty(256 << 20, dtype=torch.uint8, device=DEV)
    ms = []
    for i in range(reps + 2):
        if flush:
            FLUSH.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        if i >= 2:
            ms.append(e0.elapsed_time(e1))
    return sorted(ms)[len(ms) // 2]


def copy_peak_gbs(reps):
    a = torch.empty(2 << 30, dtype=torch.uint8, device=DEV)
    b = torch.empty_like(a)
    t = timed(lambda: b.copy_(a), reps)
    return 2.0 * a.numel() / t / 1e6


def synthetic(B, H, W, seed):
    """A blobby water mask (uint8) and a probability map whose coastline is a perturbed copy of it (float32)."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    def field(cell):
        lo = torch.randn((B, 1, H // cell + 2, W // cell + 2), generator=g, device=DEV)
        return F.interpolate(lo, size=(H, W), mode="bilinear", align_corners=False)[:, 0]
    base = field(64) + 0.3 * field(16)
    target = (base > 0).to(torch.uint8)
    prob = torch.sigmoid(4 * (base + 0.15 * field(8)))
    return prob.contiguous(), target.contiguous()


def measure(name, B, H, W, reps, peak):
    pred, target = synthetic(B, H, W, B * H)
    feats = rbunet.coastline_mask(target, 3)
    px = B * H * W
    emit()
    emit(f"{name}: B={B}, {H}x{W} ({px / 1e6:.1f} Mpixel), target coastline pixels {int((feats != 0).sum())}")
    ws_e = torch.empty(int(_lib.lib().rbu_edt_workspace_bytes(B, H, W)), dtype=torch.uint8, device=DEV)
    dist = torch.empty((B, H, W), dtype=torch.int32, device=DEV)
    t_edt = timed(lambda: _lib.call("rbu_edt", _p(feats), B, H, W, _p(dist), _p(ws_e), ws_e.numel(), _lib.stream_ptr()),
                  reps)
    del ws_e
    emit(f"  rbu_edt              {t_edt:9.3f} ms  {5.0 * px / t_edt / 1e6:6.0f} GB/s = "
         f"{5.0 * px / t_edt / 1e6 / peak:.3f} of copy peak (1 B read + 4 B written per pixel)")
    import ctypes
    tol = (ctypes.c_int * 3)(*[int((t / PIXEL) ** 2) for t in TAUS])
    ws_s = torch.empty(int(_lib.lib().rbu_coastline_stats_workspace_bytes(B, H, W)), dtype=torch.uint8, device=DEV)
    out = torch.empty((B, 2, 8), dtype=torch.float64, device=DEV)
    def stats():
        _lib.call("rbu_coastline_stats", _p(pred), 0, _p(target), 1, 0.5, B, H, W, ctypes.cast(tol, ctypes.c_void_p), 3,
                  _p(out), _p(ws_s), ws_s.numel(), _lib.stream_ptr())
    t_st = timed(stats, reps)
    emit(f"  rbu_coastline_stats  {t_st:9.3f} ms  {5.0 * px / t_st / 1e6:6.0f} GB/s = "
         f"{5.0 * px / t_st / 1e6 / peak:.3f} of copy peak (the inputs read once: 4 B + 1 B per pixel)")
    t_m = timed(lambda: rbunet.coastline_metrics(pred, target, tolerances=TAUS, pixel_size=PIXEL), reps)
    emit(f"  coastline_metrics    {t_m:9.3f} ms  (whole call: device work, one copy, the host dicts)")
    m = rbunet.coastline_metrics(pred[:1], target[:1], tolerances=TAUS, pixel_size=PIXEL)[0]
    emit("  image 0: " + ", ".join(f"{k} {v:.4g}" if isinstance(v, float) else f"{k} {v}" for k, v in m.items()))
    return pred, target, ws_s, stats


def kernel_breakdown(stats):
    stats()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        stats()
        torch.cuda.synchronize()
    rows = [(e.key, e.device_time_total / 1e3) for e in prof.key_averages() if e.device_time_total > 0]
    emit("  per kernel (torch.profiler, one call, no flush):")
    for name, ms in rows:
        short = name.replace("(anonymous namespace)::", "").replace("void ", "").split("(")[0]
        emit(f"    {short[:60]:<60} {ms:8.3f} ms")


def host_reference(pred, target):
    """scipy + NumPy on one host core: both coastlines, both EDTs, the reductions (host time, not the GPU's)."""
    from scipy import ndimage
    p = pred[0].cpu().numpy() > 0.5
    t = target[0].cpu().numpy() != 0
    t0 = time.perf_counter()
    def coast(w):
        n = np.zeros_like(w)
        n[1:] |= w[:-1]; n[:-1] |= w[1:]; n[:, 1:] |= w[:, :-1]; n[:, :-1] |= w[:, 1:]
        return n & ~w
    P, G = coast(p), coast(t)
    dG = ndimage.distance_transform_edt(~G)
    dP = ndimage.distance_transform_edt(~P)
    a, b = dG[P] * PIXEL, dP[G] * PIXEL
    res = (a.mean(), b.mean(), max(a.max(), b.max()), max(np.percentile(a, 95), np.percentile(b, 95)))
    [((a <= tau).mean(), (b <= tau).mean()) for tau in TAUS]
    return time.perf_counter() - t0, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_coastline_metrics.txt"))
    ap.add_argument("--no-host", action="store_true")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    emit(f"device: {torch.cuda.get_device_name(0)} | nvidia-smi name, power.limit, clocks.max.sm: "
         f"{q.stdout.strip() or q.stderr.strip()}")
    peak = copy_peak_gbs(args.reps)
    emit(f"device-to-device copy peak (2 GiB, read + write): {peak:.0f} GB/s")
    emit(f"tolerances {TAUS} at pixel size {PIXEL}; L2 flushed (256 MiB) before every repetition; median of {args.reps}")
    pred, target, ws, stats = measure("scene", 1, 10980, 10980, args.reps, peak)
    kernel_breakdown(stats)
    del ws, stats
    measure("patches", 64, 512, 512, args.reps, peak)
    if not args.no_host:
        torch.set_num_threads(1)
        sec, res = host_reference(pred, target)
        emit()
        emit(f"host, one core: scipy.ndimage.distance_transform_edt x2 + NumPy reductions on the 10980^2 scene: "
             f"{sec * 1e3:.0f} ms (host time; mean distances {res[0]:.4g} / {res[1]:.4g}, hausdorff {res[2]:.4g}, "
             f"hd95 {res[3]:.4g})")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("# tools/coastline_bench.py: rbunet.distance_transform / coastline_metrics\n")
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
