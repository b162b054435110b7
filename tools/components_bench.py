"""Connected components on the GPU: rbu_label_components, rbu_component_stats and rbu_remove_small_regions on
  - a 10 980^2 blobby scene with 1e-3 salt-and-pepper speckle,
  - 64 x 512^2 blobby patches,
  - a 10 980^2 random mask near the percolation threshold (0.59 water, huge fractal components at connectivity 4;
    0.41 at 8),
  - a full 10 980^2 mask (one giant component: the root aggregation's hot spot),
  - a 10 980^2 checkerboard (the most components at connectivity 4: one per water pixel).
Reports, with the GPU's name and power limit read in the same run:
  - each entry point alone: CUDA events, a 256 MiB L2 flush before every repetition, median ms, and algorithmic GB/s
    against the device-to-device copy peak measured in the same run.  Labels count 1 byte read and 4 written per pixel,
    the removal 1 read and 1 written, the statistics 4 read;
  - the per-kernel times of one labelling and one removal call (torch.profiler, a separate run, no flush);
  - for context, scipy.ndimage.label and cv2.connectedComponentsWithStats on one host core (host time).
Usage: python tools/components_bench.py [--reps N] [--out profiles/r10_components.txt] [--no-host]"""
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
SCENE = 10980
MIN_WATER, MIN_LAND = 64, 64


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


def blobby(B, H, W, seed, speckle=0.0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    def field(cell):
        lo = torch.randn((B, 1, H // cell + 2, W // cell + 2), generator=g, device=DEV)
        return F.interpolate(lo, size=(H, W), mode="bilinear", align_corners=False)[:, 0]
    m = (field(64) + 0.3 * field(16)) > 0
    if speckle:
        m ^= torch.rand((B, H, W), generator=g, device=DEV) < speckle
    return m.to(torch.uint8).contiguous()


def cases():
    g = torch.Generator(device=DEV).manual_seed(7)
    n = SCENE
    yield "scene 10980^2 blobby + 1e-3 speckle", blobby(1, n, n, 1, 1e-3), (4, 8)
    yield "patches 64 x 512^2 blobby", blobby(64, 512, 512, 2), (4, 8)
    yield "near percolation 10980^2, 0.59 water (conn 4)", \
        (torch.rand((1, n, n), generator=g, device=DEV) < 0.59).to(torch.uint8), (4,)
    yield "near percolation 10980^2, 0.41 water (conn 8)", \
        (torch.rand((1, n, n), generator=g, device=DEV) < 0.41).to(torch.uint8), (8,)
    yield "full 10980^2 (one component)", torch.ones((1, n, n), dtype=torch.uint8, device=DEV), (4, 8)
    ii = torch.arange(n, device=DEV)
    yield "checkerboard 10980^2", ((ii[:, None] + ii[None, :]) % 2 == 0).to(torch.uint8)[None].contiguous(), (4,)


def kernel_rows(fn):
    fn()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    rows = [(e.key, e.device_time_total / 1e3) for e in prof.key_averages() if e.device_time_total > 0]
    for name, ms in rows:
        short = name.replace("(anonymous namespace)::", "").replace("void ", "").split("(")[0]
        emit(f"      {short[:56]:<56} {ms:8.3f} ms")


def measure(name, m, conns, reps, peak):
    B, H, W = m.shape
    px = B * H * W
    emit()
    emit(f"{name}: B={B}, {H}x{W} ({px / 1e6:.1f} Mpixel), water fraction {float(m.float().mean()):.3f}")
    nb_l = int(_lib.lib().rbu_label_workspace_bytes(B, H, W))
    nb_r = int(_lib.lib().rbu_remove_small_regions_workspace_bytes(B, H, W))
    ws = torch.empty(max(nb_l, nb_r), dtype=torch.uint8, device=DEV)
    labels = torch.empty((B, H, W), dtype=torch.int32, device=DEV)
    counts = torch.empty((B,), dtype=torch.int32, device=DEV)
    out = torch.empty((B, H, W), dtype=torch.uint8, device=DEV)
    for conn in conns:
        def lab():
            _lib.call("rbu_label_components", _p(m), 1, 0.5, B, H, W, conn, _p(labels), _p(counts), _p(ws), nb_l,
                      _lib.stream_ptr())

        def rem():
            _lib.call("rbu_remove_small_regions", _p(m), 1, 0.5, B, H, W, conn, MIN_WATER, MIN_LAND, _p(out), _p(ws),
                      nb_r, _lib.stream_ptr())
        t_l = timed(lab, reps)
        n = counts.cpu().tolist()
        emit(f"  connectivity {conn}: components {n[0] if B == 1 else sum(n)}")
        emit(f"    rbu_label_components      {t_l:9.3f} ms  {5.0 * px / t_l / 1e6:6.0f} GB/s = "
             f"{5.0 * px / t_l / 1e6 / peak:.3f} of copy peak (1 B read + 4 B written per pixel)")
        offs = torch.cat([torch.zeros(1, dtype=torch.int64, device=DEV), counts.cumsum(0, dtype=torch.int64)])
        rows = max(int(offs[-1]), 1)
        st = torch.empty((rows, 7), dtype=torch.int64, device=DEV)
        t_s = timed(lambda: _lib.call("rbu_component_stats", _p(labels), B, H, W, _p(offs), _p(st), _lib.stream_ptr()),
                    reps)
        emit(f"    rbu_component_stats       {t_s:9.3f} ms  {4.0 * px / t_s / 1e6:6.0f} GB/s = "
             f"{4.0 * px / t_s / 1e6 / peak:.3f} of copy peak (4 B read per pixel)")
        del st
        t_r = timed(rem, reps)
        emit(f"    rbu_remove_small_regions  {t_r:9.3f} ms  {2.0 * px / t_r / 1e6:6.0f} GB/s = "
             f"{2.0 * px / t_r / 1e6 / peak:.3f} of copy peak (1 B read + 1 B written per pixel; "
             f"min_water {MIN_WATER}, min_land {MIN_LAND})")
        emit("    per kernel, labelling (torch.profiler, one call, no flush):")
        kernel_rows(lab)
        emit("    per kernel, removal:")
        kernel_rows(rem)


def host_reference(m):
    """scipy.ndimage.label and cv2.connectedComponentsWithStats on one host core (host time, not the GPU's)."""
    import cv2
    from scipy import ndimage
    cv2.setNumThreads(1)
    w = m[0].cpu().numpy()
    res = []
    for conn in (4, 8):
        t0 = time.perf_counter()
        _, n = ndimage.label(w, ndimage.generate_binary_structure(2, 1 if conn == 4 else 2))
        t1 = time.perf_counter()
        cv2.connectedComponentsWithStats(w, connectivity=conn, ltype=cv2.CV_32S)
        t2 = time.perf_counter()
        res.append((conn, n, t1 - t0, t2 - t1))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_components.txt"))
    ap.add_argument("--no-host", action="store_true")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    emit(f"device: {torch.cuda.get_device_name(0)} | nvidia-smi name, power.limit, clocks.max.sm: "
         f"{q.stdout.strip() or q.stderr.strip()}")
    peak = copy_peak_gbs(args.reps)
    emit(f"device-to-device copy peak (2 GiB, read + write): {peak:.0f} GB/s")
    emit(f"L2 flushed (256 MiB) before every repetition; median of {args.reps}")
    scene = None
    for name, m, conns in cases():
        measure(name, m, conns, args.reps, peak)
        if scene is None:
            scene = m
        del m
        torch.cuda.empty_cache()
    if not args.no_host:
        emit()
        emit("host, one core, the 10980^2 blobby scene (host time):")
        for conn, n, t_sp, t_cv in host_reference(scene):
            emit(f"  connectivity {conn}: {n} components; scipy.ndimage.label {t_sp * 1e3:.0f} ms, "
                 f"cv2.connectedComponentsWithStats {t_cv * 1e3:.0f} ms")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("# tools/components_bench.py: rbunet.label_components / component_stats / remove_small_regions\n")
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
