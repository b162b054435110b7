"""Outer contours on the GPU: rbu_trace_contours + rbu_write_contours (rbunet.find_contours) on
  - a 10 980^2 blobby scene with 1e-3 salt-and-pepper speckle,
  - 64 x 512^2 blobby patches,
  - 10 980^2 random masks near the percolation thresholds (0.41 water: foreground at 8; 0.59: background at 4),
  - a full 10 980^2 mask (one contour, the frame),
  - a 10 980^2 checkerboard (one 8-connected component; every land pixel is a hole, so most states are dropped).
Each case in both approx modes.  Reports, with the GPU's name and power limit read in the same run:
  - the trace alone and trace + write: CUDA events, a 256 MiB L2 flush before every repetition, median ms; GB/s count
    the mask (1 B per pixel) and the points written, against the device-to-device copy peak measured in the same run;
  - rbunet.find_contours end to end (workspace allocation, the count copy, the output allocation);
  - the per-kernel times of one trace + write (torch.profiler, a separate run, no flush);
  - the host path a user has without it: the device-to-host copy of the mask plus cv2.findContours on one core
    (host time).
Usage: python tools/contours_bench.py [--reps N] [--out profiles/r11_contours.txt] [--no-host]"""
import argparse
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rbunet  # noqa: E402
from rbunet import _lib  # noqa: E402
from rbunet.ops import _p  # noqa: E402
from tools.components_bench import blobby, copy_peak_gbs, timed  # noqa: E402

DEV = "cuda:0"
LINES = []
SCENE = 10980
APPROX = {"none": 1, "simple": 2}


def emit(s=""):
    print(s, flush=True)
    LINES.append(s)


def cases():
    g = torch.Generator(device=DEV).manual_seed(7)
    n = SCENE
    yield "scene 10980^2 blobby + 1e-3 speckle", blobby(1, n, n, 1, 1e-3)
    yield "patches 64 x 512^2 blobby", blobby(64, 512, 512, 2)
    yield "near percolation 10980^2, 0.41 water", (torch.rand((1, n, n), generator=g, device=DEV) < 0.41).to(torch.uint8)
    yield "near percolation 10980^2, 0.59 water", (torch.rand((1, n, n), generator=g, device=DEV) < 0.59).to(torch.uint8)
    yield "full 10980^2", torch.ones((1, n, n), dtype=torch.uint8, device=DEV)
    ii = torch.arange(n, device=DEV)
    yield "checkerboard 10980^2", ((ii[:, None] + ii[None, :]) % 2 == 0).to(torch.uint8)[None].contiguous()


def kernel_rows(fn):
    fn()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    rows = [(e.key, e.device_time_total / 1e3, e.count) for e in prof.key_averages() if e.device_time_total > 0]
    for name, ms, cnt in rows:
        short = name.replace("(anonymous namespace)::", "").replace("void ", "").split("(")[0]
        emit(f"      {short[:56]:<56} {ms:8.3f} ms  x{cnt}")


def measure(name, m, reps, peak):
    B, H, W = m.shape
    px = B * H * W
    emit()
    emit(f"{name}: B={B}, {H}x{W} ({px / 1e6:.1f} Mpixel), water fraction {float(m.float().mean()):.3f}")
    nb = int(_lib.lib().rbu_contours_workspace_bytes(B, H, W))
    emit(f"  workspace {nb / 2**30:.2f} GiB")
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    counts = torch.empty((B, 2), dtype=torch.int64, device=DEV)
    for approx, code in APPROX.items():
        def trace():
            _lib.call("rbu_trace_contours", _p(m), 1, 0.5, B, H, W, code, _p(counts), _p(ws), nb, _lib.stream_ptr())
        trace()
        n = counts.cpu()
        n_c, n_p = int(n[:, 0].sum()), int(n[:, 1].sum())
        coff = torch.cat([torch.zeros(1, dtype=torch.int64, device=DEV), (n[:, 0] + 1).cumsum(0).to(DEV)])[:B]
        poff = torch.cat([torch.zeros(1, dtype=torch.int64, device=DEV), n[:, 1].cumsum(0).to(DEV)])[:B]
        offs = torch.empty((n_c + B,), dtype=torch.int64, device=DEV)
        pts = torch.empty((max(n_p, 1), 2), dtype=torch.int32, device=DEV)

        def both():
            trace()
            _lib.call("rbu_write_contours", _p(ws), nb, B, H, W, _p(coff), _p(poff), _p(offs), _p(pts),
                      _lib.stream_ptr())
        t_t = timed(trace, reps)
        t_b = timed(both, reps)
        t_f = timed(lambda: rbunet.find_contours(m, approx), reps)
        moved = px + 8.0 * n_p + 8.0 * (n_c + B)
        emit(f"  approx {approx}: {n_c} contours, {n_p} points")
        emit(f"    rbu_trace_contours          {t_t:9.3f} ms")
        emit(f"    trace + rbu_write_contours  {t_b:9.3f} ms  {moved / t_b / 1e6:6.0f} GB/s = {moved / t_b / 1e6 / peak:.4f} "
             f"of copy peak (1 B read per pixel + 8 B per point written)")
        emit(f"    rbunet.find_contours        {t_f:9.3f} ms  (allocations and the one count copy included)")
        emit("    per kernel, one trace + write (torch.profiler, no flush):")
        kernel_rows(both)
        del offs, pts


def host_reference(m, reps):
    """The path without the device call: copy the mask to the host, cv2.findContours on one core (host time)."""
    import cv2
    cv2.setNumThreads(1)
    res = []
    for approx, mode in (("none", cv2.CHAIN_APPROX_NONE), ("simple", cv2.CHAIN_APPROX_SIMPLE)):
        tc, tf = [], []
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            w = m[0].cpu().numpy()
            t1 = time.perf_counter()
            cs = cv2.findContours(w, cv2.RETR_EXTERNAL, mode)[0]
            t2 = time.perf_counter()
            tc.append(t1 - t0)
            tf.append(t2 - t1)
        res.append((approx, len(cs), sum(len(c) for c in cs), sorted(tc)[len(tc) // 2], sorted(tf)[len(tf) // 2]))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_contours.txt"))
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
    for name, m in cases():
        measure(name, m, args.reps, peak)
        if scene is None:
            scene = m
        del m
        torch.cuda.empty_cache()
    if not args.no_host:
        emit()
        emit("host path, the 10980^2 blobby scene: device-to-host copy + cv2.findContours(RETR_EXTERNAL) on one core "
             "(host time, median of 3):")
        for approx, n_c, n_p, t_c, t_f in host_reference(scene, 3):
            emit(f"  approx {approx}: {n_c} contours, {n_p} points; copy {t_c * 1e3:.1f} ms + cv2.findContours "
                 f"{t_f * 1e3:.0f} ms = {(t_c + t_f) * 1e3:.0f} ms")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("# tools/contours_bench.py: rbunet.find_contours (rbu_trace_contours + rbu_write_contours)\n")
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
