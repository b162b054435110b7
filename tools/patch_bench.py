"""Patch sampling for native-resolution training, rbunet.PatchSampler / rbu_sample_patches, on 8 synthetic scenes of
4096^2 x 3 (640 MB with masks and coastline-band focus masks: larger than the 126 MB L2), dihedral ops on, at batch
64 x 256^2 and 256 x 512^2, focus_fraction 0 and 0.33.  Reports:
  - rbu_sample_patches alone: CUDA events around one launch, a 256 MiB L2 flush before every repetition, median; the
    algorithmic bytes B*ph*pw*(3 + 1) read and B*ph*pw*(4*nc + 1) written, against the device-to-device copy peak
    measured in the same run;
  - a whole sample() call (host draw, pinned copy, launch): CUDA events around many back-to-back calls, per call;
  - the share of a RobustUNet(3, 1, 64) training step (forward, BCE, backward, FusedAdam) at batch 64 x 256^2, measured
    in the same run;
  - the GPU's name and power limit, read in the same run.
Usage: python tools/patch_bench.py [--reps N] [--calls N] [--out profiles/r07_patch_sampler.txt]"""
import argparse
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rbunet  # noqa: E402
from rbunet import _lib  # noqa: E402
from rbunet.ops import _p  # noqa: E402
from rbunet.patches import draw_jobs  # noqa: E402
from tools.tiled_bench import DEV, copy_peak_gbs, timed  # noqa: E402

LINES = []


def emit(s=""):
    print(s, flush=True)
    LINES.append(s)


def scenes(n, H, W):
    g = torch.Generator(device=DEV).manual_seed(0)
    imgs, masks, focus = [], [], []
    for _ in range(n):
        imgs.append(torch.randint(0, 256, (H, W, 3), generator=g, device=DEV, dtype=torch.uint8))
        field = F.interpolate(torch.rand((1, 1, H // 256, W // 256), generator=g, device=DEV), size=(H, W),
                              mode="bilinear", align_corners=False)[0, 0]
        masks.append((field > 0.5).to(torch.uint8) * 255)                  # land / water blobs
        focus.append(rbunet.coastline_mask(masks[-1], 5))
    return imgs, masks, focus


def per_call_ms(fn, calls):
    """Device time per call over `calls` back-to-back calls (CUDA events around the loop)."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls


def train_step_ms(x, y, reps):
    torch.manual_seed(0)
    model = rbunet.RobustUNet(3, 1, 64).to(DEV).train()
    opt = rbunet.FusedAdam(model.parameters(), lr=1e-4, weight_decay=1e-4)
    crit = rbunet.RobustBCEDiceLoss()
    target = (y > 127).float().unsqueeze(1)

    def step():
        opt.zero_grad()
        crit(model(x), target).backward()
        opt.step()
    return timed(step, reps, flush=False)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--calls", type=int, default=100)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_patch_sampler.txt"))
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    emit(f"device: {torch.cuda.get_device_name(0)} | nvidia-smi name, power.limit, clocks.max.sm: "
         f"{q.stdout.strip() or q.stderr.strip()}")
    peak = copy_peak_gbs(5)
    emit(f"device-to-device copy peak (2 GiB, read + write): {peak:.0f} GB/s")
    S, H, W, nc = 8, 4096, 4096, 3
    imgs, masks, focus = scenes(S, H, W)
    band = sum(int(f.count_nonzero()) for f in focus) / (S * H * W)
    emit(f"{S} scenes of {H}x{W}x3 uint8 + mask + coastline-band focus (k = 5, {band:.4f} of the pixels), "
         f"n_channels {nc}, dihedral on")

    results = {}
    for B, size in ((64, 256), (256, 512)):
        for frac in (0.0, 0.33):
            s = rbunet.PatchSampler(imgs, masks, size=size, n_channels=nc, focus=focus, focus_fraction=frac,
                                    generator=torch.Generator().manual_seed(1))
            jobs = draw_jobs(B, s._sizes, size, size, round(frac * B), True, torch.Generator().manual_seed(2))
            table = s._to_device(jobs)
            x = torch.empty((B, nc, size, size), device=DEV)
            y = torch.empty((B, size, size), dtype=torch.uint8, device=DEV)
            jo = torch.empty((B, 4), dtype=torch.int32, device=DEV)
            t_kernel = timed(lambda: _lib.call("rbu_sample_patches", _p(s._table), S, _p(table), B, size, size, nc,
                                               _p(x), _p(y), _p(jo), _lib.stream_ptr()), args.reps)
            t_call = per_call_ms(lambda: s.sample(B), args.calls)
            read, written = B * size * size * 4, B * size * size * (4 * nc + 1)
            gbs = (read + written) / t_kernel / 1e6
            results[(B, size, frac)] = (t_kernel, t_call)
            emit()
            emit(f"batch {B} x {size}^2, focus_fraction {frac}: {read / 1e6:.1f} MB read + {written / 1e6:.1f} MB written")
            emit(f"  rbu_sample_patches alone   {t_kernel:8.4f} ms  {gbs:6.0f} GB/s = {gbs / peak:.2f} of copy peak")
            emit(f"  sample() call, {args.calls} back to back  {t_call:8.4f} ms per call")
            del x, y, jo, s

    s = rbunet.PatchSampler(imgs, masks, size=256, n_channels=nc, focus=focus, focus_fraction=0.33,
                            generator=torch.Generator().manual_seed(3))
    xb, yb = s.sample(64)
    t_step = train_step_ms(xb, yb, 10)
    emit()
    emit(f"RobustUNet(3, 1, 64) training step at batch 64 x 256^2 (forward, BCE, backward, FusedAdam): {t_step:.2f} ms")
    for frac in (0.0, 0.33):
        t_kernel, t_call = results[(64, 256, frac)]
        emit(f"  focus_fraction {frac}: the kernel is {t_kernel / t_step:.4f} of the step, a sample() call "
             f"{t_call / t_step:.4f}")

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("# tools/patch_bench.py: rbunet.PatchSampler on 8 scenes of 4096^2 x 3, dihedral on\n")
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
