"""Whole-scene sliding-window prediction, rbunet.predict_tiled, on an 8192^2 x 3 synthetic scene through RobustUNet(3,1,64)
in eval mode, at tile 1024 / overlap 128 and tile 512 / overlap 64 (batches of 16 tiles).  Reports:
  - the whole call (CUDA events around predict_tiled, median of the repetitions);
  - the network's share: the same batches through model() alone;
  - rbu_tile_gather (one batch) and rbu_tile_blend (the whole scene) alone: CUDA events, a 256 MiB L2 flush before every
    repetition, algorithmic GB/s (bytes read once + bytes written once) against the device-to-device copy peak measured
    in the same run;
  - the GPU's name and power limit, read in the same run.
Usage: python tools/tiled_bench.py [--reps N] [--out profiles/r06_tiled_predict.txt]"""
import argparse
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rbunet  # noqa: E402
from rbunet import _lib, tiled  # noqa: E402
from rbunet.ops import _p  # noqa: E402

DEV = "cuda:0"
FLUSH = None
LINES = []


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_tiled_predict.txt"))
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    emit(f"device: {torch.cuda.get_device_name(0)} | nvidia-smi name, power.limit, clocks.max.sm: "
         f"{q.stdout.strip() or q.stderr.strip()}")
    peak = copy_peak_gbs(args.reps)
    emit(f"device-to-device copy peak (2 GiB, read + write): {peak:.0f} GB/s")

    H = W = 8192
    nc, bs = 3, 16
    torch.manual_seed(0)
    model = rbunet.RobustUNet(nc, 1, 64).to(DEV).eval()
    g = torch.Generator(device=DEV).manual_seed(1)
    x = torch.randn((nc, H, W), generator=g, device=DEV)
    emit(f"scene {nc}x{H}x{W} fp32, RobustUNet({nc}, 1, 64) eval, batch_size {bs}, sigma_scale 0.125")

    for tile, ov in ((1024, 128), (512, 64)):
        p = tiled.plan_tiles(H, W, (tile, tile), (ov, ov), 0.125)
        T = p.ny * p.nx
        nb = -(-T // bs)
        emit()
        emit(f"tile {tile} / overlap {ov}: {p.ny}x{p.nx} = {T} tiles, {nb} batches")
        t_call = timed(lambda: rbunet.predict_tiled(model, x, tile=tile, overlap=ov, batch_size=bs), args.reps,
                       flush=False)
        batch = torch.randn((bs, nc, tile, tile), device=DEV)
        last = T - (nb - 1) * bs

        def network():
            with torch.no_grad():
                for i in range(nb):
                    model(batch if i < nb - 1 else batch[:last])
        t_net = timed(network, args.reps, flush=False)

        table = torch.from_numpy(p.table()).to(DEV)
        oy, ox, rf, rc, cf, cc, wy, wx = (_p(table[o:]) for o in p.offsets())
        gbuf = torch.empty((bs, nc, tile, tile), device=DEV)
        t_gather = timed(lambda: _lib.call("rbu_tile_gather", _p(x), nc, H, W, oy, ox, p.ny, p.nx, tile, tile, 0, bs,
                                           _p(gbuf), _lib.stream_ptr()), args.reps)
        g_bytes = 2.0 * gbuf.numel() * 4
        tiles = torch.rand((T, 1, tile, tile), device=DEV)
        labels = torch.empty((H, W), dtype=torch.uint8, device=DEV)
        out = torch.empty((1, H, W), device=DEV)
        blend = {}
        for name, o in (("labels only", None), ("labels + out", out)):
            blend[name] = timed(lambda: _lib.call("rbu_tile_blend", _p(tiles), 1, H, W, oy, ox, p.ny, p.nx, tile, tile,
                                                  rf, rc, cf, cc, wy, wx, 0.5, _p(o), _p(labels), _lib.stream_ptr()),
                                args.reps)
        emit(f"  predict_tiled call           {t_call:9.2f} ms  ({H * W / t_call / 1e3:.1f} Mpixel/s)")
        emit(f"  network alone, same batches  {t_net:9.2f} ms  = {t_net / t_call:.3f} of the call "
             f"({T / t_net * 1e3:.0f} tiles/s)")
        emit(f"  rbu_tile_gather, {bs} tiles   {t_gather:9.3f} ms  {g_bytes / t_gather / 1e6:6.0f} GB/s = "
             f"{g_bytes / t_gather / 1e6 / peak:.2f} of copy peak; x {nb} batches = {nb * t_gather / t_call:.4f} of the call")
        for name, t in blend.items():
            b_bytes = tiles.numel() * 4.0 + H * W * (1 + (4 if name == "labels + out" else 0))
            emit(f"  rbu_tile_blend, {name:<13}{t:9.3f} ms  {b_bytes / t / 1e6:6.0f} GB/s = "
                 f"{b_bytes / t / 1e6 / peak:.2f} of copy peak; {t / t_call:.4f} of the call")
        emit(f"  gather + blend (labels only) = {(nb * t_gather + blend['labels only']) / t_call:.4f} of the call")
        del tiles, gbuf, batch

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("# tools/tiled_bench.py: rbunet.predict_tiled on an 8192^2 x 3 scene, RobustUNet(3, 1, 64) eval\n")
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
