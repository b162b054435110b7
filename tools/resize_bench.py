"""Throughput of rbunet.resize / rbunet.preprocess(size=) (byte kernels) next to the host libraries the
reference uses (Pillow through torchvision, OpenCV) on one image.  CUDA events around each call, a 256 MiB L2 flush
before every repetition, median of the repetitions.  GB/s are algorithmic: source bytes once plus output bytes once,
against the measured HBM copy peak of 6 543 GB/s.  Usage: python tools/resize_bench.py [reps]"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rbunet  # noqa: E402
from rbunet import _lib, ops  # noqa: E402

COPY_PEAK_GBS = 6543.0
FLUSH = None


def timed(fns, reps):
    """Median ms of each function; the functions alternate within every repetition (same-call A/B)."""
    global FLUSH
    if FLUSH is None:
        FLUSH = torch.empty(256 << 20, dtype=torch.uint8, device="cuda:0")
    ms = [[] for _ in fns]
    for i in range(reps + 2):
        for j, fn in enumerate(fns):
            FLUSH.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            if i >= 2:
                ms[j].append(e0.elapsed_time(e1))
    return [sorted(m)[len(m) // 2] for m in ms]


def report(name, t, n_img, nbytes):
    gbs = nbytes / t / 1e6
    print(f"{name:<58} {t:8.3f} ms {n_img / t * 1e3:9.0f} img/s {gbs:7.0f} GB/s  {gbs / COPY_PEAK_GBS:.2f} of copy peak")


def kernel_fn(name, srcs, *args):
    """The bare C-ABI call on a descriptor table built once: times the kernel without the per-call host work.
    args: C, then the arguments after max_h, max_w."""
    table, max_h, max_w = ops._descriptor_table(srcs, srcs[0].device)
    return lambda: _lib.call(name, ops._p(table), len(srcs), args[0], max_h, max_w, *args[1:], _lib.stream_ptr())


def host_ms(fn, reps=5):
    fn()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    return (time.perf_counter() - t0) / reps * 1e3


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    print(f"device: {torch.cuda.get_device_name(0)} | nvidia-smi: {q.stdout.strip() or q.stderr.strip()}")
    rng = np.random.default_rng(0)
    dev = "cuda:0"

    B, S = 64, 1024
    x = torch.from_numpy(rng.integers(0, 256, size=(B, S, S, 3), dtype=np.uint8)).to(dev)
    xs = [v for v in x]
    src = B * S * S * 3
    u8 = torch.empty((B, 512, 512, 3), dtype=torch.uint8, device=dev)
    print("kernel = the C-ABI call on a prebuilt descriptor table; call = rbunet.resize / preprocess as a user calls them")
    tk, tc = timed([kernel_fn("rbu_resize_u8", xs, 3, 512, 512, 0, ops._p(u8)), lambda: rbunet.resize(x, (512, 512))], reps)
    report(f"resize bilinear {B}x{S}^2x3 -> 512^2, kernel", tk, B, src + u8.numel())
    report(f"resize bilinear {B}x{S}^2x3 -> 512^2, call", tc, B, src + u8.numel())
    for nc in (3, 6):
        tc, = timed([lambda: rbunet.preprocess(x, nc, size=(512, 512))], reps)
        report(f"preprocess(size=512, n_channels={nc}) (resize + preprocess), call", tc, B, src + B * nc * 512 * 512 * 4)

    sides = rng.integers(600, 2001, size=(64, 2))
    rag = [torch.from_numpy(rng.integers(0, 256, size=(int(h), int(w), 3), dtype=np.uint8)).to(dev) for h, w in sides]
    tk, tc = timed([kernel_fn("rbu_resize_u8", rag, 3, 512, 512, 0, ops._p(u8)), lambda: rbunet.resize(rag, (512, 512))], reps)
    nbytes = sum(r.numel() for r in rag) + u8.numel()
    report("resize bilinear ragged 64 (sides 600-2000) -> 512^2, kernel", tk, 64, nbytes)
    report("resize bilinear ragged 64 (sides 600-2000) -> 512^2, call", tc, 64, nbytes)

    big = torch.from_numpy(rng.integers(0, 256, size=(2048, 2048, 3), dtype=np.uint8)).to(dev)
    tk, tc = timed([kernel_fn("rbu_resize_u8", [big], 3, 512, 512, 0, ops._p(u8)), lambda: rbunet.resize(big, (512, 512))], reps)
    report("resize bilinear 1x2048^2x3 -> 512^2, kernel", tk, 1, big.numel() + 512 * 512 * 3)
    report("resize bilinear 1x2048^2x3 -> 512^2, call", tc, 1, big.numel() + 512 * 512 * 3)

    m = torch.from_numpy(((rng.random((512, 512)) > 0.5) * 255).astype(np.uint8)).to(dev)
    mo = torch.empty((10980, 10980), dtype=torch.uint8, device=dev)
    tk, = timed([kernel_fn("rbu_resize_u8", [m.unsqueeze(-1)], 1, 10980, 10980, 2, ops._p(mo))], reps)
    report("resize cv2_nearest mask 512^2 -> 10980^2, kernel", tk, 1, m.numel() + mo.numel())
    ms = torch.from_numpy(((rng.random((64, 1024, 1024)) > 0.5) * 255).astype(np.uint8)).to(dev)
    mo = torch.empty((64, 512, 512), dtype=torch.uint8, device=dev)
    tk, = timed([kernel_fn("rbu_resize_u8", [v.unsqueeze(-1) for v in ms], 1, 512, 512, 1, ops._p(mo))], reps)
    report("resize nearest (Pillow) masks 64x1024^2 -> 512^2, kernel", tk, 64, ms.numel() + mo.numel())

    print("host, one image, one core:")
    torch.set_num_threads(1)
    a = x[0].cpu().numpy()
    try:
        from PIL import Image
        from torchvision import transforms
        im = Image.fromarray(a)
        print(f"  Pillow resize 1024^2x3 -> 512^2 BILINEAR: {host_ms(lambda: im.resize((512, 512), Image.BILINEAR)):.2f} ms")
        tf = transforms.Compose([transforms.Resize((512, 512)), transforms.ToTensor(),
                                 transforms.Normalize([0.485, 0.456, 0.406], [0.229, 0.224, 0.225])])
        print(f"  torchvision Resize + ToTensor + Normalize 1024^2x3: {host_ms(lambda: tf(im)):.2f} ms")
        b = big.cpu().numpy()
        imb = Image.fromarray(b)
        print(f"  Pillow resize 2048^2x3 -> 512^2 BILINEAR: {host_ms(lambda: imb.resize((512, 512), Image.BILINEAR)):.2f} ms")
    except ImportError as e:
        print(f"  Pillow / torchvision not installed: {e}")
    try:
        import cv2
        mm = m.cpu().numpy()
        print(f"  OpenCV INTER_NEAREST 512^2 -> 10980^2: "
              f"{host_ms(lambda: cv2.resize(mm, (10980, 10980), interpolation=cv2.INTER_NEAREST), 2):.2f} ms")
    except ImportError as e:
        print(f"  OpenCV not installed: {e}")


if __name__ == "__main__":
    main()
