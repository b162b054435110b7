"""Throughput of the K-class head kernels (rbu_headk_forward / rbu_headk_backward) and the K-class cross-entropy
(rbu_cek_forward / rbu_cek_backward) at batch 64, 256 x 256, C = 64 input channels, for K in {1, 2, 4, 8, 16, 32}; at
K = 1 and K = 2 the specialised kernels that RobustUNet / UNet keep (rbu_head_*, rbu_head2_*, rbu_ce2_*) run in the
same repetitions.  Then a RobustUNet(3, K, 64) training step (forward, nn.BCELoss, backward, FusedAdam) at K = 1 against
K = 8, alternated.  CUDA events around each call, a 256 MiB L2 flush before every repetition, median of the
repetitions.  GB/s are algorithmic (every tensor read or written once) against the measured HBM copy peak of
6 543 GB/s.  Usage: python tools/head_bench.py [reps]"""
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rbunet  # noqa: E402
from rbunet import _lib  # noqa: E402
from rbunet._lib import call, stream_ptr  # noqa: E402
from rbunet.engine import NULL, _p  # noqa: E402

COPY_PEAK_GBS = 6543.0
B, H, W, C = 64, 256, 256, 64
FLUSH = None


def timed(fns, reps):
    """Median ms of each function; the functions alternate within every repetition."""
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


def report(name, t, nbytes):
    gbs = nbytes / t / 1e6
    print(f"{name:<44} {t:8.3f} ms {nbytes / 1e9:7.3f} GB {gbs:7.0f} GB/s  {gbs / COPY_PEAK_GBS:.2f} of copy peak")


def kernels(reps):
    P, HW = B * H * W, H * W
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn((P, C), device=dev, generator=g).to(torch.bfloat16)
    dx = torch.empty_like(x)
    s = stream_ptr()
    print(f"batch {B} x {H}x{W}, C = {C}: P = {P} pixels\n")
    for K in (1, 2, 4, 8, 16, 32):
        w = torch.randn((K, C), device=dev, generator=g) / 8
        b = torch.randn(K, device=dev, generator=g)
        out = torch.empty((B, K, HW), device=dev)
        dout = torch.randn((B, K, HW), device=dev, generator=g)
        dw, db = torch.empty_like(w), torch.empty_like(b)
        wsb = torch.empty(_lib.lib().rbu_headk_backward_workspace_bytes(P, C, K) // 4 + 1, device=dev)
        fns = {
            "headk_forward (sigmoid)": (lambda: call("rbu_headk_forward", _p(x), C, P, HW, C, K, _p(w), _p(b), 1, _p(out),
                                                      NULL, s), P * C * 2 + P * K * 4),
            "headk_backward (sigmoid)": (lambda: call("rbu_headk_backward", _p(dout), _p(out), _p(x), C, _p(dx), C, P, HW, C,
                                                       K, 1, _p(w), _p(dw), _p(db), _p(wsb), wsb.numel() * 4, s),
                                         2 * P * C * 2 + 2 * P * K * 4),
        }
        if K == 1:
            wso = torch.empty(_lib.lib().rbu_bwd_workspace_bytes(B, HW, C) // 4 + 1, device=dev)
            fns["head_forward (K = 1 kernel)"] = (lambda: call("rbu_head_forward", _p(x), C, P, C, _p(w), _p(b), _p(out),
                                                               NULL, s), P * C * 2 + P * 4)
            fns["head_backward (K = 1 kernel)"] = (lambda: call("rbu_head_backward", _p(dout), _p(out), _p(x), C, _p(dx), C,
                                                                P, C, _p(w), _p(dw), _p(db), _p(wso), wso.numel() * 4, s),
                                                   2 * P * C * 2 + 2 * P * 4)
        if K >= 2:
            t = torch.randint(0, K, (B, HW), device=dev, generator=g)
            wsc = torch.empty(_lib.lib().rbu_cek_workspace_bytes(B, HW, K) // 8 + 1, dtype=torch.int64, device=dev)
            loss = torch.empty(1, device=dev)
            cc = torch.empty((B, K, 4), dtype=torch.int64, device=dev)
            inv = torch.empty(1, dtype=torch.int64, device=dev)
            dz = torch.empty_like(out)
            fns["headk_forward (logits)"] = (lambda: call("rbu_headk_forward", _p(x), C, P, HW, C, K, _p(w), _p(b), 0,
                                                          _p(out), NULL, s), P * C * 2 + P * K * 4)
            fns["cek_forward"] = (lambda: call("rbu_cek_forward", _p(out), _p(t), B, HW, K, _p(wsc), wsc.numel() * 8,
                                               _p(loss), _p(cc), _p(inv), s), P * K * 4 + P * 8)
            fns["cek_backward"] = (lambda: call("rbu_cek_backward", _p(out), _p(t), B, HW, K, NULL, _p(dz), s),
                                   2 * P * K * 4 + P * 8)
        if K == 2:
            ws2 = torch.empty(_lib.lib().rbu_head2_backward_workspace_bytes(P, C) // 4 + 1, device=dev)
            wce = torch.empty(_lib.lib().rbu_ce2_workspace_bytes(B, HW) // 4 + 1, device=dev)
            c2 = torch.empty((B, 4), dtype=torch.int64, device=dev)
            fns["head2_forward (K = 2 kernel)"] = (lambda: call("rbu_head2_forward", _p(x), C, P, HW, C, _p(w), _p(b),
                                                                _p(out), s), P * C * 2 + P * 8)
            fns["head2_backward (K = 2 kernel)"] = (lambda: call("rbu_head2_backward", _p(dout), _p(x), C, _p(dx), C, P, HW,
                                                                 C, _p(w), _p(dw), _p(db), _p(ws2), ws2.numel() * 4, s),
                                                    2 * P * C * 2 + P * 8)
            fns["ce2_forward (K = 2 kernel)"] = (lambda: call("rbu_ce2_forward", _p(out), _p(t), B, HW, _p(wce),
                                                              wce.numel() * 4, _p(loss), _p(c2), s), P * 8 + P * 8)
            fns["ce2_backward (K = 2 kernel)"] = (lambda: call("rbu_ce2_backward", _p(out), _p(t), B, HW, NULL, _p(dz), s),
                                                  2 * P * 8 + P * 8)
        names = list(fns)
        ts = timed([fns[n][0] for n in names], reps)
        print(f"K = {K}")
        for n, tm in zip(names, ts):
            report("  " + n, tm, fns[n][1])
        print()


def steps(reps):
    from oracle import robust_unet_ref as R
    dev = torch.device("cuda:0")
    x, y = R.synthetic_inputs(B, 3, H, W, seed=123, blobby=True)
    x = x.to(dev)
    runs = []
    for K in (1, 8):
        torch.manual_seed(0)
        m = rbunet.RobustUNet(3, K, 64).to(dev).train()
        opt = rbunet.FusedAdam(m.parameters(), lr=1e-4)
        yk = y.repeat(1, K, 1, 1).to(dev)
        crit = torch.nn.BCELoss()

        def step(m=m, opt=opt, yk=yk, crit=crit):
            opt.zero_grad()
            crit(m(x), yk).backward()
            opt.step()
        runs.append(step)
    t1, t8 = timed(runs, reps)
    print(f"RobustUNet(3, K, 64) training step, batch {B} x {H}x{W} (alternated):")
    print(f"  K = 1  {t1:8.2f} ms\n  K = 8  {t8:8.2f} ms   ({(t8 / t1 - 1) * 100:+.2f} %)")


if __name__ == "__main__":
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    print(f"device: {torch.cuda.get_device_name(0)} | nvidia-smi: {q.stdout.strip() or q.stderr.strip()}")
    kernels(reps)
    steps(max(reps // 2, 5))
