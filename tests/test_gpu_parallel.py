"""GPU: rbunet.DataParallel on a single-rank NCCL group -- the bucketed gradient path (stage hooks, flat buckets,
communication stream, views as .grad) must reproduce the plain model's gradients exactly.  The multi-rank averaging
itself is covered on the CPU by tests/test_parallel_cpu.py (gloo, world size 2) and by bench.py under torchrun."""
import os
import socket

import pytest
import torch
import torch.distributed as dist

from oracle import robust_unet_ref as R

pytestmark = pytest.mark.gpu


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_data_parallel_world1_matches_plain_model():
    import rbunet
    dev = torch.device("cuda:0")
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(_free_port()))
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=dev)
    try:
        sd = R.synthetic_state_dict(R.robust_unet_shapes(3, 1, 16), seed=0)
        x, y = R.synthetic_inputs(2, 3, 32, 32, seed=3, blobby=True)
        masks = R.synthetic_drop_masks(2, 16, seed=7)
        grads = []
        for wrap in (False, True):
            model = rbunet.RobustUNet(3, 1, 16)
            model.load_state_dict(sd)
            model.to(dev).train()
            model.engine.drop_mask_fn = lambda nm, N, C: masks[nm]
            net = rbunet.DataParallel(model, bucket_bytes=64 << 10) if wrap else model
            loss = rbunet.RobustBCEDiceLoss()(net(x.to(dev)), y.to(dev))
            loss.backward()
            torch.cuda.synchronize()
            grads.append({n: p.grad.clone() for n, p in model.named_parameters()})
            if wrap:
                assert len(net.bucketer.flat) > 4
        for n in grads[0]:
            assert torch.equal(grads[0][n], grads[1][n]), n
    finally:
        dist.destroy_process_group()


def test_gradients_have_private_storage_clip_and_accumulate():
    """ADVICE r1: every parameter's .grad owns its storage (no two alias), so torch.nn.utils.clip_grad_norm_ scales each
    once, and a second micro-batch accumulates into .grad like the reference's autograd does (Main_Final.py:573-582
    with two backward calls before the step) -- checked against the oracle's accumulated gradients."""
    import rbunet
    dev = torch.device("cuda:0")
    base = 16
    sd = R.synthetic_state_dict(R.robust_unet_shapes(3, 1, base), seed=0)
    x, y = R.synthetic_inputs(4, 3, 32, 32, seed=3, blobby=True)
    masks = R.synthetic_drop_masks(4, base, seed=7)
    model = rbunet.RobustUNet(3, 1, base)
    model.load_state_dict(sd)
    model.to(dev).train()
    crit = rbunet.RobustBCEDiceLoss()
    cur = {}
    model.engine.drop_mask_fn = lambda nm, N, C: cur["m"][nm]
    singles = []
    for i in range(2):                                 # each micro-batch alone
        model.zero_grad(set_to_none=True)
        cur["m"] = {k: v[2 * i:2 * i + 2] for k, v in masks.items()}
        crit(model(x[2 * i:2 * i + 2].to(dev)), y[2 * i:2 * i + 2].to(dev)).backward()
        singles.append({n: p.grad.clone() for n, p in model.named_parameters()})
    ptrs = {}
    for n, p in model.named_parameters():
        lo = p.grad.data_ptr()
        assert lo not in ptrs, f"{n} and {ptrs[lo]} share gradient storage"
        ptrs[lo] = n
    model.zero_grad(set_to_none=True)
    for i in range(2):                                 # accumulated: .grad survives between the two backward calls
        cur["m"] = {k: v[2 * i:2 * i + 2] for k, v in masks.items()}
        crit(model(x[2 * i:2 * i + 2].to(dev)), y[2 * i:2 * i + 2].to(dev)).backward()
    for n, p in model.named_parameters():
        assert torch.allclose(p.grad, singles[0][n] + singles[1][n], rtol=1e-6, atol=1e-12), n
    before = {n: p.grad.clone() for n, p in model.named_parameters()}
    total = torch.sqrt(sum(g.double().pow(2).sum() for g in before.values())).item()
    got = torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm=0.5 * total).item()
    assert abs(got - total) < 1e-4 * total
    for n, p in model.named_parameters():              # every gradient scaled exactly once
        assert torch.allclose(p.grad, before[n] * 0.5, rtol=1e-4, atol=1e-12), n


def test_eval_mode_backward_raises_instead_of_returning_wrong_gradients():
    import rbunet
    _check_eval_mode_backward_raises(rbunet.RobustUNet(3, 1, 16), rbunet.RobustBCEDiceLoss(), lambda y: y)


def test_unet_eval_mode_backward_raises_instead_of_returning_wrong_gradients():
    import rbunet
    _check_eval_mode_backward_raises(rbunet.UNet(3, 2), rbunet.CrossEntropyArgmaxLoss(), lambda y: y[:, 0].long())


def _check_eval_mode_backward_raises(model, crit, target):
    dev = torch.device("cuda:0")
    x, y = R.synthetic_inputs(1, 3, 32, 32, seed=3, blobby=True)
    y = target(y)
    model.to(dev).eval()
    out = model(x.to(dev))                                  # forward in eval mode with grad enabled works
    with torch.no_grad():
        assert torch.equal(out, model(x.to(dev)))           # and computes what it computes without grad
    loss = crit(out, y.to(dev))
    with pytest.raises(RuntimeError, match="train-mode forward"):
        loss.backward()
    with pytest.raises(RuntimeError, match="gradient for its input"):
        model.train()(x.to(dev).requires_grad_(True))


def _two_rank_worker(rank, world, port, out_dir):
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    import rbunet
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        base, per, S = 64, 4, 64
        torch.manual_seed(0)                          # the reference's initialisation (the smoke configuration per shard)
        sd = {k: v.clone() for k, v in rbunet.RobustUNet(3, 1, base).state_dict().items()}
        x, y = R.synthetic_inputs(world * per, 3, S, S, seed=123, blobby=True)
        masks = R.synthetic_drop_masks(world * per, base, seed=7)

        def shard(r):
            sl = slice(r * per, (r + 1) * per)
            return x[sl], y[sl], {k: v[sl] for k, v in masks.items()}

        def device_grads(r, wrap):
            xs, ys, ms = shard(r)
            model = rbunet.RobustUNet(3, 1, base)
            model.load_state_dict(sd)
            model.to(dev).train()
            model.engine.drop_mask_fn = lambda nm, N, C: ms[nm]
            net = rbunet.DataParallel(model, bucket_bytes=4 << 20) if wrap else model
            outs = []
            for _ in range(2 if wrap else 1):          # two steps through the wrapper: the buckets are reused
                model.zero_grad(set_to_none=True)
                model.load_state_dict(sd)              # same BatchNorm buffers for both steps
                loss = rbunet.RobustBCEDiceLoss()(net(xs.to(dev)), ys.to(dev))
                loss.backward()
                torch.cuda.synchronize()
                outs.append({n: p.grad.clone() for n, p in model.named_parameters()})
            if wrap:
                for n in outs[0]:
                    assert torch.equal(outs[0][n], outs[1][n]), n
            return outs[-1]

        ddp = device_grads(rank, True)                                    # post-all-reduce gradients of this rank
        local = [device_grads(r, False) for r in range(world)]             # every shard on this GPU, no communication
        for n in ddp:
            want = (local[0][n] + local[1][n]) / 2 if world == 2 else sum(d[n] for d in local) / world
            assert torch.allclose(ddp[n], want, rtol=1e-6, atol=1e-12), (rank, n)    # the exchange is exact averaging
        if rank == 0:
            # ... and equal to the mean of the per-shard fp32 oracle gradients (SURVEY.md §4 tier 5: the reference run once
            # per shard with its own BatchNorm statistics and dropout masks, gradients averaged) within the bf16 bar
            acc = None
            names = list(ddp.keys())
            for r in range(world):
                xs, ys, ms = shard(r)
                s = {k: v.clone() for k, v in sd.items()}
                for n in names:
                    s[n].requires_grad_(True)
                R.bce_loss(R.robust_unet_forward(s, xs, training=True, drop_masks=ms, new_buffers={}), ys).backward()
                acc = {n: s[n].grad / world if acc is None else acc[n] + s[n].grad / world for n in names}
            a = torch.cat([ddp[n].flatten().cpu().double() for n in names])
            b = torch.cat([acc[n].flatten().double() for n in names])
            cos = (a @ b / (a.norm() * b.norm())).item()
            with open(os.path.join(out_dir, "cosine.txt"), "w") as f:
                f.write(f"{cos}\n")
            # one shard of this configuration alone: 0.982 (profiles/r02_smoke_explore.log); bf16 chaos band 0.94-0.99
            assert cos >= 0.96, cos
        torch.save(True, os.path.join(out_dir, f"ok{rank}"))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_gradients_equal_the_mean_of_the_shard_gradients(tmp_path):
    """Multi-rank gradient parity on real GPUs over NCCL: two ranks, two shards, base 64.  The post-all-reduce gradients
    equal the average of the per-shard device gradients (exact) and match the mean of the per-shard ORACLE gradients."""
    import torch.multiprocessing as mp
    world = 2
    mp.spawn(_two_rank_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    assert all(os.path.exists(os.path.join(str(tmp_path), f"ok{r}")) for r in range(world))
    print("2-rank gradient cosine vs mean of shard oracle gradients:", open(os.path.join(str(tmp_path), "cosine.txt")).read())
