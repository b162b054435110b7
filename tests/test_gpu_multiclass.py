"""GPU tests of the K-class heads (1 <= K <= 32): the 1x1 head kernels and the K-class cross-entropy on their own
against fp64 references, RobustUNet(3, 4, 16) and UNet(3, 5) against the oracle in the tolerance scheme of
tests/test_gpu_model.py / tests/test_gpu_unet.py, training with torch's own losses, determinism at the product width,
and the argument checks."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from gpu_util import Report, rel_l2
from oracle import robust_unet_ref as R
from oracle import unet_ref as U
from multiclass_ref import argmax_class_counts, class_confusion_counts

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda:0")


def _abi():
    from rbunet import _lib
    from rbunet._lib import call, stream_ptr
    from rbunet.engine import NULL, _p
    return _lib, call, stream_ptr, NULL, _p


def _bf16_ulp(v):
    a = v.abs().clamp_min(2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(a)) - 7)


# ------------------------------------------------------------------------------------------------ 1. head kernels
def _head_case(C, K, N=2, H=5, W=13, seed=0):
    g = torch.Generator().manual_seed(seed * 1000 + C * 40 + K)
    ld, off = C + 16, 8                                   # x is a channel slice of a wider buffer
    xf = torch.randn((N, H, W, C), generator=g)
    xbuf = torch.randn((N, H, W, ld), generator=g).to(torch.bfloat16)
    xbuf[..., off:off + C] = xf.to(torch.bfloat16)
    w = torch.randn((K, C), generator=g) / C ** 0.5
    b = torch.randn(K, generator=g) * 0.1
    dout = torch.randn((N, K, H * W), generator=g)
    return xbuf.to(DEV), ld, off, w.to(DEV), b.to(DEV), dout.to(DEV)


def _run_headk(xbuf, ld, off, w, b, dout, sigmoid):
    _lib, call, stream_ptr, NULL, _p = _abi()
    N, H, W, _ = xbuf.shape
    K, C = w.shape
    P, HW = N * H * W, H * W
    out = torch.empty((N, K, HW), device=DEV)
    logits = torch.empty_like(out)
    xp = xbuf.data_ptr() + off * 2
    call("rbu_headk_forward", xp, ld, P, HW, C, K, _p(w), _p(b), sigmoid, _p(out), _p(logits), stream_ptr())
    dxbuf = torch.full_like(xbuf, 7.0)                    # sentinel around the written slice
    dw, db = torch.empty_like(w), torch.empty_like(b)
    nbytes = _lib.lib().rbu_headk_backward_workspace_bytes(P, C, K)
    ws = torch.empty(nbytes // 4 + 1, device=DEV)
    call("rbu_headk_backward", _p(dout), _p(out) if sigmoid else NULL, xp, ld, dxbuf.data_ptr() + off * 2, ld, P, HW, C,
         K, sigmoid, _p(w), _p(dw), _p(db), _p(ws), ws.numel() * 4, stream_ptr())
    torch.cuda.synchronize()
    return out, logits, dxbuf, dw, db


@pytest.mark.parametrize("sigmoid", [0, 1])
@pytest.mark.parametrize("K", [1, 2, 3, 5, 8, 16, 32])
@pytest.mark.parametrize("C", [16, 64, 128])
def test_headk_kernels_against_fp64(C, K, sigmoid):
    xbuf, ld, off, w, b, dout = _head_case(C, K)
    N, H, W, _ = xbuf.shape
    out, logits, dxbuf, dw, db = _run_headk(xbuf, ld, off, w, b, dout, sigmoid)
    x = xbuf[..., off:off + C].double().cpu().reshape(-1, C)                 # the bf16-rounded input
    wd, bd = w.double().cpu(), b.double().cpu()
    z = (x @ wd.T + bd).reshape(N, H * W, K).permute(0, 2, 1)
    mag = (x.abs() @ wd.abs().T).reshape(N, H * W, K).permute(0, 2, 1)
    zl = logits.double().cpu()
    assert ((zl - z).abs() <= 1e-5 * mag + 1e-6).all()
    o = out.double().cpu()
    if sigmoid:
        assert ((o - torch.sigmoid(zl)).abs() <= 1e-6).all()
        dz = dout.double().cpu() * o * (1 - o)
    else:
        assert torch.equal(out, logits)
        dz = dout.double().cpu()
    dzp = dz.permute(0, 2, 1).reshape(-1, K)                                # [P, K]
    dx_ref = (dzp @ wd).reshape(N, H, W, C)
    dx_tol = _bf16_ulp(dx_ref) + 1e-6 * (dzp.abs() @ wd.abs()).reshape(N, H, W, C)   # one bf16 ulp + fp32 summation
    dxs = dxbuf.cpu()
    got = dxs[..., off:off + C].double()
    assert ((got - dx_ref).abs() <= dx_tol).all()
    assert (dxs[..., :off] == 7.0).all() and (dxs[..., off + C:] == 7.0).all()       # nothing written outside the slice
    assert rel_l2(dw, dzp.T @ x) <= 1e-6
    assert rel_l2(db, dzp.sum(0)) <= 1e-6
    again = _run_headk(xbuf, ld, off, w, b, dout, sigmoid)
    for a, c in zip((out, logits, dxbuf, dw, db), again):
        assert torch.equal(a, c)                                             # bit-identical reruns
    # the specialised kernels that K = 1 (RobustUNet) and K = 2 (UNet) keep agree within the same bounds
    _lib, call, stream_ptr, NULL, _p = _abi()
    P, HW, xp = N * H * W, H * W, xbuf.data_ptr() + off * 2
    if K == 1 and sigmoid:
        p1, z1 = torch.empty_like(out), torch.empty_like(out)
        call("rbu_head_forward", xp, ld, P, C, _p(w), _p(b), _p(p1), _p(z1), stream_ptr())
        dx1 = torch.zeros_like(xbuf)
        dw1, db1 = torch.empty_like(w), torch.empty_like(b)
        ws = torch.empty(_lib.lib().rbu_bwd_workspace_bytes(N, HW, C) // 4 + 1, device=DEV)
        call("rbu_head_backward", _p(dout), _p(p1), xp, ld, dx1.data_ptr() + off * 2, ld, P, C, _p(w), _p(dw1), _p(db1),
             _p(ws), ws.numel() * 4, stream_ptr())
    elif K == 2 and not sigmoid:
        z1 = torch.empty_like(out)
        p1 = z1
        call("rbu_head2_forward", xp, ld, P, HW, C, _p(w), _p(b), _p(z1), stream_ptr())
        dx1 = torch.zeros_like(xbuf)
        dw1, db1 = torch.empty_like(w), torch.empty_like(b)
        ws = torch.empty(_lib.lib().rbu_head2_backward_workspace_bytes(P, C) // 4 + 1, device=DEV)
        call("rbu_head2_backward", _p(dout), xp, ld, dx1.data_ptr() + off * 2, ld, P, HW, C, _p(w), _p(dw1), _p(db1),
             _p(ws), ws.numel() * 4, stream_ptr())
    else:
        return
    torch.cuda.synchronize()
    assert ((z1.double().cpu() - zl).abs() <= 2e-5 * mag + 2e-6).all()
    assert ((p1.double().cpu() - o).abs() <= 2e-6).all()
    assert ((dx1[..., off:off + C].double().cpu() - got).abs() <= 2 * dx_tol).all()
    assert rel_l2(dw1, dw) <= 2e-6 and rel_l2(db1, db) <= 2e-6


# ------------------------------------------------------------------------------------------------ 2. K-class CE
def _run_cek(z, t):
    _lib, call, stream_ptr, NULL, _p = _abi()
    B, K, H, W = z.shape
    HW = H * W
    ws = torch.empty(_lib.lib().rbu_cek_workspace_bytes(B, HW, K) // 8 + 1, dtype=torch.int64, device=DEV)
    loss = torch.empty(1, device=DEV)
    counts = torch.empty((B, K, 4), dtype=torch.int64, device=DEV)
    inv = torch.empty(1, dtype=torch.int64, device=DEV)
    call("rbu_cek_forward", _p(z), _p(t), B, HW, K, _p(ws), ws.numel() * 8, _p(loss), _p(counts), _p(inv), stream_ptr())
    g = torch.full((1,), 0.75, device=DEV)
    dz = torch.empty_like(z)
    call("rbu_cek_backward", _p(z), _p(t), B, HW, K, _p(g), _p(dz), stream_ptr())
    torch.cuda.synchronize()
    return loss, counts, inv, dz


@pytest.mark.parametrize("HW", [(5, 13), (61, 67)])
@pytest.mark.parametrize("K", [2, 3, 7, 32])
def test_cek_against_fp64(K, HW):
    H, W = HW
    B = 3
    gen = torch.Generator().manual_seed(K * 100 + H)
    z = torch.randn((B, K, H, W), generator=gen) * 3
    z[:, :, :2] = torch.randint(-1, 2, (B, K, 2, W), generator=gen).float()   # exact ties in the first rows
    t = torch.randint(0, K, (B, H, W), generator=gen)
    zd, td = z.to(DEV), t.to(DEV)
    loss, counts, inv, dz = _run_cek(zd, td)
    z64 = z.double().requires_grad_(True)
    ref = F.cross_entropy(z64, t)
    (0.75 * ref).backward()
    assert abs(loss.item() - ref.item()) <= 1e-6 * abs(ref.item())
    assert rel_l2(dz, z64.grad) <= 1e-6
    assert inv.item() == 0
    assert (counts.cpu().numpy() == argmax_class_counts(z.numpy(), t.numpy())).all()
    if K == 2:                                           # the two-class kernel's counts are the class-1 slice
        _lib, call, stream_ptr, NULL, _p = _abi()
        ws = torch.empty(_lib.lib().rbu_ce2_workspace_bytes(B, H * W) // 4 + 1, device=DEV)
        l2 = torch.empty(1, device=DEV)
        c2 = torch.empty((B, 4), dtype=torch.int64, device=DEV)
        call("rbu_ce2_forward", _p(zd), _p(td), B, H * W, _p(ws), ws.numel() * 4, _p(l2), _p(c2), stream_ptr())
        assert torch.equal(c2, counts[:, 1])
    # targets outside [0, K): no fault, no loss, no counts, counted as invalid
    tb = t.clone()
    tb[0, 0, :3] = torch.tensor([-1, K, -100])
    tb[2, -1, -1] = K
    loss, counts, inv, dz = _run_cek(zd, tb.to(DEV))
    valid = (tb >= 0) & (tb < K)
    per = F.cross_entropy(z.double(), tb.clamp(0, K - 1), reduction="none") * valid
    assert inv.item() == 4
    assert abs(loss.item() - per.sum().item() / tb.numel()) <= 1e-6 * per.sum().item() / tb.numel()
    z64 = z.double().requires_grad_(True)
    (0.75 * (F.cross_entropy(z64, tb.clamp(0, K - 1), reduction="none") * valid).sum() / tb.numel()).backward()
    assert rel_l2(dz, z64.grad) <= 1e-6
    assert (dz.permute(0, 2, 3, 1)[~valid.to(DEV)] == 0).all()
    assert (counts.cpu().numpy() == argmax_class_counts(z.numpy(), tb.numpy())).all()
    if K > 2:
        import rbunet
        crit = rbunet.CrossEntropyArgmaxLoss()
        crit(zd, tb.to(DEV))
        with pytest.raises(ValueError):
            crit.batch_accuracy_iou()
        with pytest.raises(ValueError):
            crit.class_iou()


# ------------------------------------------------------------------------------------------------ 3. RobustUNet(3, 4, 16)
def _four_masks(B, H, W):
    ys = [R.synthetic_inputs(B, 3, H, W, seed=123 + 11 * k, blobby=True)[1] for k in range(4)]
    return torch.cat(ys, dim=1)


def test_robust_unet_four_classes_against_oracle():
    import rbunet
    nc, K, base, B, H, W = 3, 4, 16, 2, 32, 48
    sd = R.synthetic_state_dict(R.robust_unet_shapes(nc, K, base), seed=0)
    x, _ = R.synthetic_inputs(B, nc, H, W, seed=123, blobby=True)
    y = _four_masks(B, H, W)
    masks = R.synthetic_drop_masks(B, base, seed=7)
    model = rbunet.RobustUNet(nc, K, base)
    assert list(model.state_dict().keys()) == list(R.robust_unet_shapes(nc, K, base).keys())
    model.load_state_dict(sd)
    model.to(DEV)
    # eval forward
    model.eval()
    with torch.no_grad():
        p = model(x.to(DEV))
        pf = R.robust_unet_forward(sd, x, training=False)
        pq = R.robust_unet_forward(sd, x, training=False, st=R.BF16)
        sp = {k: (v * (1 + 1e-6 * torch.randn(v.shape, generator=torch.Generator().manual_seed(1)))
                  if v.is_floating_point() else v) for k, v in sd.items()}
        pq2 = R.robust_unet_forward(sp, x, training=False, st=R.BF16)
    assert p.shape == (B, K, H, W) and p.dtype == torch.float32
    rep = Report()
    rep.check("eval probs vs fp32 oracle", p, pf, 1.5 * rel_l2(pq, pf) + 5e-3)
    rep.check("eval probs vs bf16-storage oracle", p, pq, 1.5 * rel_l2(pq2, pq) + 5e-3)
    cc = rbunet.class_confusion_counts(p, y.to(DEV))
    assert (cc.cpu().numpy() == class_confusion_counts(p.cpu().numpy(), y.numpy())).all()
    for i, per_class in enumerate(rbunet.class_metrics(p, y.to(DEV))):
        assert per_class == [R.metrics_from_counts(*c) for c in cc[i].cpu().tolist()]
    # train step with injected Dropout2d masks and RobustBCEDiceLoss(1, 0.5)
    model.train()
    model.engine.drop_mask_fn = lambda nm, N, C: masks[nm]
    crit = rbunet.RobustBCEDiceLoss(1.0, 0.5)
    p = model(x.to(DEV))
    loss = crit(p, y.to(DEV))
    loss.backward()
    torch.cuda.synchronize()
    names = [n for n, _ in model.named_parameters()]

    def oracle(st, perturb=0.0):
        s = {k: v.clone() for k, v in sd.items()}
        if perturb:
            gen = torch.Generator().manual_seed(1)
            for n in names:
                s[n].mul_(1 + perturb * torch.randn(s[n].shape, generator=gen))
        for n in names:
            s[n].requires_grad_(True)
        nb = {}
        pp = R.robust_unet_forward(s, x, training=True, drop_masks=masks, new_buffers=nb, st=st)
        ll = R.bce_dice_loss(pp, y, 1.0, 0.5)
        ll.backward()
        return pp.detach(), ll.item(), {n: s[n].grad for n in names}, nb

    pf, lf, gf, nbf = oracle(R.FP32)
    pq, _, gq, _ = oracle(R.BF16)
    pq2, _, gq2, _ = oracle(R.BF16, 1e-6)
    rep.check("train probs vs fp32 oracle", p.detach(), pf, 1.5 * rel_l2(pq, pf) + 5e-3)
    rep.check("train probs vs bf16-storage oracle", p.detach(), pq, 1.5 * rel_l2(pq2, pq) + 5e-3)
    rep.rows.append(("loss vs fp32 oracle (relative)", abs(loss.item() - lf) / abs(lf), 2e-2))
    dev_f, q_f, dev_q, q2_q = [], [], [], []
    for n, prm in model.named_parameters():
        got = prm.grad.cpu()
        assert got.shape == gf[n].shape, n
        if n.endswith(".bias") and any(t in n for t in ("bottleneck.1.conv", "W_g.0.bias", "W_x.0.bias", "psi.0.bias")):
            continue                                            # exactly-zero true gradient (tests/test_gpu_model.py)
        dev_f.append(rel_l2(got, gf[n])); q_f.append(rel_l2(gq[n], gf[n]))
        dev_q.append(rel_l2(got, gq[n])); q2_q.append(rel_l2(gq2[n], gq[n]))
    rms = lambda v: float(np.sqrt(np.mean(np.square(v))))
    rep.rows.append(("RMS grad deviation vs fp32 oracle", rms(dev_f), 1.5 * rms(q_f) + 0.01))
    rep.rows.append(("RMS grad deviation vs bf16-storage oracle", rms(dev_q), 1.5 * rms(q2_q) + 0.01))
    msd = model.state_dict()
    for k, v in nbf.items():
        if v.dtype == torch.int64:
            assert int(msd[k]) == int(v), k
        else:
            rep.check(k, msd[k], v, 3e-2)
    rep.finish()
    cc = crit.last_counts
    assert cc.shape == (B, 4)          # RobustBCEDiceLoss counts over all K planes of each image, as nn.BCELoss averages
    assert (cc.cpu().numpy() == R.confusion_counts(p.detach().cpu().numpy(), y.numpy())).all()


# ------------------------------------------------------------------------------------------------ 4. UNet(3, 5)
def test_unet_five_classes_against_oracle():
    import rbunet
    K = 5
    sd = R.synthetic_state_dict(U.unet_shapes(3, K), seed=11)
    for k in sd:
        if k.endswith(".weight") and sd[k].dim() == 1:
            sd[k] = sd[k].abs()
    x, _ = R.synthetic_inputs(2, 3, 32, 32, seed=321, blobby=True)
    t = torch.from_numpy((R._hash_uniform(2 * 32 * 32, 5) * K).astype(np.int64).clip(0, K - 1).reshape(2, 32, 32))
    model = rbunet.UNet(3, K)
    assert list(model.state_dict().keys()) == list(U.unet_shapes(3, K).keys())
    model.load_state_dict(sd)
    model.to(DEV)
    model.eval()
    with torch.no_grad():
        z = model(x.to(DEV))
        zf = U.unet_forward(sd, x, training=False)
        zq = U.unet_forward(sd, x, training=False, st=R.BF16)
        sp = {k: (v * (1 + 1e-6 * torch.randn(v.shape, generator=torch.Generator().manual_seed(1)))
                  if v.is_floating_point() else v) for k, v in sd.items()}
        zq2 = U.unet_forward(sp, x, training=False, st=R.BF16)
    assert z.shape == (2, K, 32, 32)
    rep = Report()
    rep.check("eval logits vs fp32 oracle", z, zf, 1.5 * rel_l2(zq, zf) + 5e-3)
    rep.check("eval logits vs bf16-storage oracle", z, zq, 1.5 * rel_l2(zq2, zq) + 5e-3)
    crit = rbunet.CrossEntropyArgmaxLoss()
    loss = crit(z, t.to(DEV))
    assert abs(loss.item() - U.ce_loss(z.cpu().double(), t).item()) < 1e-5 * max(1.0, loss.item())
    cc = argmax_class_counts(z.cpu().numpy(), t.numpy())
    assert (crit.last_class_counts.cpu().numpy() == cc).all()
    assert (crit.last_counts.cpu().numpy() == U.argmax_counts(z.cpu().numpy(), t.numpy())).all()
    tot = cc.sum(0)
    acc, iou = crit.batch_accuracy_iou()
    assert acc == float(tot[:, 0].sum()) / float(t.numel())
    assert iou == (1.0 if tot[1, :3].sum() == 0 else float(tot[1, 0]) / float(tot[1, :3].sum()))
    assert crit.class_iou() == [1.0 if r[:3].sum() == 0 else float(r[0]) / float(r[:3].sum()) for r in tot]
    # train step
    model.train()
    z = model(x.to(DEV))
    loss = crit(z, t.to(DEV))
    loss.backward()
    torch.cuda.synchronize()
    names = [n for n, _ in model.named_parameters()]

    def oracle(st, perturb=0.0):
        s = {k: v.clone() for k, v in sd.items()}
        if perturb:
            gen = torch.Generator().manual_seed(1)
            for n in names:
                s[n].mul_(1 + perturb * torch.randn(s[n].shape, generator=gen))
        for n in names:
            s[n].requires_grad_(True)
        nb = {}
        zz = U.unet_forward(s, x, training=True, new_buffers=nb, st=st)
        U.ce_loss(zz, t).backward()
        return zz.detach(), {n: s[n].grad for n in names}, nb

    zf, gf, nbf = oracle(R.FP32)
    zq, gq, _ = oracle(R.BF16)
    zq2, gq2, _ = oracle(R.BF16, 1e-6)
    rep.check("train logits vs fp32 oracle", z.detach(), zf, 1.5 * rel_l2(zq, zf) + 5e-3)
    rep.check("train logits vs bf16-storage oracle", z.detach(), zq, 1.5 * rel_l2(zq2, zq) + 5e-3)
    dev_f, q_f, dev_q, q2_q = [], [], [], []
    for n, prm in model.named_parameters():
        got = prm.grad.cpu()
        if n.endswith(".0.bias") or n.endswith(".3.bias"):
            assert got.abs().max() <= 1e-6 and gf[n].abs().max() < 1e-3, n
            continue
        dev_f.append(rel_l2(got, gf[n])); q_f.append(rel_l2(gq[n], gf[n]))
        dev_q.append(rel_l2(got, gq[n])); q2_q.append(rel_l2(gq2[n], gq[n]))
    rms = lambda v: float(np.sqrt(np.mean(np.square(v))))
    rep.rows.append(("RMS grad deviation vs fp32 oracle", rms(dev_f), 1.5 * rms(q_f) + 0.01))
    rep.rows.append(("RMS grad deviation vs bf16-storage oracle", rms(dev_q), 1.5 * rms(q2_q) + 0.01))
    msd = model.state_dict()
    for k, v in nbf.items():
        if v.dtype == torch.int64:
            assert int(msd[k]) == int(v), k
        else:
            rep.check(k, msd[k], v, 3e-2)
    rep.finish()


# ------------------------------------------------------------------------------------------------ 5. torch losses
@pytest.mark.parametrize("case", ["robust3_bce", "unet5_ce", "unet1_bcelogits"])
def test_trains_with_torch_losses(case):
    import rbunet
    torch.manual_seed(0)
    x, y = R.synthetic_inputs(4, 3, 64, 64, seed=9, blobby=True)
    if case == "robust3_bce":
        model = rbunet.RobustUNet(3, 3, 16)
        crit = torch.nn.BCELoss()
        tgt = _four_masks(4, 64, 64)[:, :3]
    elif case == "unet5_ce":
        model = rbunet.UNet(3, 5)
        crit = torch.nn.CrossEntropyLoss()
        tgt = (y[:, 0] * 2 + (x[:, 0] > 0.8).float() + 2 * (x[:, 1] > 1.2).float()).long().clamp(0, 4)
    else:
        model = rbunet.UNet(3, 1)
        crit = torch.nn.BCEWithLogitsLoss()
        tgt = y
    model = model.to(DEV).train()
    opt = rbunet.FusedAdam(model.parameters(), lr=1e-3)
    x, tgt = x.to(DEV), tgt.to(DEV)
    losses = []
    for _ in range(30):
        opt.zero_grad()
        loss = crit(model(x), tgt)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    assert np.isfinite(losses[-1]) and losses[-1] < 0.7 * losses[0], (losses[0], losses[-1])


# ------------------------------------------------------------------------------------------------ 6. product width
def test_product_width_deterministic_and_one_head_launch():
    import rbunet
    from rbunet import _lib
    B, H, W, base = 4, 256, 256, 64
    x, _ = R.synthetic_inputs(B, 3, H, W, seed=5, blobby=True)
    y = torch.cat([R.synthetic_inputs(B, 3, H, W, seed=40 + k, blobby=True)[1] for k in range(8)], dim=1)
    masks = R.synthetic_drop_masks(B, base, seed=7)
    x, y = x.to(DEV), y.to(DEV)

    def build(K):
        torch.manual_seed(0)
        m = rbunet.RobustUNet(3, K, base).to(DEV).train()
        m.engine.drop_mask_fn = lambda nm, N, C: masks[nm]
        return m

    model = build(8)
    crit = torch.nn.BCELoss()
    runs = []
    for _ in range(2):
        model.zero_grad(set_to_none=True)
        p = model(x)
        crit(p, y).backward()
        torch.cuda.synchronize()
        runs.append((p.detach().clone(), {n: q.grad.clone() for n, q in model.named_parameters()}))
    assert torch.equal(runs[0][0], runs[1][0])
    for n in runs[0][1]:
        assert torch.equal(runs[0][1][n], runs[1][1][n]), n

    def forward_launches(m):
        m(x)                                         # warm (weight packing)
        torch.cuda.synchronize()
        l0 = _lib.launch_count()
        m(x)
        return _lib.launch_count() - l0

    with torch.no_grad():
        k8 = forward_launches(model.eval())
        k1 = forward_launches(build(1).eval())
    assert k8 == k1, (k8, k1)


# ------------------------------------------------------------------------------------------------ 7. errors
def test_argument_errors():
    import rbunet
    for bad in (0, 33):
        with pytest.raises(ValueError):
            rbunet.RobustUNet(3, bad, 16)
        with pytest.raises(ValueError):
            rbunet.UNet(3, bad)
    with pytest.raises(ValueError):
        rbunet.CrossEntropyArgmaxLoss()(torch.zeros((2, 1, 8, 8), device=DEV), torch.zeros((2, 8, 8), dtype=torch.long,
                                                                                          device=DEV))
    _lib, call, stream_ptr, NULL, _p = _abi()
    lib = _lib.lib()
    x = torch.zeros((64, 256), dtype=torch.bfloat16, device=DEV)
    w = torch.zeros((33, 512), device=DEV)
    out = torch.zeros((64 * 33,), device=DEV)
    s = stream_ptr()
    for C, K in ((16, 0), (16, 33), (24, 2), (8, 2), (512, 2)):
        assert lib.rbu_headk_forward(_p(x), 256, 64, 64, C, K, _p(w), _p(w), 1, _p(out), NULL, s) < 0
        assert b"rbu_headk_forward" in lib.rbu_last_error()
    assert lib.rbu_headk_forward(_p(x), 256, 64, 48, 16, 2, _p(w), _p(w), 1, _p(out), NULL, s) < 0     # P % HW != 0
    assert lib.rbu_headk_backward_workspace_bytes(64, 24, 2) == 0
    ws = torch.zeros(1 << 16, device=DEV)
    assert lib.rbu_headk_backward(_p(out), _p(out), _p(x), 256, _p(x), 256, 64, 64, 16, 40, 1, _p(w), _p(w), _p(w),
                                  _p(ws), ws.numel() * 4, s) < 0
    t = torch.zeros(64, dtype=torch.int64, device=DEV)
    i1 = torch.zeros(1, dtype=torch.int64, device=DEV)
    assert lib.rbu_cek_forward(_p(out), _p(t), 1, 64, 33, _p(ws), ws.numel() * 4, _p(out), _p(i1), _p(i1), s) < 0
    assert lib.rbu_cek_forward(_p(out), _p(t), 65536, 1, 3, _p(ws), ws.numel() * 4, _p(out), _p(i1), _p(i1), s) < 0
    assert lib.rbu_cek_backward(_p(out), _p(t), 1, 64, 0, NULL, _p(out), s) < 0
    torch.cuda.synchronize()
    with pytest.raises(ValueError):
        rbunet.class_confusion_counts(torch.zeros((65536, 2, 1, 1), device=DEV), torch.zeros((65536, 2, 1, 1), device=DEV))
