"""GPU parity at the reference's own width (base 64: 64 ... 1024 channels, K up to 9 216) and at BASELINE.json's
shapes -- rbunet.RobustUNet through nn.Module -> C ABI -> sm_100a kernels against

  (a) goldens produced by the UNMODIFIED reference at base 64 (tests/golden/model_c*_b64_*.npz),
  (b) the fp32 CPU oracle (pinned to the reference's goldens, tests/test_oracle_golden.py) on the same
      weights, inputs and injected Dropout2d masks (Main_Final.py:226-321,573-582), and
  (c) the yardstick: torch's OWN `autocast(bfloat16)` execution of the reference arithmetic (eager ATen/cuDNN kernels on
      the same GPU, head + loss in fp32).

Bars (measured values in profiles/r02_parity_*.txt).  With bf16 activations the network is chaotic end to end: the
first-maximum routing of MaxPool2d / AdaptiveMaxPool2d / torch.max and the one-sided BCE saturation flip at rounding
boundaries, for torch's autocast exactly as for this path (c2 shape, reference init: torch-autocast gradients have cosine
0.984 and a per-tensor RMS rel-L2 of 0.31 against fp32; this path 0.988 and 0.28).  So the rule is relative:
  * probabilities / logits / loss: deviation from fp32 <= 1.25 x the autocast run's deviation (+ a small floor);
  * gradients, every tensor with >= 1024 elements: rel-L2 vs fp32 <= 1.25 x autocast's + 0.05;
  * smaller tensors (per-channel vectors, the 1-element BatchNorm of psi, 7x7 kernels, the inc gate MLP: one flipped arg-max moves
    them by O(1)) enter as a group: RMS of their rel-L2 <= 1.25 x autocast's RMS + 0.02;
  * all tensors: RMS rel-L2 <= 1.25 x autocast's; 1 - cosine <= max(0.02, 1.25 x autocast's) -- i.e. cosine >= 0.98
    wherever torch's own bf16 run reaches it (c2: yes; the 2-image 512x512 case with negative BatchNorm gammas: no,
    autocast 0.882, this path 0.912).
Integer results (confusion counts, thresholded masks) are bit-exact on the device probabilities; mask flips against the
fp32 reference are only allowed where the fp32 logit is inside the yardstick's worst logit error."""
import os

import numpy as np
import pytest
import torch

from gpu_util import Report, rel_l2
from oracle import robust_unet_ref as R

pytestmark = pytest.mark.gpu

NOISE_DOMINATED = 0.25     # rel-L2 of torch's own bf16-autocast gradient against fp32 from which a tensor is judged in a group
ZERO_GRAD_BIASES = ("bottleneck.1.conv", "W_g.0.bias", "W_x.0.bias", "psi.0.bias")
DEV = "cuda:0"


def _reference_init_state_dict(nc):
    """The reference's own initialisation (torch.manual_seed(0); RobustUNet(nc, 1) -- the parameter registration order of
    Main_Final.RobustUNet, hence its initial weights under the same seed) as a CPU state_dict."""
    import rbunet
    torch.manual_seed(0)
    m = rbunet.RobustUNet(nc, 1, 64)
    return {k: v.clone() for k, v in m.state_dict().items()}


def _device_model(sd, nc):
    import rbunet
    model = rbunet.RobustUNet(nc, 1, 64)
    model.load_state_dict(sd)
    return model.to(DEV)


def _oracle_train(sd, x, y, masks, w_dice, names):
    s = {k: v.clone() for k, v in sd.items()}
    for n in names:
        s[n].requires_grad_(True)
    nb = {}
    p = R.robust_unet_forward(s, x, training=True, drop_masks=masks, new_buffers=nb)
    loss = R.bce_dice_loss(p, y, 1.0, w_dice)
    loss.backward()
    return p.detach(), loss.item(), {n: s[n].grad for n in names}, nb


def _autocast_train(sd, x, y, masks, w_dice, names):
    """torch.autocast(bfloat16) run of the reference arithmetic on the GPU; the head and the loss in fp32 (PyTorch
    refuses BCELoss under CUDA autocast; SURVEY.md §8c).  nn.Dropout2d draws its noise in the input dtype, so the
    injected masks are bf16 here, as they would be inside the reference under autocast."""
    dev = torch.device(DEV)
    s = {k: v.to(dev).clone() for k, v in sd.items()}
    for n in names:
        s[n].requires_grad_(True)
    mb = {k: v.to(dev).to(torch.bfloat16) for k, v in masks.items()}
    with torch.autocast("cuda", dtype=torch.bfloat16):
        p = R.robust_unet_forward(s, x.to(dev), training=True, drop_masks=mb, new_buffers={}, fp32_head=True)
    loss = R.bce_dice_loss(p.float(), y.to(dev), 1.0, w_dice)
    loss.backward()
    torch.cuda.synchronize()
    return p.detach().float().cpu(), loss.item(), {n: s[n].grad.float().cpu() for n in names}


def _train_case(tag, nc, B, S, w_dice, init):
    import rbunet
    shapes = R.robust_unet_shapes(nc, 1, 64)
    sd = _reference_init_state_dict(nc) if init == "reference" else R.synthetic_state_dict(shapes, seed=0)
    x, y = R.synthetic_inputs(B, nc, S, S, seed=123, blobby=True)
    masks = R.synthetic_drop_masks(B, 64, seed=7)
    model = _device_model(sd, nc).train()
    model.engine.drop_mask_fn = lambda nm, N, C: masks[nm]
    crit = rbunet.RobustBCEDiceLoss(1.0, w_dice)
    p = model(x.to(DEV))
    loss = crit(p, y.to(DEV))
    loss.backward()
    torch.cuda.synchronize()
    names = [n for n, _ in model.named_parameters()]
    pf, lf, gf, nbf = _oracle_train(sd, x, y, masks, w_dice, names)
    pa, la, ga = _autocast_train(sd, x, y, masks, w_dice, names)
    rep = Report()
    ya = rel_l2(pa, pf)
    rep.check(f"{tag}: probs vs fp32 oracle (autocast yardstick {ya:.2e})", p.detach(), pf, 1.25 * ya + 2e-3)
    rep.rows.append((f"{tag}: loss vs fp32 oracle (autocast {abs(la - lf) / abs(lf):.2e})", abs(loss.item() - lf) / abs(lf),
                     1.25 * abs(la - lf) / abs(lf) + 5e-3))
    dev_f, ac_f, small_dev, small_ac, noisy_dev, noisy_ac = [], [], [], [], [], []
    dots = n1 = n2 = dots_a = n1a = 0.0
    worst = []
    for n, prm in model.named_parameters():
        got = prm.grad.cpu()
        assert got.shape == gf[n].shape, n
        if n.endswith(".bias") and any(t in n for t in ZERO_GRAD_BIASES):
            # a bias in front of a train-mode BatchNorm: the true gradient is exactly zero (the fp32 oracle leaves round-off)
            assert got.abs().max() <= 1e-6, n
            continue
        e_dev, e_ac = rel_l2(got, gf[n]), rel_l2(ga[n], gf[n])
        dev_f.append(e_dev)
        ac_f.append(e_ac)
        nf = gf[n].double().norm().item() + 1e-30
        worst.append((e_dev / (e_ac + 1e-3), n, e_dev, e_ac, got.double().norm().item() / nf, ga[n].double().norm().item() / nf))
        if got.numel() >= 1024 and e_ac < NOISE_DOMINATED:
            rep.rows.append((f"{n} grad vs fp32 (autocast {e_ac:.2e})", e_dev, 1.25 * e_ac + 0.05))
        elif got.numel() >= 1024:
            # torch's own bf16 run is >= 25 % off the fp32 gradient on this tensor (ChannelAttention's fc weights behind the
            # arg-max of AdaptiveMaxPool, the 7x7 SpatialAttention kernels): one tensor is one draw of that noise, any
            # perturbation of the summation order moves it by its own size -- judged as a group below
            noisy_dev.append(e_dev)
            noisy_ac.append(e_ac)
        else:
            small_dev.append(e_dev)
            small_ac.append(e_ac)
        dots += (got.double() * gf[n].double()).sum().item()
        n1 += got.double().pow(2).sum().item()
        n2 += gf[n].double().pow(2).sum().item()
        dots_a += (ga[n].double() * gf[n].double()).sum().item()
        n1a += ga[n].double().pow(2).sum().item()
    rms = lambda v: float(np.sqrt(np.mean(np.square(v))))          # noqa: E731
    cos, cos_a = dots / (n1 * n2) ** 0.5, dots_a / (n1a * n2) ** 0.5
    rep.rows.append((f"{tag}: RMS grad deviation vs fp32 (autocast {rms(ac_f):.2e})", rms(dev_f), 1.25 * rms(ac_f) + 1e-3))
    rep.rows.append((f"{tag}: RMS deviation of the {len(small_dev)} tensors < 1024 elements (autocast {rms(small_ac):.2e})",
                     rms(small_dev), 1.25 * rms(small_ac) + 0.02))
    if noisy_dev:
        rep.rows.append((f"{tag}: RMS deviation of the {len(noisy_dev)} noise-dominated tensors (autocast {rms(noisy_ac):.2e})",
                         rms(noisy_dev), 1.25 * rms(noisy_ac) + 0.05))
    rep.rows.append((f"{tag}: 1 - cosine(all grads, fp32) (autocast {1 - cos_a:.2e})", 1 - cos, max(0.02, 1.25 * (1 - cos_a))))
    if init == "reference":
        assert cos >= 0.98, cos                      # the product configuration: absolute bar
    # BatchNorm running statistics follow nn.BatchNorm2d (momentum 0.1, unbiased variance); counters are integers
    msd = model.state_dict()
    for k, v in nbf.items():
        if v.dtype == torch.int64:
            assert int(msd[k]) == int(v), k
        else:
            rep.check(k, msd[k], v, 2e-2)
    # integer results: bit-exact on the device probabilities
    counts = crit.last_counts.cpu().numpy()
    assert (counts == R.confusion_counts(p.detach().cpu().numpy(), y.numpy())).all()
    assert (counts.sum(1) == S * S).all()
    out_dir = os.environ.get("RBU_PARITY_REPORT_DIR")
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        with open(os.path.join(out_dir, f"parity_{tag}.txt"), "w") as f:
            f.write(f"{tag}: B={B} {nc}x{S}x{S} base 64 init={init} w_dice={w_dice}\n")
            f.write(f"probs rel-L2 vs fp32: device {rel_l2(p.detach(), pf):.3e}  torch-autocast {ya:.3e}\n")
            f.write(f"loss: device {loss.item():.6f} fp32 {lf:.6f} autocast {la:.6f}\n")
            f.write(f"grad cosine vs fp32: device {cos:.5f}  torch-autocast {cos_a:.5f}\n")
            f.write(f"RMS per-tensor grad rel-L2 vs fp32: device {rms(dev_f):.3e}  torch-autocast {rms(ac_f):.3e}\n")
            for r_, n, e_dev, e_ac, nr_d, nr_a in sorted(worst, reverse=True):
                f.write(f"{r_:7.3f}  {n:40s} device {e_dev:.3e}  autocast {e_ac:.3e}   |g|/|g_fp32| device {nr_d:.4f} autocast {nr_a:.4f}\n")
    rep.finish()


def test_c2_shaped_train_step_reference_init():
    """BASELINE configs[1] shape (3 x 256 x 256, BCE), the reference's initialisation, batch 4."""
    _train_case("c2", 3, 4, 256, 0.0, "reference")


def test_c5_shaped_train_step_4ch_dice():
    """BASELINE configs[4] shape (4 x 512 x 512, BCE + Dice 0.5), synthetic weights with negative BN gammas, batch 2."""
    _train_case("c5", 4, 2, 512, 0.5, "synthetic")


@pytest.mark.parametrize("name", ["model_c3_b64_64x64.npz", "model_c4_b64_64x96.npz"])
def test_base64_against_reference_golden(golden_dir, name):
    """The committed outputs of the unmodified reference at base 64: probabilities in full, all 173 gradients as
    (norm, first values) summaries."""
    import rbunet
    g = np.load(os.path.join(golden_dir, name))
    nc, base, B, H, W = [int(v) for v in g["config"]]
    assert base == 64
    sd = R.synthetic_state_dict(R.robust_unet_shapes(nc, 1, base), seed=0)
    x, y = R.synthetic_inputs(B, nc, H, W, seed=123, blobby=True)
    masks = R.synthetic_drop_masks(B, base, seed=7)
    w_dice = float(g["w_dice"])
    model = _device_model(sd, nc).train()
    model.engine.drop_mask_fn = lambda nm, N, C: masks[nm]
    crit = rbunet.RobustBCEDiceLoss(1.0, w_dice)
    p = model(x.to(DEV))
    loss = crit(p, y.to(DEV))
    loss.backward()
    torch.cuda.synchronize()
    names = [str(n) for n in g["param_names"]]
    pa, la, ga = _autocast_train(sd, x, y, masks, w_dice, names)
    ref = torch.from_numpy(g["probs_train"])
    rep = Report()
    rep.check("train probs vs reference golden", p.detach(), ref, 1.25 * rel_l2(pa, ref) + 2e-3)
    lref = float(g["loss_train"])
    rep.rows.append(("loss vs reference golden", abs(loss.item() - lref) / lref, 1.25 * abs(la - lref) / lref + 5e-3))
    grads = dict(model.named_parameters())
    dn, an, dh, ah, vec, ndn, nan_ = [], [], [], [], [], [], []
    for i, n in enumerate(names):
        s_ = g["grad_summary"][i]          # [norm, sum, first 8 values] of the reference gradient
        if n.endswith(".bias") and any(t in n for t in ZERO_GRAD_BIASES):
            continue
        got = grads[n].grad.double().cpu().flatten()
        k = min(8, got.numel())
        head = torch.from_numpy(s_[2:2 + k])
        # the part of the reference gradient the fixture carries: its norm and its leading values
        dn.append(abs(got.norm().item() - s_[0]) / (s_[0] + 1e-30))
        an.append(abs(ga[n].double().norm().item() - s_[0]) / (s_[0] + 1e-30))
        vec.append(got.numel() >= 8)
        if got.numel() >= 1024 and an[-1] < 0.1:
            rep.rows.append((f"{n} |grad| vs golden (autocast {an[-1]:.2e})", dn[-1], 1.5 * an[-1] + 0.15))
        elif got.numel() >= 1024:     # the norm itself is >= 10 % off under torch's bf16 autocast: judged as a group
            ndn.append(dn[-1])
            nan_.append(an[-1])
        scale = s_[0] / got.numel() ** 0.5 * k ** 0.5 + 1e-30          # expected norm of k entries
        dh.append(((got[:k] - head).norm() / scale).item())
        ah.append(((ga[n].double().flatten()[:k] - head).norm() / scale).item())
    rms = lambda v: float(np.sqrt(np.mean(np.square(v))))          # noqa: E731
    med = lambda v: float(np.median(v))                            # noqa: E731
    # The RMS runs over the tensors with at least 8 elements: the 1-element gradients (the psi BatchNorms of the attention
    # gates, |g| ~ 1e-4 = a sum of cancelling terms) move by 1-4x their own size between any two bf16 executions -- torch's
    # autocast run included, and this library with or without the fused statistics -- and one of them would decide an RMS
    # over 157 tensors; they stay in the two medians below.
    dnv = [d for d, v in zip(dn, vec) if v]
    anv = [a for a, v in zip(an, vec) if v]
    rep.rows.append((f"RMS |grad| deviation over {len(dnv)} tensors of >= 8 elements (autocast {rms(anv):.2e})", rms(dnv),
                     1.25 * rms(anv) + 0.02))
    if ndn:
        rep.rows.append((f"RMS |grad| deviation of the {len(ndn)} noise-dominated large tensors (autocast {rms(nan_):.2e})",
                         rms(ndn), 1.5 * rms(nan_) + 0.15))
    rep.rows.append((f"median |grad| deviation (autocast {med(an):.2e})", med(dn), 1.25 * med(an) + 5e-3))
    rep.rows.append((f"median deviation of grad[:8] (autocast {med(ah):.2e})", med(dh), 1.25 * med(ah) + 0.02))
    model.load_state_dict(sd)
    model.eval()
    with torch.no_grad():
        pe = model(x.to(DEV))
        se = {k: v.to(DEV) for k, v in sd.items()}
        with torch.autocast("cuda", dtype=torch.bfloat16):
            pae = R.robust_unet_forward(se, x.to(DEV), training=False, fp32_head=True).float().cpu()
    refe = torch.from_numpy(g["probs_eval"])
    rep.check("eval probs vs reference golden", pe, refe, 1.25 * rel_l2(pae, refe) + 2e-3)
    rep.finish()


def test_c4_shaped_eval_forward_counts_and_mask_flips():
    """BASELINE configs[3] path (eval forward + thresholded masks + TP/FP/FN/TN) on a 512 x 512 tile, batch 1, against
    the fp32 CPU oracle: probabilities and logits within the autocast yardstick, counts bit-exact on the device
    probabilities, no more flipped mask pixels than torch's autocast run, and every flipped pixel has an fp32 logit
    inside the yardstick's worst logit error (delta)."""
    import rbunet
    nc, S = 3, 512
    sd = R.synthetic_state_dict(R.robust_unet_shapes(nc, 1, 64), seed=0)
    x, y = R.synthetic_inputs(1, nc, S, S, seed=321, blobby=True)
    model = _device_model(sd, nc).eval()
    model.engine.keep_logits = True
    with torch.no_grad():
        p = model(x.to(DEV))
        zd = model.engine.last_logits.cpu()
        counts = rbunet.confusion_counts(p, y.to(DEV)).cpu().numpy()
        zf = R.robust_unet_forward(sd, x, training=False, return_logits=True)
        se = {k: v.to(DEV) for k, v in sd.items()}
        with torch.autocast("cuda", dtype=torch.bfloat16):
            za = R.robust_unet_forward(se, x.to(DEV), training=False, return_logits=True, fp32_head=True).float().cpu()
    torch.cuda.synchronize()
    pc = p.cpu()
    assert torch.allclose(pc, torch.sigmoid(zd), rtol=0, atol=2e-7)              # the stored logits are the head's own
    pf = torch.sigmoid(zf)
    rep = Report()
    rep.check("probs vs fp32 oracle", pc, pf, 1.25 * rel_l2(torch.sigmoid(za), pf) + 2e-3)
    rep.check("logits vs fp32 oracle", zd, zf, 1.25 * rel_l2(za, zf) + 1e-3)
    worst_dev, worst_ac = (zd - zf).abs().max().item(), (za - zf).abs().max().item()
    rep.rows.append((f"max |logit error| (autocast {worst_ac:.3f})", worst_dev, 1.25 * worst_ac))
    assert (counts == R.confusion_counts(pc.numpy(), y.numpy())).all()           # bit-exact integers
    assert counts.sum() == S * S
    m = rbunet.batch_metrics(p, y.to(DEV))[0]
    assert m == R.metrics_from_counts(*counts[0])
    flips = (pc > 0.5) != (pf > 0.5)
    flips_ac = (za > 0) != (zf > 0)
    rep.rows.append((f"flipped mask pixels (autocast {int(flips_ac.sum())})", float(flips.sum()), 1.25 * float(flips_ac.sum()) + 16))
    delta = 1.25 * worst_ac
    if flips.any():
        rep.rows.append((f"max |fp32 logit| at a flipped pixel (delta = 1.25 x autocast's worst logit error)",
                         zf[flips].abs().max().item(), delta))
    rep.finish()


def test_smoke_configuration_cosine():
    """__graft_entry__.smoke(): base 64 at 64 x 64, gradient cosine >= 0.98 against the fp32 oracle."""
    import __graft_entry__ as ge
    ge.smoke()
