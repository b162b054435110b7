"""TEST INFRASTRUCTURE — CPU fp32 restatement of the reference Robust U-Net hot path.

This file is the parity oracle: a functional (state_dict in, tensors out) restatement of
`/root/reference/Main_Final.py` in plain fp32 torch CPU ops.  It is *not* part of the
product: only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s cpu_baseline /
`--impl reference` legs may import it.  The product package never does.

Parity pinning: the reference ships no tests or golden vectors (SURVEY.md §4), so this
restatement is pinned against outputs of the reference itself run in the build container
(`oracle/make_golden.py` → `tests/golden/*.npz`, checked by `tests/test_oracle_golden.py`).
The RGB→HSV and Dice pieces have no reference code
(SURVEY.md §8c): those two are "parity unpinned" — HSV is pinned to OpenCV float semantics
and `colorsys` instead.

Each function cites the reference lines it follows.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import numpy as np
import torch
import torch.nn.functional as F

BN_EPS = 1e-5          # nn.BatchNorm2d default, Main_Final.py:158
BN_MOMENTUM = 0.1      # nn.BatchNorm2d default

RESBLOCKS = ("inc", "down1.1", "down2.1", "down3.1", "bottleneck.2", "dec4", "dec3", "dec2", "dec1")
DROPOUT_P = {"inc": 0.1, "down1.1": 0.1, "down2.1": 0.2, "down3.1": 0.2, "bottleneck.2": 0.3,
             "dec4": 0.2, "dec3": 0.2, "dec2": 0.1, "dec1": 0.1}   # Main_Final.py:233-271
IMAGENET_MEAN = (0.485, 0.456, 0.406)   # Main_Final.py:700
IMAGENET_STD = (0.229, 0.224, 0.225)


# --------------------------------------------------------------------------------------
# storage model
# --------------------------------------------------------------------------------------
class _RoundBoth(torch.autograd.Function):
    """value rounded to bf16 on the way forward, gradient rounded to bf16 on the way back."""

    @staticmethod
    def forward(ctx, x):
        return x.to(torch.bfloat16).float()

    @staticmethod
    def backward(ctx, g):
        return g.to(torch.bfloat16).float()


class _RoundGrad(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        return x.view_as(x)

    @staticmethod
    def backward(ctx, g):
        return g.to(torch.bfloat16).float()


class _RoundValue(torch.autograd.Function):
    """straight-through: the fp32 master weight receives the gradient of its bf16 copy."""

    @staticmethod
    def forward(ctx, x):
        return x.to(torch.bfloat16).float()

    @staticmethod
    def backward(ctx, g):
        return g


class Fp32Storage:
    """The reference's numerics: every tensor stays fp32 (identity hooks)."""
    name = "fp32"

    def act(self, x):      # an activation that the device path keeps in HBM
        return x

    def grad(self, x):     # a point where only the gradient is stored
        return x

    def weight(self, w):   # a tensor-core GEMM weight operand
        return w


class Bf16Storage(Fp32Storage):
    """Same algorithm, but rounding to bf16 exactly where the CUDA path stores bf16 in HBM (conv / ConvTranspose
    outputs, the BN1+ReLU+dropout output, block and gate outputs, their gradients, and the GEMM weight operands);
    statistics, gates, the head and the loss stay fp32.  Used to separate logic errors from storage rounding."""
    name = "bf16"

    def act(self, x):
        return _RoundBoth.apply(x)

    def grad(self, x):
        return _RoundGrad.apply(x)

    def weight(self, w):
        return _RoundValue.apply(w)


FP32 = Fp32Storage()
BF16 = Bf16Storage()


# --------------------------------------------------------------------------------------
# building blocks
# --------------------------------------------------------------------------------------
def batch_norm(sd: Dict[str, torch.Tensor], prefix: str, x: torch.Tensor, training: bool,
               new_buffers: Optional[dict] = None) -> torch.Tensor:
    """nn.BatchNorm2d (Main_Final.py:158,160,173,127,132,137,210): batch statistics (biased
    variance) in train mode, running statistics in eval mode; running stats are updated with
    momentum 0.1 and the *unbiased* variance.  Updated buffers go to `new_buffers`."""
    w, b = sd[prefix + ".weight"], sd[prefix + ".bias"]
    rm, rv = sd[prefix + ".running_mean"], sd[prefix + ".running_var"]
    if not training:
        return F.batch_norm(x, rm, rv, w, b, False, BN_MOMENTUM, BN_EPS)
    rm2, rv2 = rm.clone(), rv.clone()
    y = F.batch_norm(x, rm2, rv2, w, b, True, BN_MOMENTUM, BN_EPS)
    if new_buffers is not None:
        new_buffers[prefix + ".running_mean"] = rm2
        new_buffers[prefix + ".running_var"] = rv2
        new_buffers[prefix + ".num_batches_tracked"] = sd[prefix + ".num_batches_tracked"] + 1
    return y


def channel_attention(sd, prefix, x):
    """ChannelAttention.forward (Main_Final.py:97-101): x * sigmoid(fc(avgpool x) + fc(maxpool x)),
    fc = 1x1 conv C->C/16, ReLU, 1x1 conv C/16->C, no biases, shared weights."""
    w1, w2 = sd[prefix + ".fc.0.weight"], sd[prefix + ".fc.2.weight"]

    def fc(u):
        return F.conv2d(F.relu(F.conv2d(u, w1)), w2)

    avg = fc(F.adaptive_avg_pool2d(x, 1))
    mx = fc(F.adaptive_max_pool2d(x, 1))
    return x * torch.sigmoid(avg + mx)


def spatial_attention(sd, prefix, x):
    """SpatialAttention.forward (Main_Final.py:112-117): x * sigmoid(conv7x7([mean_c x, max_c x]))."""
    avg = torch.mean(x, dim=1, keepdim=True)
    mx, _ = torch.max(x, dim=1, keepdim=True)
    att = F.conv2d(torch.cat([avg, mx], dim=1), sd[prefix + ".conv1.weight"], padding=3)
    return x * torch.sigmoid(att)


def residual_block(sd, prefix, x, training, drop_mask=None, new_buffers=None, st=FP32):
    """ResidualBlock.forward (Main_Final.py:178-196).  `drop_mask` is the Dropout2d channel mask
    [B,C,1,1] with values in {0, 1/(1-p)} (train mode only; None = identity)."""
    if (prefix + ".shortcut.0.weight") in sd:
        r = st.act(F.conv2d(x, st.weight(sd[prefix + ".shortcut.0.weight"])))
        r = batch_norm(sd, prefix + ".shortcut.1", r, training, new_buffers)
    else:
        r = x
    out = st.act(F.conv2d(x, st.weight(sd[prefix + ".conv1.weight"]), padding=1))
    out = F.relu(batch_norm(sd, prefix + ".bn1", out, training, new_buffers))
    if training and drop_mask is not None:
        out = out * drop_mask
    out = st.act(out)
    out = st.act(F.conv2d(out, st.weight(sd[prefix + ".conv2.weight"]), padding=1))
    out = batch_norm(sd, prefix + ".bn2", out, training, new_buffers)
    out = channel_attention(sd, prefix + ".ca", out)
    out = spatial_attention(sd, prefix + ".sa", out)
    return st.act(F.relu(st.grad(out + r)))


def dilated_block(sd, prefix, x, training, new_buffers=None, st=FP32):
    """DilatedBlock.forward (Main_Final.py:213-223): cat(1x1, 3x3 d1, 3x3 d2, 3x3 d4) -> BN -> ReLU."""
    def w(i):
        return st.weight(sd[f"{prefix}.conv{i}.weight"])
    x1 = F.conv2d(x, w(1), sd[prefix + ".conv1.bias"])
    x2 = F.conv2d(x, w(2), sd[prefix + ".conv2.bias"], padding=1, dilation=1)
    x3 = F.conv2d(x, w(3), sd[prefix + ".conv3.bias"], padding=2, dilation=2)
    x4 = F.conv2d(x, w(4), sd[prefix + ".conv4.bias"], padding=4, dilation=4)
    out = st.act(torch.cat([x1, x2, x3, x4], dim=1))
    return st.act(F.relu(batch_norm(sd, prefix + ".bn", out, training, new_buffers)))


def attention_gate(sd, prefix, g, x, training, new_buffers=None, st=FP32):
    """AttentionGate.forward (Main_Final.py:143-148)."""
    g1 = batch_norm(sd, prefix + ".W_g.1",
                    st.act(F.conv2d(g, st.weight(sd[prefix + ".W_g.0.weight"]), sd[prefix + ".W_g.0.bias"])),
                    training, new_buffers)
    x1 = batch_norm(sd, prefix + ".W_x.1",
                    st.act(F.conv2d(x, st.weight(sd[prefix + ".W_x.0.weight"]), sd[prefix + ".W_x.0.bias"])),
                    training, new_buffers)
    t = F.relu(g1 + x1)
    q = batch_norm(sd, prefix + ".psi.1",
                   F.conv2d(t, sd[prefix + ".psi.0.weight"], sd[prefix + ".psi.0.bias"]),
                   training, new_buffers)
    return st.act(x * torch.sigmoid(q))


def robust_unet_forward(sd, x, training=False, drop_masks: Optional[dict] = None,
                        new_buffers: Optional[dict] = None, return_logits=False, st=FP32, fp32_head=False):
    """RobustUNet.forward (Main_Final.py:290-321).  Concat order is [gated skip, upsampled]
    (:303,308,313,318).  Returns probabilities [B,1,H,W] (sigmoid inside `outc`, :274-277).
    `fp32_head`: evaluate `outc` + sigmoid in fp32 outside any enclosing torch.autocast region (the bf16-autocast
    yardstick of SURVEY.md §8c: bf16-rounded logits saturate the BCE, so the head stays fp32 as on the device)."""
    dm = drop_masks or {}

    def rb(prefix, t):
        return residual_block(sd, prefix, t, training, dm.get(prefix), new_buffers, st)

    x1 = rb("inc", st.act(x))
    x2 = rb("down1.1", F.max_pool2d(x1, 2))
    x3 = rb("down2.1", F.max_pool2d(x2, 2))
    x4 = rb("down3.1", F.max_pool2d(x3, 2))
    x5 = dilated_block(sd, "bottleneck.1", F.max_pool2d(x4, 2), training, new_buffers, st)
    x5 = rb("bottleneck.2", x5)
    t = x5
    for k, skip in ((4, x4), (3, x3), (2, x2), (1, x1)):
        t = st.act(F.conv_transpose2d(t, st.weight(sd[f"up{k}.weight"]), sd[f"up{k}.bias"], stride=2))
        att = attention_gate(sd, f"att{k}", t, skip, training, new_buffers, st)
        t = rb(f"dec{k}", torch.cat([att, t], dim=1))
    if fp32_head:
        with torch.autocast(device_type=t.device.type, enabled=False):
            z = F.conv2d(t.float(), sd["outc.0.weight"].float(), sd["outc.0.bias"].float())
            return z if return_logits else torch.sigmoid(z)
    z = F.conv2d(t, sd["outc.0.weight"], sd["outc.0.bias"])
    return z if return_logits else torch.sigmoid(z)


# --------------------------------------------------------------------------------------
# loss and metrics
# --------------------------------------------------------------------------------------
def bce_loss(p: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    """nn.BCELoss() on probabilities (Main_Final.py:551,580).  Forward: mean(-(y*max(ln p,-100) +
    (1-y)*max(ln(1-p),-100))); backward (torch's binary_cross_entropy_backward):
    (p-y)/max(p(1-p),1e-12)/N — which is NOT the autograd of the clamped-log form at p in {0,1}, so the
    reference's own functional is called here."""
    return F.binary_cross_entropy(p, y)


def bce_loss_restated(p: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
    """Forward-only literal restatement of nn.BCELoss (checked against bce_loss in the CPU tests)."""
    lp = torch.clamp(torch.log(p), min=-100.0)
    l1p = torch.clamp(torch.log(1.0 - p), min=-100.0)
    return -(y * lp + (1.0 - y) * l1p).mean()


def bce_dice_loss(p, y, w_bce=1.0, w_dice=0.0, smooth=1.0):
    """Build-defined "robust" loss (no reference code, SURVEY.md §8c — parity unpinned):
    w_bce*BCE + w_dice*(1 - (2*sum(p*y)+s)/(sum(p)+sum(y)+s)).  Defaults reduce to nn.BCELoss."""
    loss = w_bce * bce_loss(p, y)
    if w_dice != 0.0:
        inter = (p * y).sum()
        dice = (2.0 * inter + smooth) / (p.sum() + y.sum() + smooth)
        loss = loss + w_dice * (1.0 - dice)
    return loss


def confusion_counts(pred: np.ndarray, target: np.ndarray, threshold: float = 0.5) -> np.ndarray:
    """Integer TP/FP/FN/TN per image for `pred > threshold` (strict, Main_Final.py:521) against a
    0/1 target.  pred/target: [B,H,W] or [B,1,H,W].  Returns int64 [B,4]."""
    pb = (np.asarray(pred) > threshold).reshape(pred.shape[0], -1)
    tb = np.asarray(target).reshape(target.shape[0], -1) != 0
    tp = np.logical_and(pb, tb).sum(1)
    fp = pb.sum(1) - tp
    fn = tb.sum(1) - tp
    tn = pb.shape[1] - tp - fp - fn
    return np.stack([tp, fp, fn, tn], axis=1).astype(np.int64)


def metrics_from_counts(tp, fp, fn, tn) -> dict:
    """ModelEvaluator.calculate_metrics (Main_Final.py:519-547) in float64 from integer counts.
    accuracy_score == (TP+TN)/HW; IoU = TP/(union+1e-8); P, R, F1 with +1e-8 each."""
    tp, fp, fn, tn = float(tp), float(fp), float(fn), float(tn)
    total = tp + fp + fn + tn
    iou = tp / (tp + fp + fn + 1e-8)
    precision = tp / (tp + fp + 1e-8)
    recall = tp / (tp + fn + 1e-8)
    f1 = 2 * precision * recall / (precision + recall + 1e-8)
    return {"accuracy": (tp + tn) / total, "iou": iou, "precision": precision,
            "recall": recall, "f1_score": f1}


def calculate_metrics(pred, target, threshold=0.5) -> dict:
    """Same signature as ModelEvaluator.calculate_metrics (Main_Final.py:519): pred/target [H,W]."""
    c = confusion_counts(np.asarray(pred)[None], np.asarray(target)[None], threshold)[0]
    return metrics_from_counts(*c)


# --------------------------------------------------------------------------------------
# input preprocessing
# --------------------------------------------------------------------------------------
def rgb_to_hsv(rgb: np.ndarray) -> np.ndarray:
    """RGB in [0,1] float32 [...,3] -> HSV with OpenCV float semantics (H in [0,360), S, V in
    [0,1]).  No reference code exists (SURVEY.md §8c): pinned to cv2.cvtColor/`colorsys`."""
    rgb = np.asarray(rgb, dtype=np.float32)
    r, g, b = rgb[..., 0], rgb[..., 1], rgb[..., 2]
    v = np.maximum(np.maximum(r, g), b)
    mn = np.minimum(np.minimum(r, g), b)
    diff = v - mn
    s = np.where(v > 0, diff / np.where(v > 0, v, 1), 0).astype(np.float32)
    safe = np.where(diff > 0, diff, 1)
    h = np.where(v == r, (g - b) / safe,
                 np.where(v == g, 2.0 + (b - r) / safe, 4.0 + (r - g) / safe)) * 60.0
    h = np.where(diff > 0, h, 0.0)
    h = np.where(h < 0, h + 360.0, h).astype(np.float32)
    return np.stack([h, s, v], axis=-1)


def preprocess(img_u8: np.ndarray, n_channels: int = 3) -> np.ndarray:
    """uint8 [B,H,W,3] -> float32 NCHW normalised input.  Channels 0-2: ToTensor + Normalize with
    ImageNet constants (Main_Final.py:697-701).  n_channels == 4 appends the HSV saturation plane
    (build-defined 4th channel, SURVEY.md §8c), n_channels == 6 appends H/360, S, V."""
    x = img_u8.astype(np.float32) / np.float32(255.0)
    mean = np.asarray(IMAGENET_MEAN, np.float32)
    std = np.asarray(IMAGENET_STD, np.float32)
    planes = [((x[..., c] - mean[c]) / std[c]) for c in range(3)]
    if n_channels > 3:
        hsv = rgb_to_hsv(x)
        if n_channels == 4:
            planes.append(hsv[..., 1])
        elif n_channels == 6:
            planes += [hsv[..., 0] / np.float32(360.0), hsv[..., 1], hsv[..., 2]]
        else:
            raise ValueError("n_channels must be 3, 4 or 6")
    return np.stack(planes, axis=1).astype(np.float32)


# --------------------------------------------------------------------------------------
# deterministic synthetic parameters (version-proof: integer hash, no torch RNG)
# --------------------------------------------------------------------------------------
def _hash_uniform(n: int, seed: int) -> np.ndarray:
    """n float64 values in [0,1) from a splitmix64-style integer hash (pure numpy uint64)."""
    with np.errstate(over="ignore"):
        z = (np.arange(n, dtype=np.uint64) + np.uint64(seed) * np.uint64(0x9E3779B97F4A7C15))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return (z >> np.uint64(11)).astype(np.float64) / float(1 << 53)


def synthetic_state_dict(shapes: Dict[str, tuple], seed: int = 0) -> Dict[str, torch.Tensor]:
    """Deterministic state_dict for the given {key: shape}: conv weights ~ U(-b,b) with
    b = sqrt(6/fan_out) (same scale as the reference's Kaiming fan_out init, Main_Final.py:285),
    biases small, BN gamma in [0.5,1.5] with ~1/4 negative, beta small, running stats non-trivial."""
    sd = {}
    for i, (k, shp) in enumerate(shapes.items()):
        n = int(np.prod(shp)) if len(shp) else 1
        u = _hash_uniform(n, seed * 1000003 + i + 1)
        if k.endswith("num_batches_tracked"):
            sd[k] = torch.tensor(3, dtype=torch.int64)
            continue
        if k.endswith("running_mean"):
            v = (u - 0.5) * 0.2
        elif k.endswith("running_var"):
            v = 0.5 + u
        elif len(shp) == 4:
            if k.startswith("up"):            # ConvTranspose2d [Cin,Cout,2,2]
                fan = shp[0] * 1.0
            else:
                fan = shp[0] * shp[2] * shp[3] * 1.0
            v = (u * 2 - 1) * math.sqrt(6.0 / fan)
        elif k.endswith(".weight"):           # BN gamma
            v = 0.5 + u
            v = np.where(_hash_uniform(n, seed * 7919 + i + 77) < 0.25, -v, v)
        else:                                 # biases, BN beta
            v = (u - 0.5) * 0.2
        sd[k] = torch.from_numpy(np.asarray(v, dtype=np.float32).reshape(shp)).clone()
    return sd


def robust_unet_shapes(n_channels=3, n_classes=1, base=64) -> Dict[str, tuple]:
    """The 290-entry state_dict schema of RobustUNet (SURVEY.md Appendix B; Main_Final.py:229-277),
    in the reference's registration order."""
    shapes: Dict[str, tuple] = {}

    def bn(p, c):
        shapes[p + ".weight"] = (c,)
        shapes[p + ".bias"] = (c,)
        shapes[p + ".running_mean"] = (c,)
        shapes[p + ".running_var"] = (c,)
        shapes[p + ".num_batches_tracked"] = ()

    def rb(p, ci, co):
        shapes[p + ".conv1.weight"] = (co, ci, 3, 3)
        bn(p + ".bn1", co)
        shapes[p + ".conv2.weight"] = (co, co, 3, 3)
        bn(p + ".bn2", co)
        shapes[p + ".ca.fc.0.weight"] = (co // 16, co, 1, 1)
        shapes[p + ".ca.fc.2.weight"] = (co, co // 16, 1, 1)
        shapes[p + ".sa.conv1.weight"] = (1, 2, 7, 7)
        if ci != co:
            shapes[p + ".shortcut.0.weight"] = (co, ci, 1, 1)
            bn(p + ".shortcut.1", co)

    def ag(p, c, fi):
        for br in ("W_g", "W_x"):
            shapes[f"{p}.{br}.0.weight"] = (fi, c, 1, 1)
            shapes[f"{p}.{br}.0.bias"] = (fi,)
            bn(f"{p}.{br}.1", fi)
        shapes[p + ".psi.0.weight"] = (1, fi, 1, 1)
        shapes[p + ".psi.0.bias"] = (1,)
        bn(p + ".psi.1", 1)

    b = base
    rb("inc", n_channels, b)
    rb("down1.1", b, 2 * b)
    rb("down2.1", 2 * b, 4 * b)
    rb("down3.1", 4 * b, 8 * b)
    shapes["bottleneck.1.conv1.weight"] = (4 * b, 8 * b, 1, 1)
    shapes["bottleneck.1.conv1.bias"] = (4 * b,)
    for i in (2, 3, 4):
        shapes[f"bottleneck.1.conv{i}.weight"] = (4 * b, 8 * b, 3, 3)
        shapes[f"bottleneck.1.conv{i}.bias"] = (4 * b,)
    bn("bottleneck.1.bn", 16 * b)
    rb("bottleneck.2", 16 * b, 16 * b)
    ag("att4", 8 * b, 4 * b)
    ag("att3", 4 * b, 2 * b)
    ag("att2", 2 * b, b)
    ag("att1", b, b // 2)
    for k, ci, co in ((4, 16 * b, 8 * b), (3, 8 * b, 4 * b), (2, 4 * b, 2 * b), (1, 2 * b, b)):
        shapes[f"up{k}.weight"] = (ci, co, 2, 2)
        shapes[f"up{k}.bias"] = (co,)
        rb(f"dec{k}", 2 * co, co)
    shapes["outc.0.weight"] = (n_classes, b, 1, 1)
    shapes["outc.0.bias"] = (n_classes,)
    return shapes


def synthetic_inputs(batch, channels, h, w, seed=123, blobby=False):
    """Seeded synthetic images (~post-Normalize distribution) and binary water masks
    (SURVEY.md §8d).  Integer-hash based, independent of torch's RNG."""
    n = batch * channels * h * w
    u1 = _hash_uniform(n, seed)
    u2 = _hash_uniform(n, seed + 17)
    x = np.sqrt(-2.0 * np.log(np.maximum(u1, 1e-12))) * np.cos(2 * np.pi * u2)
    x = torch.from_numpy(x.astype(np.float32).reshape(batch, channels, h, w))
    if blobby:
        lh, lw = max(h // 8, 1), max(w // 8, 1)
        low = _hash_uniform(batch * lh * lw, seed + 99).reshape(batch, 1, lh, lw)
        m = F.interpolate(torch.from_numpy(low.astype(np.float32)), size=(h, w), mode="bilinear",
                          align_corners=False)
        y = (m > 0.5).float()
    else:
        y = torch.from_numpy((_hash_uniform(batch * h * w, seed + 5) > 0.5).astype(np.float32)
                             .reshape(batch, 1, h, w))
    return x, y


def synthetic_drop_masks(batch, base=64, seed=7) -> Dict[str, torch.Tensor]:
    """Dropout2d channel masks [B,C,1,1] in {0,1/(1-p)} per residual block (Main_Final.py:162,184),
    drawn from the integer hash so that oracle and CUDA path see identical masks."""
    chans = {"inc": base, "down1.1": 2 * base, "down2.1": 4 * base, "down3.1": 8 * base,
             "bottleneck.2": 16 * base, "dec4": 8 * base, "dec3": 4 * base, "dec2": 2 * base,
             "dec1": base}
    out = {}
    for i, name in enumerate(RESBLOCKS):
        p = DROPOUT_P[name]
        u = _hash_uniform(batch * chans[name], seed * 31 + i)
        m = (u >= p).astype(np.float32) / np.float32(1.0 - p)
        out[name] = torch.from_numpy(m.reshape(batch, chans[name], 1, 1))
    return out
