"""Plain 2-class U-Net path of the reference (SURVEY.md §8f row 2): `train_water_segmentation.UNet`
(train_water_segmentation.py:209-288) / the network `predict_coastline.py:255-334` loads, its CrossEntropyLoss (:304) and
argmax accuracy / IoU (:384-388), on the same sm_100a kernels as the Robust U-Net.

`rbunet.UNet(n_channels=3, n_classes=2)` has the reference's constructor, parameter registration order, the 136
`state_dict` keys and `forward(x) -> logits [B,K,H,W]` (K = n_classes, 1 <= K <= 32); `rbunet.CrossEntropyArgmaxLoss()`
is interchangeable with `nn.CrossEntropyLoss()` on those logits (2 <= K <= 32) and also leaves the per-image argmax
confusion counts in `last_counts` (class 1 against the rest) and `last_class_counts` (every class).  Torch's own losses
work on the logits too (`nn.BCEWithLogitsLoss` at K = 1).  No CPU fallback.
"""
from __future__ import annotations

from ctypes import c_void_p

import torch
import torch.nn as nn

from . import _lib
from ._lib import call, stream_ptr
from .engine import NULL, Engine, _p, _vp
from .model import _Network, _Slot
from .ops import View, conv_gemm


class UNetEngine(Engine):
    LEVELS = ((1, 64), (2, 128), (3, 256), (4, 512))

    # ------------------------------------------------------------------ weight operands
    def _packed_weights(self):
        m = self.model
        out = [(m.enc1[0].weight, (5,)), (m.enc1[3].weight, (0, 1))]
        for name in ("enc2", "enc3", "enc4", "bottleneck", "dec4", "dec3", "dec2", "dec1"):
            seq = getattr(m, name)
            out += [(seq[0].weight, (0, 1)), (seq[3].weight, (0, 1))]
        return out + [(getattr(m, f"upconv{k}").weight, (2, 3)) for k in (4, 3, 2, 1)]

    # ------------------------------------------------------------------ conv_block (train_water_segmentation.py:251-260)
    def block_forward(self, seq, x: View, N, H, W, training, out: View = None, patches: View = None):
        dev = (x if x is not None else patches).base.device
        C = seq[0].out_channels
        HW, P = H * W, N * H * W
        if not training and not self._saving:
            # inference: both BatchNorm + ReLU pairs are folded into the convolutions' epilogues
            # (scale*acc + (shift + scale*bias), ReLU): the block is two GEMM launches
            src = x if x is not None else patches
            f1 = self.bn_eval_affine(seq[1], src, seq[0].bias)
            a1 = self.new(N, H, W, C, dev)
            if patches is not None:
                conv_gemm(N, H, W, [(patches, self._packs[(id(seq[0].weight), 5)], 1, 0, False)], C, a1,
                          scale=f1["scale"], bias=f1["shift"], relu=C, flops=2.0 * P * C * 9 * seq[0].in_channels)
            else:
                conv_gemm(N, H, W, [(x, self.pack(seq[0].weight, 0), 9, 1, False)], C, a1, scale=f1["scale"],
                          bias=f1["shift"], relu=C)
            f2 = self.bn_eval_affine(seq[4], a1, seq[3].bias)
            if out is None:
                out = self.new(N, H, W, C, dev)
            conv_gemm(N, H, W, [(a1, self.pack(seq[3].weight, 0), 9, 1, False)], C, out, scale=f2["scale"],
                      bias=f2["shift"], relu=C)
            return out, None
        y1 = self.new(N, H, W, C, dev)
        if patches is not None:
            conv_gemm(N, H, W, [(patches, self._packs[(id(seq[0].weight), 5)], 1, 0, False)], C, y1, bias=seq[0].bias,
                      flops=2.0 * P * C * 9 * seq[0].in_channels)
        else:
            conv_gemm(N, H, W, [(x, self.pack(seq[0].weight, 0), 9, 1, False)], C, y1, bias=seq[0].bias)
        bn1 = self.bn_stats(y1, N, HW, seq[1], training)
        a1 = self.new(N, H, W, C, dev)
        call("rbu_affine_act", _vp(y1), y1.ld, _vp(a1), a1.ld, P, HW, C, _p(bn1["scale"]), _p(bn1["shift"]), NULL, 1,
             stream_ptr())
        y2 = self.new(N, H, W, C, dev)
        conv_gemm(N, H, W, [(a1, self.pack(seq[3].weight, 0), 9, 1, False)], C, y2, bias=seq[3].bias)
        bn2 = self.bn_stats(y2, N, HW, seq[4], training)
        if out is None:
            out = self.new(N, H, W, C, dev)
        call("rbu_affine_act", _vp(y2), y2.ld, _vp(out), out.ld, P, HW, C, _p(bn2["scale"]), _p(bn2["shift"]), NULL, 1,
             stream_ptr())
        return out, {"x": x, "patches": patches, "y1": y1, "a1": a1, "y2": y2, "bn1": bn1, "bn2": bn2, "N": N, "H": H,
                     "W": W, "C": C}

    def _bn_relu_bwd(self, dy: View, y: View, bn, N, HW, C, dev):
        dx = self.new(N, 1, HW, C, dev)
        sums = self.f32(2 * C, device=dev)
        ws = self.bwd_ws(N, HW, C, dev)
        call("rbu_bn_bwd", _vp(dy), dy.ld, _vp(y), y.ld, _vp(dx), dx.ld, N, HW, C, _p(bn["scale"]), _p(bn["shift"]),
             _p(bn["mean"]), _p(bn["rstd"]), NULL, 1, _p(sums), _p(ws), ws.numel() * 4, stream_ptr())
        return dx, sums

    def block_backward(self, seq, s, dout: View, grads, prefix, need_dx=True):
        N, H, W, C = s["N"], s["H"], s["W"], s["C"]
        HW = H * W
        dev = dout.base.device
        dy2, sums2 = self._bn_relu_bwd(dout, s["y2"], s["bn2"], N, HW, C, dev)
        grads[prefix + ".4.bias"], grads[prefix + ".4.weight"] = sums2[:C], sums2[C:]
        grads[prefix + ".3.bias"] = torch.zeros(C, device=dev)          # a bias in front of a train-mode BN
        g2 = torch.empty_like(seq[3].weight)
        self.wgrad(N, H, W, dy2, s["a1"], 9, 1, False, g2)
        grads[prefix + ".3.weight"] = g2
        da1 = self.new(N, H, W, C, dev)
        conv_gemm(N, H, W, [(dy2, self.pack(seq[3].weight, 1), 9, 1, False)], C, da1)
        dy1, sums1 = self._bn_relu_bwd(da1, s["y1"], s["bn1"], N, HW, C, dev)
        grads[prefix + ".1.bias"], grads[prefix + ".1.weight"] = sums1[:C], sums1[C:]
        grads[prefix + ".0.bias"] = torch.zeros(C, device=dev)
        if s["patches"] is not None:
            pt = s["patches"]
            nc = seq[0].in_channels
            gst = self.f32(C, pt.C, device=dev)
            self.wgrad(N, H, W, dy1, pt, 1, 0, False, gst)
            self.join_side(dev)
            grads[prefix + ".0.weight"] = gst[:, :9 * nc].reshape(C, 3, 3, nc).permute(0, 3, 1, 2).contiguous()
            return None
        x = s["x"]
        g1 = torch.empty_like(seq[0].weight)
        self.wgrad(N, H, W, dy1, x, 9, 1, False, g1)
        grads[prefix + ".0.weight"] = g1
        if not need_dx:
            return None
        dx = self.new(N, H, W, x.C, dev)
        conv_gemm(N, H, W, [(dy1, self.pack(seq[0].weight, 1), 9, 1, False)], x.C, dx)
        return dx

    # ------------------------------------------------------------------ whole model (:262-288)
    def _network_forward(self, S, training: bool, save: bool):
        m = self.model
        N, H, W = S["N"], S["H"], S["W"]
        patches = S.pop("patches")
        dev = patches.base.device
        cats, h, w = {}, H, W
        cur = None
        for lvl, C in self.LEVELS:                     # encoder output k lives in the second half of concat buffer k
            cats[lvl] = self.new(N, h, w, 2 * C, dev)
            src = patches if lvl == 1 else cur
            out, st = self.block_forward(getattr(m, f"enc{lvl}"), None if lvl == 1 else src, N, h, w, training,
                                         out=cats[lvl].slice(C, C), patches=patches if lvl == 1 else None)
            if save:
                S[f"enc{lvl}"] = st
            h, w = h // 2, w // 2
            pooled = self.new(N, h, w, C, dev)
            call("rbu_maxpool2x2", _vp(out), out.ld, _vp(pooled), pooled.ld, N, h, w, C, stream_ptr())
            cur = pooled
            del st
        del patches
        cur, st = self.block_forward(m.bottleneck, cur, N, h, w, training)
        if save:
            S["bottleneck"] = st
        for lvl, C in reversed(self.LEVELS):
            cat = cats[lvl]
            st = self.up_forward(getattr(m, f"upconv{lvl}"), cur, N, h, w, cat.slice(0, C))
            if save:
                S[f"up{lvl}"] = st
            h, w = 2 * h, 2 * w
            cur, st = self.block_forward(getattr(m, f"dec{lvl}"), cat, N, h, w, training)
            if save:
                S[f"dec{lvl}"] = st
            else:
                cats[lvl] = None
            del st, cat
        K = m.final.out_channels
        logits = torch.empty((N, K, H, W), dtype=torch.float32, device=dev)
        if K == 2:
            call("rbu_head2_forward", _vp(cur), cur.ld, N * H * W, H * W, cur.C, _p(m.final.weight), _p(m.final.bias),
                 _p(logits), stream_ptr())
        else:
            call("rbu_headk_forward", _vp(cur), cur.ld, N * H * W, H * W, cur.C, K, _p(m.final.weight), _p(m.final.bias), 0,
                 _p(logits), NULL, stream_ptr())
        if save:
            S["cats"] = cats
            S["head_x"] = cur
        return logits

    def _network_backward(self, S, dlogits: torch.Tensor, allreduce_hook):
        m = self.model
        grads = {}
        N, H, W = S["N"], S["H"], S["W"]
        dev = dlogits.device
        hx = S["head_x"]
        d = self.new(N, H, W, hx.C, dev)
        gw, gb = torch.empty_like(m.final.weight), torch.empty_like(m.final.bias)
        K = m.final.out_channels
        if K == 2:
            nbytes = _lib.lib().rbu_head2_backward_workspace_bytes(N * H * W, hx.C)
            ws = self.ws(nbytes, dev)
            call("rbu_head2_backward", _p(dlogits.contiguous()), _vp(hx), hx.ld, _vp(d), d.ld, N * H * W, H * W, hx.C,
                 _p(m.final.weight), _p(gw), _p(gb), _p(ws), ws.numel() * 4, stream_ptr())
        else:
            ws = self.ws(_lib.lib().rbu_headk_backward_workspace_bytes(N * H * W, hx.C, K), dev)
            call("rbu_headk_backward", _p(dlogits.contiguous()), NULL, _vp(hx), hx.ld, _vp(d), d.ld, N * H * W, H * W,
                 hx.C, K, 0, _p(m.final.weight), _p(gw), _p(gb), _p(ws), ws.numel() * 4, stream_ptr())
        grads["final.weight"], grads["final.bias"] = gw, gb
        denc = {}
        for lvl, C in self.LEVELS:
            dcat = self.block_backward(getattr(m, f"dec{lvl}"), S[f"dec{lvl}"], d, grads, f"dec{lvl}")
            denc[lvl] = dcat.slice(C, C)
            d = self.up_backward(getattr(m, f"upconv{lvl}"), S[f"up{lvl}"], dcat.slice(0, C), grads, f"upconv{lvl}")
        d = self.block_backward(m.bottleneck, S["bottleneck"], d, grads, "bottleneck")
        cats = S["cats"]
        for lvl, C in reversed(self.LEVELS):
            src = cats[lvl].slice(C, C)                       # encoder output k = input of the pool below it
            ho, wo = S[f"enc{lvl}"]["H"] // 2, S[f"enc{lvl}"]["W"] // 2
            call("rbu_maxpool2x2_bwd", _vp(src), src.ld, _vp(d), d.ld, _vp(denc[lvl]), denc[lvl].ld, N, ho, wo, C, 1,
                 stream_ptr())
            d = self.block_backward(getattr(m, f"enc{lvl}"), S[f"enc{lvl}"], denc[lvl], grads, f"enc{lvl}", need_dx=lvl > 1)
        return grads


def _conv_block(ci, co):
    return nn.Sequential(nn.Conv2d(ci, co, 3, padding=1), nn.BatchNorm2d(co), _Slot(),
                         nn.Conv2d(co, co, 3, padding=1), nn.BatchNorm2d(co), _Slot())


class UNet(_Network):
    """B200-native plain U-Net; same public surface as train_water_segmentation.UNet (:209-288)."""

    def __init__(self, n_channels=3, n_classes=2):
        super().__init__(UNetEngine)
        if not 1 <= n_classes <= 32:
            raise ValueError(f"n_classes must be in [1, 32], got {n_classes}")
        self.enc1 = _conv_block(n_channels, 64)
        self.enc2 = _conv_block(64, 128)
        self.enc3 = _conv_block(128, 256)
        self.enc4 = _conv_block(256, 512)
        self.bottleneck = _conv_block(512, 1024)
        for k, c in ((4, 512), (3, 256), (2, 128), (1, 64)):
            setattr(self, f"upconv{k}", nn.ConvTranspose2d(2 * c, c, kernel_size=2, stride=2))
            setattr(self, f"dec{k}", _conv_block(2 * c, c))
        self.final = nn.Conv2d(64, n_classes, kernel_size=1)
        self.pool = _Slot()


class _CE2(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, target, mod):
        z = logits.detach().contiguous().float()
        t = target.detach().contiguous().long()
        B, HW = z.shape[0], z.shape[2] * z.shape[3]
        dev = z.device
        nbytes = _lib.lib().rbu_ce2_workspace_bytes(B, HW)
        ws = torch.empty(max(nbytes // 4, 1), dtype=torch.float32, device=dev)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        counts = torch.empty((B, 4), dtype=torch.int64, device=dev)
        call("rbu_ce2_forward", _p(z), _p(t), B, HW, _p(ws), nbytes, _p(loss), _p(counts), stream_ptr())
        mod.last_counts = counts
        ctx.save_for_backward(z, t)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, grad_out):
        z, t = ctx.saved_tensors
        B, HW = z.shape[0], z.shape[2] * z.shape[3]
        dz = torch.empty_like(z)
        g = grad_out.detach().contiguous().float().reshape(1)
        call("rbu_ce2_backward", _p(z), _p(t), B, HW, _p(g), _p(dz), stream_ptr())
        return dz, None, None


class _CEK(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, target, mod):
        z = logits.detach().contiguous().float()
        t = target.detach().contiguous().long()
        B, K, HW = z.shape[0], z.shape[1], z.shape[2] * z.shape[3]
        dev = z.device
        nbytes = _lib.lib().rbu_cek_workspace_bytes(B, HW, K)
        ws = torch.empty((nbytes + 7) // 8, dtype=torch.int64, device=dev)
        loss = torch.empty(1, dtype=torch.float32, device=dev)
        counts = torch.empty((B, K, 4), dtype=torch.int64, device=dev)
        invalid = torch.empty(1, dtype=torch.int64, device=dev)
        call("rbu_cek_forward", _p(z), _p(t), B, HW, K, _p(ws), ws.numel() * 8, _p(loss), _p(counts), _p(invalid),
             stream_ptr())
        mod.last_counts = counts[:, 1]
        mod._class_counts = counts
        mod._invalid = invalid
        ctx.save_for_backward(z, t)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, grad_out):
        z, t = ctx.saved_tensors
        B, K, HW = z.shape[0], z.shape[1], z.shape[2] * z.shape[3]
        dz = torch.empty_like(z)
        g = grad_out.detach().contiguous().float().reshape(1)
        call("rbu_cek_backward", _p(z), _p(t), B, HW, K, _p(g), _p(dz), stream_ptr())
        return dz, None, None


class CrossEntropyArgmaxLoss(nn.Module):
    """= nn.CrossEntropyLoss() on [B,K,H,W] logits (2 <= K <= 32) and [B,H,W] class indices
    (train_water_segmentation.py:304,381).  `last_counts` holds the per-image TP/FP/FN/TN of argmax == 1 vs target == 1
    (:384-388), `last_class_counts` the same [B,K,4] for every class (arg-max ties go to the lowest class index).

    At K = 2 any nonzero target is class 1, as in the two-class kernel.  For K > 2 a target outside [0, K) adds no loss
    and no counts (the loss is still divided by B*H*W); the methods that read counts to the host then raise ValueError.
    `forward` never synchronises."""

    def __init__(self):
        super().__init__()
        self.last_counts = None
        self._class_counts = None
        self._invalid = None

    def forward(self, logits, target):
        if not logits.is_cuda or not target.is_cuda:
            raise RuntimeError("rbunet.CrossEntropyArgmaxLoss runs on CUDA tensors only (no CPU fallback)")
        if logits.dim() != 4 or not 2 <= logits.shape[1] <= 32 or \
                tuple(target.shape) != (logits.shape[0],) + tuple(logits.shape[2:]):
            raise ValueError(f"expected logits [B,K,H,W] with 2 <= K <= 32 and class-index targets [B,H,W], got "
                             f"{tuple(logits.shape)} and {tuple(target.shape)}")
        if logits.shape[1] == 2:
            self._class_counts = self._invalid = None
            return _CE2.apply(logits, target, self)
        return _CEK.apply(logits, target, self)

    @property
    def last_class_counts(self):
        """int64 [B,K,4] TP/FP/FN/TN of each class (device tensor); at K = 2 class 0 is [TN, FN, FP, TP] of class 1."""
        if self._class_counts is None and self.last_counts is not None:
            c = self.last_counts
            return torch.stack([c.flip(1), c], dim=1)
        return self._class_counts

    def _host_counts(self):
        if self._invalid is not None:
            n = int(self._invalid.item())
            if n:
                raise ValueError(f"{n} target pixels are outside [0, {self._class_counts.shape[1]}): no counts for them")
        return self.last_class_counts.sum(0).cpu().tolist()

    def batch_accuracy_iou(self):
        """accuracy and IoU of class 1 over the whole batch as WaterSegmentationTrainer.validate_model computes them
        (:384-388, calculate_iou :341-358: union == 0 -> 1.0); accuracy is the pixel accuracy of the K-class arg-max."""
        cc = self._host_counts()
        tp, fp, fn, _ = [float(v) for v in cc[1]]
        union = tp + fp + fn
        return float(sum(c[0] for c in cc)) / float(sum(cc[0])), (1.0 if union == 0 else tp / union)

    def class_iou(self):
        """K IoUs over the whole batch, union == 0 -> 1.0 (calculate_iou, :341-358)."""
        return [1.0 if tp + fp + fn == 0 else float(tp) / float(tp + fp + fn) for tp, fp, fn, _ in self._host_counts()]
