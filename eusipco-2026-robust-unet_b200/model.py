"""Drop-in `torch.nn.Module` surface of the Robust U-Net hot path.

`RobustUNet(n_channels=3, n_classes=1, base_channels=64)` has the constructor, parameter registration
order (hence identical initial weights under the same `torch.manual_seed`), the 290 `state_dict` keys /
shapes / dtypes and the `forward(x) -> probabilities [B,K,H,W]` contract (K = n_classes, 1 <= K <= 32: a sigmoid per
class, as the reference's `outc`) of the reference model
(Main_Final.py:226-321), so reference checkpoints load unchanged and an unmodified
`torch.optim.Adam(model.parameters())` + `loss.backward()` loop (Main_Final.py:552,573-582) trains it.

The sub-modules below own the fp32 master parameters and buffers in torch layouts; none of them executes a torch op.
`RobustUNet.forward` hands the whole graph to `engine.Engine`, which schedules the sm_100a kernels of librbunet.so; the
backward pass is one `torch.autograd.Function` whose gradients come from the same library.  `ResidualBlock`,
`AttentionGate` and `DilatedBlock` are also callable on their own like the reference's modules (NCHW fp32 at the
boundary, the same block schedules inside); `ChannelAttention` / `SpatialAttention` exist only fused into the residual
block.  There is no CPU fallback.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .engine import Engine


class _Slot(nn.Identity):
    """Parameter-free position inside an nn.Sequential (keeps the reference's child indices)."""


def _no_standalone(self, *a, **k):
    raise RuntimeError(f"{type(self).__name__} has no kernel of its own: its arithmetic is fused into the ResidualBlock "
                       "schedule (channel statistics come from the convolution epilogue, the gates are applied in the "
                       "block's output pass); call the enclosing rbunet.ResidualBlock or rbunet.RobustUNet")


def _nhwc(t: torch.Tensor):
    """NCHW float CUDA tensor -> engine View (NHWC bf16)."""
    from .ops import View
    return View(t.detach().permute(0, 2, 3, 1).contiguous().to(torch.bfloat16))


def _nchw(v) -> torch.Tensor:
    return v.dense().permute(0, 3, 1, 2).float().contiguous()


class _Block(torch.autograd.Function):
    """One block-level module (ResidualBlock / AttentionGate / DilatedBlock) called on its own, as the reference's
    modules can be (Main_Final.py:143-148,178-196,213-223): NCHW fp32 at the boundary, the engine's block schedule inside."""

    @staticmethod
    def forward(ctx, mod, n_in, save, *tensors):
        xs = tensors[:n_in]
        eng = mod.__dict__.setdefault("_engine", Engine(None))
        eng._packs.clear()                      # the fp32 masters may have changed since the last call
        eng._saving = bool(save)
        for t in xs:
            if not t.is_cuda:
                raise RuntimeError(f"rbunet.{type(mod).__name__} runs on CUDA tensors only (no CPU fallback)")
        N, C, H, W = xs[0].shape
        with torch.cuda.device(xs[0].device):
            if isinstance(mod, ResidualBlock):
                if C != mod.conv1.in_channels or C % 8:
                    raise RuntimeError(f"rbunet.ResidualBlock({mod.conv1.in_channels}, ...) got {C} input channels; standalone "
                                       "calls need a multiple of 8 (the 3/4-channel stem block runs inside rbunet.RobustUNet)")
                out, st = eng.rb_forward("block", mod, _nhwc(xs[0]), N, H, W, mod.training)
            elif isinstance(mod, DilatedBlock):
                out, st = eng.dil_forward(mod, _nhwc(xs[0]), N, H, W, mod.training)
            else:                                # AttentionGate(g, x) -> x * psi
                g, x = xs
                if g.shape != x.shape:
                    raise RuntimeError("rbunet.AttentionGate: g and x must have the same shape")
                from .ops import View
                out = View(torch.empty((N, H, W, C), dtype=torch.bfloat16, device=x.device))
                st = eng.ag_forward(mod, _nhwc(g), _nhwc(x), out, N, H, W, mod.training)
            ctx.mod, ctx.st, ctx.n_in = mod, (st if save else None), n_in
            return _nchw(out)

    @staticmethod
    def backward(ctx, dout):
        mod, st = ctx.mod, ctx.st
        if st is None:
            raise RuntimeError(f"rbunet.{type(mod).__name__}: backward needs a train-mode forward with gradients enabled "
                               "(the backward kernels implement batch-statistics BatchNorm)")
        ctx.st = None
        eng = mod._engine
        grads = {}
        with torch.cuda.device(dout.device):
            d = _nhwc(dout)
            if isinstance(mod, ResidualBlock):
                dxs = (eng.rb_backward(mod, st, d, grads, "m"),)
            elif isinstance(mod, DilatedBlock):
                dxs = (eng.dil_backward(mod, st, d, grads, "m"),)
            else:
                from .ops import View
                N, H, W, C = st["N"], st["H"], st["W"], st["C"]
                dskip = View(torch.empty((N, H, W, C), dtype=torch.bfloat16, device=dout.device))
                dg = View(torch.zeros((N, H, W, C), dtype=torch.bfloat16, device=dout.device))
                eng.ag_backward(mod, st, d, dskip, dg, grads, "m")
                dxs = (dg, dskip)
            eng.join_side(dout.device)
            outs = [_nchw(v) for v in dxs]
        for name, p in mod.named_parameters():
            g = grads.get("m." + name) if p.requires_grad else None
            outs.append(g.reshape(p.shape).clone() if g is not None else None)
        return (None, None, None, *outs)


def _standalone(self, *xs):
    params = tuple(self.parameters())
    save = self.training and torch.is_grad_enabled() and (any(p.requires_grad for p in params) or any(x.requires_grad for x in xs))
    return _Block.apply(self, len(xs), save, *xs, *params)


class ChannelAttention(nn.Module):
    """Parameters of the channel gate (Main_Final.py:82-101): shared MLP C -> C/ratio -> C, no bias."""

    def __init__(self, channels, ratio=16):
        super().__init__()
        self.fc = nn.Sequential(nn.Conv2d(channels, channels // ratio, 1, bias=False), _Slot(),
                                nn.Conv2d(channels // ratio, channels, 1, bias=False))

    forward = _no_standalone


class SpatialAttention(nn.Module):
    """Parameters of the spatial gate (Main_Final.py:104-117): 7x7 conv 2 -> 1, no bias."""

    def __init__(self, kernel_size=7):
        super().__init__()
        if kernel_size != 7:
            raise ValueError("the CUDA spatial-attention kernels are specialised for kernel_size == 7")
        self.conv1 = nn.Conv2d(2, 1, kernel_size, padding=kernel_size // 2, bias=False)

    forward = _no_standalone


class AttentionGate(nn.Module):
    """Parameters of the skip-connection gate (Main_Final.py:120-148)."""

    def __init__(self, F_g, F_l, F_int):
        super().__init__()
        self.W_g = nn.Sequential(nn.Conv2d(F_g, F_int, 1), nn.BatchNorm2d(F_int))
        self.W_x = nn.Sequential(nn.Conv2d(F_l, F_int, 1), nn.BatchNorm2d(F_int))
        self.psi = nn.Sequential(nn.Conv2d(F_int, 1, 1), nn.BatchNorm2d(1), _Slot())

    def forward(self, g, x):
        """x * sigmoid(BN(psi(relu(BN(W_g g) + BN(W_x x)))))  (Main_Final.py:143-148), standalone call."""
        return _standalone(self, g, x)


class ResidualBlock(nn.Module):
    """Parameters of one residual block (Main_Final.py:151-196)."""

    def __init__(self, in_channels, out_channels, dropout_rate=0.1):
        super().__init__()
        self.conv1 = nn.Conv2d(in_channels, out_channels, 3, padding=1, bias=False)
        self.bn1 = nn.BatchNorm2d(out_channels)
        self.conv2 = nn.Conv2d(out_channels, out_channels, 3, padding=1, bias=False)
        self.bn2 = nn.BatchNorm2d(out_channels)
        self.dropout = nn.Dropout2d(dropout_rate)          # only `.p` is read; masks are drawn by the engine
        self.ca = ChannelAttention(out_channels)
        self.sa = SpatialAttention()
        if in_channels != out_channels:
            self.shortcut = nn.Sequential(nn.Conv2d(in_channels, out_channels, 1, bias=False),
                                          nn.BatchNorm2d(out_channels))
        else:
            self.shortcut = nn.Identity()

    def forward(self, x):
        """Main_Final.py:178-196, standalone call (inside RobustUNet the engine schedules the block directly)."""
        return _standalone(self, x)


class DilatedBlock(nn.Module):
    """Parameters of the dilated bottleneck (Main_Final.py:199-223): 1x1 + three 3x3 (d = 1, 2, 4)."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        q = out_channels // 4
        self.conv1 = nn.Conv2d(in_channels, q, 1)
        for i, d in ((2, 1), (3, 2), (4, 4)):
            setattr(self, f"conv{i}", nn.Conv2d(in_channels, q, 3, padding=d, dilation=d))
        self.bn = nn.BatchNorm2d(out_channels)

    def forward(self, x):
        """Main_Final.py:213-223, standalone call."""
        return _standalone(self, x)


class _Graph(torch.autograd.Function):
    """The whole network as one autograd node: forward and backward are kernel schedules of the engine."""

    @staticmethod
    def forward(ctx, model, save, x, *params):
        probs, state = model._engine.forward(x, model.training, save)
        ctx.model = model
        ctx.state = state
        return probs

    @staticmethod
    def backward(ctx, dprobs):
        model, state = ctx.model, ctx.state
        if state is None:
            raise RuntimeError(
                f"rbunet.{type(model).__name__}: backward needs a train-mode forward with gradients enabled.  Backward "
                "through an eval-mode forward (running-statistics BatchNorm) is not implemented: the backward kernels "
                "apply the batch-statistics BatchNorm formulas of the reference's training loop and would return wrong "
                "gradients, so this raises instead")
        ctx.state = None
        if model._grad_begin_hook is not None:
            model._grad_begin_hook(model._engine)
        grads = model._engine.backward(state, dprobs, allreduce_hook=model._grad_ready_hook)
        if model._grad_transform is not None:
            grads = model._grad_transform(grads)
        out = []
        for name, p in model._named_params():
            g = grads.get(name) if p.requires_grad else None
            out.append(g.reshape(p.shape) if g is not None else None)
        return (None, None, None, *out)


class _Network(nn.Module):
    """What RobustUNet and UNet share: forward() runs the whole network as one autograd node (_Graph) on the kernel
    schedule of `engine_class(self)`."""

    def __init__(self, engine_class):
        super().__init__()
        self._engine = engine_class(self)
        self._grad_begin_hook = None      # set by parallel.DataParallel: called with the engine when a backward starts
        self._grad_ready_hook = None      # set by parallel.DataParallel: called with the names of finished grads
        self._grad_transform = None       # set by parallel.DataParallel: swaps in the all-reduced gradients

    @property
    def engine(self) -> Engine:
        return self._engine

    # The module tree is fixed after construction, so the (name, Parameter) list is cached: walking 173 parameters through
    # nn.Module.named_parameters() costs ~0.5 ms of host time per call -- time the GPU idles whenever the caller has just
    # synchronised on the previous step (`loss.item()`, Main_Final.py:584).  Anything that can replace Parameter objects
    # goes through _apply / load_state_dict / register_parameter and drops the cache.
    def _named_params(self):
        c = self.__dict__.get("_param_cache")
        if c is None:
            c = tuple(self.named_parameters())
            self.__dict__["_param_cache"] = c
        return c

    def _drop_param_cache(self):
        self.__dict__["_param_cache"] = None

    def _apply(self, fn, recurse=True):
        self._drop_param_cache()
        return super()._apply(fn, recurse)

    def load_state_dict(self, *args, **kwargs):
        self._drop_param_cache()
        return super().load_state_dict(*args, **kwargs)

    def requires_grad_(self, requires_grad: bool = True):
        self._drop_param_cache()
        return super().requires_grad_(requires_grad)

    def forward(self, x):
        params = tuple(p for _, p in self._named_params())
        if torch.is_grad_enabled() and x.requires_grad:
            raise RuntimeError(f"rbunet.{type(self).__name__} does not produce a gradient for its input (the first "
                               "layer's data gradient is never computed); detach the input")
        # grad mode is off inside autograd.Function.forward, so decide here whether to keep the backward state.  Only a
        # train-mode forward keeps it: the backward kernels implement batch-statistics BatchNorm (see _Graph.backward)
        save = self.training and torch.is_grad_enabled() and any(p.requires_grad for p in params)
        return _Graph.apply(self, save, x, *params)


class RobustUNet(_Network):
    """B200-native Robust U-Net; same public surface as Main_Final.RobustUNet (Main_Final.py:226-321)."""

    def __init__(self, n_channels=3, n_classes=1, base_channels=64):
        super().__init__(Engine)
        if not 1 <= n_classes <= 32:
            raise ValueError(f"n_classes must be in [1, 32], got {n_classes}")
        b = base_channels
        if b < 16 or b & (b - 1):
            raise ValueError("base_channels must be a power of two >= 16")
        if n_classes > 1 and b > 256:
            raise ValueError("the K-class head takes at most 256 input channels: base_channels <= 256 when n_classes > 1")
        self.inc = ResidualBlock(n_channels, b, 0.1)
        self.down1 = nn.Sequential(_Slot(), ResidualBlock(b, 2 * b, 0.1))
        self.down2 = nn.Sequential(_Slot(), ResidualBlock(2 * b, 4 * b, 0.2))
        self.down3 = nn.Sequential(_Slot(), ResidualBlock(4 * b, 8 * b, 0.2))
        self.bottleneck = nn.Sequential(_Slot(), DilatedBlock(8 * b, 16 * b), ResidualBlock(16 * b, 16 * b, 0.3))
        for k, c in ((4, 8 * b), (3, 4 * b), (2, 2 * b), (1, b)):
            setattr(self, f"att{k}", AttentionGate(c, c, c // 2))
        for k, c, p in ((4, 8 * b, 0.2), (3, 4 * b, 0.2), (2, 2 * b, 0.1), (1, b, 0.1)):
            setattr(self, f"up{k}", nn.ConvTranspose2d(2 * c, c, 2, stride=2))
            setattr(self, f"dec{k}", ResidualBlock(2 * c, c, p))
        self.outc = nn.Sequential(nn.Conv2d(b, n_classes, 1), _Slot())
        self._initialize_weights()

    def _initialize_weights(self):
        """Kaiming-normal(fan_out, relu) on every Conv2d weight, BN gamma = 1 / beta = 0; ConvTranspose2d and all
        biases keep torch's defaults (Main_Final.py:281-288)."""
        for m in self.modules():
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.ones_(m.weight)
                nn.init.zeros_(m.bias)
