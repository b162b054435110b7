"""Host-side schedule of the Robust U-Net forward / backward on the CUDA kernels (one stream, no
hidden synchronisation).  Mirrors the data flow of RobustUNet.forward (Main_Final.py:290-321) and the
backward derivation in SURVEY.md Appendix C; every tensor op is a C-ABI call into librbunet.so.

Layout: activations are NHWC bf16 (`View`s, possibly channel slices of a wider buffer so that
`torch.cat` never materialises); statistics, gates, probabilities and all parameter gradients are fp32.
"""
from __future__ import annotations

import ctypes
from collections import namedtuple
from ctypes import c_void_p

import torch
import torch.nn as nn

from . import _lib
from ._lib import WgradArgs, call, stream_ptr
from .ops import View, conv_gemm, pack_dims, pack_weight

BN_EPS = 1e-5
NULL = c_void_p(0)

# One row of rbu_pack_weights_multi's job table: _packs[key] <- src (and src2), see ops.pack_dims
PackJob = namedtuple("PackJob", "key src src2 shape Nn T K mode cout")


def _p(t):
    return c_void_p(t.data_ptr()) if t is not None else NULL


def _vp(v: View):
    return c_void_p(v.ptr)


class Workspace:
    """One scratch buffer shared by all kernels of a step (they run back to back on one stream)."""

    def __init__(self, device):
        self.device = device
        self.buf = torch.empty(1 << 22, dtype=torch.float32, device=device)

    def get(self, nbytes: int):
        if nbytes > self.buf.numel() * 4:
            self.buf = torch.empty((nbytes + 3) // 4 + (1 << 20), dtype=torch.float32, device=self.device)
        return self.buf


class Engine:
    def __init__(self, model):
        self.model = model
        self._packs = {}
        self._pack_table = None
        self._pack_srcs = None
        self._pack_plan_cache = None
        self._side_stream = None
        self._side_ws = None
        self._side_dirty = False
        self._side_keep = []          # tensors read / written by side-stream kernels the compute stream is not yet ordered behind
        self._side_mark = None        # (event, len(_side_keep)) of the previous stage boundary
        self.grad_alloc = None        # optional callable(name, shape) -> fp32 tensor to receive that parameter's gradient
                                      # (parallel.DataParallel: a slice of a flat all-reduce bucket), or None
        self._saving = False
        # Weight gradients on a side stream (see wgrad()).  The profiling tools turn this off: they need per-kernel times
        # that are not inflated by a co-running kernel.
        self.overlap_wgrad = True
        self._ws = None
        self._defer_counters = False     # whole-model forward: the 39 num_batches_tracked increments become one launch
        self._pending_counters = []
        self.drop_mask_fn = None     # optional callable(name, N, C) -> float32 [N,C] device tensor (tests)
        self.keep_logits = False     # tests: also keep the fp32 logits of the head in self.last_logits
        self.last_logits = None
        self.kernel_launches = 0

    # ------------------------------------------------------------------ helpers
    def _bump(self, bn):
        """nn.BatchNorm2d's num_batches_tracked += 1 (train mode)."""
        if self._defer_counters:
            self._pending_counters.append(bn.num_batches_tracked)
        else:
            bn.num_batches_tracked += 1

    def flush_counters(self):
        if self._pending_counters:
            torch._foreach_add_(self._pending_counters, 1)
            self._pending_counters = []
        self._defer_counters = False

    def ws(self, nbytes, device):
        if self._ws is None or self._ws.device != device:
            self._ws = Workspace(device)
        return self._ws.get(int(nbytes))

    def pack(self, param: torch.Tensor, mode: int):
        """bf16 GEMM operand of a parameter (modes 0-3).  Inside the whole-model path every operand has just been rebuilt
        by refresh_packs(); standalone block calls (tests) pack on first use."""
        key = (id(param), mode)
        ent = self._packs.get(key)
        if ent is None or ent.device != param.device:
            ent = pack_weight(param.detach().contiguous(), mode)
            self._packs[key] = ent
        return ent

    def _packed_weights(self):
        """[(weight, pack modes[, second source])]: every weight the network runs as a tensor-core GEMM operand, the stem
        convolution first.  One of the three things a network supplies (with _network_forward / _network_backward)."""
        m = self.model
        out = [(m.inc.conv1.weight, (4,), m.inc.shortcut[0].weight), (m.inc.conv2.weight, (0, 1))]
        for blk in (m.down1[1], m.down2[1], m.down3[1], m.bottleneck[2], m.dec4, m.dec3, m.dec2, m.dec1):
            out += [(blk.conv1.weight, (0, 1)), (blk.conv2.weight, (0, 1))]
            if not isinstance(blk.shortcut, nn.Identity):
                out.append((blk.shortcut[0].weight, (0, 1)))
        d = m.bottleneck[1]
        out += [(cv.weight, (0, 1)) for cv in (d.conv1, d.conv2, d.conv3, d.conv4)]
        for k in (4, 3, 2, 1):
            g = getattr(m, f"att{k}")
            out += [(g.W_g[0].weight, (0, 1)), (g.W_x[0].weight, (0, 1)), (getattr(m, f"up{k}").weight, (2, 3))]
        return out

    def _pack_plan(self):
        """[PackJob] for every operand of _packed_weights(), in that order."""
        jobs = []
        for w, modes, *src2 in self._packed_weights():
            for mode in modes:
                Nn, T, K, cout, shape = pack_dims(w, mode)
                jobs.append(PackJob((id(w), mode), w, src2[0] if src2 else None, shape, Nn, T, K, mode, cout))
        return jobs

    def refresh_packs(self):
        """Rebuild every bf16 weight operand from the fp32 masters with ONE kernel launch.  Done at the start of every
        forward: optimizers that update parameters through fused multi-tensor kernels (torch.optim.Adam(fused=True))
        do not bump tensor version counters, so staleness cannot be detected -- it is simply never allowed."""
        import numpy as np
        # the job list only depends on which Parameter objects the modules hold: rebuilt when one of them is replaced
        # (model.to(), load_state_dict(assign=True)), otherwise reused -- this runs on the launching thread before the
        # first kernel of every forward, i.e. while the GPU idles whenever the caller synchronised on the previous step
        cur = tuple(t for w, _, *src2 in self._packed_weights() for t in (w, *src2))
        srcs = self._pack_srcs
        if srcs is None or len(srcs) != len(cur) or any(a is not b for a, b in zip(srcs, cur)):
            self._pack_plan_cache = self._pack_plan()
            self._pack_srcs = cur
        plan = self._pack_plan_cache
        sig = tuple(t.data_ptr() for t in cur)
        if self._pack_table is None or self._pack_table[0] != sig:
            dev = plan[0].src.device
            dt = np.dtype([("src", "<u8"), ("src2", "<u8"), ("dst", "<u8"), ("first_block", "<i8"), ("total", "<i8"),
                           ("Nn", "<i4"), ("T", "<i4"), ("K", "<i4"), ("mode", "<i4"), ("Cout", "<i4"), ("reserved", "<i4")])
            tab = np.zeros(len(plan), dtype=dt)
            first = 0
            for i, (key, src, src2, shape, Nn, T, K, mode, cout) in enumerate(plan):
                if not (src.is_cuda and src.dtype == torch.float32 and src.is_contiguous()):
                    raise RuntimeError("rbunet: parameters must be contiguous fp32 CUDA tensors")
                dst = torch.empty(shape, dtype=torch.bfloat16, device=dev)
                self._packs[key] = dst
                total = Nn * K if mode in (4, 5) else Nn * T * K   # the stem operands' T carries the channel count
                tab[i] = (src.data_ptr(), src2.data_ptr() if src2 is not None else 0, dst.data_ptr(), first, total, Nn, T, K,
                          mode, cout, 0)
                first += int(_lib.lib().rbu_pack_job_blocks(Nn, T, K, mode))
            dev_tab = torch.from_numpy(tab.view(np.uint8).copy()).to(dev)
            self._pack_table = (sig, dev_tab, len(plan), first)
        _, dev_tab, njobs, blocks = self._pack_table
        call("rbu_pack_weights_multi", _p(dev_tab), njobs, blocks, stream_ptr())

    @staticmethod
    def new(N, H, W, C, device):
        return View(torch.empty((N, H, W, C), dtype=torch.bfloat16, device=device))

    @staticmethod
    def f32(*shape, device):
        return torch.empty(shape, dtype=torch.float32, device=device)

    @staticmethod
    def _check_bn_population(N, HW, C, training):
        """torch.nn.functional.batch_norm refuses a one-value population in training mode (the reference raises there,
        e.g. batch 1 at 16 x 16 reaches the bottleneck with 1 x 1 pixels): same error, not a silent zero variance."""
        if training and N * HW <= 1:
            raise ValueError(f"Expected more than 1 value per channel when training, got input size {[N, C, 1, 1]}")

    def bn_stats(self, x: View, N, HW, bn: nn.BatchNorm2d, training, pool=False):
        self._check_bn_population(N, HW, x.C, training)
        C, dev = x.C, x.base.device
        out = {"scale": self.f32(C, device=dev), "shift": self.f32(C, device=dev),
               "mean": self.f32(C, device=dev), "rstd": self.f32(C, device=dev)}
        if pool:
            out.update(nc_mean=self.f32(N, C, device=dev), nc_max=self.f32(N, C, device=dev),
                       nc_min=self.f32(N, C, device=dev))
        nbytes = _lib.lib().rbu_bn_stats_workspace_bytes(N, HW, C)
        ws = self.ws(nbytes, dev)
        call("rbu_bn_stats", _vp(x), x.ld, N, HW, C, int(pool), int(training), _p(bn.weight), _p(bn.bias),
             _p(bn.running_mean), _p(bn.running_var), float(bn.momentum), float(bn.eps), _p(out["scale"]),
             _p(out["shift"]), _p(out["mean"]), _p(out["rstd"]), _p(out.get("nc_mean")), _p(out.get("nc_max")),
             _p(out.get("nc_min")), _p(ws), ws.numel() * 4, stream_ptr())
        if training:
            self._bump(bn)
        return out

    @staticmethod
    def tile_stats_ok(H, W, C):
        """Whether a training forward takes this 3x3 convolution's per-image statistics (sum, sum of squares, max, min per
        half-tile) from the halo kernel's epilogue (see bn_stats_tiles): BatchNorm batch statistics and ChannelAttention's
        pooled inputs without re-reading the conv output.  Measured on B200: in the training step (batch 64, 256^2) the 18
        statistics passes it replaces cost 1.34 ms, the longer epilogues 0.4 ms and the reduction of the partials 0.35 ms.
        Since the statistics are read off the staged outputs (round 2: half the epilogue cost) they are used from 64 output
        channels up -- 64->64 at 256^2: +0.059 ms in the convolution against a 0.115-0.151 ms statistics pass, step -0.2 to
        -0.4 ms (profiles/r02_tile_stats_smem.log) -- and in training mode only (inference at 1024^2, round 2: statistics
        pass -1.9 ms, convolutions +1.7 ms -- no gain)."""
        return H >= 16 and W >= 16 and C % 32 == 0 and 64 <= C <= 2048

    def tile_stats_buf(self, N, H, W, C, device):
        return torch.empty(_lib.lib().rbu_conv_tile_stats_floats(N, H, W, C), dtype=torch.float32, device=device)

    def bn_stats_tiles(self, part, N, H, W, C, bn: nn.BatchNorm2d, training, pool=False):
        """bn_stats() without the pass over the tensor: the producing 3x3 convolution wrote per-image, per-half-tile
        partial sums / extremes of what it stored (rbu_conv_gemm tile_stats)."""
        self._check_bn_population(N, H * W, C, training)
        dev = part.device
        out = {"scale": self.f32(C, device=dev), "shift": self.f32(C, device=dev),
               "mean": self.f32(C, device=dev), "rstd": self.f32(C, device=dev)}
        if pool:
            out.update(nc_mean=self.f32(N, C, device=dev), nc_max=self.f32(N, C, device=dev),
                       nc_min=self.f32(N, C, device=dev))
        ws = self.ws(N * 2 * C * 8 + 16, dev)
        chunks = int(_lib.lib().rbu_conv_tile_stats_chunks(H, W))
        call("rbu_bn_stats_from_partials", _p(part), chunks, N, H * W, C, int(pool), int(training), _p(bn.weight),
             _p(bn.bias), _p(bn.running_mean), _p(bn.running_var), float(bn.momentum), float(bn.eps), _p(out["scale"]),
             _p(out["shift"]), _p(out["mean"]), _p(out["rstd"]), _p(out.get("nc_mean")), _p(out.get("nc_max")),
             _p(out.get("nc_min")), _p(ws), ws.numel() * 4, stream_ptr())
        if training:
            self._bump(bn)
        return out

    def bn_eval_affine(self, bn: nn.BatchNorm2d, any_view: View, conv_bias=None):
        """Eval-mode BatchNorm as a per-channel (scale, shift) pair from the running statistics, with the producing
        convolution's bias folded in: BN(acc + b) = scale*acc + (shift + scale*b).  Feeds the conv epilogue."""
        st = self._bn_eval(bn, any_view)
        if conv_bias is not None:
            st = dict(st)
            st["shift"] = torch.addcmul(st["shift"], st["scale"], conv_bias.detach())
        return st

    def _bn_eval(self, bn, any_view):
        C, dev = bn.num_features, any_view.base.device
        out = {k: self.f32(C, device=dev) for k in ("scale", "shift", "mean", "rstd")}
        call("rbu_bn_stats", _vp(any_view), any_view.ld, 1, 1, C, 0, 0, _p(bn.weight), _p(bn.bias), _p(bn.running_mean),
             _p(bn.running_var), float(bn.momentum), float(bn.eps), _p(out["scale"]), _p(out["shift"]), _p(out["mean"]),
             _p(out["rstd"]), NULL, NULL, NULL, NULL, 0, stream_ptr())
        return out

    def conv_stats_buf(self, Ncols, device):
        """Scratch for the BatchNorm partial sums a convolution's epilogue emits (training only).  Training takes the batch
        statistics of the 1x1 (shortcut, attention-gate, stem, dilated-block) convolutions from the generic kernel's staged
        epilogue instead of a separate pass over the stored tensor.  Round 1's warp-transpose reduction cost as much as the
        pass it saved (44.9 vs 45.0 ms/step); read off the staged outputs (lane = channel pair, register accumulators for
        the life of the CTA) they win (profiles/r02_bn_fuse_ab.log)."""
        return torch.empty(_lib.lib().rbu_conv_stats_floats(Ncols), dtype=torch.float32, device=device)

    def bn_from_conv(self, part, Ncols, col_off, C, count, bn: nn.BatchNorm2d, off=0, out=None):
        """Train-mode BatchNorm affine from the statistics fused into the producing convolution's epilogue.  `off`
        selects a channel range of a wider BatchNorm (DilatedBlock: four convolutions feed one BN)."""
        self._check_bn_population(count, 1, C, True)
        dev = part.device
        if out is None:
            nC = bn.num_features
            out = {k: self.f32(nC, device=dev) for k in ("scale", "shift", "mean", "rstd")}

        def sl(t):
            return c_void_p(t.data_ptr() + 4 * off)

        call("rbu_bn_finalize_partials", _p(part), Ncols, col_off, C, count, sl(bn.weight), sl(bn.bias),
             sl(bn.running_mean), sl(bn.running_var), float(bn.momentum), float(bn.eps), sl(out["scale"]), sl(out["shift"]),
             sl(out["mean"]), sl(out["rstd"]), stream_ptr())
        return out

    # -- weight gradients run on a side stream: they are tensor-pipe work with no consumer inside the backward pass,
    #    so they overlap the bandwidth-bound elementwise kernels of the data-gradient chain on the main stream
    def _side(self, device):
        if self._side_stream is None or self._side_stream.device != device:
            self._side_stream = torch.cuda.Stream(device=device)
            with torch.cuda.stream(self._side_stream):      # the caching allocator ties a block to the stream it was
                self._side_ws = Workspace(device)           # allocated under: this buffer is only ever used on the side stream
        return self._side_stream

    def join_side(self, device):
        """Make the current stream wait for every weight-gradient kernel issued so far."""
        if self._side_stream is not None and self._side_dirty:
            torch.cuda.current_stream(device).wait_stream(self._side_stream)
            self._side_dirty = False
        self._side_keep.clear()      # operands may be recycled now: later main-stream work is ordered after the join
        self._side_mark = None

    def stage_boundary(self, device):
        """End of a backward stage.  Returns an event behind the weight-gradient kernels enqueued so far (None if there
        are none) -- the data-parallel all-reduce of the stage waits for it on the communication stream.  Operand
        memory is released with a lag of ONE stage: the compute stream waits for the event of the PREVIOUS boundary
        (normally long complete: the side stream trails by a few kernels) and drops the references held up to there.
        Release points are fixed in program order, so the caching allocator sees the same request sequence every step
        (releasing on event polls made cudaMalloc calls appear in random steps)."""
        if self._side_stream is None or not self._side_dirty:
            return None
        ev = torch.cuda.Event()
        ev.record(self._side_stream)
        if self._side_mark is not None:
            prev_ev, count = self._side_mark
            torch.cuda.current_stream(device).wait_event(prev_ev)
            del self._side_keep[:count]
        self._side_mark = (ev, len(self._side_keep))
        return ev

    def gbuf(self, name, like: torch.Tensor):
        """Destination of a parameter gradient: the data-parallel bucket slice when one is registered, else fresh memory."""
        if self.grad_alloc is not None:
            t = self.grad_alloc(name, like.shape)
            if t is not None:
                return t
        return torch.empty_like(like)

    def wgrad(self, N, H, W, a: View, b: View, taps, dil, gather, out: torch.Tensor):
        if self.overlap_wgrad:
            dev = out.device
            main = torch.cuda.current_stream(dev)
            side = self._side(dev)
            side.wait_stream(main)                       # operands were produced on the main stream
            # operands were allocated under the main stream: they stay referenced until a stage boundary has ordered the
            # compute stream behind this kernel (stage_boundary / join_side), so their memory cannot be recycled early
            self._side_keep.extend((a.base, b.base, out))
            with torch.cuda.stream(side):
                self._wgrad(N, H, W, a, b, taps, dil, gather, out, self._side_ws)
            self._side_dirty = True
        else:
            self._wgrad(N, H, W, a, b, taps, dil, gather, out, None)

    def _wgrad(self, N, H, W, a: View, b: View, taps, dil, gather, out: torch.Tensor, wspace):
        args = WgradArgs()
        args.N, args.H, args.W = N, H, W
        args.a, args.a_ld, args.Ca = a.ptr, a.ld, a.C
        args.b, args.b_ld, args.Cb = b.ptr, b.ld, b.C
        args.taps, args.dil, args.gather = taps, dil, int(gather)
        args.out, args.accumulate = out.data_ptr(), 0
        nbytes = _lib.lib().rbu_wgrad_workspace_bytes(ctypes.byref(args))
        ws = wspace.get(int(nbytes)) if wspace is not None else self.ws(nbytes, out.device)
        call("rbu_wgrad_gemm", ctypes.byref(args), _p(ws), ws.numel() * 4, stream_ptr(), tag="wgrad_gemm",
             flops=2.0 * N * H * W * a.C * b.C * taps,
             label=f"wgrad {N}x{H}x{W} {a.C}x{b.C} t{taps}{'g' if gather else ''}d{dil}")

    def bwd_ws(self, N, HW, C, device):
        return self.ws(_lib.lib().rbu_bwd_workspace_bytes(N, HW, max(C, 32)), device)

    def drop_mask(self, name, N, C, p, device):
        if self.drop_mask_fn is not None:
            m = self.drop_mask_fn(name, N, C)
            return m.to(device=device, dtype=torch.float32).reshape(N, C).contiguous()
        # nn.Dropout2d (Main_Final.py:162,184): per-(n,c) Bernoulli(1-p) / (1-p)
        return torch.empty((N, C), dtype=torch.float32, device=device).bernoulli_(1.0 - p).div_(1.0 - p)

    # ------------------------------------------------------------------ ResidualBlock (Main_Final.py:178-196)
    def rb_forward(self, name, blk, x: View, N, H, W, training, out: View = None, stem_patches: View = None):
        dev = x.base.device if x is not None else stem_patches.base.device
        C = blk.conv2.out_channels
        HW, P = H * W, N * H * W
        proj = not isinstance(blk.shortcut, nn.Identity)
        s = {"name": name, "x": x, "N": N, "H": H, "W": W, "C": C, "proj": proj, "patches": stem_patches}
        bns = bn1 = None
        if stem_patches is not None:
            y12 = self.new(N, H, W, 2 * C, dev)
            st12 = self.conv_stats_buf(2 * C, dev) if training else None
            conv_gemm(N, H, W, [(stem_patches, self._packs[(id(blk.conv1.weight), 4)], 1, 0, False)], 2 * C, y12,
                      flops=2.0 * N * H * W * C * 10 * blk.conv1.in_channels, stats=st12)
            y1, ys = y12.slice(0, C), y12.slice(C, C)
            if training:
                bn1 = self.bn_from_conv(st12, 2 * C, 0, C, P, blk.bn1)
                bns = self.bn_from_conv(st12, 2 * C, C, C, P, blk.shortcut[1])
                self._bump(blk.bn1)
                self._bump(blk.shortcut[1])
        else:
            folded = not training and not self._saving   # inference: BN1 + ReLU ride in conv1's epilogue, no y1
            y1 = None if folded else self.new(N, H, W, C, dev)
            # bn1 needs the batch statistics only (no per-image pooling): per-CTA register accumulators in the convolution's
            # epilogue (no per-tile exchange, no second stage over tiles)
            st1 = self.conv_stats_buf(C, dev) if training else None
            if folded:
                bn1 = self.bn_eval_affine(blk.bn1, x)
                a1 = self.new(N, H, W, C, dev)
                conv_gemm(N, H, W, [(x, self.pack(blk.conv1.weight, 0), 9, 1, False)], C, a1, scale=bn1["scale"],
                          bias=bn1["shift"], relu=C)
            else:
                conv_gemm(N, H, W, [(x, self.pack(blk.conv1.weight, 0), 9, 1, False)], C, y1, stats=st1)
            if st1 is not None:
                bn1 = self.bn_from_conv(st1, C, 0, C, P, blk.bn1)
                self._bump(blk.bn1)
            ys = None
            if proj:
                ys = self.new(N, H, W, C, dev)
                sts = self.conv_stats_buf(C, dev) if training else None
                conv_gemm(N, H, W, [(x, self.pack(blk.shortcut[0].weight, 0), 1, 0, False)], C, ys, stats=sts)
                if training:
                    bns = self.bn_from_conv(sts, C, 0, C, P, blk.shortcut[1])
                    self._bump(blk.shortcut[1])
        if y1 is not None and bn1 is None:
            bn1 = self.bn_stats(y1, N, HW, blk.bn1, training)
        drop = self.drop_mask(name, N, C, blk.dropout.p, dev) if training and blk.dropout.p > 0 else None
        if y1 is not None:
            a1 = self.new(N, H, W, C, dev)
            call("rbu_affine_act", _vp(y1), y1.ld, _vp(a1), a1.ld, P, HW, C, _p(bn1["scale"]), _p(bn1["shift"]), _p(drop), 1,
                 stream_ptr())
        y2 = self.new(N, H, W, C, dev)
        ts2 = self.tile_stats_buf(N, H, W, C, dev) if training and self.tile_stats_ok(H, W, C) else None
        conv_gemm(N, H, W, [(a1, self.pack(blk.conv2.weight, 0), 9, 1, False)], C, y2, tile_stats=ts2)
        if ts2 is not None:
            bn2 = self.bn_stats_tiles(ts2, N, H, W, C, blk.bn2, training, pool=True)
        else:
            bn2 = self.bn_stats(y2, N, HW, blk.bn2, training, pool=True)
        Ch = blk.ca.fc[0].out_channels
        ca = {k: self.f32(N, C, device=dev) for k in ("g", "A2g", "B2g", "u_avg", "u_max", "tv")}
        ca["nc_arg"] = torch.empty((N, C), dtype=torch.int32, device=dev)
        ca["h_avg"], ca["h_max"] = self.f32(N, Ch, device=dev), self.f32(N, Ch, device=dev)
        call("rbu_ca_gate", _p(bn2["nc_mean"]), _p(bn2["nc_max"]), _p(bn2["nc_min"]), _p(bn2["scale"]), _p(bn2["shift"]),
             _p(blk.ca.fc[0].weight), _p(blk.ca.fc[2].weight), N, C, Ch, _p(ca["g"]), _p(ca["A2g"]), _p(ca["B2g"]),
             _p(ca["u_avg"]), _p(ca["u_max"]), _p(ca["h_avg"]), _p(ca["h_max"]), _p(ca["tv"]), _p(ca["nc_arg"]), stream_ptr())
        sa_s = self.f32(P, 2, device=dev)
        need_arg = training or self._saving      # the arg-max bookkeeping only feeds the backward pass
        amax_c = torch.empty(P, dtype=torch.int32, device=dev) if need_arg else None
        call("rbu_sa_reduce", _vp(y2), y2.ld, P, HW, C, _p(ca["A2g"]), _p(ca["B2g"]), _p(ca["tv"]), _p(ca["nc_arg"]),
             _p(sa_s), _p(amax_c) if need_arg else NULL, stream_ptr())
        gs = self.f32(P, device=dev)
        call("rbu_sa_gate", _p(sa_s), N, H, W, _p(blk.sa.conv1.weight), _p(gs), stream_ptr())
        if proj and bns is None:
            bns = self.bn_stats(ys, N, HW, blk.shortcut[1], training)
        if out is None:
            out = self.new(N, H, W, C, dev)
        rsrc = ys if proj else x
        call("rbu_rb_out", _vp(y2), y2.ld, _vp(rsrc), rsrc.ld, _vp(out), out.ld, P, HW, C, _p(ca["A2g"]), _p(ca["B2g"]),
             _p(gs), _p(bns["scale"]) if proj else NULL, _p(bns["shift"]) if proj else NULL, stream_ptr())
        s.update(y1=y1, ys=ys, a1=a1, y2=y2, out=out, bn1=bn1, bn2=bn2, bns=bns, drop=drop, ca=ca, sa_s=sa_s,
                 amax_c=amax_c, gs=gs, Ch=Ch)
        return out, s

    def rb_backward(self, blk, s, dout: View, grads: dict, prefix: str, need_dx=True, dx: View = None):
        """dout may be overwritten (it becomes de).  Returns the View holding d(input)."""
        N, H, W, C = s["N"], s["H"], s["W"], s["C"]
        HW, P = H * W, N * H * W
        dev = dout.base.device
        proj, ys, y2, ca, bn2, bns = s["proj"], s["ys"], s["y2"], s["ca"], s["bn2"], s["bns"]
        ws = self.bwd_ws(N, HW, C, dev)
        wsb = ws.numel() * 4
        st = stream_ptr()
        de = dout
        dG = self.f32(P, device=dev)
        sraw = self.f32(2 * C, device=dev) if proj else None
        call("rbu_rb_bwd1", _vp(dout), dout.ld, _vp(s["out"]), s["out"].ld, _vp(y2), y2.ld, _vp(de), de.ld,
             _vp(ys) if proj else NULL, ys.ld if proj else 0, N, HW, C, _p(ca["A2g"]), _p(ca["B2g"]), _p(dG), _p(sraw),
             _p(ws), wsb, st)
        ds = self.f32(P, 2, device=dev)
        dk7 = self.f32(98, device=dev)
        call("rbu_sa_bwd", _p(dG), _p(s["gs"]), _p(s["sa_s"]), N, H, W, _p(blk.sa.conv1.weight), _p(ds), _p(dk7), _p(ws),
             wsb, st)
        grads[prefix + ".sa.conv1.weight"] = dk7.view(1, 2, 7, 7)
        D = torch.empty((N, 2, C), dtype=torch.float64, device=dev)
        call("rbu_rb_bwd2", _vp(de), de.ld, _vp(y2), y2.ld, N, HW, C, _p(s["gs"]), _p(ds), _p(s["amax_c"]), _p(D), _p(ws),
             wsb, st)
        Ch = s["Ch"]
        scratch = self.f32(3 * N * C + 2 * N * Ch, device=dev)
        dV1, dV2 = self.f32(Ch, C, 1, 1, device=dev), self.f32(C, Ch, 1, 1, device=dev)
        sums2 = self.f32(2 * C, device=dev)
        coef = self.f32((3 * N + 1) * C, device=dev)
        sums_s = self.f32(2 * C, device=dev) if proj else None
        coef_s = self.f32(3 * C, device=dev) if proj else None
        call("rbu_rb_mid", _p(D), _p(ca["g"]), _p(ca["h_avg"]), _p(ca["h_max"]), _p(ca["u_avg"]), _p(ca["u_max"]),
             _p(bn2["nc_mean"]), _p(ca["tv"]), _p(blk.ca.fc[0].weight), _p(blk.ca.fc[2].weight), _p(bn2["scale"]),
             _p(bn2["shift"]), _p(bn2["mean"]), _p(bn2["rstd"]), N, HW, C, Ch, _p(scratch), _p(dV1), _p(dV2), _p(sums2),
             _p(coef), _p(sraw), _p(bns["scale"]) if proj else NULL, _p(bns["mean"]) if proj else NULL,
             _p(bns["rstd"]) if proj else NULL, _p(sums_s), _p(coef_s), st)
        grads[prefix + ".ca.fc.0.weight"] = dV1
        grads[prefix + ".ca.fc.2.weight"] = dV2
        grads[prefix + ".bn2.bias"], grads[prefix + ".bn2.weight"] = sums2[:C], sums2[C:]
        # dy1 | dys share one buffer so the stem's fused GEMM sees them as one operand
        dy12 = self.new(N, H, W, 2 * C if proj else C, dev)
        dy1 = dy12.slice(0, C)
        dys = dy12.slice(C, C) if proj else None
        dy2 = self.new(N, H, W, C, dev)
        call("rbu_rb_bwd3", _vp(de), de.ld, _vp(y2), y2.ld, _vp(dy2), dy2.ld, _vp(ys) if proj else NULL,
             ys.ld if proj else 0, _vp(dys) if proj else NULL, dys.ld if proj else 0, N, HW, C, _p(s["gs"]), _p(ds),
             _p(s["amax_c"]), _p(ca["nc_arg"]), _p(coef), _p(coef_s), st)
        if proj:
            grads[prefix + ".shortcut.1.bias"], grads[prefix + ".shortcut.1.weight"] = sums_s[:C], sums_s[C:]
        # conv2
        a1 = s["a1"]
        da1 = self.new(N, H, W, C, dev)
        conv_gemm(N, H, W, [(dy2, self.pack(blk.conv2.weight, 1), 9, 1, False)], C, da1)
        gW2 = self.gbuf(prefix + ".conv2.weight", blk.conv2.weight)
        self.wgrad(N, H, W, dy2, a1, 9, 1, False, gW2)
        grads[prefix + ".conv2.weight"] = gW2
        # bn1 + relu + dropout
        bn1 = s["bn1"]
        sums1 = self.f32(2 * C, device=dev)
        call("rbu_bn_bwd", _vp(da1), da1.ld, _vp(s["y1"]), s["y1"].ld, _vp(dy1), dy1.ld, N, HW, C, _p(bn1["scale"]),
             _p(bn1["shift"]), _p(bn1["mean"]), _p(bn1["rstd"]), _p(s["drop"]), 1, _p(sums1), _p(ws), wsb, st)
        grads[prefix + ".bn1.bias"], grads[prefix + ".bn1.weight"] = sums1[:C], sums1[C:]
        # conv1 / shortcut
        if s["patches"] is not None:
            pt = s["patches"]
            nc = blk.conv1.in_channels
            gst = self.f32(2 * C, pt.C, device=dev)
            self.wgrad(N, H, W, dy12, pt, 1, 0, False, gst)
            self.join_side(dev)                    # the slicing below runs on the main stream
            grads[prefix + ".conv1.weight"] = gst[:C, :9 * nc].reshape(C, 3, 3, nc).permute(0, 3, 1, 2).contiguous()
            grads[prefix + ".shortcut.0.weight"] = gst[C:, 4 * nc:5 * nc].reshape(C, nc, 1, 1).contiguous()
            return None
        x = s["x"]
        # The data gradient goes first: two persistent tensor-core kernels cannot share the SMs, so a weight-gradient kernel
        # that grabbed them would stall the main stream; enqueued after the data gradient it runs beside the bandwidth-bound
        # kernels of the next block instead.
        if need_dx:
            if dx is None:
                dx = self.new(N, H, W, x.C, dev)
            segs = [(dy1, self.pack(blk.conv1.weight, 1), 9, 1, False)]
            if proj:
                segs.append((dys, self.pack(blk.shortcut[0].weight, 1), 1, 0, False))
            conv_gemm(N, H, W, segs, x.C, dx, addend=None if proj else de)
        gW1 = self.gbuf(prefix + ".conv1.weight", blk.conv1.weight)
        self.wgrad(N, H, W, dy1, x, 9, 1, False, gW1)
        grads[prefix + ".conv1.weight"] = gW1
        if proj:
            gWs = self.gbuf(prefix + ".shortcut.0.weight", blk.shortcut[0].weight)
            self.wgrad(N, H, W, dys, x, 1, 0, False, gWs)
            grads[prefix + ".shortcut.0.weight"] = gWs
        return dx if need_dx else None

    # ------------------------------------------------------------------ AttentionGate (Main_Final.py:143-148)
    def ag_forward(self, gate, g: View, skip: View, out: View, N, H, W, training):
        dev = g.base.device
        C, F = skip.C, gate.W_g[0].out_channels
        HW, P = H * W, N * H * W
        yg, yx = self.new(N, H, W, F, dev), self.new(N, H, W, F, dev)
        stg = self.conv_stats_buf(F, dev) if training else None
        stx = self.conv_stats_buf(F, dev) if training else None
        conv_gemm(N, H, W, [(g, self.pack(gate.W_g[0].weight, 0), 1, 0, False)], F, yg, bias=gate.W_g[0].bias, stats=stg)
        conv_gemm(N, H, W, [(skip, self.pack(gate.W_x[0].weight, 0), 1, 0, False)], F, yx, bias=gate.W_x[0].bias, stats=stx)
        if training:
            bg = self.bn_from_conv(stg, F, 0, F, P, gate.W_g[1])
            bx = self.bn_from_conv(stx, F, 0, F, P, gate.W_x[1])
            self._bump(gate.W_g[1])
            self._bump(gate.W_x[1])
        else:
            bg = self.bn_stats(yg, N, HW, gate.W_g[1], training)
            bx = self.bn_stats(yx, N, HW, gate.W_x[1], training)
        self._check_bn_population(P, 1, 1, training)
        q0 = self.f32(P, device=dev)
        stats = self.f32(4, device=dev)
        nblk = _lib.lib().rbu_ag_psi_blocks(P, F)
        part = self.ws(nblk * 8, dev)
        bnp = gate.psi[1]
        call("rbu_ag_psi", _vp(yg), yg.ld, _vp(yx), yx.ld, P, F, _p(bg["scale"]), _p(bg["shift"]), _p(bx["scale"]),
             _p(bx["shift"]), _p(gate.psi[0].weight), _p(gate.psi[0].bias), int(training), _p(bnp.weight), _p(bnp.bias),
             _p(bnp.running_mean), _p(bnp.running_var), float(bnp.momentum), float(bnp.eps), _p(q0), _p(stats), _p(part),
             stream_ptr())
        if training:
            self._bump(bnp)
        psi = self.f32(P, device=dev)
        call("rbu_ag_apply", _vp(skip), skip.ld, _vp(out), out.ld, P, C, _p(q0), _p(stats), _p(psi), stream_ptr())
        return {"g": g, "skip": skip, "yg": yg, "yx": yx, "bg": bg, "bx": bx, "q0": q0, "stats": stats, "psi": psi,
                "N": N, "H": H, "W": W, "C": C, "F": F}

    def ag_backward(self, gate, s, da: View, dskip: View, dgup: View, grads: dict, prefix: str):
        N, H, W, C, F = s["N"], s["H"], s["W"], s["C"], s["F"]
        HW, P = H * W, N * H * W
        dev = da.base.device
        ws = self.bwd_ws(N, HW, max(C, F), dev)
        dyg, dyx = self.new(N, H, W, F, dev), self.new(N, H, W, F, dev)
        dq = self.f32(P, device=dev)
        sums_psi, sums_f = self.f32(2, device=dev), self.f32(4 * F, device=dev)
        bg, bx = s["bg"], s["bx"]
        call("rbu_ag_bwd", _vp(da), da.ld, _vp(s["skip"]), s["skip"].ld, _vp(dskip), dskip.ld, _vp(s["yg"]), s["yg"].ld,
             _vp(s["yx"]), s["yx"].ld, _vp(dyg), dyg.ld, _vp(dyx), dyx.ld, N, HW, C, F, _p(s["psi"]), _p(s["q0"]),
             _p(s["stats"]), _p(bg["scale"]), _p(bg["shift"]), _p(bx["scale"]), _p(bx["shift"]), _p(bg["mean"]),
             _p(bg["rstd"]), _p(bx["mean"]), _p(bx["rstd"]), _p(gate.psi[0].weight), _p(dq), _p(sums_psi), _p(sums_f),
             _p(ws), ws.numel() * 4, stream_ptr())
        grads[prefix + ".psi.0.weight"] = sums_f[0:F].reshape(1, F, 1, 1)
        grads[prefix + ".psi.0.bias"] = torch.zeros(1, device=dev)          # BN removes the mean: exactly zero
        grads[prefix + ".psi.1.bias"], grads[prefix + ".psi.1.weight"] = sums_psi[0:1], sums_psi[1:2]
        grads[prefix + ".W_g.1.bias"], grads[prefix + ".W_g.1.weight"] = sums_f[F:2 * F], sums_f[2 * F:3 * F]
        # d(beta) of the two BatchNorms is the same sum (both see dt); every parameter still gets its OWN storage: autograd
        # adopts these tensors as .grad, and in-place users (clip_grad_norm_, gradient accumulation) must not see aliases
        grads[prefix + ".W_x.1.bias"], grads[prefix + ".W_x.1.weight"] = sums_f[F:2 * F].clone(), sums_f[3 * F:4 * F]
        grads[prefix + ".W_g.0.bias"] = torch.zeros(F, device=dev)
        grads[prefix + ".W_x.0.bias"] = torch.zeros(F, device=dev)
        conv_gemm(N, H, W, [(dyg, self.pack(gate.W_g[0].weight, 1), 1, 0, False)], C, dgup, addend=dgup)
        conv_gemm(N, H, W, [(dyx, self.pack(gate.W_x[0].weight, 1), 1, 0, False)], C, dskip, addend=dskip)
        gWg = self.gbuf(prefix + ".W_g.0.weight", gate.W_g[0].weight)
        gWx = self.gbuf(prefix + ".W_x.0.weight", gate.W_x[0].weight)
        self.wgrad(N, H, W, dyg, s["g"], 1, 0, False, gWg)        # after the data gradients (see rb_backward)
        self.wgrad(N, H, W, dyx, s["skip"], 1, 0, False, gWx)
        grads[prefix + ".W_g.0.weight"], grads[prefix + ".W_x.0.weight"] = gWg, gWx

    # ------------------------------------------------------------------ DilatedBlock (Main_Final.py:213-223)
    def dil_forward(self, blk, x: View, N, H, W, training):
        dev = x.base.device
        Cq = blk.conv1.out_channels
        C = 4 * Cq
        HW, P = H * W, N * H * W
        ycat = self.new(N, H, W, C, dev)
        convs = (blk.conv1, blk.conv2, blk.conv3, blk.conv4)
        bn = None
        for i, cv in enumerate(convs):
            taps = 1 if i == 0 else 9
            sti = self.conv_stats_buf(Cq, dev) if training else None
            conv_gemm(N, H, W, [(x, self.pack(cv.weight, 0), taps, cv.dilation[0], False)], Cq, ycat.slice(i * Cq, Cq),
                      bias=cv.bias, stats=sti)
            if training:
                bn = self.bn_from_conv(sti, Cq, 0, Cq, P, blk.bn, off=i * Cq, out=bn)
        if training:
            self._bump(blk.bn)
        else:
            bn = self.bn_stats(ycat, N, HW, blk.bn, training)
        out = self.new(N, H, W, C, dev)
        call("rbu_affine_act", _vp(ycat), ycat.ld, _vp(out), out.ld, P, HW, C, _p(bn["scale"]), _p(bn["shift"]), NULL, 1,
             stream_ptr())
        return out, {"x": x, "ycat": ycat, "bn": bn, "N": N, "H": H, "W": W, "C": C, "Cq": Cq}

    def dil_backward(self, blk, s, dout: View, grads: dict, prefix: str):
        N, H, W, C, Cq = s["N"], s["H"], s["W"], s["C"], s["Cq"]
        HW = H * W
        dev = dout.base.device
        x, ycat, bn = s["x"], s["ycat"], s["bn"]
        ws = self.bwd_ws(N, HW, C, dev)
        dycat = self.new(N, H, W, C, dev)
        sums = self.f32(2 * C, device=dev)
        call("rbu_bn_bwd", _vp(dout), dout.ld, _vp(ycat), ycat.ld, _vp(dycat), dycat.ld, N, HW, C, _p(bn["scale"]),
             _p(bn["shift"]), _p(bn["mean"]), _p(bn["rstd"]), NULL, 1, _p(sums), _p(ws), ws.numel() * 4, stream_ptr())
        grads[prefix + ".bn.bias"], grads[prefix + ".bn.weight"] = sums[:C], sums[C:]
        convs = (blk.conv1, blk.conv2, blk.conv3, blk.conv4)
        segs = []
        for i, cv in enumerate(convs):
            taps = 1 if i == 0 else 9
            segs.append((dycat.slice(i * Cq, Cq), self.pack(cv.weight, 1), taps, cv.dilation[0], False))
        dx = self.new(N, H, W, x.C, dev)
        conv_gemm(N, H, W, segs[:2], x.C, dx)
        conv_gemm(N, H, W, segs[2:], x.C, dx, addend=dx)
        for i, cv in enumerate(convs):          # weight gradients after the data gradients (see rb_backward)
            g = self.gbuf(f"{prefix}.conv{i + 1}.weight", cv.weight)
            self.wgrad(N, H, W, segs[i][0], x, segs[i][2], cv.dilation[0], False, g)
            grads[f"{prefix}.conv{i + 1}.weight"] = g
            grads[f"{prefix}.conv{i + 1}.bias"] = torch.zeros(Cq, device=dev)   # a bias before a train-mode BN
        return dx

    # ------------------------------------------------------------------ ConvTranspose2d(2, stride 2) up-sampling
    def up_forward(self, up, x: View, N, H, W, out: View):
        """up(x) for x [N,H,W,Cin], scattered into out [N,2H,2W,Cout] (a channel slice of the decoder's concat buffer).
        Returns the state up_backward needs."""
        C = up.out_channels
        conv_gemm(N, H, W, [(x, self.pack(up.weight, 2), 1, 0, False)], 4 * C, out, scatter=True, Cout=C, bias=up.bias)
        return {"x": x, "N": N, "H": H, "W": W}

    def up_backward(self, up, s, dout: View, grads: dict, prefix: str):
        """Puts up's bias and weight gradients into grads; returns d(x)."""
        N, H, W, x = s["N"], s["H"], s["W"], s["x"]
        C, dev = dout.C, dout.base.device
        gb = torch.empty_like(up.bias)
        ws = self.bwd_ws(N, 4 * H * W, C, dev)
        call("rbu_chan_sum", _vp(dout), dout.ld, 4 * N * H * W, C, _p(gb), _p(ws), ws.numel() * 4, stream_ptr())
        dx = self.new(N, H, W, x.C, dev)
        conv_gemm(N, H, W, [(dout, self.pack(up.weight, 3), 4, 0, True)], x.C, dx)
        gw = self.gbuf(prefix + ".weight", up.weight)
        self.wgrad(N, H, W, x, dout, 4, 0, True, gw)             # after the data gradient (see rb_backward)
        grads[prefix + ".bias"], grads[prefix + ".weight"] = gb, gw
        return dx

    # ------------------------------------------------------------------ whole network
    def forward(self, x: torch.Tensor, training: bool, save: bool):
        """The whole network on an NCHW input: (output [N,K,H,W] fp32, the state backward() needs if `save`, else None).
        What differs between networks is _packed_weights and _network_forward."""
        name = f"rbunet.{type(self.model).__name__}"
        if not x.is_cuda:
            raise RuntimeError(f"{name} runs on CUDA tensors only (no CPU fallback)")
        N, nc, H, W = x.shape
        if H % 16 or W % 16:
            raise RuntimeError(f"{name}: input H,W must be multiples of 16, got {H}x{W}")
        self._pending_counters = []
        self._defer_counters = True
        try:
            with torch.cuda.device(x.device):        # stream_ptr() and the library's per-device state follow the tensors
                x = x.contiguous().float()
                self.refresh_packs()
                stem = self._pack_plan_cache[0]    # _packed_weights() lists the stem convolution first
                if nc != stem.T:
                    raise RuntimeError(f"{name}: expected {stem.T} input channels, got {nc}")
                self._saving = bool(save)
                patches = self.new(N, H, W, stem.K, x.device)
                call("rbu_stem_im2col", _p(x), N, nc, H, W, stem.K, _vp(patches), stream_ptr())
                # handed over inside S so that the body holds the only reference: inference frees the patches as soon as
                # the first block has run
                S = {"N": N, "H": H, "W": W, "patches": patches}
                del patches
                out = self._network_forward(S, training, save)
                return out, (S if save else None)
        finally:
            self.flush_counters()

    def backward(self, S, dout: torch.Tensor, allreduce_hook=None):
        """Returns {param_name: fp32 gradient} from the state of forward(..., save=True) and d(output).  A network may call
        `allreduce_hook(names, grads, event)` as soon as the gradients of a top-level child are complete (reverse
        execution order) so data-parallel buckets can overlap.  The network-specific part is _network_backward."""
        with torch.cuda.device(dout.device):
            grads = self._network_backward(S, dout, allreduce_hook)
            self.join_side(dout.device)
        return grads

    def _network_forward(self, S, training: bool, save: bool):
        """RobustUNet.forward (Main_Final.py:290-321) from the stem patches (S["patches"], taken out of S) to the
        probabilities; fills S with the backward state when `save`."""
        m = self.model
        N, H, W = S["N"], S["H"], S["W"]
        patches = S.pop("patches")
        dev = patches.base.device
        enc = []

        def keep(key, st):          # inference: intermediates are released as soon as their block has run
            if save:
                S[key] = st

        cur, st = self.rb_forward("inc", m.inc, None, N, H, W, training, stem_patches=patches)
        keep("inc", st)
        del st, patches
        enc.append(cur)
        h, w = H, W
        pools = []
        for i, name in enumerate(("down1", "down2", "down3")):
            h, w = h // 2, w // 2
            pooled = self.new(N, h, w, cur.C, dev)
            call("rbu_maxpool2x2", _vp(cur), cur.ld, _vp(pooled), pooled.ld, N, h, w, cur.C, stream_ptr())
            if save:
                pools.append(pooled)
            cur, st = self.rb_forward(name + ".1", getattr(m, name)[1], pooled, N, h, w, training)
            keep(name, st)
            del st, pooled
            enc.append(cur)
        h, w = h // 2, w // 2
        pooled = self.new(N, h, w, cur.C, dev)
        call("rbu_maxpool2x2", _vp(cur), cur.ld, _vp(pooled), pooled.ld, N, h, w, cur.C, stream_ptr())
        if save:
            pools.append(pooled)
        x5a, st = self.dil_forward(m.bottleneck[1], pooled, N, h, w, training)
        keep("dil", st)
        cur, st = self.rb_forward("bottleneck.2", m.bottleneck[2], x5a, N, h, w, training)
        keep("bott", st)
        del st, pooled, x5a
        S["pools"] = pools
        if save:
            S["enc"] = enc
        for k in (4, 3, 2, 1):
            up = getattr(m, f"up{k}")
            C = up.out_channels
            skip = enc[k - 1]
            cat = self.new(N, 2 * h, 2 * w, 2 * C, dev)
            keep(f"up{k}", self.up_forward(up, cur, N, h, w, cat.slice(C, C)))
            h, w = 2 * h, 2 * w
            st = self.ag_forward(getattr(m, f"att{k}"), cat.slice(C, C), skip, cat.slice(0, C), N, h, w, training)
            keep(f"att{k}", st)
            if not save:
                enc[k - 1] = None            # the skip tensor has been consumed
            cur, st = self.rb_forward(f"dec{k}", getattr(m, f"dec{k}"), cat, N, h, w, training)
            keep(f"dec{k}", st)
            del st, cat, skip
        P = N * H * W
        hc = m.outc[0]
        K = hc.out_channels
        probs = torch.empty((N, K, H, W), dtype=torch.float32, device=dev)
        logits = torch.empty_like(probs) if self.keep_logits else None
        if K == 1:
            call("rbu_head_forward", _vp(cur), cur.ld, P, cur.C, _p(hc.weight), _p(hc.bias), _p(probs), _p(logits),
                 stream_ptr())
        else:                                      # a sigmoid per class, as the reference's outc
            call("rbu_headk_forward", _vp(cur), cur.ld, P, H * W, cur.C, K, _p(hc.weight), _p(hc.bias), 1, _p(probs),
                 _p(logits), stream_ptr())
        self.last_logits = logits
        S["head_x"] = cur
        S["probs"] = probs
        return probs

    def _network_backward(self, S, dprobs: torch.Tensor, allreduce_hook):
        m = self.model
        grads = {}
        N, H, W = S["N"], S["H"], S["W"]
        dev = dprobs.device
        P = N * H * W
        hx = S["head_x"]
        hc = m.outc[0]
        d = self.new(N, H, W, hx.C, dev)
        gw, gb = torch.empty_like(hc.weight), torch.empty_like(hc.bias)
        K = hc.out_channels
        if K == 1:
            ws = self.bwd_ws(N, H * W, hx.C, dev)
            call("rbu_head_backward", _p(dprobs.contiguous()), _p(S["probs"]), _vp(hx), hx.ld, _vp(d), d.ld, P, hx.C,
                 _p(hc.weight), _p(gw), _p(gb), _p(ws), ws.numel() * 4, stream_ptr())
        else:
            ws = self.ws(_lib.lib().rbu_headk_backward_workspace_bytes(P, hx.C, K), dev)
            call("rbu_headk_backward", _p(dprobs.contiguous()), _p(S["probs"]), _vp(hx), hx.ld, _vp(d), d.ld, P, H * W,
                 hx.C, K, 1, _p(hc.weight), _p(gw), _p(gb), _p(ws), ws.numel() * 4, stream_ptr())
        grads["outc.0.weight"], grads["outc.0.bias"] = gw, gb

        def done(*prefixes):
            # the hook gets an event behind the stage's weight-gradient kernels (side stream): the all-reduce waits for it
            # on the communication stream; the compute stream only ever waits for the PREVIOUS stage's event
            ev = self.stage_boundary(dev)
            if allreduce_hook is not None:
                allreduce_hook([k for k in grads if any(k == p or k.startswith(p + ".") for p in prefixes)], grads, ev)

        done("outc")
        enc = S["enc"]
        denc = [None] * 4
        for k in (1, 2, 3, 4):
            sd = S[f"dec{k}"]
            dcat = self.rb_backward(getattr(m, f"dec{k}"), sd, d, grads, f"dec{k}")
            C = sd["C"]
            denc[k - 1] = self.new(N, sd["H"], sd["W"], C, dev)
            self.ag_backward(getattr(m, f"att{k}"), S[f"att{k}"], dcat.slice(0, C), denc[k - 1], dcat.slice(C, C), grads,
                             f"att{k}")
            d = self.up_backward(getattr(m, f"up{k}"), S[f"up{k}"], dcat.slice(C, C), grads, f"up{k}")
            done(f"dec{k}", f"att{k}", f"up{k}")
        d = self.rb_backward(m.bottleneck[2], S["bott"], d, grads, "bottleneck.2")
        d = self.dil_backward(m.bottleneck[1], S["dil"], d, grads, "bottleneck.1")
        done("bottleneck")
        pools = S["pools"]
        for lvl in (3, 2, 1, 0):
            src = enc[lvl]                      # x_{lvl+1}: input of the pool
            pl = pools[lvl]
            n_, ho, wo, _ = pl.base.shape
            call("rbu_maxpool2x2_bwd", _vp(src), src.ld, _vp(d), d.ld, _vp(denc[lvl]), denc[lvl].ld, N, ho, wo, src.C, 1,
                 stream_ptr())
            if lvl > 0:
                name = f"down{lvl}"
                d = self.rb_backward(getattr(m, name)[1], S[name], denc[lvl], grads, name + ".1")
                done(name)
            else:
                self.rb_backward(m.inc, S["inc"], denc[0], grads, "inc", need_dx=False)
                done("inc")
        return grads
