#!/usr/bin/env python
"""bench.py -- Robust U-Net hot-path benchmark (contract: see DESIGN.md "Measurement").

  python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's sm_100a path
  python bench.py --impl reference [--gpus N] [--steps K] ...    # the UNMODIFIED reference on the host cores
  python bench.py ... --dump-outputs DIR                         # also save the last timed step's outputs as .npy

Own arm.  A step is one pass of the training hot path over one synthetic batch: forward, BCE loss (+ confusion
counts), backward, (N > 1: bucketed gradient all-reduce overlapped with the backward) and the Adam update of
Main_Final.py:552,573-582.  The headline workload at every N is BASELINE.json configs[1] per GPU -- bf16 storage / fp32
accumulate, batch 64 at 256x256, 3 channels (weak scaling).  `value` is images/s with the batch resident in HBM; `e2e` is
the same loop fed from pinned host memory (H2D of images + masks and D2H of the loss inside the timed region) through
the public nn.Module API.  The other BASELINE configurations ride in the same JSON line under `extra`:
  extra.c3        configs[2]: 512x512, GLOBAL batch 256 split over the N GPUs (strong scaling; N = 1 runs the two
                  128-image halves back to back with gradient accumulation -- the arithmetic of the N = 2 job)
  extra.c5        configs[4]: 4-channel input, BCE + Dice, 512x512, batch 32 per GPU (weak scaling)
  extra.c4_infer  configs[3]: eval forward on 1024x1024 tiles, batch 32 per GPU, thresholded masks + TP/FP/FN/TN
  torch_eager_same_gpu (N = 1)  the reference arithmetic through eager PyTorch / cuDNN on the same GPU (informational)

Reference arm.  `Main_Final.RobustUNet` itself -- the reference's eight scripts are copied verbatim into the
git-ignored baseline/_ref/ by __graft_entry__.build() when /root/reference is present -- trained with the loop of
Main_Final.py:573-582 (fp32, torch CPU kernels, all host threads) on a bounded sample of the workload.  Only when
baseline/_ref/ is absent does it fall back to the bit-identical oracle port (`kind: "port"`).
"""
import argparse
import json
import os
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

TRAIN_GFLOP_PER_IMG_256 = 323.6      # SURVEY.md §2.2 / BASELINE.md: fwd + dgrad + wgrad conv FLOPs per image at 256x256
FWD_GFLOP_PER_IMG_256 = 107.9
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
DUMP_MAX_ELEMS = 1 << 22     # per --dump-outputs array (16 MiB in float32): at most three arrays of this size per workload


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p["bf16_tflops_sustained"],
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs.  NVML is initialised once, up
    front (nvmlInit inside the timed region stalls kernel launches for ~100 ms)."""
    _nv = None
    _handles = {}

    @classmethod
    def prepare(cls, index):
        try:
            import pynvml as nv
            if cls._nv is None:
                nv.nvmlInit()
                cls._nv = nv
            if index not in cls._handles:
                cls._handles[index] = nv.nvmlDeviceGetHandleByIndex(index)
        except Exception as e:
            cls._nv = None
            cls._err = f"nvml_unavailable:{type(e).__name__}"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        self.recording = False     # the thread polls from before the warm-up (first NVML queries are slow and hold a
                                   # driver lock); samples and throttle reasons count only inside the timed region

    def run(self):
        nv = ClockSampler._nv
        if nv is None:
            self.reasons.add(getattr(ClockSampler, "_err", "nvml_unavailable"))
            return
        try:
            h = ClockSampler._handles[self.index]
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksEventReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap"}
            while not self.stop_flag:
                mhz = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                if self.recording:
                    self.samples.append(mhz)
                    for bit, nm in names.items():
                        if r & bit:
                            self.reasons.add(nm)
                time.sleep(0.05)
        except Exception as e:   # NVML trouble: report that instead of failing the bench
            self.reasons.add(f"nvml_error:{type(e).__name__}")

    def result(self):
        self.stop_flag = True
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------------ own arm
class Env:
    """Process-wide state of the own arm: rank, device, process group, L2-flush buffer."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from rbunet import _lib
        self.args = args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        _lib.check(_lib.lib().rbu_device_check(), "rbu_device_check")
        ClockSampler.prepare(self.local)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)     # > 126 MB L2
        self.flush.zero_()     # first use loads torch's fill-kernel module (lazy CUDA module loading: 200-400 ms)

    def barrier(self):
        import torch
        import torch.distributed as dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        import torch
        import torch.distributed as dist
        if self.world > 1:
            t = torch.tensor([ms], device=self.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms


class Case:
    """One workload: model + criterion + optimizer + resident and pinned synthetic inputs for this rank.
    kind: "train" | "infer" | "unet".  `accum` > 1 splits the per-rank batch into that many micro-batches whose
    gradients accumulate before the optimizer step (each micro-batch has its own BatchNorm statistics, exactly like
    one rank of a data-parallel job)."""

    def __init__(self, env, kind, nc, S, B, w_dice=0.0, accum=1, ddp=True):
        import torch
        import rbunet
        from tools.synthetic import synthetic_batch
        self.env, self.kind, self.nc, self.S, self.B, self.w_dice, self.accum = env, kind, nc, S, B, w_dice, accum
        dev = env.dev
        torch.manual_seed(0)
        unet = kind == "unet"
        self.model = (rbunet.UNet(nc, 2) if unet else rbunet.RobustUNet(nc, 1, 64)).to(dev)
        self.crit = rbunet.CrossEntropyArgmaxLoss() if unet else rbunet.RobustBCEDiceLoss(1.0, w_dice)
        self.net = self.model
        self.opt = None
        if kind == "infer":
            self.model.eval()
        else:
            self.model.train()
            if env.world > 1 and not unet and ddp:
                self.net = rbunet.DataParallel(self.model)
            self.opt = rbunet.FusedAdam(self.model.parameters(), lr=1e-4, weight_decay=1e-4)   # = Adam of Main_Final.py:552
        x_cpu, y_cpu = synthetic_batch(B, nc, S, S, seed=123 + env.rank)
        if unet:
            y_cpu = y_cpu[:, 0].long()           # class-index masks, nn.CrossEntropyLoss style
        self.x_pin, self.y_pin = x_cpu.pin_memory(), y_cpu.pin_memory()
        self.x_dev, self.y_dev = x_cpu.to(dev), y_cpu.to(dev)
        # e2e: double-buffered input staging -- the H2D copy of step i+1 runs on a copy stream while step i computes (what
        # a pin_memory DataLoader + prefetcher does); every step's inputs are copied from pinned host memory inside the
        # timed region and every step ends with a D2H read of its result
        self.stage = [(torch.empty_like(self.x_dev), torch.empty_like(self.y_dev)) for _ in range(2)]
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.staged = {"i": 0, "ev": None}
        self.keep_last = False     # --dump-outputs: step() keeps its network output and result for outputs()
        self.last = self.dumped = None

    # -- one step on device-resident inputs
    def step(self, x=None, y=None):
        import torch
        import rbunet
        x = self.x_dev if x is None else x
        y = self.y_dev if y is None else y
        if self.kind == "infer":
            with torch.no_grad():
                p = self.net(x)
                counts = rbunet.confusion_counts(p, y)
            if self.keep_last:
                self.last = (p, counts)
            return counts
        self.opt.zero_grad(set_to_none=True)
        if self.accum == 1:
            p = self.net(x)
            loss = self.crit(p, y)
            loss.backward()
            if self.keep_last:
                self.last = (p, loss)
        else:
            mb = self.B // self.accum
            loss = None
            for i in range(self.accum):
                li = self.crit(self.net(x[i * mb:(i + 1) * mb]), y[i * mb:(i + 1) * mb]) / self.accum
                li.backward()
                loss = li.detach() if loss is None else loss + li.detach()
        self.opt.step()
        return loss

    def _stage_next(self):
        import torch
        xs, ys = self.stage[self.staged["i"] & 1]
        self.copy_stream.wait_stream(torch.cuda.current_stream(self.env.dev))   # the buffer's previous consumer is enqueued
        with torch.cuda.stream(self.copy_stream):
            xs.copy_(self.x_pin, non_blocking=True)
            ys.copy_(self.y_pin, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
        self.staged["ev"] = ev
        return xs, ys

    def step_e2e(self):
        import torch
        st = self.staged
        if st["ev"] is None:
            st["cur"] = self._stage_next()                           # first step: nothing to overlap with
        xs, ys = st["cur"]
        torch.cuda.current_stream(self.env.dev).wait_event(st["ev"])
        st["i"] += 1
        st["cur"] = self._stage_next()                               # next step's inputs, behind this step's compute
        out = self.step(xs, ys)
        return out.cpu() if self.kind == "infer" else out.item()

    def outputs(self):
        """{name: float32/float64 numpy array} of what the last step() computed: the network output, the loss and
        confusion counts and, for training, the gradients, the updated parameters and the BatchNorm running statistics.
        An array above DUMP_MAX_ELEMS elements is reduced to a fixed seeded sample of its flattened values (the same
        positions in every run of the same workload)."""
        import numpy as np
        import torch
        torch.cuda.synchronize(self.env.dev)
        p, res = self.last

        def host(t):
            t = t.detach()
            if t.numel() > DUMP_MAX_ELEMS:
                idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_MAX_ELEMS, replace=False))
                t = t.flatten()[torch.from_numpy(idx).to(t.device)]
            t = t.double() if t.dtype in (torch.int64, torch.float64) else t.float()    # integers exact in float64
            return t.cpu().numpy()

        out = {"logits" if self.kind == "unet" else "probs": host(p)}
        if self.kind == "infer":
            out["confusion_counts"] = host(res)
            return out
        out["loss"] = host(res)
        out["confusion_counts"] = host(self.crit.last_counts)
        params = [q for q in self.model.parameters() if q.grad is not None]
        out["grads"] = host(torch.cat([q.grad.flatten() for q in params]))
        out["params"] = host(torch.cat([q.detach().flatten() for q in params]))
        stats = [b.flatten() for n, b in self.model.named_buffers() if n.endswith(("running_mean", "running_var"))]
        if stats:
            out["bn_running_stats"] = host(torch.cat(stats))
        return out

    def io_bytes(self):
        h2d = self.x_pin.numel() * 4 + self.y_pin.numel() * self.y_pin.element_size()
        d2h = (self.B * 4 * 8) if self.kind == "infer" else 4
        return h2d, d2h

    def timed(self, fn, steps, warmup):
        import torch
        from rbunet import _lib
        env = self.env
        sampler = ClockSampler(env.local)
        sampler.start()
        for _ in range(warmup):
            fn()
        env.barrier()
        sampler.recording = True
        l0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        marks = []
        for _ in range(steps):
            if not env.args.no_flush:
                env.flush.zero_()               # L2 flush between timed iterations
            fn()
            m = torch.cuda.Event(enable_timing=True)
            m.record()
            marks.append(m)
        e1.record()
        env.barrier()
        ms = e0.elapsed_time(e1)
        prev, per = e0, []
        for m in marks:                     # per-step durations (diagnostic: outliers show up here, not in the mean)
            per.append(round(prev.elapsed_time(m), 2))
            prev = m
        launches = _lib.launch_count() - l0
        clocks = sampler.result()
        return env.max_over_ranks(ms), launches, clocks, per

    def measure(self, steps, warmup, e2e=True):
        """{value, ms_per_step, e2e, ...} of this case (images/s over all ranks, max-over-ranks device time)."""
        ms, launches, clocks, per = self.timed(self.step, steps, warmup)
        if self.keep_last:
            self.dumped = self.outputs()         # before the e2e steps below train the model further
            self.keep_last, self.last = False, None
        imgs = self.B * self.env.world * steps
        rec = {"value": round(imgs / (ms / 1e3), 2), "unit": "img/s", "ms_per_step": round(ms / steps, 3), "steps": steps,
               "warmup": warmup, "gpu_launches": int(launches), "clocks": clocks, "ms_each_step": per}
        if e2e:
            ms2, _, _, _ = self.timed(self.step_e2e, steps, max(1, warmup // 2))
            h2d, d2h = self.io_bytes()
            rec["e2e"] = {"value": round(imgs / (ms2 / 1e3), 2), "unit": "img/s", "h2d_bytes_per_step": h2d,
                          "d2h_bytes_per_step": d2h, "ms_per_step": round(ms2 / steps, 3)}
        return rec

    def close(self):
        import torch
        self.model = self.net = self.opt = self.crit = None
        self.x_dev = self.y_dev = self.stage = self.x_pin = self.y_pin = None
        self.staged = {"i": 0, "ev": None}
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


def _workload_name(kind, nc, S, B, w_dice=0.0):
    if kind == "infer":
        return f"Robust U-Net inference {S}x{S} batch {B}/GPU, thresholded masks + TP/FP/FN/TN counts"
    if kind == "unet":
        return f"plain 2-class U-Net (train_water_segmentation.py) training step (fwd+CE+bwd+Adam), batch {B}/GPU at {S}x{S}"
    loss = "BCE" if not w_dice else f"BCE+{w_dice}*Dice"
    return f"Robust U-Net bf16 training step (fwd+{loss}+bwd+Adam), batch {B}/GPU at {S}x{S}, {nc} channels, base 64"


def profile_step(case, peaks, detail_path=None):
    """Per-kernel-class device times of one extra step (CUDA events around every C-ABI call on the launching stream).
    The weight-gradient side stream is switched off for this pass: kernels running concurrently slow each other down
    and the per-kernel times (the roofline numerators) would be those of the mix, not of the kernel."""
    from rbunet import _lib
    prof = _lib.Profiler()
    eng = getattr(case.model, "engine", None)
    was_overlap = getattr(eng, "overlap_wgrad", None)
    if was_overlap:
        eng.overlap_wgrad = False
    _lib.PROFILER = prof
    try:
        case.step()
    finally:
        _lib.PROFILER = None
        if was_overlap:
            eng.overlap_wgrad = True
    summ = prof.summary()
    if detail_path and case.env.rank == 0:
        with open(detail_path, "w") as f:
            for lab, ms_, fl, nb_ in prof.detail():
                f.write(f"{ms_:8.3f} ms  {fl / ms_ / 1e9 if fl and ms_ else 0:8.1f} TF/s  "
                        f"{nb_ / ms_ / 1e6 if nb_ and ms_ else 0:8.0f} GB/s  {lab}\n")
    gemm = {k: v for k, v in summ.items() if v["flops"] > 0}
    gemm_ms = sum(v["ms"] for v in gemm.values())
    gemm_flops = sum(v["flops"] for v in gemm.values())
    lib_ms = sum(v["ms"] for v in summ.values())
    top = max(gemm.items(), key=lambda kv: kv[1]["ms"])
    peak_tf = peaks["bf16_tflops_sustained"]
    roof = {"bound": "tensor", "kernel": top[0], "achieved": top[1]["flops"] / top[1]["ms"] / 1e9 if top[1]["ms"] else None,
            "peak": peak_tf, "unit": "TFLOP/s", "frac": None, "traffic": None, "peak_source": peaks["source"] + " (sustained)",
            "launches_per_step": top[1]["calls"], "avg_launch_ms": top[1]["ms"] / max(1, top[1]["calls"]),
            "share_of_step": top[1]["ms"] / lib_ms if lib_ms else None,
            "all_gemm_tflops": gemm_flops / gemm_ms / 1e9 if gemm_ms else None,
            "all_gemm_frac": gemm_flops / gemm_ms / 1e9 / peak_tf if gemm_ms else None}
    if roof["achieved"]:
        roof["frac"] = roof["achieved"] / peak_tf
    # DRAM bytes per launch of the dominant kernel from the committed ncu capture (dram__bytes_read/write.sum) of the same
    # step (tools/ncu_traffic.py -> profiles/traffic.json)
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tr = json.load(f).get(top[0])
        if tr and case.kind == "train" and case.B == 64 and case.S == 256:
            roof["traffic"] = tr["dram_bytes_per_launch"]
            roof["traffic_source"] = tr["source"]
            roof["algorithmic_bytes_per_launch"] = top[1]["bytes"] / max(1, top[1]["calls"]) if top[1].get("bytes") else None
    except (OSError, ValueError):
        pass
    classes = {k: {"calls": v["calls"], "ms": round(v["ms"], 3), "share": round(v["ms"] / lib_ms, 4) if lib_ms else None,
                   **({"tflops": round(v["flops"] / v["ms"] / 1e9, 1),
                       "tensor_frac": round(v["flops"] / v["ms"] / 1e9 / peak_tf, 3)} if v["flops"] and v["ms"] else {}),
                   **({"gbps": round(v["bytes"] / v["ms"] / 1e6, 0),
                       "hbm_frac": round(v["bytes"] / v["ms"] / 1e6 / peaks["hbm_gbs"], 3)} if v["bytes"] and v["ms"] else {})}
               for k, v in sorted(summ.items(), key=lambda kv: -kv[1]["ms"])}
    ew_ms = sum(v["ms"] for v in summ.values() if v["bytes"] and not v["flops"])
    ew_bytes = sum(v["bytes"] for v in summ.values() if v["bytes"] and not v["flops"])
    hbm = {"ms": round(ew_ms, 3), "gbps": round(ew_bytes / ew_ms / 1e6, 0) if ew_ms else None,
           "hbm_frac": round(ew_bytes / ew_ms / 1e6 / peaks["hbm_gbs"], 3) if ew_ms else None,
           "peak": peaks["hbm_gbs"], "peak_source": peaks["source"],
           "note": "all bandwidth-bound kernels of one step: algorithmic bytes / summed CUDA-event time"}
    return roof, classes, hbm


def run_extra(env, name, kind, nc, S, B, steps, warmup, w_dice=0.0, accum=1, scaling="weak", note=None):
    """One BASELINE configuration as a sub-record; a failure (e.g. out of memory) is reported, never raised."""
    import torch
    case = None
    try:
        case = Case(env, kind, nc, S, B, w_dice=w_dice, accum=accum)
        rec = case.measure(steps, warmup)
        rec.update({"metric": "infer_images_per_sec" if kind == "infer" else "train_images_per_sec", "scaling": scaling,
                    "n_gpus": env.world,
                    "config": {"workload": _workload_name(kind, nc, S, B // accum if accum > 1 else B, w_dice),
                               "global_batch": B * env.world, "per_gpu_batch": B, "image": [nc, S, S],
                               "parallelism": f"dp{env.world}"}})
        if accum > 1:
            rec["config"]["micro_batches"] = accum
        if note:
            rec["config"]["note"] = note
        rec["peak_mem_gb"] = round(torch.cuda.max_memory_allocated(env.dev) / 2 ** 30, 1)
    except Exception as e:          # noqa: BLE001  (report, do not fail the headline line)
        rec = {"error": f"{type(e).__name__}: {str(e)[:160]}"}
    if case is not None:
        case.close()
    torch.cuda.reset_peak_memory_stats(env.dev)
    ok = torch.tensor([0 if "error" in rec else 1], device=env.dev)
    if env.world > 1:
        import torch.distributed as dist
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if not ok.item() and "error" not in rec:
        rec = {"error": "another rank failed"}
    return rec


def write_outputs(path, arrays):
    """--dump-outputs: one DIR/<name>.npy per array of Case.outputs()."""
    import numpy as np
    assert sum(a.nbytes for a in arrays.values()) <= 64 * 10 ** 6, {k: a.nbytes for k, a in arrays.items()}
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_ours(args):
    import torch
    import torch.distributed as dist
    env = Env(args)
    world, rank, dev = env.world, env.rank, env.dev
    kind = args.workload
    infer, unet = kind == "infer", kind == "unet"
    B = args.batch or (32 if infer else 64)
    S = args.size or (1024 if infer else 256)
    nc = args.channels
    peaks = load_peaks()
    peak_tf = peaks["bf16_tflops_sustained"]

    torch.cuda.reset_peak_memory_stats(dev)
    case = Case(env, kind, nc, S, B, w_dice=args.w_dice)
    case.keep_last = bool(args.dump_outputs)
    main = case.measure(args.steps, args.warmup)
    dumped = case.dumped
    mem_per_px = torch.cuda.max_memory_allocated(dev) / (B * S * S)        # bytes per input pixel of the per-GPU batch
    # host time to ENQUEUE one step (no synchronisation inside): how close the launching thread is to being the bottleneck
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    case.step()
    host_enqueue_ms = (time.perf_counter() - t0) * 1e3
    torch.cuda.synchronize()
    roof, classes, hbm = profile_step(case, peaks, args.detail)
    ddp = None
    if world > 1 and kind == "train":
        # what the data-parallel machinery costs: the same step without the gradient hooks (no buckets, no all-reduce),
        # timed after everything else because the replicas diverge from here on
        hook, tr, bg = case.model._grad_ready_hook, case.model._grad_transform, case.model._grad_begin_hook
        case.model._grad_ready_hook = case.model._grad_transform = case.model._grad_begin_hook = None
        case.net = case.model
        ms_local, _, _, _ = case.timed(case.step, min(args.steps, 5), 2)
        case.model._grad_ready_hook, case.model._grad_transform, case.model._grad_begin_hook = hook, tr, bg
        local_ms = ms_local / min(args.steps, 5)
        ddp = {"local_step_ms": round(local_ms, 3), "ddp_step_ms": main["ms_per_step"],
               "exposed_comm_ms_per_step": round(main["ms_per_step"] - local_ms, 3),
               "allreduce_bytes_per_step": 4 * sum(p.numel() for p in case.model.parameters()),
               "note": "max over ranks; exposed = data-parallel step minus the same step without gradient hooks"}
    case.close()

    gflop_img = (FWD_GFLOP_PER_IMG_256 if infer else (289.2 if unet else TRAIN_GFLOP_PER_IMG_256)) * (S * S) / (256 * 256)
    out = {"metric": "infer_images_per_sec" if infer else "train_images_per_sec", "value": main["value"], "unit": "img/s",
           "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"],
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
           "config": {"workload": _workload_name(kind, nc, S, B, args.w_dice),
                      "global_batch": B * world, "image": [nc, S, S], "parallelism": f"dp{world}",
                      "l2": "256 MiB flush buffer written between timed steps; per-step activations exceed L2",
                      "weights": "reference init (seed 0), random",
                      "optimizer": "rbunet.FusedAdam (= torch.optim.Adam, coupled L2) lr 1e-4 wd 1e-4"},
           "clocks": main["clocks"], "ms_each_step": main["ms_each_step"], "host_enqueue_ms_per_step": round(host_enqueue_ms, 2),
           "e2e": main["e2e"], "gpu_launches": main["gpu_launches"],
           "model_tflops": round(main["value"] * gflop_img / 1e3, 1),
           "model_frac_of_sustained_peak": round(main["value"] * gflop_img / 1e3 / peak_tf, 4),
           "roofline": roof, "hbm_kernels": hbm, "kernel_classes": classes}
    if ddp:
        out["ddp"] = ddp

    if kind == "train" and not args.no_extras and nc == 3 and S == 256 and B == 64:
        xs, xw = min(args.steps, 5), 3
        extra = {}
        # configs[2]: global batch 256 at 512x512 split over the GPUs.  One GPU cannot hold 256 images' activations
        # (~0.9 GB per image): N = 1 runs two 128-image micro-batches (= the arithmetic of the N = 2 job).
        per_gpu = 256 // world
        accum = 1
        total_mem = torch.cuda.get_device_properties(dev).total_memory
        while per_gpu // accum > 1 and mem_per_px * (per_gpu // accum) * 512 * 512 > 0.8 * total_mem:
            accum *= 2             # same decision on every rank: it depends on shapes and the measured bytes per pixel
        if world > 1:
            t = torch.tensor([accum], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            accum = int(t.item())
        extra["c3"] = run_extra(env, "c3", "train", 3, 512, per_gpu, min(xs, 3), 2, accum=accum, scaling="strong",
                                note="BASELINE configs[2]: global batch 256 at 512x512 (strong scaling over N)")
        extra["c5"] = run_extra(env, "c5", "train", 4, 512, 32, xs, xw, w_dice=0.5, scaling="weak",
                                note="BASELINE configs[4]: 4-channel input, BCE + 0.5*Dice, batch 32 per GPU")
        extra["c4_infer"] = run_extra(env, "c4_infer", "infer", 3, 1024, 32, xs, 6, scaling="weak",
                                      note="BASELINE configs[3]: independent replicas, no collective")
        out["extra"] = extra

    if rank == 0:
        if dumped is not None:
            write_outputs(args.dump_outputs, dumped)
        if world == 1 and not args.no_cpu_baseline and not unet:
            out["cpu_baseline"] = cpu_reference(infer, nc, S, budget_s=20.0)
        if world == 1 and not args.no_eager_baseline and kind == "train":
            torch.cuda.empty_cache()
            out["torch_eager_same_gpu"] = eager_cuda_leg(nc, B, S, dev)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out


# ------------------------------------------------------------------------------------------------ CPU reference
def load_reference_module():
    """Main_Final from baseline/_ref/ (verbatim copies of the reference scripts made by __graft_entry__.build()), with
    the plotting / GDAL imports it does not need on this path stubbed (Main_Final.py:19).  None when absent."""
    if not os.path.isfile(os.path.join(REF_DIR, "Main_Final.py")):
        return None
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.patches", "matplotlib.colors", "matplotlib.gridspec"):
        if name not in sys.modules:
            mod = types.ModuleType(name)
            mod.__path__ = []
            sys.modules[name] = mod
    sys.modules["matplotlib"].rcParams = {}
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    try:
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):       # the module prints "Using device: ..." at import
            import Main_Final
        return Main_Final
    except Exception:        # noqa: BLE001  (a missing optional dependency on this box: fall back to the port)
        return None


def cpu_reference(infer, nc, S, budget_s, steps=None, warmup=1, batch=None):
    """Times the reference's own CPU implementation (fp32 torch CPU kernels, all host threads) on a bounded sample of
    the workload: the unmodified Main_Final.RobustUNet from baseline/_ref/ with the training loop body of
    Main_Final.py:573-582 (kind "reference"), else the bit-identical oracle port (kind "port")."""
    import torch
    from tools.synthetic import synthetic_batch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    MF = load_reference_module()
    if MF is not None:
        kind = "reference"
        torch.manual_seed(0)
        model = MF.RobustUNet(n_channels=nc, n_classes=1)
        criterion = torch.nn.BCELoss()                                                       # Main_Final.py:551
        optimizer = None if infer else torch.optim.Adam(model.parameters(), lr=1e-4, weight_decay=1e-4)   # :552
        evaluator = MF.ModelEvaluator(torch.device("cpu"))
        model.eval() if infer else model.train()

        def one(bs):
            x, y = synthetic_batch(bs, nc, S, S, seed=5)
            t0 = time.perf_counter()
            if infer:
                with torch.no_grad():                                                        # Main_Final.py:639-657
                    outputs = model(x)
                    for i in range(outputs.shape[0]):
                        evaluator.calculate_metrics(outputs[i, 0], y[i, 0])
            else:
                optimizer.zero_grad()                                                        # Main_Final.py:576-582
                outputs = model(x)
                loss = criterion(outputs, y)
                loss.backward()
                optimizer.step()
            return time.perf_counter() - t0
    else:
        kind = "port"
        from oracle import robust_unet_ref as R
        sd = R.synthetic_state_dict(R.robust_unet_shapes(nc, 1, 64), seed=0)
        names = [k for k, v in sd.items() if v.is_floating_point() and "running" not in k]
        params = [sd[n].requires_grad_(not infer) for n in names]
        opt = None if infer else torch.optim.Adam(params, lr=1e-4, weight_decay=1e-4)
        masks = R.synthetic_drop_masks(64, 64, seed=7)

        def one(bs):
            x, y = synthetic_batch(bs, nc, S, S, seed=5)
            t0 = time.perf_counter()
            if infer:
                with torch.no_grad():
                    p = R.robust_unet_forward(sd, x, training=False)
                R.confusion_counts(p.numpy(), y.numpy())
            else:
                opt.zero_grad()
                dm = {k: v[:bs] for k, v in masks.items()}
                p = R.robust_unet_forward(sd, x, training=True, drop_masks=dm, new_buffers={})
                loss = R.bce_loss(p, y)
                loss.backward()
                opt.step()
            return time.perf_counter() - t0

    b = batch or (1 if S >= 1024 else 2)
    t_probe = one(b)                                   # also the warm-up
    n_steps = steps or 2
    if batch is None:                                  # size the sample to the time budget
        per_img = t_probe / b
        b = int(max(1, min(8, budget_s / max(per_img * (n_steps + warmup), 1e-9))))
    for _ in range(max(0, warmup - 1)):
        one(b)
    times = [one(b) for _ in range(n_steps)]
    total = sum(times)
    what = "eval forward + calculate_metrics per image" if infer else "zero_grad+forward+BCELoss+backward+Adam.step"
    src = "unmodified Main_Final.RobustUNet (baseline/_ref)" if kind == "reference" else "oracle port of Main_Final.RobustUNet"
    return {"value": round(b * n_steps / total, 4), "unit": "img/s", "cores": cores, "kind": kind,
            "sample": f"{n_steps} steps of batch {b} at {S}x{S}, {nc} channels ({what}), {src}, fp32 torch CPU kernels "
                      f"({torch.__version__}), {cores} threads",
            "ms_per_step": round(1e3 * total / n_steps, 1), "batch": b}


def eager_cuda_leg(nc, B, S, dev, steps=3):
    """Informational: the reference itself (Main_Final.RobustUNet from baseline/_ref when present, else the oracle's
    functional restatement -- the same torch ops) executed by eager PyTorch on the SAME GPU: cuDNN/ATen kernels,
    autocast(bfloat16) + channels_last and plain fp32 (SURVEY.md §2.1: the existing-Blackwell-kernel bar)."""
    import torch
    from tools.synthetic import synthetic_batch
    MF = load_reference_module()
    out = {"implementation": "Main_Final.RobustUNet (baseline/_ref), eager" if MF is not None else "oracle functional ops, eager"}
    for mode in ("bf16_autocast_channels_last", "fp32"):
        try:
            x, y = synthetic_batch(B, nc, S, S, seed=5)
            x, y = x.to(dev), y.to(dev)
            if MF is not None:
                torch.manual_seed(0)
                model = MF.RobustUNet(n_channels=nc, n_classes=1).to(dev).train()
                if mode != "fp32":
                    model = model.to(memory_format=torch.channels_last)
                    x = x.contiguous(memory_format=torch.channels_last)
                opt = torch.optim.Adam(model.parameters(), lr=1e-4, weight_decay=1e-4, fused=True)
                crit = torch.nn.BCELoss()

                def one():
                    opt.zero_grad(set_to_none=True)
                    if mode == "fp32":
                        p = model(x)
                    else:
                        with torch.autocast("cuda", dtype=torch.bfloat16):
                            p = model(x)
                        p = p.float()            # nn.BCELoss is refused inside a CUDA autocast region: the loss runs outside
                    loss = crit(p, y)
                    loss.backward()
                    opt.step()
            else:
                from oracle import robust_unet_ref as R
                sd = {k: v.to(dev) for k, v in R.synthetic_state_dict(R.robust_unet_shapes(nc, 1, 64), seed=0).items()}
                names = [k for k, v in sd.items() if v.is_floating_point() and "running" not in k]
                params = [sd[n].requires_grad_(True) for n in names]
                opt = torch.optim.Adam(params, lr=1e-4, weight_decay=1e-4, fused=True)
                if mode != "fp32":
                    x = x.contiguous(memory_format=torch.channels_last)

                def one():
                    opt.zero_grad(set_to_none=True)
                    if mode == "fp32":
                        p = R.robust_unet_forward(sd, x, training=True, new_buffers={})
                    else:
                        with torch.autocast("cuda", dtype=torch.bfloat16):
                            p = R.robust_unet_forward(sd, x, training=True, new_buffers={}, fp32_head=True)
                    loss = R.bce_loss(p.float(), y)
                    loss.backward()
                    opt.step()

            one()
            one()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                one()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out[mode] = {"img_per_s": round(B / ms * 1e3, 1), "ms_per_step": round(ms, 2), "batch": B}
        except Exception as e:      # noqa: BLE001  e.g. out of memory at this batch: report, do not fail the bench
            out[mode] = {"error": f"{type(e).__name__}: {str(e)[:120]}"}
        one = opt = model = sd = params = None
        torch.cuda.empty_cache()
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    infer = args.workload == "infer"
    S = args.size or (1024 if infer else 256)
    nc = args.channels
    steps, warmup = args.steps, max(1, args.warmup)
    r = cpu_reference(infer, nc, S, budget_s=150.0, steps=steps, warmup=warmup)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    out = {"impl": "reference", "metric": "infer_images_per_sec" if infer else "train_images_per_sec", "value": r["value"],
           "unit": "img/s", "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": r["ms_per_step"],
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": (f"Robust U-Net inference {S}x{S}" if infer else
                                   f"Robust U-Net training step (fwd+BCE+bwd+Adam) at {S}x{S}, {nc} channels, base 64")
                      + f"; bounded sample: batch {r['batch']} per step on the host CPU", "parallelism": "cpu"},
           "cpu_baseline": {k: r[k] for k in ("value", "unit", "cores", "kind", "sample")},
           "e2e": {"value": r["value"], "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train", choices=["train", "infer", "unet"])
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--size", type=int, default=0)
    ap.add_argument("--channels", type=int, default=3)
    ap.add_argument("--w-dice", type=float, default=0.0, dest="w_dice")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true",
                    help="skip the eager PyTorch (cuDNN) run of the reference on the same GPU (N = 1, informational)")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra.c3 / extra.c5 / extra.c4_infer sub-records")
    ap.add_argument("--no-flush", action="store_true", help="skip the 256 MiB L2-flush write between timed steps")
    ap.add_argument("--detail", default="", help="write the per-call device times of one profiled step to this file")
    ap.add_argument("--dump-outputs", default="", dest="dump_outputs", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float32/float64, a fixed seeded "
                         "sample of arrays above 4 Mi elements): outputs of two builds compare one to one")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs saves the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        if args.workload == "infer" and args.warmup < 6:
            args.warmup = 6        # 1024x1024 activations: the caching allocator needs a few passes to settle
        run_ours(args)


if __name__ == "__main__":
    main()
