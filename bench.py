#!/usr/bin/env python
"""Benchmark of the MRFP hot path (BASELINE.json metric) — one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one forward+backward pass of the whole MRFP path over one batch of synthetic stem / layer1
features at BASELINE config[1] shapes (per GPU: batch 8, 768x768 crop -> 64ch and 256ch @192x192):
    NP+ call 1 fwd (deepv3.py:318) -> HRFP chain fwd incl. OCout+x (deepv3.py:320-330) -> NP+ call 2 fwd
    (deepv3.py:335) -> backward of all three with gradients for x, OCout_dec (HRFP+, deepv3.py:357) and the
    layer1 feature.
The path shards by batch with no collective (SURVEY.md §8e): under torchrun every rank runs the same step on
its own batch-8 shard ("weak" scaling) and `value` is the aggregate images/s.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_PER_GPU, H_IMG, W_IMG = 8, 768, 768
XH = XW = 192
N_CLASSES = 19
HRFP_FLOP_FWD_PER_SAMPLE = 192.70e9        # needed-only MACs x2 (SURVEY.md §8d); dgrad the same
METRIC = "mrfp_fwd_bwd_throughput"
UNIT = "img/s"
CONFIG = {
    "workload": "mrfp_fwd_bwd: NP+ on (8,64,192,192) and (8,256,192,192) + HRFP/HRFP+ chain 64ch@192^2 -> 256ch@384^2 -> "
                "64ch@192^2, the HRFP+ tail THROUGH the classifier (deepv3.py:356-361: bilinear Upsample of the decoder feature, "
                "HRFP+ add, final2 = Conv2d(256, 19, 1)), fwd + bwd (gradients to xp, the layer1 feature, dec1, W2, b2), per-GPU "
                "batch 8 (BASELINE config[1], 768x768 crop).  Round 1 timed the step up to the HRFP+ sum; this step does "
                "strictly more work (step_r1_definition carries the old one)",
    "per_gpu_batch": N_PER_GPU, "crop": [H_IMG, W_IMG], "hrfp_math": "bf16 tcgen05 (fp32 accumulate)", "np_plus_math": "fp32",
    "cache": "inputs larger than L2 (302 MB / 1.2 GB tensors per step); the per-kernel roofline launches flush L2 first",
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs and gradients of the last one as DIR/<name>.npy "
                         "(float32; arrays of more than 2^20 elements as the same seeded sample of 2^20 on every run)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    return args


DUMP_SAMPLES = 1 << 20


def dump_outputs(out_dir, arrays):
    """Writes every array as out_dir/<name>.npy in float32: whole if it has at most DUMP_SAMPLES elements, otherwise the
    elements at DUMP_SAMPLES flat indices drawn without replacement by numpy's PCG64 seeded with 0, in ascending order —
    the same positions on every run, so two builds can be compared output for output (at most 4 MB per array)."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLES:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_SAMPLES, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


# ----------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's CPU implementation of the path (oracle/torch_port.py)
# ----------------------------------------------------------------------------------------------------------
def cpu_reference_run(steps, warmup, batch=N_PER_GPU, budget_s=150.0):
    """The reference's CPU implementation of the step (oracle/torch_port.py: the reference's own torch operators) at the
    SAME per-GPU batch and shapes as the GPU arm, all host threads.  Bounded: at most `steps` timed passes and no more
    than fit into `budget_s` seconds (never fewer than 3); the line reports the passes actually timed."""
    import torch
    from oracle import torch_port as T
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(1)
    convs, bns = T.make_layers()
    g = torch.Generator().manual_seed(0)
    xp = torch.relu(torch.randn(batch, 64, XH, XW, generator=g))
    f2 = torch.relu(torch.randn(batch, 256, XH, XW, generator=g))
    draws = [(1 + 0.75 * torch.randn(batch, c, 1, 1, generator=g), 0.75 * torch.randn(batch, c, 1, 1, generator=g)) for c in (64, 256)]
    grads = (torch.randn(batch, 64, XH, XW, generator=g), torch.randn(batch, 256, H_IMG // 2, W_IMG // 2, generator=g),
             torch.randn(batch, 256, XH, XW, generator=g))
    d1 = torch.randn(batch, 256, XH, XW, generator=g)                   # decoder feature before the Upsample of deepv3.py:356
    final2 = torch.nn.Conv2d(256, N_CLASSES, 1, bias=True)              # deepv3.py:219-220
    grads = (grads[0], torch.randn(batch, N_CLASSES, H_IMG // 2, W_IMG // 2, generator=g), grads[2])
    t_w = time.perf_counter()
    for _ in range(max(1, warmup)):
        final2.zero_grad(set_to_none=True)
        T.mrfp_step(convs, bns, xp, f2, d1, draws, grads, H_IMG, W_IMG, final2)
    per = (time.perf_counter() - t_w) / max(1, warmup)
    steps = max(3, min(steps, int(budget_s / max(per, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(steps):
        final2.zero_grad(set_to_none=True)
        T.mrfp_step(convs, bns, xp, f2, d1, draws, grads, H_IMG, W_IMG, final2)
    dt = time.perf_counter() - t0
    return dict(value=batch * steps / dt, unit=UNIT, cores=torch.get_num_threads(), kind="port", batch=batch, timed_passes=steps,
                sample=f"the same step at the same per-GPU batch ({batch}) and shapes, {steps} timed + {max(1, warmup)} warm-up passes "
                       "of oracle/torch_port.py (the reference's torch operators on all host cores; its throughput is the "
                       "host's, whatever the number of GPUs in the other arm); the reference itself is a Python package "
                       "under /root/reference that does not exist on the GPU box"), dt / steps * 1e3, steps


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    warm = max(1, min(args.warmup, 2))
    base, ms, steps = cpu_reference_run(args.steps, warm)
    line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": steps, "warmup": warm, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": CONFIG, "cpu_baseline": base,
            "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def traffic_from_profiles(kernel_substr, file_hints=("",), prefixes=("R2c_", "R2b_", "R2_", "r9_", "r5_", "r3_")):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch of the kernel, read from the newest committed
    `ncu --set full` export under profiles/ (`ncu -i ... --page raw --csv`: header row, unit row, one value row)."""
    import csv
    import glob
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    for pre in prefixes:
        for path in sorted(glob.glob(os.path.join(ROOT, "profiles", pre + "*_raw.csv")), reverse=True):
            try:
                rows = list(csv.reader(open(path)))
                h, u, v = rows[0], rows[1], rows[2]
                if kernel_substr not in v[h.index("Kernel Name")] or not any(fh in os.path.basename(path) for fh in file_hints):
                    continue
                tot = 0.0
                for key in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    i = h.index(key)
                    tot += float(v[i].replace(",", "")) * scale[u[i]]
                return int(tot), os.path.relpath(path, ROOT)
            except Exception:          # noqa: BLE001  (a file of another layout: skip it)
                continue
    return None, None


# ----------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled through NVML every ~5 ms DURING the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.err = index, [], False, None
        self.max_mhz, self.nv, self.h = None, None, None
        try:                              # NVML start-up takes longer than a short timed region: do it up front
            import pynvml as nv
            nv.nvmlInit()
            self.nv, self.h = nv, nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        except Exception as e:          # noqa: BLE001
            self.err = repr(e)

    def run(self):
        try:
            nv, h = self.nv, self.h
            if nv is None:
                return
            while not self.stop_flag:
                self.rows.append((nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM),
                                  nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons")
                                  else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)))
                time.sleep(0.005)
        except Exception as e:          # noqa: BLE001
            self.err = repr(e)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable: %s" % self.err]}
        sm = sorted(r[0] for r in self.rows)
        bits = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                "hw_power_brake_slowdown": 0x80}
        reasons = [n for n, b in bits.items() if any(r[1] & b for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(self.rows)}


def _use_reference_ops(model):
    """Swap the three MRFP insertion points of `model` for the reference's own op sequence (eager ATen / cuDNN on the
    GPU, deepv3.py:268-277 and :320-330, :357) — the practical bar the kernels must beat inside a training step."""
    import math
    import torch
    import torch.nn.functional as F
    from mrfp_b200 import hrfp as H

    def np_eager(feat):
        m = feat.mean((2, 3), keepdim=True)
        d = torch.std(m, 0, keepdim=True)
        s = d / d.max() * 1.5
        a = torch.normal(torch.ones_like(m), 0.75 * torch.ones_like(m))
        b = 1 + torch.normal(torch.zeros_like(m), 0.75 * torch.ones_like(m)) * s
        return a * feat - a * m + b * m

    def stem(xp, h, w, training, p, p2, p3):
        c, b = model.hrfp_modules()
        x = np_eager(xp) if (training and p2 < 0.5) else xp
        o = F.relu(b[0](F.interpolate(c[0](xp), scale_factor=(1.205, 1.205))))
        o = F.relu(b[1](F.interpolate(c[1](o), scale_factor=(1.2, 1.2))))
        o = F.relu(b[2](F.interpolate(c[2](o), scale_factor=(1.2, 1.2))))
        dec = F.relu(b[3](F.interpolate(c[3](o), size=(int(h / 2), int(w / 2)))))
        o = F.relu(b[4](F.interpolate(c[4](dec), size=(int(h / 2), int(w / 2)))))
        o = F.relu(b[5](F.interpolate(c[5](o), scale_factor=(0.838, 0.838))))
        o = F.relu(b[6](F.interpolate(c[6](o), scale_factor=(0.798, 0.798))))
        o = F.relu(b[7](F.interpolate(c[7](o), size=(math.ceil(h / 4), math.ceil(w / 4)))))
        if training and p < 0.5:
            x = torch.add(o, x)
        return x, dec

    model.Normalization_Perturbation_Plus = np_eager
    model.mrfp_stem = stem
    model._plus_add = lambda a, d: torch.add(d, a)
    model.fuse_layer1_np = False        # NP+ call 2: the eager sequence above, not the producer-fused kernels


def train_bench(world, rank, dev, steps=30, warmup=10, global_batch=16, reference_ops=False, trunk="resnet-50", graphs=True,
                ddp_eager=False):
    """BASELINE config[2]: MRFP+ DeepLabV3+/ResNet-50 training step (main.py:845-871 recipe) on synthetic GTAV-shaped
    768x768 crops, 19 classes, `global_batch` sharded over the ranks.  The gradient all-reduce over NCCL is the only
    collective; BatchNorm and the MRFP statistics stay per rank (SURVEY.md §8e).

    graphs=True: mrfp_b200.train_step.GraphedTrainStep — forward+backward replayed as a CUDA graph per gate combination,
    one flat-buffer all-reduce, eager SGD step.  graphs=False: the same class without capture (eager launches).
    ddp_eager=True: torch DistributedDataParallel + eager launches (round 1's configuration), for comparison.
    The three MRFP gates are drawn ONCE PER GLOBAL STEP (same Python seed on every rank), as in the reference where one
    forward call — one (p, p2, p3) — covers the whole batch (deepv3.py:281-283); alpha / eps / HRFP weights use per-rank
    torch streams."""
    import random
    import torch
    import torch.distributed as dist
    from mrfp_b200.model import MRFPPlus
    from mrfp_b200.train_step import GraphedTrainStep
    from mrfp_b200 import dist as D
    # host trunk: let cuDNN pick its fastest algorithms for the fixed shapes (applies equally to both MRFP-op variants)
    torch.backends.cudnn.benchmark = os.environ.get("MRFP_BENCH_CUDNN_AUTOTUNE", "1") != "0"
    lo, hi = D.shard_bounds(global_batch, world, rank)
    nb = hi - lo
    D.seed_rank_streams(3, rank)
    random.seed(100)                                            # gates: one draw per global step, identical on every rank
    from mrfp_b200 import model as M
    M.FUSE_INSTNORM = (not reference_ops) and os.environ.get("MRFP_FUSE_INSTNORM", "1") != "0"   # reference arm: ATen InstanceNorm + ReLU
    model = MRFPPlus(19, trunk=trunk, criterion=torch.nn.CrossEntropyLoss(ignore_index=255)).to(dev)
    if reference_ops:
        _use_reference_ops(model)
    if world > 1:
        for p_ in model.parameters():                       # same start on every rank (DDP would broadcast rank 0 anyway)
            dist.broadcast(p_.data, 0)
    net = model
    if ddp_eager and world > 1:
        net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[dev.index], broadcast_buffers=False)
    opt = torch.optim.SGD([p_ for p_ in model.parameters() if p_.requires_grad], lr=1e-2, momentum=0.9, weight_decay=5e-4)
    img = torch.rand(nb, 3, H_IMG, W_IMG, device=dev) * 255.0       # the reference feeds un-normalised pixels
    lab = torch.randint(0, 19, (nb, H_IMG, W_IMG), device=dev)
    lab[torch.rand(nb, H_IMG, W_IMG, device=dev) < 0.05] = 255

    if ddp_eager or reference_ops:
        def one():
            opt.zero_grad(set_to_none=True)
            loss = net(img, lab, training=True)
            loss.backward()
            opt.step()
            return loss
        mode = "torch DDP, eager launches" if ddp_eager else "eager launches"
    else:
        stepper = GraphedTrainStep(model, opt, img, lab, eager_steps=2, use_graphs=graphs)
        if graphs:
            stepper.warm_all(img, lab)                          # untimed: every gate combination captured
        def one():
            return stepper(img, lab)
        mode = "CUDA graph per gate combination (8), flat-buffer all-reduce, eager SGD" if graphs else "eager launches, flat-buffer all-reduce"

    for _ in range(warmup):
        one()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        loss = one()
    e1.record()
    host_ms = (time.perf_counter() - t0) * 1e3 / steps
    torch.cuda.synchronize()
    ms = D.max_over_ranks(e0.elapsed_time(e1), dev)
    out = {"metric": "deeplabv3plus_%s_mrfp_plus_train_throughput" % {"resnet-50": "r50", "resnet-101": "r101", "mobilenetv2": "mobilenetv2", "shufflenetv2": "shufflenetv2"}[trunk],
           "mrfp_ops": "reference eager ATen/cuDNN" if reference_ops else "libmrfp_b200", "value": global_batch * steps / (ms * 1e-3), "unit": "img/s",
           "global_batch": global_batch, "per_gpu_batch": nb, "steps": steps, "warmup": warmup, "ms_per_step": ms / steps,
           "host_enqueue_ms_per_step": host_ms, "launch_mode": mode,
           "parallelism": f"dp{world}", "loss_finite": bool(torch.isfinite(loss).item()),
           "instance_norm": "mrfp_instnorm cluster kernels" if M.FUSE_INSTNORM else "ATen",
           "precision": "fp32 host model (cuDNN TF32 default, as the reference on this torch; cudnn.benchmark=%s), bf16 tcgen05 HRFP, fp32 NP+" % torch.backends.cudnn.benchmark,
           "gates": "natural Bernoulli(0.5) x3, one draw per global step (python random, seed 100 on every rank)",
           "data": "synthetic U[0,255) images, 19 classes, 5% ignore"}
    del model, net, opt, img, lab
    if not (ddp_eager or reference_ops):
        del stepper
    M.FUSE_INSTNORM = os.environ.get("MRFP_FUSE_INSTNORM", "1") != "0"
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    from mrfp_b200 import build, _lib
    import torch.nn.functional as F
    from mrfp_b200 import hrfp as H
    from mrfp_b200 import npplus as NP

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (the MRFP kernels have no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        build.build()
    if world > 1:
        dist.barrier()
    lib = _lib.load()

    n = N_PER_GPU
    from mrfp_b200 import dist as D
    D.seed_rank_streams(1, rank)
    from mrfp_b200.model import HRFP_CONVS, init_hrfp_module
    chans, dils = [64, 64, 64, 128, 256, 128, 64, 64, 64], [1, 1, 2, 2, 1, 1, 2, 2]
    convs = [torch.nn.Conv2d(chans[k], chans[k + 1], 3, padding=dils[k], dilation=dils[k]).to(dev).requires_grad_(False)
             for k in range(len(HRFP_CONVS))]
    bns = [torch.nn.BatchNorm2d(chans[k + 1]).to(dev).requires_grad_(False) for k in range(len(HRFP_CONVS))]
    for c, b in zip(convs, bns):            # the reference initialiser (network/mynn.py:57-74), random-init weights
        init_hrfp_module(c); init_hrfp_module(b)
    sig = 0.5 + torch.rand(1, 256, 1, 1, device=dev)
    mu = torch.randn(1, 256, 1, 1, device=dev)
    xp = torch.relu(torch.randn(n, 64, XH, XW, device=dev) * sig[:, :64] + mu[:, :64])
    f2 = torch.relu(torch.randn(n, 256, XH, XW, device=dev) * sig + mu)
    draws = [(1 + 0.75 * torch.randn(n, c, 1, 1, device=dev), 0.75 * torch.randn(n, c, 1, 1, device=dev)) for c in (64, 256)]
    g_x = torch.randn(n, 64, XH, XW, device=dev)
    g_dec = torch.randn(n, N_CLASSES, H_IMG // 2, W_IMG // 2, device=dev)     # gradient wrt dec2 = final2(HRFP+ sum)
    g_dec_r1 = torch.randn(n, 256, H_IMG // 2, W_IMG // 2, device=dev)        # (round-1 step: gradient wrt the HRFP+ sum)
    g_f2 = torch.randn(n, 256, XH, XW, device=dev)
    dec1_up = torch.randn(n, 256, XH, XW, device=dev)   # the decoder feature BEFORE the reference's bilinear Upsample (deepv3.py:356)
    final2 = torch.nn.Conv2d(256, N_CLASSES, 1, bias=True).to(dev)            # deepv3.py:219-220

    def step(xp_, f2_, d1_, gx_, gdec_, gf2_):
        """Public API path: autograd Functions over the C ABI (the same calls MRFPPlus.forward makes)."""
        a = xp_.detach().requires_grad_(True)
        b = f2_.detach().requires_grad_(True)
        d = d1_.detach().requires_grad_(True)
        final2.weight.grad = None; final2.bias.grad = None
        # deepv3.py:316-330: x = OCout + NP+(xp); NP+ call 1 rides on the chain's passes (SURVEY.md 8f-1)
        x, dec = H.hrfp_chain(a, convs, bns, H_IMG, W_IMG, np_draws=draws[0], math_mode=H.MATH_BF16, lazy_dec=True)
        y2 = NP.np_plus_with_draws(b, *draws[1])                                       # :335
        d2 = H.hrfp_plus_final2(d, final2, dec)                                        # :356-361 (Upsample + add + classifier)
        torch.autograd.backward([x, d2, y2], [gx_, gdec_, gf2_])
        return x, d2, y2, a.grad, b.grad, d.grad

    def step_r1(xp_, f2_, d1_, gx_, gdec_, gf2_):
        """Round 1's step definition (up to the HRFP+ sum, no gradient to dec1), kept for comparison."""
        a = xp_.detach().requires_grad_(True)
        b = f2_.detach().requires_grad_(True)
        x, dec = H.hrfp_chain(a, convs, bns, H_IMG, W_IMG, np_draws=draws[0], math_mode=H.MATH_BF16, lazy_dec=True)
        y2 = NP.np_plus_with_draws(b, *draws[1])
        d1 = H.hrfp_plus_add_upsampled(d1_, dec)
        torch.autograd.backward([x, d1, y2], [gx_, gdec_, gf2_])
        return x, d1, y2, a.grad, b.grad

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step(xp, f2, dec1_up, g_x, g_dec, g_f2)
    sampler = ClockSampler(local) if rank == 0 else None
    sync_all()
    if sampler:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps - 1):
        step(xp, f2, dec1_up, g_x, g_dec, g_f2)
    last = step(xp, f2, dec1_up, g_x, g_dec, g_f2)
    e1.record()
    sync_all()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    if sampler:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    total_ms = float(ms.item())
    value = world * n * args.steps / (total_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(("x", "dec2", "np_plus_layer1", "grad_xp", "grad_layer1", "grad_dec1"), last),
                                             grad_final2_weight=final2.weight.grad, grad_final2_bias=final2.bias.grad))
    del last
    # round 1's step definition, same timing rules
    for _ in range(3):
        step_r1(xp, f2, dec1_up, g_x, g_dec_r1, g_f2)
    sync_all()
    e0.record()
    for _ in range(args.steps):
        step_r1(xp, f2, dec1_up, g_x, g_dec_r1, g_f2)
    e1.record()
    sync_all()
    ms_r1 = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms_r1, op=dist.ReduceOp.MAX)
    step_r1_ms = float(ms_r1.item()) / args.steps
    del g_dec_r1

    # ---- e2e: same step through the same API with HOST (pinned) buffers, copies inside the timed region ----
    # Every step copies ITS inputs host->device and ITS five results device->host.  The copies run on their own
    # streams over double-buffered device inputs / pinned host outputs, so the H2D of step i+1 and the D2H of step
    # i-1 overlap the kernels of step i (PCIe is full duplex); the timed region ends when the last D2H has landed.
    host_in = [t.cpu().pin_memory() for t in (xp, f2, dec1_up, g_x, g_dec, g_f2)]
    dev_in = [[torch.empty_like(t) for t in (xp, f2, dec1_up, g_x, g_dec, g_f2)] for _ in range(2)]
    outs = step(xp, f2, dec1_up, g_x, g_dec, g_f2)
    host_out = [[torch.empty(o.shape, dtype=o.dtype).pin_memory() for o in outs] for _ in range(2)]
    h2d = sum(t.numel() * 4 for t in host_in)
    d2h = sum(t.numel() * 4 for t in host_out[0])
    del outs
    cur = torch.cuda.current_stream()
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()
    in_ready = [torch.cuda.Event() for _ in range(2)]
    in_free = [torch.cuda.Event() for _ in range(2)]
    out_ready = [torch.cuda.Event() for _ in range(2)]
    out_done = [torch.cuda.Event() for _ in range(2)]

    def e2e_step(i):
        b = i & 1
        with torch.cuda.stream(s_in):
            s_in.wait_event(in_free[b])                  # step i-2 has consumed this input buffer
            for d, h in zip(dev_in[b], host_in):
                d.copy_(h, non_blocking=True)
            in_ready[b].record(s_in)
        cur.wait_event(in_ready[b])
        o = step(*dev_in[b])
        in_free[b].record(cur)
        out_ready[b].record(cur)
        with torch.cuda.stream(s_out):
            s_out.wait_event(out_ready[b])
            s_out.wait_event(out_done[b])                # (host buffer b was last written by step i-2: same stream, ordered)
            for h, d in zip(host_out[b], o):
                d.record_stream(s_out)
                h.copy_(d, non_blocking=True)
            out_done[b].record(s_out)

    e2e_steps = args.steps                           # ~25 ms each: PCIe-bound; the fill / drain of the three-stage pipeline is inside the region
    for i in range(4):                               # warm-up: both buffer sets twice (first-touch of the pinned pages, copy-engine set-up)
        e2e_step(i)
    cur.wait_stream(s_out)
    sync_all()
    e0.record()
    for i in range(e2e_steps):
        e2e_step(i)
    cur.wait_stream(s_out)
    e1.record()
    sync_all()
    ms2 = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_value = world * n * e2e_steps / (float(ms2.item()) * 1e-3)

    # ---- BASELINE config[2] / [3]: the training step that hosts the path (all ranks) ----
    train = None
    if os.environ.get("MRFP_BENCH_TRAIN", "1") != "0":
        del host_in, host_out, dev_in
        torch.cuda.empty_cache()
        keys = ("value", "unit", "ms_per_step", "host_enqueue_ms_per_step", "steps", "warmup", "global_batch", "per_gpu_batch",
                "launch_mode", "mrfp_ops", "loss_finite")
        try:
            # strong scaling: global batch 16 (the configuration the BASELINE metric names), SURVEY §8d: 10 warm-up + 50 timed
            train = train_bench(world, rank, dev, steps=50, warmup=10)
            train["scaling"] = "strong (global batch 16)"
            eager = train_bench(world, rank, dev, steps=10, warmup=5, graphs=False)
            train["same_step_eager_launches"] = {k: eager[k] for k in keys}
            if world > 1:
                ddp = train_bench(world, rank, dev, steps=10, warmup=5, ddp_eager=True)
                train["same_step_torch_ddp_eager"] = {k: ddp[k] for k in keys}
            ref_t = train_bench(world, rank, dev, steps=10, warmup=5, reference_ops=True)
            train["same_step_with_reference_mrfp_ops"] = {k: ref_t[k] for k in keys}
            # weak scaling: per-GPU batch 8 (BASELINE config[1]'s per-GPU batch), global batch 8 x n_gpus
            weak = train_bench(world, rank, dev, steps=30, warmup=10, global_batch=8 * world)
            train["weak_scaling_per_gpu_batch_8"] = {k: weak[k] for k in keys}
            if os.environ.get("MRFP_BENCH_TRAIN_R101", "1") != "0":
                # BASELINE config[3] per-GPU shard: ResNet-101 host, global batch 32 at 8 GPUs = 4 per GPU
                r101 = train_bench(world, rank, dev, steps=30, warmup=10, global_batch=4 * world, trunk="resnet-101")
                train["resnet101_config3_shard"] = {k: r101[k] for k in ("metric",) + keys}
            if os.environ.get("MRFP_BENCH_TRAIN_MOBILE", "1") != "0":
                # BASELINE config[4]: MRFP+ on the narrow-stem trunks (16 ch @ stride 2 / 24 ch @ stride 4), global batch 16
                for tr in ("mobilenetv2", "shufflenetv2"):
                    mb = train_bench(world, rank, dev, steps=20, warmup=5, trunk=tr)
                    train[tr + "_config4"] = {k: mb[k] for k in ("metric",) + keys}
        except Exception as e:          # noqa: BLE001  (e.g. out of memory on a smaller GPU): report, do not hide
            import traceback
            train = dict(train or {}, error=repr(e)[:400], traceback=traceback.format_exc()[-800:])

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- per-kernel roofline measurements (rank 0, CUDA events on the launching stream, L2 flushed) ----
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    tf_peak = float(peaks.get("bf16_tflops", 1590.0))
    tf_sustained = float(peaks.get("bf16_tflops_sustained", tf_peak))
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream().cuda_stream

    def time_launch(fn, iters=10):
        ts = []
        for i in range(iters + 3):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record(); torch.cuda.synchronize()
            if i >= 3:
                ts.append(a.elapsed_time(b))
        ts.sort()
        return ts[len(ts) // 2]          # median: one preempted launch must not move a per-kernel figure

    np_rows = {}
    for name, x_t, (al, ep) in (("npplus_64ch", xp, draws[0]), ("npplus_256ch", f2, draws[1])):
        nn_, c = x_t.shape[0], x_t.shape[1]
        out = torch.empty_like(x_t)
        mean = torch.empty(nn_, c, device=dev); beta = torch.empty(nn_, c, device=dev)
        al2, ep2 = al.reshape(nn_, c).contiguous(), ep.reshape(nn_, c).contiguous()
        wsb = lib.mrfp_npplus_ws_bytes(nn_, c, XH * XW)
        wsp = torch.zeros(wsb, dtype=torch.uint8, device=dev)         # control block zero on first use (mrfp_npplus_ws_init)
        bytes_alg = 2 * x_t.numel() * 4
        t_f = time_launch(lambda: _lib.check(lib.mrfp_npplus_fwd_f32(x_t.data_ptr(), al2.data_ptr(), ep2.data_ptr(), out.data_ptr(),
                                                                     mean.data_ptr(), beta.data_ptr(), wsp.data_ptr(), wsb, nn_, c, XH * XW, st), "np fwd"))
        t_b = time_launch(lambda: _lib.check(lib.mrfp_npplus_bwd_f32(x_t.data_ptr(), al2.data_ptr(), ep2.data_ptr(), mean.data_ptr(),
                                                                     out.data_ptr(), wsp.data_ptr(), wsb, nn_, c, XH * XW, st), "np bwd"))
        np_rows[name] = {"fwd_us": t_f * 1e3, "bwd_us": t_b * 1e3, "fwd_gbs": bytes_alg / t_f / 1e6, "bwd_gbs": bytes_alg / t_b / 1e6,
                         "algorithmic_bytes": bytes_alg}
    np_bytes = sum(2 * r["algorithmic_bytes"] for r in np_rows.values())
    np_time = sum(r["fwd_us"] + r["bwd_us"] for r in np_rows.values()) * 1e-6
    big = np_rows["npplus_256ch"]
    roof_np = {"kernel": "npplus_ring_kernel<fwd> on (8,256,192,192)", "bound": "hbm", "achieved": big["fwd_gbs"], "peak": hbm_peak,
               "unit": "GB/s", "frac": big["fwd_gbs"] / hbm_peak,
               "traffic": traffic_from_profiles("npplus_ring_kernel")[0],   # dram__bytes_read.sum + dram__bytes_write.sum per launch
               "traffic_source": "%s (ncu --set full, one launch of this kernel); algorithmic bytes per launch = 603979776"
                                 % traffic_from_profiles("npplus_ring_kernel")[1],
               "peak_source": peak_src,
               "all_four_np_kernels_gbs": np_bytes / np_time / 1e9, "per_call": np_rows}

    # NP+ with its statistics taken by the producer (SURVEY.md 8f-1): layer1's last ReLU leaves the plane sums, NP+ forward
    # is one streaming pass.  Timed: the ReLU-with-sums kernel next to ATen's relu (same 1R+1W), and the pre-summed NP+.
    try:
        pre = torch.randn(n, 256, XH, XW, device=dev)
        y_r = torch.empty_like(pre)
        psum = torch.empty(n, 256, device=dev, dtype=torch.float64)
        al2, ep2 = draws[1][0].reshape(n, 256).contiguous(), draws[1][1].reshape(n, 256).contiguous()
        out_p = torch.empty_like(pre); mean_p = torch.empty(n, 256, device=dev)
        wsb_p = lib.mrfp_npplus_presummed_ws_bytes(n, 256)
        ws_p = torch.empty(wsb_p, dtype=torch.uint8, device=dev)
        t_relu = time_launch(lambda: _lib.check(lib.mrfp_relu_psum_f32(pre.data_ptr(), y_r.data_ptr(), psum.data_ptr(), n * 256, XH * XW, st), "relu_psum"))
        t_aten = time_launch(lambda: torch.relu(pre))
        t_pre = time_launch(lambda: _lib.check(lib.mrfp_npplus_fwd_presummed_f32(y_r.data_ptr(), psum.data_ptr(), al2.data_ptr(), ep2.data_ptr(), out_p.data_ptr(),
                                                                                 mean_p.data_ptr(), None, ws_p.data_ptr(), wsb_p, n, 256, XH * XW, st), "np presummed"))
        b_alg = 2 * pre.numel() * 4
        roof_np["producer_fused"] = {
            "what": "layer1's last ReLU also takes the plane sums (mrfp_relu_psum_f32), NP+ forward = coefficient block + one streaming pass "
                    "(mrfp_npplus_fwd_presummed_f32); the path MRFPPlus.forward uses for call 2; the backward stays on the ring kernel",
            "relu_psum_us": t_relu * 1e3, "aten_relu_us": t_aten * 1e3, "npplus_fwd_presummed_us": t_pre * 1e3,
            "npplus_fwd_presummed_gbs": b_alg / t_pre / 1e6, "frac": b_alg / t_pre / 1e6 / hbm_peak,
            "fwd_plus_bwd_gbs": 2 * b_alg / (t_pre + big["bwd_us"] * 1e-3) / 1e6,
            "fwd_plus_bwd_frac": 2 * b_alg / (t_pre + big["bwd_us"] * 1e-3) / 1e6 / hbm_peak}
        del pre, y_r, out_p
    except Exception as e_:          # noqa: BLE001
        roof_np["producer_fused"] = {"error": repr(e_)[:200]}

    # InstanceNorm2d(affine)+ReLU of the trunk next to the insertion points (SURVEY.md 8f-3): layer1's site, the producer of NP+ call 2
    roof_in = None
    try:
        xin = torch.randn(n, 256, XH, XW, device=dev) * 2 + 1
        gin_ = torch.randn_like(xin)
        w_in = 1 + 0.2 * torch.randn(256, device=dev); b_in = 0.2 * torch.randn(256, device=dev)
        y_in = torch.empty_like(xin); gx_in = torch.empty_like(xin)
        m_in = torch.empty(n, 256, device=dev); i_in = torch.empty(n, 256, device=dev)
        dg_in = torch.empty(n, 256, device=dev); db_in = torch.empty(n, 256, device=dev)
        ps_in = torch.empty(n, 256, device=dev, dtype=torch.float64)
        t_if = time_launch(lambda: _lib.check(lib.mrfp_instnorm_fwd_f32(xin.data_ptr(), w_in.data_ptr(), b_in.data_ptr(), y_in.data_ptr(), m_in.data_ptr(),
                                                                        i_in.data_ptr(), ps_in.data_ptr(), n, 256, XH * XW, 1e-5, 1, st), "instnorm fwd"))
        t_ib = time_launch(lambda: _lib.check(lib.mrfp_instnorm_bwd_f32(gin_.data_ptr(), xin.data_ptr(), w_in.data_ptr(), b_in.data_ptr(), m_in.data_ptr(),
                                                                        i_in.data_ptr(), gx_in.data_ptr(), dg_in.data_ptr(), db_in.data_ptr(), n, 256,
                                                                        XH * XW, 1, st), "instnorm bwd"))
        t_ia = time_launch(lambda: F.relu(F.instance_norm(xin, weight=w_in, bias=b_in)))
        nb_in = xin.numel() * 4
        roof_in = {"kernel": "instnorm_fwd_kernel / instnorm_bwd_kernel on (8,256,192,192), ReLU and NP+ plane sums fused", "bound": "hbm",
                   "fwd_us": t_if * 1e3, "fwd_gbs": 2 * nb_in / t_if / 1e6, "fwd_frac": 2 * nb_in / t_if / 1e6 / hbm_peak,
                   "bwd_us": t_ib * 1e3, "bwd_gbs": 3 * nb_in / t_ib / 1e6, "bwd_frac": 3 * nb_in / t_ib / 1e6 / hbm_peak,
                   "algorithmic_bytes": {"fwd": 2 * nb_in, "bwd": 3 * nb_in}, "aten_instance_norm_relu_fwd_us": t_ia * 1e3, "peak": hbm_peak}
        del xin, gin_, y_in, gx_in
    except Exception as e_:          # noqa: BLE001
        roof_in = {"error": repr(e_)[:200]}

    # tcgen05 conv kernels of the chain at the step's shapes, each through the debug hook of the kernel the chain launches
    # for it: forward stage 0 = conv3x3_tc_kernel on the stem feature; forward stages 1-7 = conv3x3_gather_kernel<fwd> (the
    # resample + BN + ReLU of the previous stage built into the operand, BN statistics in the epilogue); dgrads of the
    # wide up-sampling stages 2-3 = conv3x3_tc_kernel on dY; the other dgrads = conv3x3_gather_kernel<bwd | bwd-rep> (BN-backward
    # apply built into the operand; stage 4 also takes the classifier tail's gradient as a rank-K k-block)
    import ctypes
    fn = lib.mrfp_debug_conv3x3_bf16
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_int] * 6 + [ctypes.c_void_p] * 4
    gfn = lib.mrfp_debug_conv3x3_gather_fwd
    gfn.restype = ctypes.c_int
    gfn.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int] + [ctypes.c_void_p] * 5 + [ctypes.c_int] * 6 + [ctypes.c_void_p] * 4
    bfn = lib.mrfp_debug_conv3x3_gather_bwd
    bfn.restype = ctypes.c_int
    bfn.argtypes = ([ctypes.c_void_p] * 2 + [ctypes.c_int] * 2 + [ctypes.c_void_p] * 4 + [ctypes.c_int] + [ctypes.c_void_p] * 3 +
                    [ctypes.c_double] + [ctypes.c_void_p] * 2 + [ctypes.c_int] * 6 + [ctypes.c_void_p] * 2)
    rfn = lib.mrfp_debug_conv3x3_gather_bwd_rk     # stage 4: the classifier tail's gradient joins as a rank-K k-block
    rfn.restype = ctypes.c_int
    rfn.argtypes = ([ctypes.c_void_p] * 2 + [ctypes.c_int] * 2 + [ctypes.c_void_p] * 7 + [ctypes.c_double] + [ctypes.c_void_p] * 2 +
                    [ctypes.c_int] * 6 + [ctypes.c_void_p] * 3)
    plan = H.get_plan(n, 64, XH, XW, H_IMG, W_IMG, dev, H.MATH_BF16)

    def nearest_idx(src, dst):          # ATen's rule in float32 (size= form; the tables only shape the access pattern here)
        sc = torch.tensor(src / dst, dtype=torch.float32)
        return torch.clamp(torch.floor(torch.arange(dst, dtype=torch.float32) * sc).to(torch.int64), max=src - 1)

    def padded_ones(size):
        c = torch.zeros((size + 15) // 16 * 16 + 16, dtype=torch.int32, device=dev)
        c[:size] = 1
        return c

    def ok(rc):
        assert rc == 0, f"conv debug hook returned {rc}"

    conv_rows, dgrad_rows, conv_time, conv_flop = [], [], 0.0, 0.0
    stats_t = torch.zeros(4, 256, device=dev)
    stats_t[1] = 1.0; stats_t[2] = 0.5 + torch.rand(256, device=dev); stats_t[3] = 0.2 * torch.randn(256, device=dev)
    gamma_t = torch.ones(256, device=dev)
    for k, (cin, cout, dil, ch, cw, oh, ow) in enumerate(plan.stages):
        fl = 2.0 * n * ch * cw * cout * 9 * cin
        wp = (torch.randn(9, cout, cin, device=dev) * (2.0 / (9 * cin)) ** 0.5).to(torch.bfloat16)
        y = torch.empty(n, ch, cw, cout, device=dev, dtype=torch.bfloat16)
        cnth, cntw = padded_ones(ch), padded_ones(cw)
        acc_t = torch.zeros(2 * 256, dtype=torch.float64, device=dev)
        if k == 0:
            a_in = torch.randn(n, ch, cw, cin, device=dev).to(torch.bfloat16)
            t = time_launch(lambda: ok(fn(a_in.data_ptr(), wp.data_ptr(), y.data_ptr(), n, ch, cw, cin, cout, dil, cnth.data_ptr(),
                                          cntw.data_ptr(), acc_t.data_ptr(), st)), 5)
            kern = f"conv3x3_tc_kernel<{cout}>"
        else:
            sh, sw = plan.stages[k - 1][3], plan.stages[k - 1][4]
            a_in = torch.randn(n, sh, sw, cin, device=dev).to(torch.bfloat16)
            ih, iw = nearest_idx(sh, ch).to(torch.int32).to(dev), nearest_idx(sw, cw).to(torch.int32).to(dev)
            t = time_launch(lambda: ok(gfn(a_in.data_ptr(), sh, sw, ih.data_ptr(), iw.data_ptr(), stats_t.data_ptr(), wp.data_ptr(),
                                           y.data_ptr(), n, ch, cw, cin, cout, dil, cnth.data_ptr(), cntw.data_ptr(), acc_t.data_ptr(), st)), 5)
            kern = f"conv3x3_gather_kernel<{cout}, fwd>"
        conv_rows.append({"stage": k, "kernel": kern, "cin": cin, "cout": cout, "hw": [ch, cw], "us": t * 1e3, "tflops": fl / t / 1e9})
        conv_time += t; conv_flop += fl
        del a_in, y
        # dgrad of the stage: cout channels in, cin channels out, same resolution and FLOPs
        wpb = (torch.randn(9, cin, cout, device=dev) * (2.0 / (9 * cout)) ** 0.5).to(torch.bfloat16)
        gout = torch.empty(n, ch, cw, cin, device=dev, dtype=torch.bfloat16)
        if k in (2, 3):
            dy = torch.randn(n, ch, cw, cout, device=dev).to(torch.bfloat16)
            t = time_launch(lambda: ok(fn(dy.data_ptr(), wpb.data_ptr(), gout.data_ptr(), n, ch, cw, cout, cin, dil, None, None, None, st)), 5)
            kern = f"conv3x3_tc_kernel<{cin}>"
            del dy
        else:
            yk = torch.randn(n, ch, cw, cout, device=dev).to(torch.bfloat16)
            da = torch.randn(n, oh, ow, cout, device=dev).to(torch.bfloat16)
            ih, iw = nearest_idx(ch, oh), nearest_idx(cw, ow)
            loh_c = torch.searchsorted(ih, torch.arange(ch + 1)).to(torch.int32).contiguous()     # host copies size the extras stage
            low_c = torch.searchsorted(iw, torch.arange(cw + 1)).to(torch.int32).contiguous()
            loh, low = loh_c.to(dev), low_c.to(dev)
            rep = 2 if k < 4 else 1                     # up-sampling stages: up to 2 x 2 replicas of a source pixel
            if k == 4:      # as the chain launches it: + G (pixels, 64) . W2T (256, 64)^T, the classifier tail's gradient
                g64 = torch.zeros(n, ch, cw, 64, device=dev, dtype=torch.bfloat16)
                g64[..., :N_CLASSES] = torch.randn(n, ch, cw, N_CLASSES, device=dev).to(torch.bfloat16)
                w2t = torch.zeros(cin, 64, device=dev, dtype=torch.bfloat16)
                w2t[:, :N_CLASSES] = (0.05 * torch.randn(cin, N_CLASSES, device=dev)).to(torch.bfloat16)
                t = time_launch(lambda: ok(rfn(yk.data_ptr(), da.data_ptr(), oh, ow, loh.data_ptr(), low.data_ptr(), loh_c.data_ptr(),
                                               low_c.data_ptr(), stats_t.data_ptr(), gamma_t.data_ptr(), acc_t.data_ptr(),
                                               float(n * oh * ow), wpb.data_ptr(), gout.data_ptr(), n, ch, cw, cout, cin, dil,
                                               g64.data_ptr(), w2t.data_ptr(), st)), 5)
                del g64, w2t
            else:
                t = time_launch(lambda: ok(bfn(yk.data_ptr(), da.data_ptr(), oh, ow, loh.data_ptr(), low.data_ptr(), loh_c.data_ptr(),
                                               low_c.data_ptr(), rep, stats_t.data_ptr(), gamma_t.data_ptr(), acc_t.data_ptr(),
                                               float(n * oh * ow), wpb.data_ptr(), gout.data_ptr(), n, ch, cw, cout, cin, dil,
                                               None, st)), 5)
            kern = f"conv3x3_gather_kernel<{cin}, {'bwd-rep' if k < 4 else 'bwd'}{', rank-K' if k == 4 else ''}>"
            del yk, da
        dgrad_rows.append({"stage": k, "kernel": kern, "cin": cout, "cout": cin, "hw": [ch, cw], "us": t * 1e3, "tflops": fl / t / 1e9})
        del wp, wpb, gout
    top = max(conv_rows + dgrad_rows, key=lambda r: r["us"])
    is_dgrad = top in dgrad_rows
    hint = ("gather_d4",) if is_dgrad else ("gather_s4",)
    roofline = {"kernel": f"{top['kernel']} stage {top['stage']} {'dgrad' if is_dgrad else 'forward'} "
                          f"({top['cin']}->{top['cout']} @{top['hw'][0]}x{top['hw'][1]}) — the longest single launch of the step",
                "bound": "tensor", "achieved": top["tflops"], "peak": tf_peak, "unit": "TFLOP/s", "frac": top["tflops"] / tf_peak,
                "traffic": traffic_from_profiles("conv3x3_gather_kernel", hint)[0],   # dram read + write bytes per launch
                "traffic_source": "%s (ncu --set full, one launch of this kernel inside the step)"
                                  % traffic_from_profiles("conv3x3_gather_kernel", hint)[1],
                "peak_source": peak_src, "peak_sustained": tf_sustained,
                "all_conv_fwd_tflops": conv_flop / conv_time / 1e9, "per_stage": conv_rows, "per_stage_dgrad": dgrad_rows}

    # chain-level numbers through the public API
    def t_api(fn_, iters=5):
        for _ in range(2):
            fn_()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn_()
        b.record(); torch.cuda.synchronize()
        return a.elapsed_time(b) / iters

    xr = xp.detach().requires_grad_(True)
    with torch.no_grad():
        t_chain_f = t_api(lambda: H.hrfp_plus_final2(dec1_up, final2, H.hrfp_chain(xr, convs, bns, H_IMG, W_IMG, math_mode=H.MATH_BF16, lazy_dec=True)[1]))

    def chain_fb():
        xr.grad = None
        o, d = H.hrfp_chain(xr, convs, bns, H_IMG, W_IMG, math_mode=H.MATH_BF16, lazy_dec=True)
        torch.autograd.backward([o, H.hrfp_plus_final2(dec1_up, final2, d)], [g_x, g_dec])
    t_chain_fb = t_api(chain_fb)
    def chain_fb_tf32():
        xr.grad = None
        o, d = H.hrfp_chain(xr, convs, bns, H_IMG, W_IMG, math_mode=H.MATH_TF32, lazy_dec=True)
        torch.autograd.backward([o, final2(H.hrfp_plus_add_upsampled(dec1_up, d))], [g_x, g_dec])
    try:
        t_chain_fb_tf32 = t_api(chain_fb_tf32, 3)
    except Exception as e_:          # noqa: BLE001
        t_chain_fb_tf32 = repr(e_)[:200]
    hrfp = {"fwd_ms": t_chain_f, "fwd_bwd_ms": t_chain_fb, "fwd_bwd_ms_tf32_mode": t_chain_fb_tf32,
            "fwd_tflops_needed_only": HRFP_FLOP_FWD_PER_SAMPLE * n / t_chain_f / 1e9,
            "fwd_bwd_tflops_needed_only": 2 * HRFP_FLOP_FWD_PER_SAMPLE * n / t_chain_fb / 1e9}

    base = cpu_reference_run(3, 1, budget_s=30.0)[0] if world == 1 else None

    # kernels launched per step (ours; memsets and the host's two library GEMMs W2 . dec1 / its backward excluded):
    # NP+ call 2 fwd + bwd (call 1 is folded into the chain: +1 coefficient block each way); HRFP fwd 1 weight pack + 1
    # NCHW->NHWC + 8 conv (stages 1-7 build their operand from the previous conv output, BN finalised by the last CTA) + 1
    # NHWC->NCHW epilogue (OCout + x); tail through the classifier 1 fwd + 1 bwd + 1 bilinear-transpose gather; HRFP bwd
    # 1 NCHW->NHWC + 8 BN-bwd reductions + 2 BN-bwd apply passes (stages 2-3; the others build dY inside the dgrad) + 8 dgrad
    # + 1 NHWC->NCHW
    launches_per_step = 2 + (1 + 1 + 1 + 8 + 1) + 3 + (1 + 1 + 8 + 2 + 8 + 1)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16 (HRFP tensor-core operands, fp32 accumulate) / f32 (NP+)", "data": "synthetic", "config": CONFIG,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                    "pipeline": "H2D / kernels / D2H on three streams, double-buffered; every step moves its own inputs and results"},
            "gpu_launches": launches_per_step * args.steps,
            "step_r1_definition": {"ms_per_step": step_r1_ms, "value": world * n / (step_r1_ms * 1e-3), "unit": UNIT,
                                   "what": "round 1's step (tail up to the HRFP+ sum, (N,256,384,384) fp32 output and gradient, no gradient to dec1)"},
            "roofline": roofline, "roofline_npplus": roof_np, "roofline_instnorm": roof_in, "hrfp_chain": hrfp, "train": train,
            "clocks": sampler.summary() if sampler else None}
    if base is not None:
        line["cpu_baseline"] = base
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
