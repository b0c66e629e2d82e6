#!/usr/bin/env python
"""bench.py -- entropy-model images/sec of the DCAE slice loop on B200 (BASELINE.json metric).

    python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--math tf32x3|tf32|fp32]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the channel-slice loop (dcae.py:638-670: 5 x [dictionary cross-attention,
cc_mean/cc_scale, GaussianConditional quantise+likelihood+index, LRP]) over one batch of synthetic
Kodak-shaped latents: BASELINE config #2, 16 images of 768x512 per GPU -> y/latent_scales/latent_means
[16, 320, 32, 48].  Images are independent, so N GPUs run N independent shards (weak scaling, no
data-path collective); NCCL is used for the barrier, the max-over-ranks time and the bpp reduction.

Printed JSON line: see DESIGN.md section "Measurement".
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

FLOP_PER_TOKEN = 163.76e6        # SURVEY §8d: whole slice loop, 2*MAC
GC_BYTES_PER_ELEM = 28           # y, mu, scale in; lik, y_hat, sym, idx out (compress variant)

# BASELINE.json configs that are bench lines (the others are parity-test cases).  #2 is the one the metric is quoted on
# and the default; #3 and #5 are the "larger images" of the north star.  H x W are padded to multiples of 128 as
# eval.py:3583-3598 does before the model sees them; tokens = (H_pad / 16) * (W_pad / 16).
CONFIGS = {
    1: dict(H=256, W=256, batch=1, mode="forward", tag="256x256",
            workload="DCAE entropy-model forward (slice loop), one synthetic 256x256 image (BASELINE config #1)"),
    2: dict(H=512, W=768, batch=16, mode="forward", tag="768x512",
            workload="DCAE entropy-model forward (slice loop), batch 16 synthetic Kodak-shaped 768x512 images per GPU (BASELINE config #2)"),
    3: dict(H=1365, W=2048, batch=4, mode="compress", tag="2048x1365",
            workload="DCAE compress() slice loop (quantize + build_indexes + likelihoods), synthetic CLIC-shaped 2048x1365 images, 4 per GPU per step (BASELINE config #3)"),
    4: dict(H=256, W=256, batch=8, mode="train", tag="256x256 crops (training)",
            workload="DCAE entropy-model rate-distortion training step (MSE lambda = 0.013: forward, train.py:82-88 loss, backward, grad clip 1.0, Adam) on 8 x 256x256 crops per GPU, DDP gradient all-reduce over NCCL (BASELINE config #4)"),
    5: dict(H=2160, W=3840, batch=4, mode="forward", tag="3840x2160",
            workload="DCAE entropy-model forward (slice loop), synthetic 4K 3840x2160 images, 4 per GPU per step (BASELINE config #5)"),
    # beyond the north star (SURVEY 8f N3 / N4): the WHOLE model -- g_a, h_a, entropy bottleneck, h_z_s1 / h_z_s2, slice loop, g_s
    6: dict(H=512, W=768, batch=16, mode="codec", tag="768x512 (whole codec)",
            workload="whole DCAE.forward (g_a, h_a, EntropyBottleneck, h_z_s1, h_z_s2, slice loop, g_s: dcae.py:623-677), batch 16 synthetic 768x512 images per GPU"),
}


def latent_hw(cfg):
    pad = lambda v: (v + 127) // 128 * 128
    return pad(cfg["H"]) // 16, pad(cfg["W"]) // 16


def ncu_traffic(kernel_csv):
    """Mean DRAM bytes (read + write) per launch from a committed `ncu --set full` summary (tools/ncu_summary.py), or None."""
    import csv
    path = os.path.join(ROOT, "profiles", "r02", kernel_csv)
    if not os.path.exists(path):
        path = os.path.join(ROOT, "profiles", "r01", kernel_csv)
    try:
        rows = list(csv.reader(open(path)))
        hdr, units, data = rows[0], rows[1], rows[2:]
        mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
        tot = []
        for r in data:
            b = 0.0
            for name in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                i = hdr.index(name)
                b += float(r[i]) * mult[units[i]]
            tot.append(b)
        return sum(tot) / len(tot) if tot else None
    except Exception:                                   # noqa: BLE001
        return None


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm": d["hbm_gbs"], "tc_burst": d["bf16_tflops"], "tc_sustained": d["bf16_tflops_sustained"], "src": "measured"}
    return {"hbm": 6650.0, "tc_burst": 1590.0, "tc_sustained": 1400.0, "src": "fallback"}


DUMP_BYTES = 60 << 20            # --dump-outputs: data bytes of all files together (< 64 MB with the .npy headers)


def _flat_outputs(outputs, prefix=""):
    for k, v in outputs.items():
        if isinstance(v, dict):
            yield from _flat_outputs(v, f"{prefix}{k}.")
        else:
            yield prefix + k, v


def dump_outputs(path, outputs, budget=DUMP_BYTES, seed=0):
    """Write every tensor of `outputs` (nested dicts: names joined by '.') as `path/<name>.npy`: float64 for float64 and
    integer tensors (exact), float32 otherwise.  Within `budget` bytes in all: the smaller arrays are written whole, and
    each array above the byte cap that leaves becomes a 1-D sample of its flattened elements at sorted indices drawn
    with `seed`, the same indices on every run (and for every array of the same size), so that the files of two builds
    compare element for element."""
    import numpy as np
    arrays = [(n, t.detach(), np.float64 if t.dtype == torch.float64 or not t.is_floating_point() else np.float32)
              for n, t in _flat_outputs(outputs)]
    sizes = sorted(t.numel() * np.dtype(d).itemsize for _, t, d in arrays)
    cap, left = None, budget
    for i, s in enumerate(sizes):
        if s * (len(sizes) - i) > left:
            cap = left // (len(sizes) - i)
            break
        left -= s
    os.makedirs(path, exist_ok=True)
    for name, t, dtype in arrays:
        keep = t.numel() if cap is None else min(t.numel(), cap // np.dtype(dtype).itemsize)
        if keep < t.numel():
            idx = np.sort(np.random.default_rng(seed).choice(t.numel(), keep, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.cpu().numpy().astype(dtype))


def synth_latents(B, h, w, seed=1234, pin=False):
    """SURVEY §8d 'direct' synthetic inputs: y = 4 randn, latents = randn."""
    g = torch.Generator().manual_seed(seed)
    ts = [4.0 * torch.randn(B, 320, h, w, generator=g), torch.randn(B, 320, h, w, generator=g),
          torch.randn(B, 320, h, w, generator=g)]
    return [t.pin_memory() for t in ts] if pin else ts


class ClockSampler:
    """SM clock, power and throttle reasons sampled DURING the timed region through NVML in a thread of this
    process (nvidia-smi -lms was measured to stall the GPU by tens of ms per query on this box, which is not
    acceptable inside a 0.6 s timed region; the NVML calls below are the same counters without that cost)."""

    def __init__(self, index, period_s=0.1):
        self.rows, self.ok, self._stop = [], False, threading.Event()
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv, self.h = nv, nv.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:                      # noqa: BLE001
            self.err = repr(e)
            return
        self.period = period_s
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:                   # noqa: BLE001
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((sm, pw, rs))
            except Exception:                       # noqa: BLE001
                pass
            self._stop.wait(self.period)

    def mark(self):
        """Only samples taken after this call count (call right before the timed region)."""
        self.start = len(self.rows)

    def stop(self):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "")]}
        self._stop.set()
        self.t.join(timeout=2)
        nv = self.nv
        rows = self.rows[getattr(self, "start", 0):]
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        reasons = sorted(n for n, bit in names.items() if any(r[2] & bit for r in rows))
        sm = sorted(r[0] for r in rows)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_sm, "reasons": reasons,
                "power_w_max": max((r[1] for r in rows), default=None), "samples": len(rows), "source": "nvml"}


def bind_rank_to_cores(local: int, local_world: int):
    """e2e at N > 1 is a host-side question (r01: 8 ranks x 220 MB per 14 ms step through one NUMA node).  Before any
    pinned buffer is allocated, bind this process to its own slice of the GPU's NUMA-local cores (NVML's CPU affinity of
    the device; the ranks split it evenly), so that first-touch places the pinned pages next to the GPU and the ranks'
    copy / launch threads do not migrate over each other.  Returns a description for the JSON line."""
    info = {"bound": False}
    try:
        allowed = sorted(os.sched_getaffinity(0))
        cpus = allowed
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(local)
            words = nv.nvmlDeviceGetCpuAffinity(h, (max(allowed) + 64) // 64)
            near = [i for i in allowed if (words[i // 64] >> (i % 64)) & 1]
            if near:
                cpus = near
            info["gpu_cpu_affinity"] = f"{cpus[0]}-{cpus[-1]} ({len(cpus)} cores)"
        except Exception as e:                      # noqa: BLE001
            info["nvml"] = repr(e)[:80]
        n = max(len(cpus) // max(local_world, 1), 1)
        mine = cpus[(local * n) % len(cpus): (local * n) % len(cpus) + n] or cpus
        os.sched_setaffinity(0, mine)
        info.update(bound=True, cores=f"{mine[0]}-{mine[-1]}", n_cores=len(mine))
    except Exception as e:                          # noqa: BLE001
        info["error"] = repr(e)[:120]
    return info


class _ReferenceLoop:
    """The reference's own implementation of the path, for the baseline legs only (never on the product path).
    kind "reference": the UNMODIFIED classes of /root/reference/models/dcae.py (staged into oracle/_ref/ by build()):
    `DCAE.forward` / `DCAE.compress` run as written on injected (y, latent_scales, latent_means) -- everything outside
    the slice loop is replaced by injectors that cost nothing (oracle/reference_loader.py); compressai is absent, so
    `GaussianConditional` is the oracle restatement and, in compress mode, the rANS encoder is a recorder (the
    `.tolist()` hand-off of dcae.py:742-743 is part of the reference's path and stays inside the timed region).
    kind "port": the functional restatement oracle/entropy_model.py, when the reference file is not available."""

    def __init__(self, params, device, mode):
        from oracle import reference_loader as rl
        self.mode, self.device = mode, torch.device(device)
        if rl.reference_available():
            self.kind = "reference"
            self.rl = rl
            self.net = rl.build_reference_net(params).to(self.device)
        else:
            from oracle.entropy_model import SliceLoopOracle
            self.kind = "port"
            p = {k: v.to(self.device) for k, v in params.items()}
            self.orc = SliceLoopOracle(p, scale_table=None)
            self.orc.scale_table = self.orc.scale_table.to(self.device)

    def step(self, y, ls, lm):
        with torch.no_grad():
            if self.kind == "port":
                return self.orc.compress(y, ls, lm) if self.mode == "compress" else self.orc.forward(y, ls, lm)
            x = self.rl.inject_latents(self.net, y, ls, lm)
            if self.mode == "forward":
                return self.net(x)
            import tempfile
            cwd = os.getcwd()
            with tempfile.TemporaryDirectory() as td:           # compress() writes debug dumps to ./output/debug (dcae.py:707, 758)
                os.makedirs(os.path.join(td, "output", "debug"))
                os.chdir(td)
                try:
                    return self.net.compress(x)
                finally:
                    os.chdir(cwd)


def cpu_reference_rate(cfg, n_images, steps, warmup, seed=0):
    """The reference's CPU path on all host threads, `steps` steps of `n_images` images.
    -> (images/s, threads, seconds per step, kind)."""
    from dcae_b200.params import init_entropy_params
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    h, w = latent_hw(cfg)
    loop = _ReferenceLoop(init_entropy_params(seed, "lively"), "cpu", cfg["mode"])
    y, ls, lm = synth_latents(n_images, h, w)
    for _ in range(warmup):
        loop.step(y, ls, lm)
    t0 = time.perf_counter()
    for _ in range(steps):
        loop.step(y, ls, lm)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return n_images / dt, threads, dt, loop.kind


def gpu_eager_rate(cfg, dev, n_images, steps, warmup, seed=0, tf32=False):
    """The same reference classes run by eager PyTorch ON THE GPU with the reference's evaluation flags (TF32 off,
    cuDNN off: eval.py:3182-3187, 3904): what a user of the reference gets on this B200 without this library.  A
    baseline leg like cpu_baseline; `tf32=True` is the reduced-precision fair-fight variant (TF32 + cuDNN on).
    -> (images/s, seconds per step, kind)."""
    from dcae_b200.params import init_entropy_params
    saved = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.enabled)
    torch.backends.cuda.matmul.allow_tf32 = tf32
    torch.backends.cudnn.allow_tf32 = tf32
    torch.backends.cudnn.enabled = tf32
    try:
        h, w = latent_hw(cfg)
        loop = _ReferenceLoop(init_entropy_params(seed, "lively"), dev, cfg["mode"])
        y, ls, lm = (t.to(dev) for t in synth_latents(n_images, h, w))
        for _ in range(warmup):
            loop.step(y, ls, lm)
        torch.cuda.synchronize()
        t0 = time.perf_counter()                      # wall clock: compress mode has host work (.tolist()) on its path
        for _ in range(steps):
            loop.step(y, ls, lm)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / max(steps, 1)
        return n_images / dt, dt, loop.kind
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.enabled = saved


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path on the box's host cores; every step is the
    same batch the GPU arm processes per GPU (same config), same warm-up count."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    n_img = args.batch or cfg["batch"]
    warm = max(args.warmup, 3) if args.config == 2 else min(args.warmup, 1)
    if args.config == 4:
        torch.set_num_threads(os.cpu_count() or 1)
        rate, dt, kind = reference_train_rate(cfg, "cpu", n_img, args.steps, warm)
        threads = os.cpu_count() or 1
        if rate is None:
            print(json.dumps({"impl": "reference", "unavailable": "reference models/dcae.py not staged in oracle/_ref"}), flush=True)
            return
    else:
        rate, threads, dt, kind = cpu_reference_rate(cfg, n_img, args.steps, warm)
    what = ("unmodified /root/reference/models/dcae.py classes (DCAE.%s slice loop on injected latents; GaussianConditional = oracle restatement, compressai absent)" % cfg["mode"]
            if kind == "reference" else "torch-CPU fp32 oracle port of dcae.py:638-670")
    line = {
        "impl": "reference", "metric": "entropy-model training images/sec @256x256 crops" if args.config == 4 else f"entropy-model images/sec @{cfg['tag']}", "value": rate, "unit": "images/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": warm, "ms_per_step": dt * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg["workload"], "batch_per_gpu": n_img, "mode": cfg["mode"], "where": "host CPU, torch fp32, all threads"},
        "cpu_baseline": {"value": rate, "unit": "images/s", "cores": threads, "kind": kind,
                         "sample": f"{args.steps} steps x {n_img} images of {cfg['tag']}: {what}"},
        "e2e": {"value": rate, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---- BASELINE config #4: the training step ---------------------------------------------------------------------------
def _train_loss(lik, y_hat, target, pixels):
    """train.py:82-88 (type mse, lambda 0.013) on the slice loop's outputs; the synthesis transform is outside the hot path,
    so the distortion is measured on y_hat against y."""
    import math
    bpp = torch.log(lik).sum() / (-math.log(2) * pixels)
    return 0.013 * 255 ** 2 * torch.mean((y_hat - target) ** 2) + bpp


def reference_train_rate(cfg, device, n_images, steps, warmup, seed=0):
    """The reference's own classes (oracle/_ref) doing the same step with torch autograd: DCAE.forward in train() mode on
    injected latents, loss, backward, clip, Adam over the hot-path parameters.  -> (images/s, s/step, kind)."""
    from dcae_b200.params import init_entropy_params
    from oracle import reference_loader as rl
    if not rl.reference_available():
        return None, None, "unavailable"
    h, w = latent_hw(cfg)
    dev = torch.device(device)
    net = rl.build_reference_net(init_entropy_params(seed, "lively")).to(dev).train()
    hot = [p for k, p in net.named_parameters() if k.split(".")[0] in rl.HOT_PREFIXES]
    opt = torch.optim.Adam(hot, lr=1e-4)
    y, ls, lm = (t.to(dev) for t in synth_latents(n_images, h, w))
    pixels = n_images * cfg["H"] * cfg["W"]

    def step():
        opt.zero_grad(set_to_none=True)
        out = net(rl.inject_latents(net, y, ls, lm))
        loss = _train_loss(out["likelihoods"]["y"], out["x_hat"], y, pixels)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(hot, 1.0)
        opt.step()
        return loss

    for _ in range(warmup):
        step()
    if dev.type == "cuda":
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        loss = step()
    float(loss.detach())
    if dev.type == "cuda":
        torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return n_images / dt, dt, "reference"


def run_training(args):
    """config #4 on N GPUs: one process per GPU, `dcae_b200.EntropyModel` under DistributedDataParallel
    (find_unused_parameters=True as train.py:424), every step = H2D of the batch, forward on the library's kernels,
    loss, backward (torch-graph recompute + dcae_gc_backward), NCCL gradient all-reduce, clip, Adam, D2H of the loss."""
    cfg = CONFIGS[4]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.backends.cuda.matmul.allow_tf32 = False          # the backward recompute is the fp32 graph
    torch.backends.cudnn.allow_tf32 = False
    from dcae_b200.params import init_entropy_params
    from dcae_b200.training import EntropyModel
    B = args.batch or cfg["batch"]
    h, w = latent_hw(cfg)
    model = EntropyModel(init_entropy_params(0, "lively"), device=dev, math=args.math).train()
    ddp = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local], find_unused_parameters=True) if world > 1 else model
    params = list(model.parameters())
    opt = torch.optim.Adam(params, lr=1e-4)
    host_in = synth_latents(B, h, w, seed=1234 + rank, pin=True)
    dev_in = [torch.empty_like(t, device=dev) for t in host_in]
    pixels = B * cfg["H"] * cfg["W"]
    host_loss = torch.empty(1).pin_memory()
    n_params = sum(p.numel() for p in params)

    def step(sync=True, copy=True):
        if copy:
            for d, s_ in zip(dev_in, host_in):
                d.copy_(s_, non_blocking=True)
        opt.zero_grad(set_to_none=True)
        ctx = ddp.no_sync() if (world > 1 and not sync) else _null()
        with ctx:
            out = ddp(*dev_in)
            loss = _train_loss(out["likelihoods"], out["y_hat"], dev_in[0], pixels)
            loss.backward()
        torch.nn.utils.clip_grad_norm_(params, 1.0)
        opt.step()
        if copy:
            host_loss.copy_(loss.detach().reshape(1), non_blocking=True)
        return loss

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms) / steps, out

    sampler = ClockSampler(local) if rank == 0 and not args.no_clock_sampler else None
    for _ in range(max(args.warmup, 3)):
        step()
    if sampler:
        sampler.mark()
    ms_step, loss = timed(lambda: step(copy=False), args.steps)    # inputs resident
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": loss, "params": dict(model.named_parameters())})
    launches = model.engine[0].last_launches
    t0 = time.perf_counter()
    barrier()
    ms_e2e, _ = timed(step, args.steps)                            # H2D of the batch + D2H of the loss inside
    loss_value = float(host_loss[0])
    ms_nosync = timed(lambda: step(sync=False, copy=False), args.steps)[0] if world > 1 else ms_step
    # the gradient all-reduce alone: one flat fp32 buffer of all hot-path gradients
    ar_ms = None
    if world > 1:
        flat = torch.zeros(n_params, device=dev)
        for _ in range(3):
            dist.all_reduce(flat)
        ar_ms = timed(lambda: dist.all_reduce(flat), 10)[0]
        del flat
    # where the step goes on one rank: forward (kernels), backward (recompute + autograd), optimizer + repack
    def phase_times():
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        for d, s_ in zip(dev_in, host_in):
            d.copy_(s_)
        opt.zero_grad(set_to_none=True)
        torch.cuda.synchronize()
        ev[0].record()
        model.sync()
        ev[1].record()
        out = model(*dev_in)
        loss = _train_loss(out["likelihoods"], out["y_hat"], dev_in[0], pixels)
        ev[2].record()
        loss.backward()
        ev[3].record()
        torch.nn.utils.clip_grad_norm_(params, 1.0)
        opt.step()
        ev[4].record()
        torch.cuda.synchronize()
        return {k: ev[i].elapsed_time(ev[i + 1]) for i, k in enumerate(("repack_weights", "forward_kernels", "backward_recompute", "clip_adam"))}
    phases = phase_times() if rank == 0 else None

    cpu_baseline = torch_gpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        rate, dt, kind = reference_train_rate(cfg, "cpu", B, 1, 1)
        if rate:
            cpu_baseline = {"value": rate, "unit": "images/s", "cores": os.cpu_count(), "kind": kind, "ms_per_step": dt * 1e3,
                            "sample": f"1 step x {B} crops after 1 warm-up: the reference's own classes, torch autograd, fp32, all host threads"}
    if rank == 0 and not args.no_gpu_baseline:
        try:
            rate, dt, kind = reference_train_rate(cfg, dev, B, args.gpu_baseline_steps, 2)
            torch_gpu_baseline = {"value": rate, "unit": "images/s", "ms_per_step": dt * 1e3, "kind": kind,
                                  "sample": f"{args.gpu_baseline_steps} steps x {B} crops: the reference's own classes trained by eager PyTorch on this GPU (fp32, TF32 off)"}
        except Exception as e:                      # noqa: BLE001
            torch_gpu_baseline = {"value": None, "error": repr(e)[:200]}
    if rank == 0:
        imgs = B * world
        line = {
            "metric": "entropy-model training images/sec @256x256 crops", "value": imgs / (ms_step * 1e-3), "unit": "images/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (forward: fp16 hi+lo planes, 3-pass tcgen05; backward: fp32 torch ops)", "data": "synthetic",
            "config": {"workload": cfg["workload"], "config": 4, "mode": "train", "batch_per_gpu": B, "tokens_per_gpu": B * h * w, "math": args.math,
                       "parallelism": f"DDP x{world}, find_unused_parameters=True (train.py:424)", "hot_path_parameters": n_params,
                       "l2": "working set (weights 333 MB fp32 + packed planes) >> 126 MB L2; no flush needed"},
            "e2e": {"value": imgs / (ms_e2e * 1e-3), "unit": "images/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": sum(t.numel() * 4 for t in host_in), "d2h_bytes_per_step": 4,
                    "how": "per step: pinned host batch -> device, forward, loss, backward, all-reduce, clip, Adam, loss -> host"},
            "gpu_launches": launches * args.steps, "gpu_launches_per_step": launches,
            "gpu_launches_note": "launches of this library's kernels in the forward pass of a step (the backward recompute runs torch kernels + dcae_gc_backward)",
            "clocks": clocks,
            "roofline": {"kernel": "forward slice loop (see config #2 for the per-kernel rooflines)", "bound": "tensor", "achieved": None, "peak": None, "unit": "TFLOP/s", "frac": None, "traffic": None,
                         "note": "the training step is dominated by the torch-op backward (phases below); the library's kernels are the forward phase"},
            "phases_ms": phases,
            "allreduce": {"gradient_bytes": n_params * 4, "alone_ms": ar_ms, "exposed_ms": (ms_step - ms_nosync) if world > 1 else 0.0,
                          "note": "alone = one flat fp32 all-reduce of all hot-path gradients; exposed = step time with DDP sync minus the same step under no_sync()"},
            "loss": loss_value,
            "cpu_baseline": cpu_baseline, "torch_gpu_baseline": torch_gpu_baseline,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ---- config 6: the whole model on the library (SURVEY 8f N3 / N4) ------------------------------------------------------
def _codec_params(seed=0):
    from dcae_b200.params import init_entropy_params
    from dcae_b200.transforms import init_transform_params
    P = dict(init_entropy_params(seed, "lively"))
    P.update(init_transform_params(seed))
    return P


def reference_codec_rate(cfg, device, n_images, steps, warmup):
    """The reference's own `DCAE.forward` (unmodified models/dcae.py staged in oracle/_ref; EntropyBottleneck = the loader's
    stub, GaussianConditional = the oracle restatement: compressai is absent) by eager PyTorch, fp32, the reference's
    evaluation flags.  -> (images/s, seconds per step) or (None, None) without the staged file."""
    from oracle import reference_loader as rl
    if not rl.reference_available():
        return None, None
    saved = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.enabled)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cudnn.enabled = False
    try:
        net = rl.build_reference_net(_codec_params()).to(device)
        x = torch.rand(n_images, 3, (cfg["H"] + 127) // 128 * 128, (cfg["W"] + 127) // 128 * 128, generator=torch.Generator().manual_seed(1234)).to(device)
        cuda = torch.device(device).type == "cuda"
        with torch.no_grad():
            for _ in range(warmup):
                net(x)
            if cuda:
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                net(x)
            if cuda:
                torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / max(steps, 1)
        return n_images / dt, dt
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32, torch.backends.cudnn.enabled = saved


def run_codec(args):
    """config 6: `dcae_b200.DCAECodec.forward` = the reference's whole `DCAE.forward` on the library, images sharded over
    the ranks like the slice loop (no data-path collective)."""
    cfg = CONFIGS[6]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from dcae_b200 import _lib
    from dcae_b200.codec import DCAECodec
    lib = _lib.load()
    B = args.batch or cfg["batch"]
    H, W = (cfg["H"] + 127) // 128 * 128, (cfg["W"] + 127) // 128 * 128
    codec = DCAECodec(_codec_params(), device=dev, math=args.math, lanes=args.lanes)
    host_x = torch.rand(B, 3, H, W, generator=torch.Generator().manual_seed(1234 + rank)).pin_memory()
    dev_x = host_x.to(dev)
    host_out = torch.empty(B, 3, H, W).pin_memory()
    host_bits = torch.empty(2).pin_memory()

    def step_resident():
        return codec.forward(dev_x)

    def step_e2e():
        x = host_x.to(dev, non_blocking=True)
        o = codec.forward(x)
        host_out.copy_(o["x_hat"], non_blocking=True)
        host_bits.copy_(torch.stack([o["log2_lik_sum_y"].reshape(()), torch.log2(o["likelihoods"]["z"]).sum()]), non_blocking=True)
        return o

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms) / steps, out

    sampler = ClockSampler(local) if rank == 0 and not args.no_clock_sampler else None
    warm = max(args.warmup, 3)
    t_w = time.perf_counter()
    n_warm = 0
    while n_warm < warm or (time.perf_counter() - t_w) < args.warmup_seconds:
        step_resident()
        torch.cuda.synchronize()
        n_warm += 1
    if sampler:
        sampler.mark()
    ms_step, out = timed(step_resident, args.steps)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)
    del out                                     # held, it would make the first e2e step allocate a second output set
    ms_e2e, _ = timed(step_e2e, args.steps)

    # launches of one step: the library's counter restarts when the slice loop loads its inputs, so read it on both sides
    torch.cuda.synchronize()
    c_prev = int(lib.dcae_launch_count())
    y = codec.stacks["g_a"](dev_x)
    z = codec.stacks["h_a"](y)
    z_hat, _ = codec.entropy_bottleneck(z, training=False)
    ls, lm = codec.stacks["h_z_s1"](z_hat), codec.stacks["h_z_s2"](z_hat)
    c_front = int(lib.dcae_launch_count()) - c_prev
    o = codec.loop.forward(y, ls, lm)
    codec.stacks["g_s"](o["y_hat"])
    launches = c_front + int(lib.dcae_launch_count())
    torch.cuda.synchronize()

    # where the step goes: CUDA events around the stages, and the library's per-family profile (every op timed alone)
    def stage_times():
        names = ("g_a", "h_a", "entropy_bottleneck", "h_z_s1", "h_z_s2", "slice_loop", "g_s")
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
        ev[0].record()
        y = codec.stacks["g_a"](dev_x); ev[1].record()
        z = codec.stacks["h_a"](y); ev[2].record()
        z_hat, _ = codec.entropy_bottleneck(z, training=False); ev[3].record()
        ls = codec.stacks["h_z_s1"](z_hat); ev[4].record()
        lm = codec.stacks["h_z_s2"](z_hat); ev[5].record()
        o = codec.loop.forward(y, ls, lm); ev[6].record()
        codec.stacks["g_s"](o["y_hat"]); ev[7].record()
        torch.cuda.synchronize()
        return {n: ev[i].elapsed_time(ev[i + 1]) for i, n in enumerate(names)}
    stages = stage_times() if rank == 0 else None
    fam = None
    if rank == 0:
        import ctypes as C
        ms = (C.c_double * 4)(); work = (C.c_double * 4)(); ln = (C.c_int64 * 4)()
        saved_lanes = codec.loop.lanes
        codec.loop.lanes = 1
        _lib.check(lib.dcae_profile_start(), "profile_start")
        codec.forward(dev_x)
        torch.cuda.synchronize()
        _lib.check(lib.dcae_profile_stop(ms, work, ln), "profile_stop")
        codec.loop.lanes = saved_lanes
        fam = {n: {"ms_per_step": ms[i], "launches_per_step": int(ln[i]), "work_per_step": work[i]} for i, n in enumerate(("gemm", "attention", "gc", "other"))}
    peaks = load_peaks()
    cpu_baseline = torch_gpu_baseline = None
    if rank == 0 and not args.no_gpu_baseline:
        try:
            n_g = min(B, 4)
            rate, dt = reference_codec_rate(cfg, dev, n_g, 3, 1)
            if rate:
                torch_gpu_baseline = {"value": rate, "unit": "images/s", "ms_per_step": dt * 1e3, "kind": "reference",
                                      "sample": f"3 steps x {n_g} images of 768x512 after 1 warm-up: the reference's own DCAE.forward by eager PyTorch on this GPU (fp32, TF32 off, cuDNN off: eval.py:3182-3187, 3904)"}
        except Exception as e:                      # noqa: BLE001
            torch_gpu_baseline = {"value": None, "error": repr(e)[:200]}
    if rank == 0 and not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        rate, dt = reference_codec_rate(cfg, "cpu", 1, 1, 0)
        if rate:
            cpu_baseline = {"value": rate, "unit": "images/s", "cores": os.cpu_count(), "kind": "reference", "ms_per_step": dt * 1e3,
                            "sample": "1 step x 1 image of 768x512, no warm-up: the reference's own DCAE.forward, torch fp32 on all host threads"}
    if rank == 0:
        imgs = B * world
        g = fam["gemm"] if fam else None
        achieved = (g["work_per_step"] / (g["ms_per_step"] * 1e-3) / 1e12) if g and g["ms_per_step"] > 0 else None
        peak = peaks["tc_sustained"]
        line = {
            "metric": "whole-codec images/sec @768x512", "value": imgs / (ms_step * 1e-3), "unit": "images/s",
            "n_gpus": world, "steps": args.steps, "warmup": warm, "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (fp16 hi+lo planes = 22-bit operands, 3-pass tcgen05, fp32 accumulate)" if args.math == "f16x3" else args.math, "data": "synthetic",
            "config": {"workload": cfg["workload"], "config": 6, "mode": "codec", "batch_per_gpu": B, "math": args.math,
                       "weights": "random-init (seeded: init_entropy_params + init_transform_params)", "lanes_per_gpu": args.lanes,
                       "l2": "no flush needed: per-step working set (several GB of activations) >> 126 MB L2", "warmup_steps_run": n_warm,
                       "parallelism": f"{world} independent image shards"},
            "e2e": {"value": imgs / (ms_e2e * 1e-3), "unit": "images/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": host_x.numel() * 4, "d2h_bytes_per_step": host_out.numel() * 4 + 8,
                    "how": "per step: pinned host images -> device, DCAECodec.forward, x_hat and the two log2-likelihood sums -> pinned host (copies on the compute stream, not overlapped)"},
            "gpu_launches": launches * args.steps, "gpu_launches_per_step": launches,
            "clocks": clocks, "stages_ms": stages, "kernel_families": fam,
            "roofline": {"kernel": "gemm_f16x3 family over the whole model", "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                         "frac": (achieved / peak) if achieved and peak else None, "traffic": None,
                         "note": "achieved = algorithmic 2*T*N*K flop of every dense-layer launch (zero-padded channels and the zero taps of the space-to-depth / 4-phase forms included) / their summed CUDA-event time; 3-pass fp16 ceiling = 1/3 of the peak"},
            "cpu_baseline": cpu_baseline, "torch_gpu_baseline": torch_gpu_baseline,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


class _null:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False



def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--math", default="f16x3", choices=["f16x3", "f16", "tf32x3", "tf32", "fp32"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS), help="BASELINE.json config number (2 = the headline)")
    ap.add_argument("--mode", default=None, choices=["forward", "compress"], help="override the config's mode")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (default: the config's)")
    ap.add_argument("--cpu-steps", type=int, default=2, help="steps of the in-line cpu_baseline leg (same batch as the GPU arm for config #2, one image otherwise)")
    ap.add_argument("--gpu-baseline-steps", type=int, default=5)
    ap.add_argument("--lanes", type=int, default=2, help="sub-batches run on separate streams by EntropySliceLoop.forward")
    ap.add_argument("--warmup-seconds", type=float, default=1.5, help="keep warming up until the device has been busy this long (0 under ncu)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="skip the eager-PyTorch-on-GPU oracle leg")
    ap.add_argument("--no-clock-sampler", action="store_true", help="diagnostic: do not poll NVML during the timed region")
    ap.add_argument("--gc-micro-mb", type=int, default=1024, help="footprint of the kernel-3 HBM microbenchmark")
    ap.add_argument("--no-whole-codec", action="store_true", help="skip the secondary whole-model figure of the default line")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed on rank 0 (the outputs; for --config 4 the loss "
                         "and the updated parameters) as DIR/<name>.npy, float32 / float64, under 64 MB in all: a larger "
                         "array becomes a fixed seeded sample (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what this library computes: not with --impl reference")
    if args.mode:
        CONFIGS[args.config] = dict(CONFIGS[args.config], mode=args.mode)
    if args.impl == "reference":
        return run_reference(args)
    if args.config == 4:
        return run_training(args)
    if args.config == 6:
        return run_codec(args)
    cfg = CONFIGS[args.config]
    compress = cfg["mode"] == "compress"

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    binding = bind_rank_to_cores(local, int(os.environ.get("LOCAL_WORLD_SIZE", world))) if world > 1 else {"bound": False}
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from dcae_b200 import _lib
    from dcae_b200.entropy_model import EntropySliceLoop
    from dcae_b200.params import init_entropy_params
    from dcae_b200.sharding import max_over_ranks

    B = args.batch or cfg["batch"]
    h, w = latent_hw(cfg)
    T = B * h * w
    eng = EntropySliceLoop(init_entropy_params(0, "lively"), device=dev, math=args.math, lanes=args.lanes)
    host_in = synth_latents(B, h, w, seed=1234 + rank, pin=True)
    dev_in = [t.to(dev) for t in host_in]
    lib = _lib.load()

    out_buf = eng.forward(*dev_in, want_symbols=compress)   # outputs are allocated once and overwritten in place (forward(out=...)):
                                               # a cudaMalloc inside the timed region synchronises the device (measured:
                                               # 150-400 ms in the one step that had to grow the caching allocator's pool)
    def step_resident():
        return eng.forward(*dev_in, want_symbols=compress, out=out_buf)

    from dcae_b200.pipeline import HostPipeline
    pipe = HostPipeline(eng, B, h, w, mode=cfg["mode"])      # the public host-facing call: pinned host in, pinned host out

    def run_e2e(steps):
        last = None
        for last in pipe.run(host_in for _ in range(steps)):
            pass
        return last

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dbg = [] if os.environ.get("DCAE_BENCH_DEBUG") else None
        e0.record()
        for _ in range(steps):
            out = fn()
            if dbg is not None:
                ev = torch.cuda.Event(enable_timing=True); ev.record(); dbg.append((ev, time.perf_counter()))
        e1.record()
        torch.cuda.synchronize()
        if dbg:
            ts = [e0.elapsed_time(ev) for ev, _ in dbg]
            print(f"[rank {rank}] per-step device ms: {[round(b - a, 1) for a, b in zip([0.0] + ts[:-1], ts)]}", file=sys.stderr, flush=True)
            print(f"[rank {rank}] host enqueue ms since first: {[round((t - dbg[0][1]) * 1e3, 1) for _, t in dbg]}", file=sys.stderr, flush=True)
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if os.environ.get("DCAE_BENCH_DEBUG"):
            print(f"[rank {rank}] timed region {float(ms) / steps:.3f} ms/step", file=sys.stderr, flush=True)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        barrier()
        return float(ms) / steps, out

    # the sampler starts BEFORE the warm-up (NVML start-up must not land inside the timed region)
    sampler = ClockSampler(local) if rank == 0 and not args.no_clock_sampler else None
    # warm-up: W steps (>= 3), and keep going until the device has been busy for ~1.5 s -- a fresh box needs that long
    # to page in, ramp its clocks and settle under the power cap (three 15 ms steps do not)
    n_warm, t_warm = 0, time.perf_counter()
    while n_warm < max(args.warmup, 3) or time.perf_counter() - t_warm < args.warmup_seconds:
        step_resident()
        torch.cuda.synchronize()
        n_warm += 1
    if sampler:
        sampler.mark()
    ms_step, out = timed(step_resident, args.steps)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out)
    launches = eng.last_launches
    run_e2e(3)
    barrier()
    t0 = time.perf_counter()
    host_res = run_e2e(args.steps)             # returns after the last result is in host memory
    ms_e2e = (time.perf_counter() - t0) * 1e3 / args.steps
    if world > 1:
        ms_e2e = max_over_ranks(ms_e2e, dev)
    barrier()
    # the copies of a step alone (no compute), all ranks at once: the host-side ceiling of the e2e figure
    def copies_only():
        for d, s_ in zip(dev_in, host_in):
            d.copy_(s_, non_blocking=True)
        for key, dst in pipe.host_out[0].items():
            dst.copy_(pipe.dev_out[0][key], non_blocking=True)
    for _ in range(2):
        copies_only()
    barrier()
    t0c = time.perf_counter()
    for _ in range(5):
        copies_only()
    torch.cuda.synchronize()
    ms_copy = (time.perf_counter() - t0c) * 1e3 / 5
    if world > 1:
        ms_copy = max_over_ranks(ms_copy, dev)
    barrier()
    if compress:
        assert int(host_res["overflow"][0]) == 0 and int(host_res["indexes8"].max()) <= 63
    else:
        assert bool(torch.isfinite(host_res["likelihoods"]).all())

    # bpp over all ranks: the only data-path reduction (SURVEY §8e) -- one scalar all-reduce
    from dcae_b200.sharding import reduce_bpp
    bpp = reduce_bpp(out["log2_lik_sum"], B * cfg["H"] * cfg["W"])

    # per-kernel-family device time of one instrumented step (CUDA events on the launching stream)
    ms = (C.c_double * 4)(); work = (C.c_double * 4)(); cnt = (C.c_int64 * 4)()
    # (one lane, no side stream: every kernel runs ALONE here, so its event time is its own duration; with lanes the
    # kernels of two sub-batches overlap and per-kernel event times would count each other's SM time)
    eng_prof = eng if args.lanes == 1 else EntropySliceLoop(init_entropy_params(0, "lively"), device=dev, math=args.math, lanes=1)
    for _ in range(2):
        eng_prof.forward(*dev_in, want_symbols=compress)
    torch.cuda.synchronize()
    lib.dcae_profile_start()
    for _ in range(2):
        eng_prof.forward(*dev_in, want_symbols=compress)
    lib.dcae_profile_stop(ms, work, cnt)
    del eng_prof
    fam = {n: {"ms_per_step": ms[i] / 2, "launches_per_step": cnt[i] // 2, "work_per_step": work[i] / 2}
           for i, n in enumerate(("gemm", "attention", "gc", "other"))}
    peaks = load_peaks()
    gemm_tflops = fam["gemm"]["work_per_step"] / (fam["gemm"]["ms_per_step"] * 1e-3) / 1e12 if fam["gemm"]["ms_per_step"] else 0.0
    tc_peak = peaks["tc_sustained"]
    roofline = {
        "kernel": {"f16x3": "gemm_f16x3_kernel (+ split_f16_planes_kernel)", "f16": "gemm_f16x3_kernel, single pass (hi planes only)", "tf32x3": "gemm_tcgen05_kernel / gemm_tcgen05_2cta_kernel",
                   "tf32": "gemm_tcgen05_kernel", "fp32": "gemm_simt_kernel"}[args.math],
        "bound": "tensor", "achieved": gemm_tflops, "peak": tc_peak, "unit": "TFLOP/s", "frac": gemm_tflops / tc_peak,
        "traffic": ncu_traffic("prof_gemm_final_summary.csv") if args.math == "f16x3" else None,
        "traffic_note": "mean dram__bytes_read + write per launch over the launches of profiles/r02/prof_gemm_final_summary.csv (ncu --set full, same command); operands are L2-resident between layers, so DRAM traffic is below the algorithmic operand bytes",
        "note": (f"achieved = algorithmic 2*T*N*K flop of all {fam['gemm']['launches_per_step']} dense-layer launches of a step / "
                 f"their summed CUDA-event time; peak = {peaks['src']} sustained dense bf16 (kernel timed inside a long step). "
                 + {"f16": "Reduced-precision fast mode: one fp16 MMA per algorithmic MAC (hi planes only).",
                    "f16x3": "Arithmetic is 3 fp16 MMAs (hi/lo operand planes, fp32 accumulate) per algorithmic MAC: ceiling = 1/3 of this peak; the fp16 plane split of each operand is included in the timed launches.",
                    "tf32x3": "Arithmetic is 3 TF32 MMAs per algorithmic MAC at half the bf16 rate: ceiling = 1/6 of this peak.",
                    "tf32": "Arithmetic is TF32 (half the bf16 rate): ceiling = 1/2 of this peak.",
                    "fp32": "FFMA reference mode: tensor cores unused."}[args.math]),
        "share_of_step": fam["gemm"]["ms_per_step"] / max(sum(f["ms_per_step"] for f in fam.values()), 1e-9),
    }

    # kernel 3 alone at an HBM-sized footprint (SURVEY §7: per-slice launches are L2-resident at B=16)
    roofline_gc = None
    if rank == 0:
        roofline_gc = gc_microbench(dev, lib, args.gc_micro_mb, peaks, variant="compress" if compress else "forward")
        other = gc_microbench(dev, lib, args.gc_micro_mb, peaks, variant="forward" if compress else "compress")
        ref_math = gc_microbench(dev, lib, args.gc_micro_mb, peaks, variant="compress", lik_math="reference")
        roofline_gc["other_variants"] = [{k: r[k] for k in ("variant", "lik_math", "achieved", "frac", "ms")} for r in (other, ref_math)]
        roofline_gc["in_loop"] = {"ms_per_step": fam["gc"]["ms_per_step"], "launches_per_step": fam["gc"]["launches_per_step"],
                                  "GB/s": fam["gc"]["work_per_step"] / max(fam["gc"]["ms_per_step"], 1e-9) / 1e6,
                                  "traffic": ncu_traffic("prof_gc_final_summary.csv"),
                                  "traffic_note": "DRAM bytes per in-loop launch (ncu --set full): the 18.9 MB of inputs; the 25 MB of outputs stay in L2"}

    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        n_cpu = B if args.config == 2 else 1            # bounded sample: ~10-30 s of host work
        rate, threads, dt, kind = cpu_reference_rate(cfg, n_cpu, args.cpu_steps, 1)
        cpu_baseline = {"value": rate, "unit": "images/s", "cores": threads, "kind": kind, "ms_per_step": dt * 1e3,
                        "sample": f"{args.cpu_steps} steps x {n_cpu} images of {cfg['tag']} after 1 warm-up, torch fp32 on all host threads: "
                                  + ("the unmodified reference classes of models/dcae.py (oracle/_ref), DCAE.%s slice loop on injected latents" % cfg["mode"]
                                     if kind == "reference" else "oracle port of dcae.py:638-670")}

    h2d_bytes, d2h_bytes = pipe.h2d_bytes, pipe.d2h_bytes
    torch_gpu_baseline = None
    if rank == 0 and not args.no_gpu_baseline:
        del eng, pipe, out_buf, out, host_res       # free the plans' workspaces before the eager run needs its temporaries
        torch.cuda.empty_cache()
        try:
            gs = args.gpu_baseline_steps if not compress else 2
            rate, dt, kind = gpu_eager_rate(cfg, dev, B, gs, 2)
            rate_tf32, dt_tf32, _ = gpu_eager_rate(cfg, dev, B, gs, 2, tf32=True)
            torch_gpu_baseline = {"value": rate, "unit": "images/s", "ms_per_step": dt * 1e3, "kind": kind,
                                  "sample": f"{gs} steps x {B} images of {cfg['tag']} after 2 warm-ups: the reference's own classes (DCAE.{cfg['mode']} slice loop on injected latents) "
                                            "run by eager PyTorch on this GPU with the reference's evaluation flags (fp32, TF32 off, cuDNN off: eval.py:3182-3187, 3904)",
                                  "tf32_on": {"value": rate_tf32, "ms_per_step": dt_tf32 * 1e3,
                                              "note": "same with TF32 and cuDNN on (reduced precision: not the parity setting)"}}
        except Exception as e:                      # noqa: BLE001  (a baseline leg must never take the bench line down)
            torch_gpu_baseline = {"value": None, "error": repr(e)[:200]}

    # secondary figure (never the headline): the WHOLE model on the library, SURVEY 8f N3 / N4 -- see `--config 6` for the full line
    whole_codec = None
    if rank == 0 and world == 1 and args.config == 2 and not args.no_whole_codec:
        try:
            torch.cuda.empty_cache()
            whole_codec = whole_codec_figure(dev, args.math, B, cfg)
        except Exception as e:                      # noqa: BLE001
            whole_codec = {"value": None, "error": repr(e)[:200]}

    if rank == 0:
        imgs = B * world
        line = {
            "metric": f"entropy-model images/sec @{cfg['tag']}", "value": imgs / (ms_step * 1e-3), "unit": "images/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"f16": "f16 operands (hi planes only), fp32 accumulate: reduced-precision fast mode, NOT the parity mode",
                      "f16x3": "f32 (fp16 hi+lo planes = 22-bit operands, 3-pass tcgen05, fp32 accumulate)",
                      "tf32x3": "f32 (3xTF32 error-compensated tcgen05, fp32 accumulate)", "tf32": "tf32", "fp32": "f32"}[args.math],
            "data": "synthetic",
            "config": {"workload": cfg["workload"], "config": args.config, "mode": cfg["mode"],
                       "batch_per_gpu": B, "tokens_per_gpu": T, "math": args.math, "weights": "random-init (seeded, lively profile)",
                       "l2": f"no flush needed: per-step working set {T * 110e3 / 1e9:.1f} GB >> 126 MB L2" if T >= 4096 else "working set is L2-sized at this config (latency-bound single image)", "parallelism": f"{world} independent image shards", "lanes_per_gpu": args.lanes,
                       "warmup_steps_run": n_warm},
            "e2e": {"value": imgs / (ms_e2e * 1e-3), "unit": "images/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                    "copies_only_ms_per_step": ms_copy, "copies_only_GBps_per_rank": (h2d_bytes + d2h_bytes) / (ms_copy * 1e-3) / 1e9,
                    "host_binding": binding,
                    "how": "dcae_b200.HostPipeline(mode=%r): pinned host tensors in and out, H2D / compute / D2H of consecutive batches overlapped on 3 streams (wall clock over the K steps, last result on the host)" % cfg["mode"]
                           + ("; results = int16 symbols + uint8 indexes in coder order (what DCAE.compress hands to the range coder), y_hat stays on the device" if compress else "; results = y_hat, means, scales, likelihoods fp32")},
            "gpu_launches": launches * args.steps,
            "gpu_launches_per_step": launches,
            "clocks": clocks,
            "roofline": roofline,
            "roofline_gc": roofline_gc,
            "kernel_families": fam,
            "step_tflops": FLOP_PER_TOKEN * T / (ms_step * 1e-3) / 1e12,
            "bpp": bpp,
            "cpu_baseline": cpu_baseline,
            "torch_gpu_baseline": torch_gpu_baseline,
            "whole_codec": whole_codec,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def whole_codec_figure(dev, math, B, cfg):
    """`DCAECodec.forward` (g_a, h_a, entropy bottleneck, h_z_s1 / h_z_s2, slice loop, g_s) on B images of the config's size:
    5 device-timed steps after 3 warm-ups, plus the per-stage CUDA-event times of one more."""
    from dcae_b200.codec import DCAECodec
    codec = DCAECodec(_codec_params(), device=dev, math=math)
    H, W = (cfg["H"] + 127) // 128 * 128, (cfg["W"] + 127) // 128 * 128
    x = torch.rand(B, 3, H, W, generator=torch.Generator().manual_seed(1234)).to(dev)
    for _ in range(3):
        codec.forward(x)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        codec.forward(x)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    names = ("g_a", "h_a", "entropy_bottleneck", "h_z_s1", "h_z_s2", "slice_loop", "g_s")
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
    ev[0].record()
    y = codec.stacks["g_a"](x); ev[1].record()
    z = codec.stacks["h_a"](y); ev[2].record()
    z_hat, _ = codec.entropy_bottleneck(z, training=False); ev[3].record()
    ls = codec.stacks["h_z_s1"](z_hat); ev[4].record()
    lm = codec.stacks["h_z_s2"](z_hat); ev[5].record()
    o = codec.loop.forward(y, ls, lm); ev[6].record()
    codec.stacks["g_s"](o["y_hat"]); ev[7].record()
    torch.cuda.synchronize()
    return {"metric": "whole-codec images/sec @768x512 (secondary figure; `bench.py --config 6` prints the full line)", "value": B / (ms * 1e-3), "unit": "images/s",
            "ms_per_step": ms, "batch": B, "stages_ms": {n: ev[i].elapsed_time(ev[i + 1]) for i, n in enumerate(names)},
            "what": "DCAECodec.forward = the reference's whole DCAE.forward (dcae.py:623-677) on libdcae_b200.so, inputs resident, 5 steps after 3 warm-ups"}


def gc_microbench(dev, lib, mb, peaks, variant="compress", lik_math="fast"):
    """Kernel 3 timed alone on inputs far larger than L2.  variant "compress": y, mu, scale in; lik, y_hat, sym, idx out
    = 28 B/element (SURVEY 8d); "forward": no int32 stores = 20 B/element."""
    from dcae_b200 import _lib
    bpe = GC_BYTES_PER_ELEM if variant == "compress" else 20
    n = mb * (1 << 20) // bpe // 64 * 64
    rows = n // 64
    g = torch.Generator(device=dev).manual_seed(1)
    y = 4 * torch.randn(rows, 64, device=dev, generator=g)
    mu = 2 * torch.randn(rows, 64, device=dev, generator=g)
    sc = torch.exp(torch.empty(rows, 64, device=dev).uniform_(-3.0, 5.7, generator=g))
    from dcae_b200.entropy_model import get_scale_table
    table = get_scale_table().to(dev)
    outs = [torch.empty(rows, 64, device=dev), torch.empty(rows, 64, device=dev)]
    a = _lib.GcArgs()
    a.y, a.y_ld, a.mu, a.mu_ld, a.scale, a.scale_ld = y.data_ptr(), 64, mu.data_ptr(), 64, sc.data_ptr(), 64
    a.scale_table, a.n_table, a.scale_bound, a.lik_bound, a.mode = table.data_ptr(), 64, 0.11, 1e-9, 0
    a.rows, a.inner = rows, 64
    a.lik_math = _lib.GC_LIK[lik_math]
    a.y_hat, a.y_hat_ld, a.lik, a.lik_ld = outs[0].data_ptr(), 64, outs[1].data_ptr(), 64
    if variant == "compress":
        outs += [torch.empty(rows, 64, device=dev, dtype=torch.int32), torch.empty(rows, 64, device=dev, dtype=torch.int32)]
        a.sym, a.sym_ld, a.idx, a.idx_ld = outs[2].data_ptr(), 64, outs[3].data_ptr(), 64
    s = _lib.current_stream(dev)
    torch.cuda.synchronize()
    time.sleep(0.3)                 # a kernel timed ALONE: let the power state of the preceding GEMM loop settle
    for _ in range(3):
        _lib.check(lib.dcae_gc_fused(a, s))
    reps, rounds = 10, []
    for _ in range(3):              # three rounds of 10 launches, the median round is reported
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            lib.dcae_gc_fused(a, s)
        e1.record()
        torch.cuda.synchronize()
        rounds.append(e0.elapsed_time(e1) / reps)
    ms = sorted(rounds)[1]
    gbs = n * bpe / (ms * 1e-3) / 1e9
    return {"kernel": "gc_fused_kernel", "bound": "hbm", "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s",
            "frac": gbs / peaks["hbm"], "traffic": None, "elements": n, "ms": ms, "variant": variant, "lik_math": lik_math,
            "note": f"kernel 3 alone, {n * bpe / 2**20:.0f} MiB algorithmic footprint ({bpe} B/element, {variant} variant, likelihood math {lik_math!r}), peak = {peaks['src']} copy bandwidth"}


if __name__ == "__main__":
    main()
