"""One training step of the whole DCAE (train.py:165-179) at the crops of config #4 (8 and 16 crops of 256x256 per step).

    python tools/dcae_train_step.py [--batches 8 16] [--rounds 5] [--iters 3] [--metric {mse,ms-ssim}]
                                    [--out profiles/r03/dcae_train_step.log]

1. Median step time (CUDA events; one warm-up step, then the median over rounds of `iters` steps) and peak memory
   (max_memory_allocated) of forward, main backward, aux backward and both Adam steps, two ways:
     library   dcae_b200.DCAEModel
     eager     the same graph in eager torch, fp32, TF32 off: transform_graph stacks, torch_graph.slice_loop with a torch
               Gaussian likelihood, and a torch entropy bottleneck
   with the loss of --metric: mse (default) or ms-ssim (library: dcae_rate_distortion_loss(metric="ms-ssim") on the MS-SSIM
   kernels; eager: the same loss with oracle/msssim.py's torch MS-SSIM).
2. The entropy-bottleneck backward kernel alone (dcae_eb_backward) at the training shape of z and at 4 x 3840x2160
   (z = 4 x 192 x 60 x 34 after padding to multiples of 128), against torch autograd of the same likelihood.
The device name and power limit are read in the same run and printed first.
"""
from __future__ import annotations

import argparse
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from dcae_b200 import _lib, torch_graph, transform_graph  # noqa: E402
from dcae_b200.modules import HOT_PREFIXES  # noqa: E402
from oracle import entropy_bottleneck as oeb  # noqa: E402
from oracle import gaussian_conditional as ogc  # noqa: E402
from oracle import msssim as oms  # noqa: E402

C = 192


def timed(fn, iters, rounds):
    """(median ms per call, peak bytes) over `rounds` rounds of `iters` calls, after one warm-up call."""
    fn()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    times = []
    for _ in range(rounds):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b) / iters)
    times.sort()
    return times[len(times) // 2], torch.cuda.max_memory_allocated() - base


def eb_likelihood(p, z, noise):
    """EntropyBottleneck likelihood of z [B, C, h, w] in torch ops (training mode: out = z + noise)."""
    B, _, h, w = z.shape
    lik, _, _ = oeb.likelihood(p, (z + noise).transpose(0, 1).reshape(C, 1, -1))
    return ogc.lower_bound(lik, 1e-9).reshape(C, B, h, w).transpose(0, 1)


def eager_forward(P, x, y_noise, z_noise):
    def sub(pre):
        return {k[len(pre) + 1:]: v for k, v in P.items() if k.startswith(pre + ".")}
    y = transform_graph.stack("g_a", sub("g_a"), x)
    z = transform_graph.stack("h_a", sub("h_a"), y)
    ebp = sub("entropy_bottleneck")
    z_lik = eb_likelihood(ebp, z, z_noise)
    med = ebp["quantiles"][:, 0, 1].detach().reshape(1, C, 1, 1)
    z_hat = torch_graph.ste_round(z - med) + med
    ls, lm = transform_graph.stack("h_z_s1", sub("h_z_s1"), z_hat), transform_graph.stack("h_z_s2", sub("h_z_s2"), z_hat)
    hot = {k: v for k, v in P.items() if k.split(".")[0] in HOT_PREFIXES}
    gc = lambda ys, sc, mu, nz: ogc.lower_bound(ogc.likelihood(ys + nz, sc, mu), 1e-9)      # noqa: E731
    y_hat, mu, sc, y_lik = torch_graph.slice_loop(hot, y, ls, lm, gc, y_noise)
    return {"x_hat": transform_graph.stack("g_s", sub("g_s"), y_hat), "likelihoods": {"y": y_lik, "z": z_lik}}


def eager_aux_loss(P):
    """compressai's aux loss: density parameters detached, the gradient reaches the quantiles only."""
    p = {k[len("entropy_bottleneck."):]: (v if k.endswith(".quantiles") else v.detach()) for k, v in P.items()
         if k.startswith("entropy_bottleneck.")}
    target = math.log(2 / oeb.TAIL_MASS - 1)
    return torch.abs(oeb.logits_cumulative(p, p["quantiles"]) - torch.tensor([-target, 0.0, target], device=p["quantiles"].device)).sum()


def eager_ms_ssim_loss(out, target, lmbda=0.013):
    """dcae_rate_distortion_loss(metric="ms-ssim") with the torch MS-SSIM of the oracle."""
    bpp = sum(torch.log(lik).sum() / (-math.log(2) * target.shape[0] * target.shape[2] * target.shape[3])
              for lik in out["likelihoods"].values())
    msssim = oms.ms_ssim(out["x_hat"], target, data_range=1.0)
    return lmbda * (1 - msssim) + bpp, bpp, msssim


def step_fn(kind, B, dev, metric="mse"):
    from dcae_b200.training import DCAEModel, dcae_rate_distortion_loss
    model = DCAEModel(device=dev, seed=0).train()
    g = torch.Generator(device=dev).manual_seed(B)
    x = torch.rand(B, 3, 256, 256, device=dev, generator=g)
    y_noise = torch.rand(B, 320, 16, 16, device=dev, generator=g) - 0.5
    z_noise = torch.rand(B, C, 4, 4, device=dev, generator=g) - 0.5
    if kind == "library":
        main, aux = model.parameter_groups()
        run, aux_loss = (lambda: model(x, y_noise=y_noise, z_noise=z_noise)), model.aux_loss
    else:
        buffers = {f"entropy_bottleneck.{n}" for n, _ in model.entropy_bottleneck.named_buffers()}
        P = {k: v.detach().clone().requires_grad_(True) for k, v in model.reference_state_dict().items()
             if k not in buffers and not k.startswith("gaussian_conditional.")}
        main = [v for k, v in P.items() if not k.endswith(".quantiles")]
        aux = [v for k, v in P.items() if k.endswith(".quantiles")]
        run, aux_loss = (lambda: eager_forward(P, x, y_noise, z_noise)), (lambda: eager_aux_loss(P))
        del model
    opt, aux_opt = torch.optim.Adam(main, lr=1e-4), torch.optim.Adam(aux, lr=1e-3)
    if kind == "eager" and metric == "ms-ssim":
        loss_fn = eager_ms_ssim_loss
    else:
        loss_fn = lambda out, target: dcae_rate_distortion_loss(out, target, metric=metric)      # noqa: E731

    def fn():
        opt.zero_grad()
        aux_opt.zero_grad()
        loss, _, _ = loss_fn(run(), x)
        loss.backward()
        opt.step()
        aux_loss().backward()
        aux_opt.step()
    return fn


def eb_rows(dev, iters, rounds, batches):
    from dcae_b200.training import EntropyBottleneckModel
    eb = EntropyBottleneckModel(C)
    eb.load_state_dict(oeb.init_params(C, seed=5, trained_like=True), strict=False)
    eb.to(dev).train()
    p = {k: v.detach().clone().requires_grad_(not k.startswith("quantiles")) for k, v in eb.named_parameters()}
    rows = []
    for B, h, w, label in [(b, 4, 4, f"{b}x256x256") for b in batches] + [(4, 34, 60, "4x3840x2160")]:
        g = torch.Generator(device=dev).manual_seed(h * w)
        z = eb.quantiles[:, 0, 1].detach().reshape(1, C, 1, 1) + 4 * torch.randn(B, C, h, w, device=dev, generator=g)
        noise = torch.rand(B, C, h, w, device=dev, generator=g) - 0.5
        cot = torch.randn(B, C, h, w, device=dev, generator=g)
        packed, med = eb._pack(dev)
        lik = eb(z, training=True, noise=noise)[1]
        a = _lib.EbBwdArgs()
        gz, gp = torch.empty_like(z), torch.empty_like(packed)
        a.z, a.noise, a.params, a.medians, a.grad_lik = z.data_ptr(), noise.data_ptr(), packed.data_ptr(), med.data_ptr(), cot.data_ptr()
        a.mode, a.B, a.C, a.HW, a.lik_bound = _lib.GC_NOISE, B, C, h * w, 1e-9
        a.grad_z, a.grad_params = gz.data_ptr(), gp.data_ptr()
        lib, stream = _lib.load(), _lib.current_stream(dev)
        t_k, _ = timed(lambda: _lib.check(lib.dcae_eb_backward(a, stream), "dcae_eb_backward"), iters * 20, rounds)
        zt = z.clone().requires_grad_(True)

        def torch_bwd():
            for v in p.values():
                v.grad = None
            zt.grad = None
            eb_likelihood(p, zt, noise).backward(cot)
        t_t, _ = timed(torch_bwd, iters * 4, rounds)
        n = B * C * h * w
        rows.append(f"dcae_eb_backward z {B}x{C}x{h}x{w} ({label}, {n} elements): {t_k * 1e3:.1f} us ({n / t_k / 1e6:.2f} G elements/s) | "
                    f"torch forward+backward of the same likelihood {t_t * 1e3:.1f} us | lik min {float(lik.min()):.1e}")
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[8, 16])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--metric", choices=["mse", "ms-ssim"], default="mse")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("dcae_train_step.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True).stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        smi = "nvidia-smi unavailable"
    emit(f"device: {torch.cuda.get_device_name(dev)} | {smi} | torch {torch.__version__}")
    for B in args.batches:
        parts = []
        for kind in ("library", "eager"):
            t, mem = timed(step_fn(kind, B, dev, args.metric), args.iters, args.rounds)
            parts.append(f"{kind} {t:.2f} ms {mem / 2**30:.2f} GiB")
            torch.cuda.empty_cache()
        emit(f"train step (forward, main + aux backward, both Adam steps) B={B}x256x256, {args.metric} loss: " + " | ".join(parts))
    for row in eb_rows(dev, args.iters, args.rounds, args.batches):
        emit(row)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
