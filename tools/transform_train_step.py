"""Forward + backward of the transform stacks at the training crops of config #4 (8 and 16 crops of 256x256 per step).

    python tools/transform_train_step.py [--batches 8 16] [--rounds 5] [--iters 3] [--out profiles/r03/transform_train_step.log]

1. Per stack and for g_a + g_s: median step time (CUDA events; warm-up, then the median over rounds of `iters` steps)
   and peak memory (max_memory_allocated) of one forward + backward, three ways:
     library   dcae_b200.TransformModel (kernels forward, recompute backward with the window-attention kernel)
     eager     the same graph (dcae_b200.transform_graph) in eager torch, TF32 off
     reference the reference's own modules, when models/dcae.py is staged (TF32 off)
2. The attention core alone at each Swin level's shape: WindowAttentionFunction forward + backward against torch autograd
   of transform_graph.window_attention, with the achieved rate from 4 T P^2 C (forward) and 10 T P^2 C (backward) flop.
The device name and power limit are read in the same run and printed first.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from dcae_b200 import transform_graph  # noqa: E402
from dcae_b200.transforms import ARCH, init_transform_params  # noqa: E402

# input of each stack for a 256 x 256 crop (dcae.py:623-677: y = g_a(x) is 16 x 16, z = h_a(y) is 4 x 4)
INPUT = {"g_a": (3, 256, 256), "g_s": (320, 16, 16), "h_a": (320, 16, 16), "h_z_s1": (192, 4, 4), "h_z_s2": (192, 4, 4)}


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


def step_fn(kind, stacks, B, dev, ref_net=None):
    """One forward + backward of the chain of `stacks` (g_a + g_s: g_s(g_a(x))) with a fixed cotangent."""
    first = stacks[0]
    x = torch.rand(B, *INPUT[first], device=dev) if first == "g_a" else torch.randn(B, *INPUT[first], device=dev)
    if kind == "library":
        from dcae_b200.training import TransformModel
        mods = [TransformModel(s, init_transform_params(0, (s,)), device=dev) for s in stacks]
        params = [p for m in mods for p in m.parameters()]
        run = lambda t: [t := m(t) for m in mods][-1]                                                  # noqa: E731
    elif kind == "eager":
        P = [{k: v.to(dev).requires_grad_(True) for k, v in init_transform_params(0, (s,), prefixed=False).items()} for s in stacks]
        params = [v for p in P for v in p.values()]
        run = lambda t: [t := transform_graph.stack(s, p, t) for s, p in zip(stacks, P)][-1]           # noqa: E731
    else:
        mods = [getattr(ref_net, s) for s in stacks]
        params = [p for m in mods for p in m.parameters()]
        run = lambda t: [t := m(t) for m in mods][-1]                                                  # noqa: E731
    with torch.no_grad():
        cot = torch.randn_like(run(x))

    def fn():
        for p in params:
            p.grad = None
        y = run(x)
        y.backward(cot)
    return fn


def attention_rows(B, dev, iters, rounds):
    from dcae_b200.training import WindowAttentionFunction
    rows, seen = [], set()
    for stack in ("g_a", "h_a"):
        h, w = INPUT[stack][1:]
        for spec in ARCH[stack]:
            if spec[0] in ("rbws", "conv_s2"):
                h, w = h // 2, w // 2
            if spec[0] != "swin":
                continue
            _, C, hd, win, _n = spec
            key = (C, hd, win, h, w)
            if key in seen:
                continue
            seen.add(key)
            qkv = torch.randn(B, h, w, 3 * C, device=dev, requires_grad=True)
            rel = torch.randn(C // hd, 2 * win - 1, 2 * win - 1, device=dev, requires_grad=True)
            cot = torch.randn(B, h, w, C, device=dev)
            T = B * h * w
            fwd_flop, bwd_flop = 4.0 * T * win * win * C, 10.0 * T * win * win * C
            res = {}
            for name, f in (("kernel", lambda a, r: WindowAttentionFunction.apply(a, hd, win, win // 2, r)),
                            ("torch", lambda a, r: transform_graph.window_attention(a, hd, win, win // 2, r))):
                t_f, _ = timed(lambda: f(qkv, rel), iters, rounds)

                def fb():
                    qkv.grad = rel.grad = None
                    f(qkv, rel).backward(cot)
                t_fb, mem = timed(fb, iters, rounds)
                res[name] = (t_f, t_fb - t_f, mem)
            kf, kb, km = res["kernel"]
            tf, tb, tm = res["torch"]
            rows.append(f"attention {h}x{w} C={C} hd={hd} P={win} SW B={B}: kernel fwd {kf:.3f} ms ({fwd_flop / kf / 1e9:.1f} TFLOP/s) "
                        f"bwd {kb:.3f} ms ({bwd_flop / kb / 1e9:.1f} TFLOP/s) peak {km / 2**20:.0f} MiB | torch fwd {tf:.3f} ms bwd {tb:.3f} ms "
                        f"peak {tm / 2**20:.0f} MiB | backward speed-up {tb / kb:.1f}x")
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[8, 16])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--iters", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("transform_train_step.py needs a CUDA device")
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
    ref_net = None
    try:
        from oracle.reference_loader import load_reference_dcae_module, reference_available
        if reference_available():
            torch.manual_seed(0)
            ref_net = load_reference_dcae_module().DCAE().to(dev).train()
            torch.nn.Module.load_state_dict(ref_net, init_transform_params(0), strict=False)
    except Exception as e:                      # the reference leg is optional: report why it is missing
        emit(f"reference modules unavailable: {e!r}")
    kinds = ["library", "eager"] + (["reference"] if ref_net is not None else [])
    for B in args.batches:
        for stacks in (["g_a"], ["g_s"], ["h_a"], ["h_z_s1"], ["h_z_s2"], ["g_a", "g_s"]):
            parts = []
            for kind in kinds:
                t, mem = timed(step_fn(kind, stacks, B, dev, ref_net), args.iters, args.rounds)
                parts.append(f"{kind} {t:.2f} ms {mem / 2**30:.2f} GiB")
                torch.cuda.empty_cache()
            emit(f"step fwd+bwd {'+'.join(stacks)} B={B}x256x256: " + " | ".join(parts))
        for row in attention_rows(B, dev, args.iters * 3, args.rounds):
            emit(row)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
