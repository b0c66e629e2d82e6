"""MS-SSIM on the library against the same math in torch (oracle/msssim.py, fp32, cuDNN on, TF32 off so that both sides
compute in fp32).

    python tools/msssim_bench.py [--rounds 7] [--iters 10] [--out profiles/r03/msssim_bench.log]

For 16 x 3 x 512x768 and 8 x 3 x 256x256 (the reference's training crop): median time (CUDA events, after warm-up)
of the forward value and of forward + backward, both ways; the value and gradient differences against the fp64 oracle;
and achieved bytes/s of the library from the byte model below, with the share of the B200's 7.7 TB/s it implies.
The 16 x 3 x 512x768 pair (151 MB) does not fit the 126 MB L2; the 8 x 3 x 256x256 pair (6.3 MB) does, and stays in
L2 between iterations.  The device name and power limit are read in the same run and printed first.
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from dcae_b200.msssim import ms_ssim  # noqa: E402
from oracle import msssim as oms  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
SHAPES = [(16, 3, 512, 768), (8, 3, 256, 256)]


def levels(H, W):
    out = [(H, W)]
    for _ in range(4):
        h, w = out[-1]
        out.append(((h + 1) // 2, (w + 1) // 2))
    return out


def model(B, C, H, W):
    """(forward bytes, backward bytes, forward flops, backward flops) the algorithm needs, fp32.
    Bytes: forward reads X and Y of every level and writes the pooled X and Y of the next (the level's second read of
    the same tile for pooling is an L1/L2 hit and not counted); backward reads X, Y and the coarser dX and writes dX of
    every level.  Flops: 11-tap separable passes at 2 flop per tap -- forward five moments horizontally over h x (w-10)
    and vertically over the valid map; backward the same moments again plus three maps through the full correlation
    (horizontally over (h+10) x w, vertically over h x w).  The per-pixel epilogues (~20 flop) are left out."""
    P = B * C
    fb = bb = ff = bf = 0
    lv = levels(H, W)
    for i, (h, w) in enumerate(lv):
        hv, wv = h - 10, w - 10
        fb += 8 * h * w + (8 * lv[i + 1][0] * lv[i + 1][1] if i < 4 else 0)
        bb += 8 * h * w + 4 * h * w + (4 * lv[i + 1][0] * lv[i + 1][1] if i < 4 else 0)
        moments = 5 * 22 * (h * wv + hv * wv)
        ff += moments
        bf += moments + 3 * 22 * ((h + 10) * w + h * w)
    return fb * P, bb * P, ff * P, bf * P


def timed(fn, iters, rounds):
    fn()
    torch.cuda.synchronize()
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
    return times[len(times) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("msssim_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.backends.cudnn.enabled = True
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    lines = []

    def emit(s):
        print(s, flush=True)
        lines.append(s)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                             text=True).stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        smi = "nvidia-smi unavailable"
    emit(f"device: {torch.cuda.get_device_name(dev)} | {smi} | torch {torch.__version__} | cudnn {torch.backends.cudnn.version()}")
    for B, C, H, W in SHAPES:
        g = torch.Generator(device=dev).manual_seed(H + W)
        X = torch.rand(B, C, H, W, device=dev, generator=g)
        Y = (X + 0.08 * torch.randn(B, C, H, W, device=dev, generator=g)).clamp(0, 1)
        Xr = X.clone().requires_grad_(True)

        def lib_fwd():
            with torch.no_grad():
                ms_ssim(X, Y)

        def lib_fwd_bwd():
            Xr.grad = None
            ms_ssim(Xr, Y).backward()

        def torch_fwd():
            with torch.no_grad():
                oms.ms_ssim(X, Y)

        def torch_fwd_bwd():
            Xr.grad = None
            oms.ms_ssim(Xr, Y).backward()

        t = {name: timed(fn, args.iters, args.rounds) for name, fn in
             (("lib_fwd", lib_fwd), ("lib_fb", lib_fwd_bwd), ("torch_fwd", torch_fwd), ("torch_fb", torch_fwd_bwd))}
        # parity at the timed size
        Xr.grad = None
        v = ms_ssim(Xr, Y)
        v.backward()
        g_lib = Xr.grad.detach().clone()
        Xr.grad = None
        v32 = oms.ms_ssim(Xr, Y)
        v32.backward()
        g_t32 = Xr.grad.detach().clone()
        X64 = X.double().requires_grad_(True)
        v64 = oms.ms_ssim(X64, Y.double())
        v64.backward()

        def rel(a):
            return float((a.double() - X64.grad).norm() / X64.grad.norm())
        fb, bb, ff, bf = model(B, C, H, W)
        t_bwd = t["lib_fb"] - t["lib_fwd"]
        emit(f"{B}x{C}x{H}x{W}: forward library {t['lib_fwd'] * 1e3:.1f} us | torch (cuDNN, fp32) {t['torch_fwd'] * 1e3:.1f} us | "
             f"x{t['torch_fwd'] / t['lib_fwd']:.1f}")
        emit(f"{B}x{C}x{H}x{W}: forward+backward library {t['lib_fb'] * 1e3:.1f} us | torch (cuDNN, fp32) {t['torch_fb'] * 1e3:.1f} us | "
             f"x{t['torch_fb'] / t['lib_fb']:.1f}")
        emit(f"{B}x{C}x{H}x{W}: library forward {fb / 1e6:.1f} MB, {ff / 1e9:.2f} GFLOP -> {fb / t['lib_fwd'] / 1e6:.0f} GB/s "
             f"({100 * fb / t['lib_fwd'] * 1e3 / HBM_BYTES_PER_S:.1f}% of 7.7 TB/s), {ff / t['lib_fwd'] / 1e9:.1f} TFLOP/s; "
             f"backward (fwd+bwd minus fwd, {t_bwd * 1e3:.1f} us) {bb / 1e6:.1f} MB, {bf / 1e9:.2f} GFLOP -> "
             f"{bb / t_bwd / 1e6:.0f} GB/s ({100 * bb / t_bwd * 1e3 / HBM_BYTES_PER_S:.1f}%), {bf / t_bwd / 1e9:.1f} TFLOP/s")
        emit(f"{B}x{C}x{H}x{W}: vs fp64 oracle: value library {abs(float(v) - float(v64)):.1e} | torch fp32 {abs(float(v32) - float(v64)):.1e}; "
             f"gradient ||d||/||g|| library {rel(g_lib):.1e} | torch fp32 {rel(g_t32):.1e}")
        del X, Y, Xr, X64
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
