"""The y range coder: the opt-in ilv1 format on the GPU (csrc/rans_gpu.cu) against the host coder (libdcae_rans.so).

    python tools/rans_gpu_bench.py [--reps N]

1. Coder only, on the symbols / indexes the library's own slice loop produces for random images (random-init weights,
   `init_entropy_params(7, "lively")` + `init_transform_params(2)`), at 768x512 (B = 1 and 16), 2048x1365 and 3840x2160:
   - GPU encode: `EntropySliceLoop.encode_symbols_interleaved` (device symbols -> B strings on the host, both copies and
     syncs included), L = 32;
   - host encode: the reference format (`BufferedRansEncoder` over the packed host arrays the default path codes) and the
     host ilv1 coder (`ans.encode_interleaved`, one call per image), D2H copies excluded;
   - GPU decode: `decode_symbols_interleaved` (upload, five slice launches, status read) given the indexes;
   - host decode: `RansDecoder.decode_array` over the five slices, indexes already on the host.
2. Whole `DCAECodec.encode_image / decode_image` per coder at 768x512 and 2048x1365.
3. Bytes per image for each L against the reference format, at 768x512 and 2048x1365 (random-init weights code far
   more bits than a trained model, so the relative overhead here understates what a trained model would see).
Each time is the median of --reps calls after two warm-up calls, a host clock around work that ends in a device sync.
"""
from __future__ import annotations

import argparse
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SIZES = [("768x512", 512, 768, 1), ("768x512", 512, 768, 16), ("2048x1365", 1365, 2048, 1), ("3840x2160", 2160, 3840, 1)]


def timed(fn, reps):
    import torch
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return 1e3 * statistics.median(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("rans_gpu_bench.py measures the GPU coder: no CUDA device")
    import __graft_entry__ as ge
    ge.build()
    from dcae_b200 import DCAECodec, ans, container
    from dcae_b200.params import init_entropy_params
    from dcae_b200.transforms import init_transform_params
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(f"device: {gpu[0] if gpu else torch.cuda.get_device_name(0)}  (name, power limit, max SM clock)")
    P = init_entropy_params(7, "lively")
    P.update(init_transform_params(2))
    codec = DCAECodec(P, device="cuda:0")
    codec.update()
    loop, gc = codec.loop, codec.gaussian_conditional
    tables = loop._coder_tables(gc)

    print("\n1. coder only (ms, median)")
    print(f"{'size':>10} {'B':>3} {'symbols':>9} | {'GPU enc':>8} {'host enc ref':>12} {'host enc ilv':>12} | {'GPU dec':>8} {'host dec ref':>12}")
    for name, H, W, B in SIZES:
        g = torch.Generator().manual_seed(H * W + B)
        x = torch.rand(B, 3, H, W, generator=g).cuda()
        xp, _ = container.pad(x)
        with torch.no_grad():
            y, z = codec._latents(xp)
            z_hat = codec.entropy_bottleneck.decompress(codec.entropy_bottleneck.compress(z), z.shape[-2:])
            ls, lm = codec.stacks["h_z_s1"](z_hat), codec.stacks["h_z_s2"](z_hat)
            out = loop.compress(y, ls, lm)
        sym, idx = out["symbols"], out["indexes"]
        hs, hi = sym.cpu().numpy(), idx.cpu().numpy()
        strings = loop.encode_symbols_interleaved(sym, idx, gc)
        assert torch.equal(loop.decode_symbols_interleaved(strings, idx, gc), sym)
        assert strings[0] == ans.encode_interleaved(hs[:, 0].reshape(5, -1), hi[:, 0].reshape(5, -1), *tables)

        def host_enc_ref():
            e = ans.BufferedRansEncoder()
            e.encode_with_indexes(hs.astype(np.int16) if np.abs(hs).max() < 32768 else hs, hi.astype(np.uint8), *tables)
            return e.flush()

        ref = host_enc_ref()
        t_gpu_enc = timed(lambda: loop.encode_symbols_interleaved(sym, idx, gc), args.reps)
        t_host_ref = timed(host_enc_ref, args.reps)
        t_host_ilv = timed(lambda: [ans.encode_interleaved(hs[:, b].reshape(5, -1), hi[:, b].reshape(5, -1), *tables)
                                    for b in range(B)], args.reps)
        t_gpu_dec = timed(lambda: loop.decode_symbols_interleaved(strings, idx, gc), args.reps)

        def host_dec_ref():
            d = ans.RansDecoder()
            d.set_stream(ref)
            for s in range(5):
                d.decode_array(hi[s].reshape(-1), *tables)

        t_host_dec = timed(host_dec_ref, args.reps)
        print(f"{name:>10} {B:>3} {sym.numel():>9} | {t_gpu_enc:8.2f} {t_host_ref:12.2f} {t_host_ilv:12.2f} | {t_gpu_dec:8.2f} {t_host_dec:12.2f}")

    print("\n2. whole encode_image / decode_image (ms, median, B = 1)")
    for name, H, W, _ in SIZES[:3:2]:
        x = torch.rand(1, 3, H, W, generator=torch.Generator().manual_seed(3)).cuda()
        for coder in ("reference", "interleaved"):
            blob = codec.encode_image(x, coder=coder)
            assert torch.equal(codec.decode_image(blob, coder=coder), codec.decode_image(codec.encode_image(x)))
            te = timed(lambda: codec.encode_image(x, coder=coder), args.reps)
            td = timed(lambda: codec.decode_image(blob, coder=coder), args.reps)
            print(f"{name:>10} {coder:>11}: encode_image {te:8.2f}  decode_image {td:8.2f}  ({len(blob)} bytes)")

    print("\n3. y bytes per image by L (random-init weights; fixed cost 4 + 5 (4 + 8 L) against 8 for the reference format)")
    for name, H, W, _ in SIZES[:3:2]:
        x = torch.rand(1, 3, H, W, generator=torch.Generator().manual_seed(4)).cuda()
        xp, _ = container.pad(x)
        ref = len(codec.compress(xp)["strings"][0][0])
        row = []
        for lanes in (1, 2, 4, 8, 16, 32):
            n = len(codec.compress(xp, coder="interleaved", lanes=lanes)["strings"][0][0])
            row.append(f"L={lanes}: {n} (+{n - ref}, {100.0 * (n - ref) / ref:+.3f} %)")
        print(f"{name:>10}: reference {ref} bytes; " + "; ".join(row))


if __name__ == "__main__":
    main()
