"""A/B of the tensor-core GEMM and dictionary-attention kernels between two builds of libdcae_b200.so.

    python tools/gemm_ab.py --lib PATH --out DIR          # GPU box: seeded cases through dcae_op_gemm /
                                                          # dcae_op_dict_attention -> DIR/outputs.pt, DIR/times.json
    python tools/gemm_ab.py --compare DIR_A DIR_B         # every output torch.equal? times side by side

The cases reach every kernel path: tf32x3 on one CTA (short K) and on a thread-block pair (K >= 4096, including an odd
number of token tiles, whose last pair has a tile past the batch) and its one-CTA fallback for a single token tile;
tf32; f16x3 and f16 on one CTA and on a pair with fp32, fp16-plane and GELU-plane outputs; the dictionary attention
in tf32x3, tf32 and f16x3.  One library per process: `_lib` loads one file."""
import argparse
import json
import os
import subprocess
import sys
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# (name, math, B, h, w, K, N, taps, outputs): outputs "o" = fp32, "p" = fp16 planes, "g" = GELU(result) planes
GEMM_CASES = [
    ("tf32x3_k640", "tf32x3", 16, 32, 48, 640, 640, 1, "o"),
    ("tf32x3_k2016_t9", "tf32x3", 16, 32, 48, 2016, 128, 9, "o"),
    ("tf32x3_pair_k8640_t9", "tf32x3", 16, 32, 48, 8640, 672, 9, "o"),
    ("tf32x3_pair_odd_tiles", "tf32x3", 3, 8, 16, 4320, 256, 9, "o"),
    ("tf32x3_k4320_one_tile", "tf32x3", 1, 8, 16, 4320, 256, 9, "o"),
    ("tf32x3_pair_ragged", "tf32x3", 2, 13, 19, 4608, 96, 9, "o"),
    ("tf32_k640", "tf32", 16, 32, 48, 640, 640, 1, "o"),
    ("tf32_k2016_t9", "tf32", 16, 32, 48, 2016, 128, 9, "o"),
    ("tf32_k8640_t9", "tf32", 16, 32, 48, 8640, 672, 9, "o"),
    ("tf32_ragged", "tf32", 2, 13, 19, 576, 64, 9, "o"),
    ("f16x3_k640", "f16x3", 16, 32, 48, 640, 640, 1, "opg"),
    ("f16x3_n320_t9", "f16x3", 16, 32, 48, 576, 320, 9, "o"),
    ("f16x3_pair_k2016_t9", "f16x3", 16, 32, 48, 2016, 128, 9, "opg"),
    ("f16x3_pair_k8640_t9", "f16x3", 16, 32, 48, 8640, 672, 9, "o"),
    ("f16_n64_t9", "f16", 16, 32, 48, 576, 64, 9, "opg"),
    ("f16_pair_k640", "f16", 16, 32, 48, 640, 640, 1, "opg"),
    ("f16_pair_k8640_t9", "f16", 2, 13, 19, 8640, 672, 9, "o"),
]
ATT_CASES = [("att_tf32x3", "tf32x3", 24576), ("att_tf32", "tf32", 24576), ("att_f16x3", "f16x3", 24576),
             ("att_f16x3_ragged", "f16x3", 1000), ("att_tf32x3_ragged", "tf32x3", 1000)]


def gemm_case(lib, _lib, torch, name, math, B, h, w, K, N, taps, outs, dev, s):
    from _cabi import split_weight
    from dcae_b200.weights import f16_weight_planes
    g = torch.Generator(device="cpu").manual_seed(zlib.crc32(name.encode()))
    T, C = B * h * w, K // taps
    x = torch.randn(T, C, generator=g).to(dev)
    wt = (torch.randn(N, K, generator=g) * (1.0 / K ** 0.5)).to(dev)
    bias = (torch.randn(N, generator=g) * 0.1).to(dev)
    res = torch.randn(T, N, generator=g).to(dev)
    hi, lo = split_weight(wt)
    h16, l16, K16, descale = f16_weight_planes(lib, wt, taps, s)
    nbytes = lib.dcae_planes_bytes(T, C)
    scratch = torch.empty(nbytes + 128, dtype=torch.uint8, device=dev)
    a = _lib.Operand(x.data_ptr(), C, 0, C, 0, 0, taps, B, h, w, (scratch.data_ptr() + 127) // 128 * 128, nbytes)
    W = _lib.Weight(wt.data_ptr(), hi.data_ptr(), lo.data_ptr(), N, K, h16.data_ptr(), l16.data_ptr(), K16, descale)
    e = _lib.Epilogue()
    e.bias, e.act = bias.data_ptr(), _lib.ACT_GELU if taps == 9 else _lib.ACT_NONE
    e.residual, e.residual_ld = res.data_ptr(), N
    result = {}
    out = torch.zeros(T, N, device=dev)
    e.out, e.out_ld = out.data_ptr(), N
    result["out"] = out
    keep = [x, wt, bias, res, hi, lo, h16, l16, scratch]
    for tag, field in (("p", "out16"), ("g", "out16_act")):
        if tag in outs:
            ph, pl = (torch.zeros(T, N, dtype=torch.float16, device=dev) for _ in range(2))
            setattr(e, field, _lib.Planes(ph.data_ptr(), pl.data_ptr(), N))
            result[f"{field}_hi"], result[f"{field}_lo"] = ph, pl
    e.act2 = _lib.ACT_GELU if "g" in outs else _lib.ACT_NONE
    run = lambda: lib.dcae_op_gemm(a, W, e, _lib.MATH[math], s)
    _lib.check(run(), name)
    torch.cuda.synchronize()
    flop = 2.0 * T * N * K
    return {k: v.cpu().clone() for k, v in result.items()}, run, flop, keep


def att_case(lib, _lib, torch, name, math, T, dev, s):
    from _cabi import split_weight
    from dcae_b200.weights import f16_weight_planes
    g = torch.Generator(device="cpu").manual_seed(zlib.crc32(name.encode()))
    q = torch.randn(T, 640, generator=g).to(dev)
    Kh = torch.randn(20, 128, 32, generator=g).to(dev)
    Vh = torch.randn(20, 128, 32, generator=g).to(dev)
    hs = (torch.rand(20, generator=g) * 0.3 + 0.05).to(dev)
    Vt = Vh.transpose(1, 2).contiguous()
    khi, klo = split_weight(Kh)
    vhi, vlo = split_weight(Vt)
    kv = _lib.DictKV(Kh.data_ptr(), Vh.data_ptr(), khi.data_ptr(), klo.data_ptr(), vhi.data_ptr(), vlo.data_ptr(), hs.data_ptr())
    keep = [q, Kh, Vh, hs, Vt, khi, klo, vhi, vlo]
    q16 = None
    if math == "f16x3":
        k_hi, k_lo, _, kv.k_descale = f16_weight_planes(lib, Kh.permute(1, 0, 2).reshape(128, -1).contiguous(), 1, s)
        v_hi, v_lo, _, kv.v_descale = f16_weight_planes(lib, Vh.permute(0, 2, 1).reshape(-1, 128).contiguous(), 1, s)
        kv.K16_hi, kv.K16_lo, kv.Vt16_hi, kv.Vt16_lo = k_hi.data_ptr(), k_lo.data_ptr(), v_hi.data_ptr(), v_lo.data_ptr()
        q_hi = q.half()
        q_lo = (q - q_hi.float()).half()
        q16 = _lib.Planes(q_hi.data_ptr(), q_lo.data_ptr(), 640)
        keep += [k_hi, k_lo, v_hi, v_lo, q_hi, q_lo]
    out = torch.zeros(T, 640, device=dev)
    ph, pl = (torch.zeros(T, 640, dtype=torch.float16, device=dev) for _ in range(2))
    p16 = _lib.Planes(ph.data_ptr(), pl.data_ptr(), 640)
    run = lambda: lib.dcae_op_dict_attention(q.data_ptr(), 640, q16, kv, T, out.data_ptr(), 640, p16, _lib.MATH[math], s)
    _lib.check(run(), name)
    torch.cuda.synchronize()
    return {"out": out.cpu().clone(), "out16_hi": ph.cpu().clone(), "out16_lo": pl.cpu().clone()}, run, 2.0 * T * 20 * 128 * 32 * 2, keep


def time_it(torch, run, windows=5, target_ms=40.0):
    """median over `windows` CUDA-event windows of back-to-back launches, each window about target_ms long"""
    for _ in range(3):
        run()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); run(); e1.record(); torch.cuda.synchronize()
    reps = max(5, min(2000, int(target_ms / max(e0.elapsed_time(e1), 1e-3))))
    ts = []
    for _ in range(windows):
        e0.record()
        for _ in range(reps):
            run()
        e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3 / reps)
    ts.sort()
    return ts[len(ts) // 2], reps


def measure(lib_path, out_dir):
    import torch
    from dcae_b200 import _lib
    _lib.LIB_PATH = os.path.abspath(lib_path)
    lib = _lib.load()
    dev = torch.device("cuda:0")
    s = _lib.current_stream(dev)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    outputs, times = {}, {"lib": _lib.LIB_PATH, "device": torch.cuda.get_device_name(dev), "nvidia_smi": smi[:1], "us": {}}
    cases = [("gemm",) + c for c in GEMM_CASES] + [("att",) + c for c in ATT_CASES]
    for c in cases:
        if c[0] == "gemm":
            res, run, flop, keep = gemm_case(lib, _lib, torch, *c[1:], dev, s)
        else:
            res, run, flop, keep = att_case(lib, _lib, torch, *c[1:], dev, s)
        name = c[1]
        for k, v in res.items():
            outputs[f"{name}/{k}"] = v
        us, reps = time_it(torch, run)
        times["us"][name] = us
        print(json.dumps({"case": name, "us": round(us, 2), "reps": reps, "TFLOPs": round(flop / us * 1e-6, 1)}), flush=True)
        del keep
    os.makedirs(out_dir, exist_ok=True)
    torch.save(outputs, os.path.join(out_dir, "outputs.pt"))
    with open(os.path.join(out_dir, "times.json"), "w") as f:
        json.dump(times, f, indent=1)


def compare(dir_a, dir_b):
    """exit status 1 when an output differs in any bit"""
    import torch
    a, b = torch.load(os.path.join(dir_a, "outputs.pt")), torch.load(os.path.join(dir_b, "outputs.pt"))
    bad = sorted(k for k in set(a) | set(b) if k not in a or k not in b or not torch.equal(a[k], b[k]))
    print(f"{len(set(a) & set(b))} outputs compared, {len(bad)} differ" + ("".join(f"\n  differs: {k}" for k in bad)))
    ta, tb = (json.load(open(os.path.join(d, "times.json"))) for d in (dir_a, dir_b))
    print(f"{ta['device']} {ta['nvidia_smi']} | {tb['device']} {tb['nvidia_smi']}")
    for k in ta["us"]:
        print(f"{k:28s} {ta['us'][k]:10.2f} us {tb['us'].get(k, float('nan')):10.2f} us")
    return 1 if bad else 0


if __name__ == "__main__":
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--lib", help="libdcae_b200.so to load")
    ap.add_argument("--out", help="directory for outputs.pt and times.json")
    ap.add_argument("--compare", nargs=2, metavar=("DIR_A", "DIR_B"))
    args = ap.parse_args()
    if args.compare:
        sys.exit(compare(*args.compare))
    if not (args.lib and args.out):
        ap.error("--lib and --out, or --compare")
    measure(args.lib, args.out)
