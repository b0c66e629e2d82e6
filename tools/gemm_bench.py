"""GEMM microbenchmark through the C ABI: python tools/gemm_bench.py  (GPU box)."""
import os, sys, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import torch
import _cabi as K
from dcae_b200 import _lib

B, h, w = 16, 32, 48
T = B * h * w
lib = _lib.load()
dev = torch.device("cuda:0")


def bench(Kd, N, math, taps=1, reps=10):
    C = Kd // taps
    buf = torch.randn(T, C, device=dev)
    wt = torch.randn(N, Kd, device=dev) * 0.02
    hi, lo = K.split_weight(wt)
    out = torch.empty(T, N, device=dev)
    a = _lib.Operand(buf.data_ptr(), C, 0, C, 0, 0, taps, B, h, w)
    W = _lib.Weight(wt.data_ptr(), hi.data_ptr(), lo.data_ptr(), N, Kd)
    e = _lib.Epilogue(); e.out, e.out_ld = out.data_ptr(), N
    s = _lib.current_stream(dev)
    for _ in range(3):
        _lib.check(lib.dcae_op_gemm(a, W, e, _lib.MATH[math], s))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record()
    for _ in range(reps):
        lib.dcae_op_gemm(a, W, e, _lib.MATH[math], s)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    tf = 2.0 * T * N * Kd / (ms * 1e-3) / 1e12
    print(json.dumps({"K": Kd, "N": N, "taps": taps, "math": math, "ms": round(ms, 4), "algo_TFLOPs": round(tf, 1),
                      "mma_TFLOPs": round(tf * (3 if math == "tf32x3" else 1), 1)}), flush=True)


for math in ("tf32x3", "tf32"):
    for Kd, N, taps in [(640, 640, 1), (2560, 640, 1), (640, 2560, 1), (8640, 672, 9), (2016, 128, 9), (1152, 64, 9)]:
        bench(Kd, N, math, taps)
