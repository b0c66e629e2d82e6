"""The transform stacks around the entropy model on libdcae_b200.so (SURVEY 8f N3 / N4):
`h_a`, `h_z_s1`, `h_z_s2` (hyper path) and `g_a`, `g_s` (analysis / synthesis) of the reference
`DCAE` (/root/reference/models/dcae.py:541-582), built from its blocks (:152-383).

Host side only: every arithmetic operation is a C-ABI call (include/dcae_b200.h) --

  nn.Linear / 1x1 conv / 3x3 conv             dcae_op_gemm (kernel 2: tcgen05, 3x3 = implicit GEMM over shifted TMA boxes)
  conv k=5|3, stride 2 (conv(), :35-42)       dcae_op_space_to_depth + dcae_op_gemm(taps=9) on re-indexed weights
  deconv k=5|3, stride 2 (deconv(), :44-52)   dcae_op_gemm(taps=9) producing the 4 output phases + dcae_op_depth_to_space
  LayerNorm                                   dcae_op_layernorm
  WMSA core, W / SW windows (:228-298)        dcae_op_window_attention
  DWConv + GELU * gate (:300-327)             dcae_op_dwconv3x3
  ReLU / residual / Scale                     GEMM epilogue

Activations stay token-major `[T, ld]` fp32 between operators (T = B*h*w tokens); every channel count is padded to a
multiple of 32 columns (144 -> 160, 72 -> 96, 48 -> 64) with zero weights behind the padding, so the padded columns
hold exact zeros.  NCHW appears at stack entry and exit only.

The kernels are reached through a small backend object (`LibKernels`); tests/ substitutes a torch-CPU restatement of
each operator's contract to check the weight re-indexing and the composition without a GPU.  There is no CPU
fallback in the product: `TransformStack` with the default backend raises without the CUDA library.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib

# ---- architecture (dcae.py:520-582): (kind, args) per nn.Sequential index ---------------------------------------
_FEAT = (96, 144, 256)
_HEAD_DIM = (8, 16, 32, 32, 16, 8)
_BLOCKS = (1, 2, 12)
N_HYPER, M_LATENT = 192, 320

ARCH: Dict[str, List[Tuple]] = {
    "g_a": [("rbws", 3, _FEAT[0]), ("swin", _FEAT[0], _HEAD_DIM[0], 8, _BLOCKS[0]),
            ("rbws", _FEAT[0], _FEAT[1]), ("swin", _FEAT[1], _HEAD_DIM[1], 8, _BLOCKS[1]),
            ("rbws", _FEAT[1], _FEAT[2]), ("swin", _FEAT[2], _HEAD_DIM[2], 8, _BLOCKS[2]),
            ("conv_s2", _FEAT[2], M_LATENT, 5)],
    "g_s": [("deconv_s2", M_LATENT, _FEAT[2], 5), ("swin", _FEAT[2], _HEAD_DIM[3], 8, _BLOCKS[2]),
            ("rbwu", _FEAT[2], _FEAT[1]), ("swin", _FEAT[1], _HEAD_DIM[4], 8, _BLOCKS[1]),
            ("rbwu", _FEAT[1], _FEAT[0]), ("swin", _FEAT[0], _HEAD_DIM[5], 8, _BLOCKS[0]),
            ("rbwu", _FEAT[0], 3)],
    "h_a": [("rbws", M_LATENT, N_HYPER), ("swin", N_HYPER, 32, 4, 1), ("conv_s2", N_HYPER, 192, 3)],
    "h_z_s1": [("deconv_s2", 192, N_HYPER, 3), ("swin", N_HYPER, 32, 4, 1), ("rbwu", N_HYPER, M_LATENT)],
    "h_z_s2": [("deconv_s2", 192, N_HYPER, 3), ("swin", N_HYPER, 32, 4, 1), ("rbwu", N_HYPER, M_LATENT)],
}
STACKS = tuple(ARCH)


def pad32(c: int) -> int:
    return (c + 31) // 32 * 32


def pad8(c: int) -> int:
    return (c + 7) // 8 * 8


def transform_param_shapes(stack: str) -> Dict[str, Tuple[int, ...]]:
    """State-dict keys (relative to the stack's prefix, e.g. 'g_a.') and shapes of a stack, as `DCAE()` creates them."""
    out: Dict[str, Tuple[int, ...]] = {}

    def rbb(p, c):
        mid = c // 2
        out[p + "conv1.weight"], out[p + "conv1.bias"] = (mid, c, 1, 1), (mid,)
        out[p + "conv2.weight"], out[p + "conv2.bias"] = (mid, mid, 3, 3), (mid,)
        out[p + "conv3.weight"], out[p + "conv3.bias"] = (c, mid, 1, 1), (c,)

    for idx, spec in enumerate(ARCH[stack]):
        p = f"{idx}."
        kind = spec[0]
        if kind == "rbws":
            _, cin, cout = spec
            out[p + "conv.weight"], out[p + "conv.bias"] = (cout, cin, 5, 5), (cout,)
            for r in (1, 2, 3):
                rbb(p + f"res{r}.", cout)
        elif kind == "rbwu":
            _, cin, cout = spec
            for r in (1, 2, 3):
                rbb(p + f"res{r}.", cin)
            out[p + "conv.weight"], out[p + "conv.bias"] = (cin, cout, 5, 5), (cout,)
        elif kind == "conv_s2":
            _, cin, cout, k = spec
            out[p + "weight"], out[p + "bias"] = (cout, cin, k, k), (cout,)
        elif kind == "deconv_s2":
            _, cin, cout, k = spec
            out[p + "weight"], out[p + "bias"] = (cin, cout, k, k), (cout,)
        elif kind == "swin":
            _, c, hd, win, n = spec
            for i in range(n):
                q = p + f"layers.{i}."
                for ln in ("ln1", "ln2"):
                    out[q + ln + ".weight"], out[q + ln + ".bias"] = (c,), (c,)
                out[q + "msa.embedding_layer.weight"], out[q + "msa.embedding_layer.bias"] = (3 * c, c), (3 * c,)
                out[q + "msa.relative_position_params"] = (c // hd, 2 * win - 1, 2 * win - 1)
                out[q + "msa.linear.weight"], out[q + "msa.linear.bias"] = (c, c), (c,)
                out[q + "mlp.fc1.weight"], out[q + "mlp.fc1.bias"] = (4 * c, c), (4 * c,)
                out[q + "mlp.dwconv.dwconv.weight"], out[q + "mlp.dwconv.dwconv.bias"] = (2 * c, 1, 3, 3), (2 * c,)
                out[q + "mlp.fc2.weight"], out[q + "mlp.fc2.bias"] = (c, 2 * c), (c,)
                out[q + "res_scale_1.scale"], out[q + "res_scale_2.scale"] = (c,), (c,)
            out[p + "conv.weight"], out[p + "conv.bias"] = (c, c, 3, 3), (c,)
    return out


def init_transform_params(seed: int = 0, stacks: Sequence[str] = STACKS, prefixed: bool = True) -> Dict[str, torch.Tensor]:
    """Deterministic random weights with the reference's state-dict keys and shapes (synthetic benchmarks / tests; there
    are no checkpoints offline).  Dense and conv weights are uniform in +-1/sqrt(fan_in) like torch's default init; the
    parameters that default init leaves trivial (Scale = 1, LayerNorm affine, relative position bias ~ 0.02) are made
    lively so that every term of the blocks matters."""
    out: Dict[str, torch.Tensor] = {}
    for stack in stacks:
        g = torch.Generator().manual_seed(1000 * (1 + STACKS.index(stack)) + seed)     # per stack: a subset gives the same weights
        for key, shape in transform_param_shapes(stack).items():
            if key.endswith("scale"):
                t = 0.75 + 0.5 * torch.rand(shape, generator=g)
            elif key.endswith("relative_position_params"):
                t = 0.3 * torch.randn(shape, generator=g)
            elif ".ln1." in key or ".ln2." in key:
                t = (1.0 if key.endswith("weight") else 0.0) + 0.1 * torch.randn(shape, generator=g)
            else:
                if key.endswith("bias"):
                    bound = 0.05
                else:
                    kind = ARCH[stack][int(key.split(".")[0])][0]
                    rest = key.split(".", 1)[1]
                    is_deconv = (kind == "deconv_s2" and rest == "weight") or (kind == "rbwu" and rest == "conv.weight")
                    fan_in = (shape[0] if is_deconv else shape[1]) * (shape[2] * shape[3] if len(shape) == 4 else 1)
                    if is_deconv:
                        fan_in = fan_in / 4.0          # a stride-2 transposed conv sums a quarter of its taps per output
                    bound = 1.0 / math.sqrt(fan_in)
                t = (2.0 * torch.rand(shape, generator=g) - 1.0) * bound
            out[(f"{stack}." if prefixed else "") + key] = t
    return out


# ---- weight re-indexing (pure tensor rearrangement, CPU or GPU) ---------------------------------------------------

def _pad_to(t: torch.Tensor, dim: int, size: int) -> torch.Tensor:
    if t.shape[dim] == size:
        return t
    shape = list(t.shape)
    shape[dim] = size - t.shape[dim]
    return torch.cat([t, t.new_zeros(shape)], dim=dim)


def linear_to_gemm(w: torch.Tensor, n_pad: int, k_pad: int) -> torch.Tensor:
    """[N, K] (or [N, K, 1, 1]) -> [n_pad, k_pad], zero padded."""
    w = w.reshape(w.shape[0], -1)
    return _pad_to(_pad_to(w, 0, n_pad), 1, k_pad).contiguous()


def conv3x3_to_gemm(w: torch.Tensor, n_pad: int, c_pad: int) -> torch.Tensor:
    """[N, C, 3, 3] -> [n_pad, 9 * c_pad], K ordered tap-major (tap = 3 ky + kx), channels zero padded."""
    w = _pad_to(_pad_to(w, 0, n_pad), 1, c_pad)
    return w.permute(0, 2, 3, 1).reshape(n_pad, 9 * c_pad).contiguous()


def conv_s2_to_gemm(w: torch.Tensor, n_pad: int, cs: int) -> torch.Tensor:
    """Stride-2 conv weight [N, C, k, k] (k = 3 or 5, pad k // 2) -> the stride-1 3x3 conv weight over the
    space-to-depth image, [n_pad, 9 * 4 * cs]: tap (by, bx) in {-1, 0, 1}^2, K index (sy*2 + sx) * cs + c, and
    original tap ky = 2 by + sy + k // 2 (zero where that falls outside the k x k kernel)."""
    N, C, k, _ = w.shape
    pad = k // 2
    out = w.new_zeros(n_pad, 3, 3, 2, 2, cs)
    for by in (-1, 0, 1):
        for sy in (0, 1):
            ky = 2 * by + sy + pad
            if not 0 <= ky < k:
                continue
            for bx in (-1, 0, 1):
                for sx in (0, 1):
                    kx = 2 * bx + sx + pad
                    if 0 <= kx < k:
                        out[:N, by + 1, bx + 1, sy, sx, :C] = w[:, :, ky, kx]
    return out.reshape(n_pad, 9 * 4 * cs).contiguous()


def deconv_s2_to_gemm(w: torch.Tensor, cs_out: int, c_pad: int) -> torch.Tensor:
    """Stride-2 transposed conv weight [C_in, C_out, k, k] (k = 3 or 5, pad k // 2, output_padding 1) -> the stride-1 3x3
    conv weight that produces the four output phases, [4 * cs_out, 9 * c_pad]: row (py*2 + px) * cs_out + co, tap
    (by, bx) reads input (y + by, x + bx) for output (2y + py, 2x + px), original tap ky = py - 2 by + k // 2."""
    Cin, Cout, k, _ = w.shape
    pad = k // 2
    out = w.new_zeros(2, 2, cs_out, 3, 3, c_pad)
    for py in (0, 1):
        for by in (-1, 0, 1):
            ky = py - 2 * by + pad
            if not 0 <= ky < k:
                continue
            for px in (0, 1):
                for bx in (-1, 0, 1):
                    kx = px - 2 * bx + pad
                    if 0 <= kx < k:
                        out[py, px, :Cout, by + 1, bx + 1, :Cin] = w[:, :, ky, kx].t()
    return out.reshape(4 * cs_out, 9 * c_pad).contiguous()


# ---- activations and the kernel backend ----------------------------------------------------------------------------

F32, P16 = 1, 2          # which forms of a result its consumers read: fp32 [T, ld] and / or fp16 hi/lo planes


@dataclass
class Act:
    """Token-major activation on the token grid (B, h, w): `buf` = fp32 [T, ld] (ld = padded channel count) and / or
    `p16` = (hi, lo) fp16 planes [T, pad64(ld)], the form the f16x3 GEMMs read by TMA (value = hi + lo, 22 bits)."""
    buf: Optional[torch.Tensor]
    B: int
    h: int
    w: int
    p16: Optional[Tuple[torch.Tensor, torch.Tensor]] = None

    @property
    def T(self) -> int:
        return self.B * self.h * self.w

    @property
    def ld(self) -> int:
        return self.buf.shape[1] if self.buf is not None else self.p16[0].shape[1]


class PackedGemm:
    """One dense layer in the layouts dcae_op_gemm reads: fp32 [N, K], its TF32 hi/lo split or its scaled fp16 hi/lo planes
    (whichever the math mode needs), bias [N]."""

    def __init__(self, N: int, K: int, taps: int):
        self.N, self.K, self.taps = N, K, taps
        self.w = self.bias = None
        self.struct = None
        self.keep: list = []


def pad64(c: int) -> int:
    return (c + 63) // 64 * 64


class LibKernels:
    """The operators on libdcae_b200.so (device tensors in, device tensors out, everything on the current stream).

    Data flow in the f16x3 / f16 modes: every producer writes the form(s) its consumers read (`want` = F32 | P16) --
    fp16 hi/lo planes for GEMM operands, straight from the producing kernel (LayerNorm, window attention, depthwise
    conv, GEMM epilogue, space-to-depth / depth-to-space), fp32 for residuals and element-wise consumers -- so no
    conversion pass runs between layers and nothing is written that nobody reads.  Other math modes stay fp32.

    Buffers with padding columns (planes are pad64(columns) wide because the GEMM's 64-column TMA boxes over-read the
    padding against zero weights; LayerNorm / attention outputs of the 144-channel level) come from a pool keyed by
    (kind, rows, columns, written columns, stream): zeroed once, no kernel ever writes the padding, and a buffer whose
    only reference is the pool's is free (reuse is ordered by the stream).  Everything else is torch.empty."""

    def __init__(self, device="cuda:0", math: str = "f16x3"):
        if math not in _lib.MATH:
            raise ValueError(f"math must be one of {sorted(_lib.MATH)}")
        self.device = torch.device(device)
        self.math = math
        self.planes = math in ("f16x3", "f16")
        self.lib = _lib.load()
        self._scratch: Optional[torch.Tensor] = None
        self._pool: Dict[tuple, list] = {}
        self._pool_bytes = 0
        self.max_pool_bytes = 64 << 30

    # -- helpers
    def _s(self) -> int:
        return _lib.current_stream(self.device)

    def tensor(self, t: torch.Tensor) -> torch.Tensor:
        return t.detach().to(self.device, torch.float32).contiguous()

    def _take(self, key, make):
        import sys
        key = key + (self._s(),)                      # reuse is ordered by the stream: one pool per stream
        lst = self._pool.setdefault(key, [])
        for i in range(len(lst)):
            if sys.getrefcount(lst[i]) == 2:          # the list and getrefcount's own argument: nobody else holds it
                return lst[i]
        if self._pool_bytes > self.max_pool_bytes:    # many different input shapes: drop what is free before growing further
            self.clear_pool(only_free=True)
            lst = self._pool.setdefault(key, [])
        t = make()
        self._pool_bytes += t.numel() * t.element_size()
        lst.append(t)
        return t

    def clear_pool(self, only_free: bool = False) -> None:
        import sys
        if not only_free:
            self._pool.clear()
            self._pool_bytes = 0
            return
        for key in list(self._pool):
            kept = []
            for i in range(len(self._pool[key])):
                if sys.getrefcount(self._pool[key][i]) > 2:
                    kept.append(self._pool[key][i])
            self._pool[key] = kept
        self._pool_bytes = sum(t.numel() * t.element_size() for lst in self._pool.values() for t in lst)

    def _f32(self, T: int, ld: int, cols: int) -> torch.Tensor:
        """fp32 [T, ld] of which a kernel writes the first `cols` columns; the rest stays zero (pooled: zeroed once).
        Fully written buffers come from torch's caching allocator, which shares memory across shapes."""
        if ld == cols:
            return torch.empty(T, ld, device=self.device)
        return self._take(("f32", T, ld, cols), lambda: torch.zeros(T, ld, device=self.device))

    def _p16(self, T: int, cols: int) -> torch.Tensor:
        """[2, T, pad64(cols)] fp16: hi = [0], lo = [1]."""
        ld = pad64(cols)
        if ld == cols:
            return torch.empty(2, T, ld, dtype=torch.float16, device=self.device)
        return self._take(("p16", T, ld, cols), lambda: torch.zeros(2, T, ld, dtype=torch.float16, device=self.device))

    @staticmethod
    def _pl(p16) -> _lib.Planes:
        return _lib.Planes(p16[0].data_ptr(), p16[1].data_ptr(), p16[0].stride(0))

    def _outs(self, T: int, ld: int, cols: int, want: int):
        """(fp32 buffer or None, planes or None) for a result of `cols` written columns."""
        if not self.planes:
            want = F32
        buf = self._f32(T, ld, cols) if want & F32 else None
        p16 = self._p16(T, ld) if want & P16 else None
        return buf, p16

    def _planes_scratch(self, T: int, k: int) -> Tuple[int, int]:
        n = int(self.lib.dcae_planes_bytes(T, k))
        if self._scratch is None or self._scratch.numel() < n + 128:
            self._scratch = torch.empty(n + 128, dtype=torch.uint8, device=self.device)
        return (self._scratch.data_ptr() + 127) // 128 * 128, n

    # -- weights
    def pack_gemm(self, w2d: torch.Tensor, bias: torch.Tensor, taps: int = 1) -> PackedGemm:
        w = self.tensor(w2d)
        N, K = w.shape
        pg = PackedGemm(N, K, taps)
        pg.w, pg.bias = w, self.tensor(_pad_to(bias.reshape(-1), 0, N))
        W = _lib.Weight()
        W.w, W.N, W.K = w.data_ptr(), N, K
        with torch.cuda.device(self.device):
            if self.math in ("tf32x3", "tf32"):
                hi, lo = torch.empty_like(w), torch.empty_like(w)
                _lib.check(self.lib.dcae_split_tf32(w.data_ptr(), hi.data_ptr(), lo.data_ptr(), w.numel(), self._s()), "dcae_split_tf32")
                W.w_hi, W.w_lo = hi.data_ptr(), lo.data_ptr()
                pg.keep += [hi, lo]
            elif self.planes:
                from .weights import f16_weight_planes
                h16, l16, K16, descale = f16_weight_planes(self.lib, w, taps, self._s())
                W.w16_hi, W.w16_lo, W.K16, W.descale = h16.data_ptr(), l16.data_ptr(), K16, descale
                pg.keep += [h16, l16]
        pg.struct = W
        return pg

    def vector(self, t: torch.Tensor, n_pad: Optional[int] = None, fill: float = 0.0) -> torch.Tensor:
        t = t.detach().reshape(-1).to(torch.float32)
        if n_pad is not None and t.numel() < n_pad:
            t = torch.cat([t, t.new_full((n_pad - t.numel(),), fill)])
        return self.tensor(t)

    # -- operators
    def to_tokens(self, x: torch.Tensor, ld: int, want: int = F32) -> Act:
        """NCHW -> token-major with `ld` columns (columns >= C are zero)."""
        B, C, H, W = x.shape
        x = self.tensor(x)
        buf, p16 = self._outs(B * H * W, ld, C, want)
        _lib.check(self.lib.dcae_op_nchw_to_tokens(x.data_ptr(), B, C, H * W, _lib.ptr(buf), ld, self._pl(p16) if p16 is not None else None,
                                                   self._s()), "dcae_op_nchw_to_tokens")
        return Act(buf, B, H, W, p16)

    def to_nchw(self, a: Act, C: int) -> torch.Tensor:
        out = torch.empty(a.B, C, a.h, a.w, device=self.device, dtype=torch.float32)
        _lib.check(self.lib.dcae_op_tokens_to_nchw(a.buf.data_ptr(), a.ld, a.B, C, a.h * a.w, out.data_ptr(), self._s()), "dcae_op_tokens_to_nchw")
        return out

    def gemm(self, a: Act, pg: PackedGemm, act: int = _lib.ACT_NONE, residual: Optional[Act] = None,
             res_scale: Optional[torch.Tensor] = None, want: int = F32) -> Act:
        """out[T, N] = act(A[T, taps*k] W^T + bias) + residual * res_scale, A = the first K / taps columns of `a`."""
        k = pg.K // pg.taps
        assert k <= a.ld and k % 32 == 0, (k, a.ld)
        buf, p16 = self._outs(a.T, pg.N, pg.N, want)
        A = _lib.Operand()
        A.col0, A.k0, A.taps, A.B, A.h, A.w = 0, k, pg.taps, a.B, a.h, a.w
        if self.planes and a.p16 is not None:
            A.src16 = self._pl(a.p16)                 # the producer wrote the operand planes: no split pass
            A.ld = a.p16[0].stride(0)
        else:
            A.base, A.ld = a.buf.data_ptr(), a.buf.shape[1]
            if self.planes:
                A.planes, A.planes_bytes = self._planes_scratch(a.T, k)
        e = _lib.Epilogue()
        e.bias = pg.bias.data_ptr()
        if residual is not None:
            assert residual.buf is not None and residual.buf.shape[1] >= pg.N and residual.T == a.T
            e.residual, e.residual_ld = residual.buf.data_ptr(), residual.buf.shape[1]
            e.res_scale = _lib.ptr(res_scale)
        e.act = act
        if buf is not None:
            e.out, e.out_ld = buf.data_ptr(), pg.N
        if p16 is not None:
            e.out16 = self._pl(p16)
        _lib.check(self.lib.dcae_op_gemm(A, pg.struct, e, _lib.MATH[self.math], self._s()), "dcae_op_gemm")
        return Act(buf, a.B, a.h, a.w, p16)

    def layernorm(self, a: Act, gamma: torch.Tensor, beta: torch.Tensor, C: int, want: int = F32) -> Act:
        ld = a.buf.shape[1]
        buf, p16 = self._outs(a.T, ld, C, want)
        _lib.check(self.lib.dcae_op_layernorm(a.buf.data_ptr(), ld, gamma.data_ptr(), beta.data_ptr(), C, a.T, _lib.ptr(buf), ld,
                                              self._pl(p16) if p16 is not None else None, self._s()), "dcae_op_layernorm")
        return Act(buf, a.B, a.h, a.w, p16)

    def window_attention(self, qkv: Act, C: int, c_pad: int, head_dim: int, window: int, shift: int, rel: torch.Tensor, want: int = F32) -> Act:
        buf, p16 = self._outs(qkv.T, c_pad, C, want)
        _lib.check(self.lib.dcae_op_window_attention(qkv.buf.data_ptr(), qkv.buf.shape[1], 0, c_pad, 2 * c_pad, C, head_dim, window, shift,
                                                     rel.data_ptr(), qkv.B, qkv.h, qkv.w, _lib.ptr(buf), c_pad,
                                                     self._pl(p16) if p16 is not None else None, self._s()), "dcae_op_window_attention")
        return Act(buf, qkv.B, qkv.h, qkv.w, p16)

    def dwconv_glu(self, f: Act, wt9c: torch.Tensor, bias: torch.Tensor, hid: int, want: int = F32) -> Act:
        """gelu(dw3x3(f[:, :hid]) + bias) * f[:, hid:2 hid]   (ConvolutionalGLU, dcae.py:323-326)."""
        buf, p16 = self._outs(f.T, hid, hid, want)
        ld = f.buf.shape[1]
        _lib.check(self.lib.dcae_op_dwconv3x3(f.buf.data_ptr(), ld, wt9c.data_ptr(), bias.data_ptr(), hid, f.B, f.h, f.w, _lib.ACT_GELU,
                                              f.buf.data_ptr() + 4 * hid, ld, _lib.ptr(buf), hid, self._pl(p16) if p16 is not None else None,
                                              self._s()), "dcae_op_dwconv3x3")
        return Act(buf, f.B, f.h, f.w, p16)

    def space_to_depth(self, a: Act, C: int, cs: int, want: int = F32) -> Act:
        h2, w2 = (a.h + 1) // 2, (a.w + 1) // 2
        buf, p16 = self._outs(a.B * h2 * w2, 4 * cs, 4 * cs, want)
        _lib.check(self.lib.dcae_op_space_to_depth(a.buf.data_ptr(), a.buf.shape[1], C, cs, a.B, a.h, a.w, _lib.ptr(buf), 4 * cs,
                                                   self._pl(p16) if p16 is not None else None, self._s()), "dcae_op_space_to_depth")
        return Act(buf, a.B, h2, w2, p16)

    def depth_to_space(self, a: Act, cs: int, C: int, c_pad: int, want: int = F32) -> Act:
        buf, p16 = self._outs(4 * a.T, c_pad, c_pad, want)
        _lib.check(self.lib.dcae_op_depth_to_space(a.buf.data_ptr(), a.buf.shape[1], cs, C, c_pad, a.B, a.h, a.w, _lib.ptr(buf), c_pad,
                                                   self._pl(p16) if p16 is not None else None, self._s()), "dcae_op_depth_to_space")
        return Act(buf, a.B, 2 * a.h, 2 * a.w, p16)


# ---- blocks -----------------------------------------------------------------------------------------------------------
# `want` of a block = the forms its successor reads (NEEDS below); inside a block every intermediate is written in the
# one form its single consumer reads.

class _ResidualBottleneck:
    """ResidualBottleneckBlock(c, c) (dcae.py:152-190): 1x1 -> ReLU -> 3x3 -> ReLU -> 1x1, + x (skip is Identity)."""
    needs = F32 | P16          # x: residual (fp32) and the operand of conv1 (planes)

    def __init__(self, K, P, p: str, c: int):
        mid, cp = c // 2, pad32(c)
        mp = pad32(mid)
        self.c1 = K.pack_gemm(linear_to_gemm(P[p + "conv1.weight"], mp, cp), P[p + "conv1.bias"])
        self.c2 = K.pack_gemm(conv3x3_to_gemm(P[p + "conv2.weight"], mp, mp), P[p + "conv2.bias"], taps=9)
        self.c3 = K.pack_gemm(linear_to_gemm(P[p + "conv3.weight"], cp, mp), P[p + "conv3.bias"])

    def __call__(self, K, x: Act, want: int = F32) -> Act:
        t = K.gemm(x, self.c1, act=_lib.ACT_RELU, want=P16)
        t = K.gemm(t, self.c2, act=_lib.ACT_RELU, want=P16)
        return K.gemm(t, self.c3, residual=x, want=want)


class _ConvS2:
    """conv(cin, cout, k, stride 2) (dcae.py:35-42) = space-to-depth + stride-1 3x3 implicit GEMM."""
    needs = F32

    def __init__(self, K, w: torch.Tensor, b: torch.Tensor, cin: int, cout: int):
        self.cin, self.cout = cin, cout
        self.cs = pad8(cin)
        self.g = K.pack_gemm(conv_s2_to_gemm(w, pad32(cout), self.cs), b, taps=9)

    def __call__(self, K, x: Act, want: int = F32) -> Act:
        return K.gemm(K.space_to_depth(x, self.cin, self.cs, want=P16), self.g, want=want)


class _DeconvS2:
    """deconv(cin, cout, k, stride 2) (dcae.py:44-52) = stride-1 3x3 implicit GEMM to the 4 output phases + depth-to-space."""
    needs = P16

    def __init__(self, K, w: torch.Tensor, b: torch.Tensor, cin: int, cout: int):
        self.cin, self.cout = cin, cout
        self.cs = pad8(cout)
        bias4 = _pad_to(b.reshape(-1), 0, self.cs).repeat(4)
        self.g = K.pack_gemm(deconv_s2_to_gemm(w, self.cs, pad32(cin)), bias4, taps=9)

    def __call__(self, K, x: Act, want: int = F32, c_pad: Optional[int] = None) -> Act:
        return K.depth_to_space(K.gemm(x, self.g, want=F32), self.cs, self.cout, c_pad or pad32(self.cout), want=want)


class _SwinLayer:
    """ResScaleConvolutionGateBlock (dcae.py:338-360): x = s1 x + WMSA(LN1 x); x = s2 x + ConvGLU(LN2 x)."""

    def __init__(self, K, P, p: str, c: int, head_dim: int, window: int, shifted: bool):
        cp = pad32(c)
        self.c, self.cp, self.hd, self.window, self.shift = c, cp, head_dim, window, (window // 2 if shifted else 0)
        self.ln1 = (K.vector(P[p + "ln1.weight"]), K.vector(P[p + "ln1.bias"]))
        self.ln2 = (K.vector(P[p + "ln2.weight"]), K.vector(P[p + "ln2.bias"]))
        # embedding_layer rows are (q heads | k heads | v heads) (dcae.py:275-276): each third on its own padded window
        we, be = P[p + "msa.embedding_layer.weight"], P[p + "msa.embedding_layer.bias"]
        wq = torch.cat([_pad_to(_pad_to(we[j * c:(j + 1) * c], 1, cp), 0, cp) for j in range(3)], dim=0)
        bq = torch.cat([_pad_to(be[j * c:(j + 1) * c], 0, cp) for j in range(3)], dim=0)
        self.qkv = K.pack_gemm(wq, bq)
        rel = P[p + "msa.relative_position_params"]
        assert tuple(rel.shape) == (c // head_dim, 2 * window - 1, 2 * window - 1), tuple(rel.shape)
        self.rel = K.tensor(rel)
        self.proj = K.pack_gemm(linear_to_gemm(P[p + "msa.linear.weight"], cp, cp), P[p + "msa.linear.bias"])
        hid = 2 * c
        assert hid % 32 == 0
        self.hid = hid
        self.fc1 = K.pack_gemm(linear_to_gemm(P[p + "mlp.fc1.weight"], 2 * hid, cp), P[p + "mlp.fc1.bias"])
        self.dw_w = K.tensor(P[p + "mlp.dwconv.dwconv.weight"].reshape(hid, 9).t())
        self.dw_b = K.vector(P[p + "mlp.dwconv.dwconv.bias"])
        self.fc2 = K.pack_gemm(linear_to_gemm(P[p + "mlp.fc2.weight"], cp, hid), P[p + "mlp.fc2.bias"])
        self.s1 = K.vector(P[p + "res_scale_1.scale"], cp, 1.0)
        self.s2 = K.vector(P[p + "res_scale_2.scale"], cp, 1.0)

    def __call__(self, K, x: Act, want: int = F32) -> Act:
        t = K.layernorm(x, *self.ln1, self.c, want=P16)
        t = K.gemm(t, self.qkv, want=F32)
        t = K.window_attention(t, self.c, self.cp, self.hd, self.window, self.shift, self.rel, want=P16)
        x = K.gemm(t, self.proj, residual=x, res_scale=self.s1, want=F32)
        t = K.layernorm(x, *self.ln2, self.c, want=P16)
        t = K.gemm(t, self.fc1, want=F32)
        t = K.dwconv_glu(t, self.dw_w, self.dw_b, self.hid, want=P16)
        return K.gemm(t, self.fc2, residual=x, res_scale=self.s2, want=want)


class _Swin:
    """SwinBlockWithConvMulti (dcae.py:362-383): n alternating W / SW layers, then conv3x3 + x."""
    needs = F32

    def __init__(self, K, P, p: str, c: int, head_dim: int, window: int, n: int):
        self.c, self.window = c, window
        self.layers = [_SwinLayer(K, P, p + f"layers.{i}.", c, head_dim, window, shifted=(i % 2 == 1)) for i in range(n)]
        cp = pad32(c)
        self.conv = K.pack_gemm(conv3x3_to_gemm(P[p + "conv.weight"], cp, cp), P[p + "conv.bias"], taps=9)

    def __call__(self, K, x: Act, want: int = F32) -> Act:
        if x.h <= self.window or x.w <= self.window or x.h % self.window or x.w % self.window:
            # dcae.py:374-377 pads inputs no larger than the window (and its `trans_x + x` then only works when the padded
            # and the original sizes agree); grids that are not a multiple of the window fail in the reference's rearrange
            raise _lib.DcaeError(f"Swin block: token grid {x.h}x{x.w} must be a multiple of the window {self.window} and larger than it")
        t = x
        for j, layer in enumerate(self.layers):
            t = layer(K, t, want=P16 if j == len(self.layers) - 1 else F32)      # the last layer feeds the 3x3 conv only
        return K.gemm(t, self.conv, residual=x, want=want)


class TransformStack:
    """One of g_a / g_s / h_a / h_z_s1 / h_z_s2 with the reference's weights.

    params: state dict holding the stack's keys, either relative ('0.conv.weight') or with the stack prefix
    ('g_a.0.conv.weight').  forward(x [B, C_in, H, W]) -> [B, C_out, H', W'] like the reference nn.Sequential."""

    def __init__(self, stack: str, params: Dict[str, torch.Tensor], device="cuda:0", math: str = "f16x3", kernels=None):
        if stack not in ARCH:
            raise ValueError(f"unknown stack {stack!r}; one of {STACKS}")
        self.stack = stack
        self.K = kernels if kernels is not None else LibKernels(device, math)
        self._pack(params)
        first, last = ARCH[stack][0], ARCH[stack][-1]
        self.c_in = first[1]
        self.c_out = last[2]

    def _pack(self, params: Dict[str, torch.Tensor]) -> None:
        stack = self.stack
        P = {}
        for key, shape in transform_param_shapes(stack).items():
            t = params.get(key, params.get(f"{stack}.{key}"))
            if t is None:
                raise KeyError(f"{stack}: missing parameter {key}")
            if tuple(t.shape) != shape:
                raise ValueError(f"{stack}.{key}: expected shape {shape}, got {tuple(t.shape)}")
            P[key] = t.detach().to(torch.float32)
        K = self.K
        blocks: list = []
        for idx, spec in enumerate(ARCH[stack]):
            p = f"{idx}."
            kind = spec[0]
            if kind == "rbws":
                _, cin, cout = spec
                blocks.append(("conv", _ConvS2(K, P[p + "conv.weight"], P[p + "conv.bias"], cin, cout)))
                blocks += [("rbb", _ResidualBottleneck(K, P, p + f"res{r}.", cout)) for r in (1, 2, 3)]
            elif kind == "rbwu":
                _, cin, cout = spec
                blocks += [("rbb", _ResidualBottleneck(K, P, p + f"res{r}.", cin)) for r in (1, 2, 3)]
                blocks.append(("deconv", _DeconvS2(K, P[p + "conv.weight"], P[p + "conv.bias"], cin, cout)))
            elif kind == "conv_s2":
                _, cin, cout, _k = spec
                blocks.append(("conv", _ConvS2(K, P[p + "weight"], P[p + "bias"], cin, cout)))
            elif kind == "deconv_s2":
                _, cin, cout, _k = spec
                blocks.append(("deconv", _DeconvS2(K, P[p + "weight"], P[p + "bias"], cin, cout)))
            elif kind == "swin":
                _, c, hd, win, n = spec
                blocks.append(("swin", _Swin(K, P, p, c, hd, win, n)))
        self.blocks = blocks

    def refresh(self, params: Dict[str, torch.Tensor]) -> None:
        """Repack the weights in place from a new state dict (same keys as the constructor takes), e.g. after an optimizer
        step or `load_state_dict`.  The previous packed tensors are released once no queued launch uses them."""
        if isinstance(self.K, LibKernels):
            torch.cuda.synchronize(self.K.device)
        self._pack(params)

    # widest intermediate of a stack, in fp32 elements per input position (tokens of the finest level x its widest buffer,
    # the fc1 output of 4 C columns): the element-wise kernels address with 32-bit offsets, so one call must stay below 2^32
    _ELEMS_PER_INPUT_POSITION = {"g_a": 4 * 96 / 4, "g_s": 64 * 4 * 96, "h_a": 4 * 192 / 4, "h_z_s1": 16 * 4 * 320, "h_z_s2": 16 * 4 * 320}

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if x.dim() != 4 or x.shape[1] != self.c_in:
            raise ValueError(f"{self.stack}: expected [B, {self.c_in}, H, W], got {tuple(x.shape)}")
        per_image = x.shape[2] * x.shape[3] * self._ELEMS_PER_INPUT_POSITION[self.stack]
        max_b = max(1, int((1 << 31) // max(per_image, 1)))           # half of the limit: headroom for padded widths
        if x.shape[0] > max_b:                                         # images are independent: run the batch in slices
            return torch.cat([self._forward(x[i:i + max_b]) for i in range(0, x.shape[0], max_b)], dim=0)
        return self._forward(x)

    def _forward(self, x: torch.Tensor) -> torch.Tensor:
        K = self.K
        blocks = self.blocks
        # the first operator decides the entry layout: a stride-2 conv reads C fp32 columns of any ld, a GEMM reads pad32(C)
        ld_in = pad32(self.c_in) if blocks[0][0] != "conv" else (self.c_in + 3) // 4 * 4
        a = K.to_tokens(x, ld_in, want=blocks[0][1].needs)
        for j, (kind, blk) in enumerate(blocks):
            last = j == len(blocks) - 1
            want = F32 if last else blocks[j + 1][1].needs            # the forms the successor reads
            if kind == "deconv" and last:
                a = blk(K, a, want=want, c_pad=(self.c_out + 3) // 4 * 4)     # nothing reads padded columns behind the last operator
            else:
                a = blk(K, a, want=want)
        return K.to_nchw(a, self.c_out)

    __call__ = forward


def accelerate_transforms(net: torch.nn.Module, device="cuda:0", math: str = "f16x3", stacks: Sequence[str] = STACKS) -> Dict[str, TransformStack]:
    """Redirect `net.g_a / g_s / h_a / h_z_s1 / h_z_s2` of a reference `DCAE` instance to the CUDA library, in place
    (instance-level `forward`, the modules and their parameters stay where they are, like `accelerate`).  The packed
    weights follow the module's parameters: they are repacked when a parameter's version counter or address changed
    (an optimizer step, `load_state_dict`).  Under autograd a call becomes one `training.TransformStackFunction` node
    over the module's own parameters -- kernels forward, recompute backward -- so gradients land in `net.parameters()`."""
    out = {}
    for name in stacks:
        mod = getattr(net, name)
        tracked = dict(list(mod.named_parameters()) + list(mod.named_buffers()))
        ts = TransformStack(name, {k: v.detach() for k, v in mod.state_dict().items()}, device=device, math=math)
        sig = [tuple((t.data_ptr(), t._version) for t in tracked.values())]

        def fwd(x, ts=ts, tracked=tracked, sig=sig):
            now = tuple((t.data_ptr(), t._version) for t in tracked.values())
            if now != sig[0]:
                ts.refresh({k: v.detach() for k, v in tracked.items()})
                sig[0] = now
            if torch.is_grad_enabled() and (x.requires_grad or any(t.requires_grad for t in tracked.values())):
                from .training import TransformStackFunction
                return TransformStackFunction.apply(ts, list(tracked), x, *tracked.values())
            return ts.forward(x)

        mod.forward = fwd
        out[name] = ts
    return out


__all__ = ["TransformStack", "init_transform_params", "LibKernels", "Act", "ARCH", "STACKS", "accelerate_transforms", "transform_param_shapes",
           "conv_s2_to_gemm", "deconv_s2_to_gemm", "conv3x3_to_gemm", "linear_to_gemm", "pad32", "pad8", "F32", "P16"]
