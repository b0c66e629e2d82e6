"""The transform stacks g_a / g_s / h_a / h_z_s1 / h_z_s2 in differentiable PyTorch ops -- used ONLY to DIFFERENTIATE.

This file is to `dcae_b200.transforms` what `torch_graph` is to the slice loop: `dcae_b200.training.TransformStackFunction`
runs a stack's forward pass on the library's kernels and, in backward, recomputes the same graph here under autograd.
Parameters arrive as a dict with the reference's state-dict keys relative to the stack prefix ('0.conv.weight'), as
`transforms.transform_param_shapes` lists them, so gradients map one to one onto the reference's parameters.

The windowed attention core is a parameter of the graph: `window_attention` below is the pure-torch form (the CPU and
fp64 reference); `training.WindowAttentionFunction` runs the library's forward and backward kernels
(dcae_op_window_attention / dcae_op_window_attention_backward) and is what the GPU recompute uses.
"""
from __future__ import annotations

import math
from typing import Callable, Dict

import torch
import torch.nn.functional as F

from .transforms import ARCH

P = Dict[str, torch.Tensor]
# attn(qkv [B, h, w, 3C], head_dim, window, shift, rel [n_heads, 2P-1, 2P-1]) -> [B, h, w, C]
Attention = Callable[[torch.Tensor, int, int, int, torch.Tensor], torch.Tensor]


def window_attention(qkv: torch.Tensor, head_dim: int, window: int, shift: int, rel: torch.Tensor) -> torch.Tensor:
    """WMSA core (dcae.py:262-291), vectorised: roll by -shift (:270), windows of window x window tokens, per head
    q k^T / sqrt(hd) + relative position bias (:293-296), SW mask (generate_mask, :244-260), softmax, p v, roll back (:289).
    qkv: [B, h, w, 3C] in embedding_layer's '(threeh c)' column order (q heads | k heads | v heads)."""
    B, h, w, C3 = qkv.shape
    C, Pw = C3 // 3, window
    nh, ny, nx = C // head_dim, h // Pw, w // Pw
    if shift:
        qkv = torch.roll(qkv, shifts=(-shift, -shift), dims=(1, 2))
    x = qkv.reshape(B, ny, Pw, nx, Pw, 3, nh, head_dim).permute(5, 0, 1, 3, 6, 2, 4, 7).reshape(3, B, ny, nx, nh, Pw * Pw, head_dim)
    q, k, v = x[0], x[1], x[2]
    pos = torch.stack(torch.meshgrid(torch.arange(Pw), torch.arange(Pw), indexing="ij"), -1).reshape(-1, 2).to(qkv.device)
    d = pos[:, None, :] - pos[None, :, :] + Pw - 1
    sim = q @ k.transpose(-1, -2) / math.sqrt(head_dim) + rel[:, d[..., 0], d[..., 1]]
    if shift:
        sp = Pw - shift
        side = pos < sp                                                     # [PP, 2]: which part of a split window
        cross = side[:, None, :] != side[None, :, :]                        # [PP, PP, 2]
        mask = torch.zeros(ny, nx, Pw * Pw, Pw * Pw, dtype=torch.bool, device=qkv.device)
        mask[-1] |= cross[..., 0]
        mask[:, -1] |= cross[..., 1]
        sim = sim.masked_fill(mask[None, :, :, None], float("-inf"))
    o = sim.softmax(-1) @ v                                                 # [B, ny, nx, nh, PP, hd]
    o = o.reshape(B, ny, nx, nh, Pw, Pw, head_dim).permute(0, 1, 4, 2, 5, 3, 6).reshape(B, h, w, C)
    if shift:
        o = torch.roll(o, shifts=(shift, shift), dims=(1, 2))
    return o


def conv(x, w, b):
    """conv(cin, cout, k, stride 2), dcae.py:35-42."""
    return F.conv2d(x, w, b, stride=2, padding=w.shape[-1] // 2)


def deconv(x, w, b):
    """deconv(cin, cout, k, stride 2), dcae.py:44-52."""
    return F.conv_transpose2d(x, w, b, stride=2, padding=w.shape[-1] // 2, output_padding=1)


def residual_bottleneck(x, p: P, pre: str):
    """ResidualBottleneckBlock(c, c), dcae.py:152-190: 1x1 -> ReLU -> 3x3 -> ReLU -> 1x1, + x (the skip is Identity); NCHW."""
    t = F.relu(F.conv2d(x, p[pre + "conv1.weight"], p[pre + "conv1.bias"]))
    t = F.relu(F.conv2d(t, p[pre + "conv2.weight"], p[pre + "conv2.bias"], padding=1))
    return F.conv2d(t, p[pre + "conv3.weight"], p[pre + "conv3.bias"]) + x


def swin_layer(x, p: P, pre: str, head_dim: int, window: int, shift: int, attn: Attention):
    """ResScaleConvolutionGateBlock, dcae.py:338-360, with WMSA (:228-298) and ConvolutionalGLU (:300-327); x: [B, h, w, C].
    x = s1 x + linear(attn(embedding(LN1 x))); x = s2 x + fc2(GELU(dwconv(a)) * v), (a, v) = fc1(LN2 x)."""
    C = x.shape[-1]
    t = F.layer_norm(x, (C,), p[pre + "ln1.weight"], p[pre + "ln1.bias"], 1e-5)
    qkv = F.linear(t, p[pre + "msa.embedding_layer.weight"], p[pre + "msa.embedding_layer.bias"])
    t = F.linear(attn(qkv, head_dim, window, shift, p[pre + "msa.relative_position_params"]), p[pre + "msa.linear.weight"], p[pre + "msa.linear.bias"])
    x = x * p[pre + "res_scale_1.scale"] + t
    t = F.layer_norm(x, (C,), p[pre + "ln2.weight"], p[pre + "ln2.bias"], 1e-5)
    a, v = F.linear(t, p[pre + "mlp.fc1.weight"], p[pre + "mlp.fc1.bias"]).chunk(2, dim=-1)
    a = F.conv2d(a.permute(0, 3, 1, 2), p[pre + "mlp.dwconv.dwconv.weight"], p[pre + "mlp.dwconv.dwconv.bias"], padding=1, groups=a.shape[-1])
    t = F.linear(F.gelu(a.permute(0, 2, 3, 1)) * v, p[pre + "mlp.fc2.weight"], p[pre + "mlp.fc2.bias"])
    return x * p[pre + "res_scale_2.scale"] + t


def swin_block(x, p: P, pre: str, head_dim: int, window: int, n: int, attn: Attention):
    """SwinBlockWithConvMulti, dcae.py:362-383: n alternating W / SW layers on [B, h, w, C], then conv3x3 + x; NCHW in / out.
    Like `transforms._Swin`, grids that are no multiple of the window or not larger than it are refused (dcae.py:374-377)."""
    h, w = x.shape[-2:]
    if h <= window or w <= window or h % window or w % window:
        raise ValueError(f"Swin block: token grid {h}x{w} must be a multiple of the window {window} and larger than it")
    t = x.permute(0, 2, 3, 1)
    for i in range(n):
        t = swin_layer(t, p, pre + f"layers.{i}.", head_dim, window, window // 2 if i % 2 else 0, attn)
    return F.conv2d(t.permute(0, 3, 1, 2), p[pre + "conv.weight"], p[pre + "conv.bias"], padding=1) + x


def stack(name: str, p: P, x: torch.Tensor, attn: Attention = window_attention) -> torch.Tensor:
    """One of g_a / g_s / h_a / h_z_s1 / h_z_s2 (dcae.py:541-582) on NCHW x, blocks as `transforms.ARCH` lists them:
    ResidualBlockWithStride = conv + 3 bottlenecks, ResidualBlockUpsample = 3 bottlenecks + deconv."""
    for idx, spec in enumerate(ARCH[name]):
        pre, kind = f"{idx}.", spec[0]
        if kind == "rbws":
            x = conv(x, p[pre + "conv.weight"], p[pre + "conv.bias"])
            for r in (1, 2, 3):
                x = residual_bottleneck(x, p, pre + f"res{r}.")
        elif kind == "rbwu":
            for r in (1, 2, 3):
                x = residual_bottleneck(x, p, pre + f"res{r}.")
            x = deconv(x, p[pre + "conv.weight"], p[pre + "conv.bias"])
        elif kind == "conv_s2":
            x = conv(x, p[pre + "weight"], p[pre + "bias"])
        elif kind == "deconv_s2":
            x = deconv(x, p[pre + "weight"], p[pre + "bias"])
        else:
            _, _, hd, win, n = spec
            x = swin_block(x, p, pre, hd, win, n, attn)
    return x


__all__ = ["window_attention", "stack", "conv", "deconv", "residual_bottleneck", "swin_layer", "swin_block"]
