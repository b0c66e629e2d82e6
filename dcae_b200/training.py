"""Training support for the hot path (BASELINE config #4: rate-distortion step, train.py:165-179).

Forward runs on the library's kernels; backward recomputes the same operator graph in PyTorch ops under autograd
(`dcae_b200.torch_graph`: gradient checkpointing with a fast forward -- SURVEY section 7's plan) with kernel 3
differentiated analytically on the device (`dcae_gc_backward`).  Three entry points:

  GaussianLikelihoodFunction   lik = GaussianConditional(y, scale, mu) with grad (kernel 3 forward + backward kernel)
  SliceLoopFunction            the whole slice loop of DCAE.forward (dcae.py:638-670) as one autograd node
  EntropyModel                 nn.Module owning the hot-path parameters under the reference's keys; what DDP wraps
                               (train.py:413-426) when only the entropy model trains or is benchmarked

and the same pattern for the transform stacks g_a / g_s / h_a / h_z_s1 / h_z_s2 (`dcae_b200.transform_graph` is their
recompute graph; the windowed attention core keeps a kernel backward, `dcae_op_window_attention_backward`):

  WindowAttentionFunction      the WMSA core with the library's forward and backward kernels
  TransformStackFunction       one stack call as one autograd node (forward = `TransformStack.forward`)
  TransformModel               nn.Module owning one stack's parameters, the transform counterpart of EntropyModel

Gradients are the exact gradients of the fp32 graph (the forward values agree with it to 1e-5, tests/test_gpu_training.py
pins gradient parity against the reference's own modules under torch autograd).
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.nn as nn

from . import _lib, torch_graph, transform_graph
from .entropy_model import EntropySliceLoop
from .params import init_entropy_params
from .transforms import TransformStack, init_transform_params, transform_param_shapes


def _rows(t: torch.Tensor):
    """(contiguous tensor, rows, inner) of an NCHW tensor for the row-strided kernel-3 ABI."""
    t = t.contiguous()
    return t, t.shape[0], t[0].numel()


class GaussianLikelihoodFunction(torch.autograd.Function):
    """likelihood of compressai GaussianConditional.forward (dcae.py:657; math :839-857) for [B, C, h, w] tensors.
    noise=None: eval-mode quantisation (no gradient to y / mu through the likelihood, as with torch.round);
    noise given: training mode, out = y + noise."""

    @staticmethod
    def forward(ctx, y, scale, mu, noise, scale_bound: float, lik_bound: float, lik_math: str):
        lib = _lib.load()
        y, rows, inner = _rows(y)
        scale, mu = scale.contiguous(), mu.contiguous()
        if inner % 4:
            raise _lib.DcaeError("GaussianLikelihoodFunction: C*h*w must be a multiple of 4")
        lik = torch.empty_like(mu)
        a = _lib.GcArgs()
        a.y, a.y_ld, a.mu, a.mu_ld, a.scale, a.scale_ld = y.data_ptr(), inner, mu.data_ptr(), inner, scale.data_ptr(), inner
        a.scale_bound, a.lik_bound, a.rows, a.inner = scale_bound, lik_bound, rows, inner
        a.lik, a.lik_ld, a.lik_math = lik.data_ptr(), inner, _lib.GC_LIK[lik_math]
        a.mode = _lib.GC_EVAL
        if noise is not None:
            noise = noise.contiguous()
            a.mode, a.noise, a.noise_ld = _lib.GC_NOISE, noise.data_ptr(), inner
        with torch.cuda.device(y.device):
            _lib.check(lib.dcae_gc_fused(a, _lib.current_stream(y.device)), "dcae_gc_fused")
        ctx.save_for_backward(y, scale, mu, noise if noise is not None else y.new_empty(0))
        ctx.bounds = (scale_bound, lik_bound, noise is not None)
        return lik

    @staticmethod
    def backward(ctx, g):
        y, scale, mu, noise = ctx.saved_tensors
        scale_bound, lik_bound, noisy = ctx.bounds
        lib = _lib.load()
        g = g.contiguous()
        rows, inner = y.shape[0], y[0].numel()
        gy, gm, gs = torch.empty_like(y), torch.empty_like(y), torch.empty_like(y)
        a = _lib.GcBwdArgs()
        a.y, a.y_ld, a.mu, a.mu_ld, a.scale, a.scale_ld = y.data_ptr(), inner, mu.data_ptr(), inner, scale.data_ptr(), inner
        a.grad_lik, a.grad_lik_ld = g.data_ptr(), inner
        a.scale_bound, a.lik_bound, a.rows, a.inner = scale_bound, lik_bound, rows, inner
        a.mode = _lib.GC_NOISE if noisy else _lib.GC_EVAL
        if noisy:
            a.noise, a.noise_ld = noise.data_ptr(), inner
        a.grad_y, a.grad_y_ld, a.grad_mu, a.grad_mu_ld, a.grad_scale, a.grad_scale_ld = gy.data_ptr(), inner, gm.data_ptr(), inner, gs.data_ptr(), inner
        with torch.cuda.device(y.device):
            _lib.check(lib.dcae_gc_backward(a, _lib.current_stream(y.device)), "dcae_gc_backward")
        return gy, gs, gm, None, None, None, None


def gaussian_likelihood(y, scale, mu, noise=None, scale_bound=0.11, lik_bound=1e-9, lik_math="fast"):
    return GaussianLikelihoodFunction.apply(y, scale, mu, noise, scale_bound, lik_bound, lik_math)


class SliceLoopFunction(torch.autograd.Function):
    """(y_hat, means, scales, likelihoods) = slice loop(y, latent_scales, latent_means[, noise]; params) as ONE autograd
    node: forward = `EntropySliceLoop.forward` (the CUDA kernels), backward = recompute in `torch_graph` + autograd."""

    @staticmethod
    def forward(ctx, engine: EntropySliceLoop, keys, noise, y, ls, lm, *params):
        out = engine.forward(y, ls, lm, noise=noise)
        ctx.engine, ctx.keys = engine, keys
        ctx.save_for_backward(y, ls, lm, noise if noise is not None else y.new_empty(0), *params)
        return out["y_hat"], out["means"], out["scales"], out["likelihoods"]

    @staticmethod
    def backward(ctx, g_yhat, g_mu, g_sc, g_lik):
        y, ls, lm, noise, *params = ctx.saved_tensors
        noise = noise if noise.numel() else None
        eng = ctx.engine
        with torch.enable_grad():
            leaves = [t.detach().requires_grad_(True) for t in (y, ls, lm)]
            plist = [p.detach().requires_grad_(True) for p in params]
            P = dict(zip(ctx.keys, plist))
            gc = lambda ys, sc, mu, nz: gaussian_likelihood(ys, sc, mu, nz, lik_math=eng.likelihood_math)   # noqa: E731
            outs = torch_graph.slice_loop(P, leaves[0], leaves[1], leaves[2], gc, noise)
            grads = torch.autograd.grad(outs, leaves + plist, [g_yhat, g_mu, g_sc, g_lik], allow_unused=True)
        return (None, None, None) + tuple(grads)


class ModuleFunction(torch.autograd.Function):
    """One hot-path sub-module of a reference DCAE (dt_cross_attention[i], cc_*_transforms[i], lrp_transforms[i]) as an
    autograd node: forward = the library call `fast(*inputs)`, backward = recompute `graph(inputs, params)` in torch ops.
    Used by `dcae_b200.accelerate` when a call happens under autograd, so that the reference's own train.py step
    (train.py:165-179) differentiates through the redirected modules into the reference's own parameters."""

    @staticmethod
    def forward(ctx, fast, graph, keys, n_in, *tensors):
        ins = tensors[:n_in]
        ctx.graph, ctx.keys, ctx.n_in = graph, keys, n_in
        ctx.save_for_backward(*tensors)
        return fast(*[t.detach() for t in ins])

    @staticmethod
    def backward(ctx, g):
        tensors = ctx.saved_tensors
        with torch.enable_grad():
            leaves = [t.detach().requires_grad_(True) for t in tensors]
            out = ctx.graph(leaves[:ctx.n_in], dict(zip(ctx.keys, leaves[ctx.n_in:])))
            grads = torch.autograd.grad(out, leaves, g, allow_unused=True)
        return (None, None, None, None) + tuple(grads)


class EntropyModel(nn.Module):
    """The hot path as a trainable module: parameters in a ParameterList, `keys` holds the reference's state-dict key of
    each (`reference_state_dict()` gives the mapping back), forward = the slice loop.  Eval / no-grad calls run
    the inference kernels only; training calls go through `SliceLoopFunction`.  The packed device weights follow the
    parameters (repacked when their version counters change, i.e. after an optimizer step or load)."""

    def __init__(self, params: Optional[Dict[str, torch.Tensor]] = None, device="cuda:0", math: str = "f16x3", lanes: int = 1, seed: int = 0,
                 likelihood_math: str = "fast"):
        super().__init__()
        params = params if params is not None else init_entropy_params(seed)
        self.keys = list(params)
        self.plist = nn.ParameterList([nn.Parameter(params[k].detach().clone().to(device, torch.float32)) for k in self.keys])
        self.engine = [EntropySliceLoop({k: p.detach() for k, p in zip(self.keys, self.plist)}, device=device, math=math, lanes=lanes,
                                        likelihood_math=likelihood_math)]
        self._sig = self._signature()

    def _signature(self):
        return tuple((p.data_ptr(), p._version) for p in self.plist)

    def reference_state_dict(self) -> Dict[str, torch.Tensor]:
        return {k: p.detach() for k, p in zip(self.keys, self.plist)}

    def sync(self) -> None:
        if self._signature() != self._sig:
            self.engine[0].refresh(self.reference_state_dict())
            self._sig = self._signature()

    def forward(self, y, latent_scales, latent_means, noise: Optional[torch.Tensor] = None):
        """-> dict(y_hat, means, scales, likelihoods); noise: U(-1/2, 1/2) tensor like y for the training-mode likelihood
        (drawn here when the module is in train() mode and none is given)."""
        self.sync()
        if self.training and noise is None:
            noise = torch.empty_like(y).uniform_(-0.5, 0.5)
        needs_grad = torch.is_grad_enabled() and (any(p.requires_grad for p in self.plist) or y.requires_grad or latent_scales.requires_grad or latent_means.requires_grad)
        if not needs_grad:
            out = self.engine[0].forward(y, latent_scales, latent_means, noise=noise)
            return {k: out[k] for k in ("y_hat", "means", "scales", "likelihoods")}
        y_hat, mu, sc, lik = SliceLoopFunction.apply(self.engine[0], self.keys, noise, y, latent_scales, latent_means, *self.plist)
        return {"y_hat": y_hat, "means": mu, "scales": sc, "likelihoods": lik}


class WindowAttentionFunction(torch.autograd.Function):
    """out [B, h, w, C] = WMSA core of qkv [B, h, w, 3C] ('(threeh c)' columns) with relative position bias rel
    [n_heads, 2 window - 1, 2 window - 1]: forward dcae_op_window_attention (fp32 output), backward
    dcae_op_window_attention_backward (dq / dk / dv and drel).  The signature of `transform_graph.window_attention`."""

    @staticmethod
    def forward(ctx, qkv, head_dim: int, window: int, shift: int, rel):
        lib = _lib.load()
        qkv, rel = qkv.contiguous(), rel.contiguous()
        B, h, w, C3 = qkv.shape
        C = C3 // 3
        out = qkv.new_empty(B, h, w, C)
        with torch.cuda.device(qkv.device):
            _lib.check(lib.dcae_op_window_attention(qkv.data_ptr(), C3, 0, C, 2 * C, C, head_dim, window, shift, rel.data_ptr(), B, h, w,
                                                    out.data_ptr(), C, None, _lib.current_stream(qkv.device)), "dcae_op_window_attention")
        ctx.save_for_backward(qkv, rel)
        ctx.cfg = (head_dim, window, shift)
        return out

    @staticmethod
    def backward(ctx, g):
        qkv, rel = ctx.saved_tensors
        head_dim, window, shift = ctx.cfg
        lib = _lib.load()
        g = g.contiguous()
        B, h, w, C3 = qkv.shape
        C = C3 // 3
        dqkv, drel = torch.empty_like(qkv), torch.empty_like(rel)
        n = int(lib.dcae_window_attention_backward_scratch_bytes(B, h, w, C, head_dim, window))
        scratch = torch.empty(max(n, 16), dtype=torch.uint8, device=qkv.device)
        with torch.cuda.device(qkv.device):
            _lib.check(lib.dcae_op_window_attention_backward(qkv.data_ptr(), C3, 0, C, 2 * C, C, head_dim, window, shift, rel.data_ptr(), B, h, w,
                                                             g.data_ptr(), C, dqkv.data_ptr(), C3, drel.data_ptr(), scratch.data_ptr(), n,
                                                             _lib.current_stream(qkv.device)), "dcae_op_window_attention_backward")
        return dqkv, None, None, None, drel


def window_attention(qkv, head_dim: int, window: int, shift: int, rel):
    return WindowAttentionFunction.apply(qkv, head_dim, window, shift, rel)


class TransformStackFunction(torch.autograd.Function):
    """y = stack(x; params) as ONE autograd node: forward = `TransformStack.forward` (the kernels, in the stack's math mode),
    backward = recompute `transform_graph.stack` on the saved input with `WindowAttentionFunction` + torch.autograd.grad.
    `keys`: the state-dict key of each parameter, with or without the stack prefix.  The recompute's dense layers and
    convolutions are torch ops and follow torch's TF32 settings."""

    @staticmethod
    def forward(ctx, engine: TransformStack, keys, x, *params):
        ctx.engine, ctx.keys = engine, [k[len(engine.stack) + 1:] if k.startswith(engine.stack + ".") else k for k in keys]
        ctx.save_for_backward(x, *params)
        return engine.forward(x)

    @staticmethod
    def backward(ctx, g):
        x, *params = ctx.saved_tensors
        with torch.enable_grad():
            leaf = x.detach().requires_grad_(True)
            plist = [p.detach().requires_grad_(True) for p in params]
            out = transform_graph.stack(ctx.engine.stack, dict(zip(ctx.keys, plist)), leaf, attn=window_attention)
            grads = torch.autograd.grad(out, [leaf] + plist, g, allow_unused=True)
        return (None, None) + tuple(grads)


class TransformModel(nn.Module):
    """One transform stack (g_a / g_s / h_a / h_z_s1 / h_z_s2) as a trainable module: parameters in a ParameterList, `keys`
    holds the reference's state-dict key of each ('g_a.0.conv.weight'; `reference_state_dict()` gives the mapping back),
    forward(x NCHW) = the stack.  No-grad calls run the kernels only (the bits of `TransformStack.forward`); calls under
    autograd go through `TransformStackFunction`.  The packed device weights follow the parameters (repacked when their
    version counters or addresses change, i.e. after an optimizer step or load)."""

    def __init__(self, stack: str, params: Optional[Dict[str, torch.Tensor]] = None, device="cuda:0", math: str = "f16x3", seed: int = 0):
        super().__init__()
        params = params if params is not None else init_transform_params(seed, (stack,))
        self.stack = stack
        self.keys = [f"{stack}.{k}" for k in transform_param_shapes(stack)]
        vals = [params.get(k, params.get(k[len(stack) + 1:])) for k in self.keys]
        missing = [k for k, v in zip(self.keys, vals) if v is None]
        if missing:
            raise KeyError(f"{stack}: missing parameters {missing[:3]}")
        self.plist = nn.ParameterList([nn.Parameter(v.detach().clone().to(device, torch.float32)) for v in vals])
        self.engine = [TransformStack(stack, self.reference_state_dict(), device=device, math=math)]
        self._sig = self._signature()

    def _signature(self):
        return tuple((p.data_ptr(), p._version) for p in self.plist)

    def reference_state_dict(self) -> Dict[str, torch.Tensor]:
        return {k: p.detach() for k, p in zip(self.keys, self.plist)}

    def sync(self) -> None:
        if self._signature() != self._sig:
            self.engine[0].refresh(self.reference_state_dict())
            self._sig = self._signature()

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        self.sync()
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.plist)):
            return TransformStackFunction.apply(self.engine[0], self.keys, x, *self.plist)
        return self.engine[0].forward(x)


def rate_distortion_loss(likelihoods: torch.Tensor, y_hat: torch.Tensor, target: torch.Tensor, num_pixels: int, lmbda: float = 0.013):
    """train.py:82-88 with type='mse': bpp = sum(log lik) / (-ln 2 * pixels); loss = lmbda * 255^2 * mse + bpp.  (In the
    reference the distortion is measured on g_s(y_hat) against the image; for the entropy-model-only step the synthesis
    transform is the identity and `target` is y.)"""
    import math
    bpp = torch.log(likelihoods).sum() / (-math.log(2) * num_pixels)
    mse = torch.mean((y_hat - target) ** 2)
    return lmbda * 255 ** 2 * mse + bpp, bpp, mse
