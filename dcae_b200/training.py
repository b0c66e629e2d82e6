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

and for the hyper-latent entropy bottleneck and the whole model:

  EntropyBottleneckFunction    the bottleneck's likelihood with the library's forward and backward kernels
                               (`dcae_eb_fused`, `dcae_eb_backward`)
  EntropyBottleneckModel       `EntropyBottleneck` that trains (same keys); aux loss with compressai's stop_gradient
  DCAEModel                    the whole DCAE (dcae.py:623-677) as one trainable nn.Module over the reference's keys

Gradients are the exact gradients of the fp32 graph (the forward values agree with it to 1e-5, tests/test_gpu_training.py
pins gradient parity against the reference's own modules under torch autograd).
"""
from __future__ import annotations

import math as _math
from typing import Dict, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, torch_graph, transform_graph
from .entropy_bottleneck import EntropyBottleneck
from .entropy_model import EntropySliceLoop, get_scale_table
from .gaussian_conditional import GaussianConditional
from .modules import HOT_PREFIXES
from .msssim import ms_ssim
from .params import init_entropy_params
from .transforms import STACKS, TransformStack, init_transform_params, transform_param_shapes


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


def dcae_rate_distortion_loss(out: dict, target: torch.Tensor, lmbda: float = 0.013, metric: str = "mse"):
    """train.py:82-88 for the whole model: bpp = sum over BOTH likelihood tensors (y and z) of
    sum(log lik) / (-ln 2 * pixels), pixels = N * H * W of the image.
      metric="mse"      loss = lmbda * 255^2 * mse(x_hat, target) + bpp              -> (loss, bpp, mse)
      metric="ms-ssim"  loss = lmbda * (1 - ms_ssim(x_hat, target, data_range=1)) + bpp  -> (loss, bpp, ms_ssim)
    (the ms-ssim form of the TCM-lineage RateDistortionLoss; MS-SSIM on the library's kernels, dcae_b200/msssim.py)."""
    if metric not in ("mse", "ms-ssim"):
        raise ValueError(f"dcae_rate_distortion_loss: metric must be 'mse' or 'ms-ssim', got {metric!r}")
    N, _, H, W = target.shape
    pixels = N * H * W
    bpp = sum(torch.log(lik).sum() / (-_math.log(2) * pixels) for lik in out["likelihoods"].values())
    if metric == "ms-ssim":
        msssim = ms_ssim(out["x_hat"], target, data_range=1.0)
        return lmbda * (1 - msssim) + bpp, bpp, msssim
    mse = F.mse_loss(out["x_hat"], target)
    return lmbda * 255 ** 2 * mse + bpp, bpp, mse


# ---- the hyper-latent entropy bottleneck ---------------------------------------------------------------------------------

class EntropyBottleneckFunction(torch.autograd.Function):
    """(lik, z_hat) = compressai EntropyBottleneck likelihood of z [B, C, h, w] (dcae.py:630) with the packed density
    `params` [C, 58] (softplus(_matrix*) | _bias* | tanh(_factor*), as `EntropyBottleneck._pack` lays them out) and
    `medians` [C] (no gradient, compressai detaches them).  noise given: training mode, out = z + noise; None: eval mode,
    out = round(z - median) + median.  Forward dcae_eb_fused, backward dcae_eb_backward; the packed tensor is built under
    autograd by the caller, so torch chains its gradient back to _matrix* / _bias* / _factor*.  z_hat = round(z - median)
    + median in both modes, not differentiable (the caller attaches the straight-through gradient)."""

    @staticmethod
    def forward(ctx, z, noise, params, medians, lik_bound: float):
        z, params, medians = z.contiguous().float(), params.contiguous().float(), medians.contiguous().float()
        noise = noise.contiguous().float() if noise is not None else None
        B, C, h, w = z.shape
        lik, z_hat = torch.empty_like(z), torch.empty_like(z)
        a = _lib.EbArgs()
        a.z, a.params, a.medians = z.data_ptr(), params.data_ptr(), medians.data_ptr()
        a.mode = _lib.GC_NOISE if noise is not None else _lib.GC_EVAL
        if noise is not None:
            a.noise = noise.data_ptr()
        a.B, a.C, a.HW, a.lik_bound = B, C, h * w, lik_bound
        a.z_hat, a.lik = z_hat.data_ptr(), lik.data_ptr()
        if z.numel():
            with torch.cuda.device(z.device):
                _lib.check(_lib.load().dcae_eb_fused(a, _lib.current_stream(z.device)), "dcae_eb_fused")
        ctx.save_for_backward(z, noise if noise is not None else z.new_empty(0), params, medians)
        ctx.lik_bound = lik_bound
        ctx.mark_non_differentiable(z_hat)
        return lik, z_hat

    @staticmethod
    def backward(ctx, g_lik, _g_zhat):
        z, noise, params, medians = ctx.saved_tensors
        noisy = noise.numel() > 0
        B, C, h, w = z.shape
        g_lik = g_lik.contiguous().float()
        gz, gp = torch.empty_like(z), torch.empty_like(params)
        a = _lib.EbBwdArgs()
        a.z, a.params, a.medians, a.grad_lik = z.data_ptr(), params.data_ptr(), medians.data_ptr(), g_lik.data_ptr()
        a.mode = _lib.GC_NOISE if noisy else _lib.GC_EVAL
        if noisy:
            a.noise = noise.data_ptr()
        a.B, a.C, a.HW, a.lik_bound = B, C, h * w, ctx.lik_bound
        a.grad_z, a.grad_params = gz.data_ptr(), gp.data_ptr()
        with torch.cuda.device(z.device):
            _lib.check(_lib.load().dcae_eb_backward(a, _lib.current_stream(z.device)), "dcae_eb_backward")
        return gz, None, gp, None, None


class EntropyBottleneckModel(EntropyBottleneck):
    """`dcae_b200.EntropyBottleneck` that trains: the same parameter and buffer names (state dicts move either way between
    it, `EntropyBottleneck` and `DCAECodec`).  Calls under autograd go through `EntropyBottleneckFunction` with the packed
    density built differentiably; calls without autograd are `EntropyBottleneck.forward`'s launch, bit for bit.
    `loss()` is compressai's aux loss: stop_gradient=True, so its gradient reaches `quantiles` only."""

    def _pack_graph(self, device) -> torch.Tensor:
        """[C, 58] as `_pack` builds it, under autograd."""
        parts = [F.softplus(getattr(self, f"_matrix{i}")).reshape(self.channels, -1) for i in range(5)]
        parts += [getattr(self, f"_bias{i}").reshape(self.channels, -1) for i in range(5)]
        parts += [torch.tanh(getattr(self, f"_factor{i}")).reshape(self.channels, -1) for i in range(4)]
        return torch.cat(parts, dim=1).to(device, torch.float32)

    def forward_parts(self, x: torch.Tensor, training: Optional[bool] = None, noise: Optional[torch.Tensor] = None):
        """-> (outputs, likelihood, z_hat): outputs as compressai's forward returns them (x + noise in training mode,
        round(x - median) + median otherwise) and z_hat = round(x - median) + median, the value dcae.py:631-633 passes on."""
        if training is None:
            training = self.training
        if training and noise is None:
            noise = torch.empty_like(x).uniform_(-0.5, 0.5)
        if not training:
            noise = None
        if not x.is_cuda:
            raise _lib.DcaeError("dcae_b200.EntropyBottleneckModel runs on CUDA tensors only (no CPU fallback)")
        if len(x.shape) != 4 or x.shape[1] != self.channels:
            raise ValueError(f"expected [B, {self.channels}, h, w], got {tuple(x.shape)}")
        if not (torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters()))):
            o = self._run(_lib.GC_NOISE if noise is not None else _lib.GC_EVAL, x, noise=noise, want=("z_hat", "lik"))
            return (x + noise if noise is not None else o["z_hat"]), o["lik"], o["z_hat"]
        med = self.quantiles[:, 0, 1].detach().to(x.device, torch.float32)
        lik, z_hat = EntropyBottleneckFunction.apply(x, noise, self._pack_graph(x.device), med, self.likelihood_bound)
        return (x + noise if noise is not None else z_hat), lik, z_hat

    def forward(self, x: torch.Tensor, training: Optional[bool] = None, noise: Optional[torch.Tensor] = None):
        """-> (outputs, likelihood) like compressai (dcae.py:630)."""
        out, lik, _ = self.forward_parts(x, training, noise)
        return out, lik

    def loss(self) -> torch.Tensor:
        """aux loss (train.py:177) as compressai computes it: sum |logits_cumulative(quantiles) - target| with the density
        parameters detached."""
        return torch.abs(self._logits_cumulative(self.quantiles, stop_gradient=True) - self.target).sum()


def init_entropy_bottleneck_params(seed: int = 0, channels: int = 192) -> Dict[str, torch.Tensor]:
    """compressai's EntropyBottleneck initialisation (matrices log(expm1(1 / scale / fan)), biases U(-1/2, 1/2), factors 0,
    quantiles [-10, 0, 10]) from a fixed seed, under the reference's `entropy_bottleneck.` keys (parameters only)."""
    with torch.random.fork_rng(devices=[]):
        torch.manual_seed(seed)
        eb = EntropyBottleneck(channels)
    return {f"entropy_bottleneck.{k}": v.detach() for k, v in eb.named_parameters()}


# ---- the whole model ---------------------------------------------------------------------------------------------------

class DCAEModel(nn.Module):
    """The whole DCAE as one trainable module (dcae.py:623-677): five `TransformModel`s (g_a, g_s, h_a, h_z_s1, h_z_s2), the
    slice loop as an `EntropyModel` (one lane), an `EntropyBottleneckModel(192)` and a `GaussianConditional` holding the
    scale table.  `params`: a reference state dict (the keys `DCAECodec` takes); missing -> seeded initialisation.
    Every hot path runs on the library's kernels forward; backward is the kernels' backward (likelihoods, window attention)
    and torch recompute elsewhere.  `reference_state_dict()` loads into `DCAECodec` (compress / decompress) and back."""

    def __init__(self, params: Optional[Dict[str, torch.Tensor]] = None, device="cuda:0", math: str = "f16x3", seed: int = 0,
                 likelihood_math: str = "fast"):
        super().__init__()
        if params is None:
            params = dict(init_entropy_params(seed))
            params.update(init_transform_params(seed))
            params.update(init_entropy_bottleneck_params(seed))
        for name in STACKS:
            self.add_module(name, TransformModel(name, params, device=device, math=math))
        hot = {k: v for k, v in params.items() if k.split(".")[0] in HOT_PREFIXES}
        self.entropy = EntropyModel(hot, device=device, math=math, lanes=1, likelihood_math=likelihood_math)
        self.entropy_bottleneck = EntropyBottleneckModel(192)
        eb = {k[len("entropy_bottleneck."):]: v for k, v in params.items() if k.startswith("entropy_bottleneck.")}
        if eb:
            self.entropy_bottleneck.load_state_dict(eb, strict=False)
        self.entropy_bottleneck.to(device)
        table = params.get("gaussian_conditional.scale_table")
        table = table if table is not None and table.numel() else get_scale_table()
        self.gaussian_conditional = GaussianConditional(table.tolist(), likelihood_math=likelihood_math)
        gc = {k[len("gaussian_conditional."):]: v for k, v in params.items() if k.startswith("gaussian_conditional.")}
        if gc:
            self.gaussian_conditional.load_state_dict(gc, strict=False)
        self.gaussian_conditional.to(device)

    def forward(self, x: torch.Tensor, y_noise: Optional[torch.Tensor] = None, z_noise: Optional[torch.Tensor] = None) -> dict:
        """-> {"x_hat", "likelihoods": {"y", "z"}, "para": {"means", "scales", "y"}} (dcae.py:623-677).  A given noise tensor
        (U(-1/2, 1/2), shaped like y / z) selects the training-mode likelihood for its part; in train() mode missing
        noise is drawn, in eval() mode the latents are rounded."""
        y = self.g_a(x)
        z = self.h_a(y)
        if self.training and z_noise is None:
            z_noise = torch.empty_like(z).uniform_(-0.5, 0.5)
        _, z_lik, z_hat = self.entropy_bottleneck.forward_parts(z, training=z_noise is not None, noise=z_noise)
        if torch.is_grad_enabled() and z.requires_grad:
            z_hat = z_hat + (z - z.detach())           # ste_round(z - median) + median: the value round() gives, gradient 1
        latent_scales, latent_means = self.h_z_s1(z_hat), self.h_z_s2(z_hat)
        o = self.entropy(y, latent_scales, latent_means, noise=y_noise)
        x_hat = self.g_s(o["y_hat"])
        return {"x_hat": x_hat, "likelihoods": {"y": o["likelihoods"], "z": z_lik},
                "para": {"means": o["means"], "scales": o["scales"], "y": y}}

    def aux_loss(self) -> torch.Tensor:
        """train.py:177: the bottleneck's aux loss (gradient to `quantiles` only)."""
        return self.entropy_bottleneck.loss()

    def parameter_groups(self):
        """-> (main, aux): the optimizer split of train.py -- every `*.quantiles` in aux, everything else in main."""
        named = list(self.named_parameters())
        return ([p for n, p in named if not n.endswith(".quantiles")], [p for n, p in named if n.endswith(".quantiles")])

    def reference_state_dict(self) -> Dict[str, torch.Tensor]:
        """Every parameter under the reference's key, plus the entropy bottleneck's and the Gaussian conditional's buffers:
        what `DCAECodec` consumes, and what this class's constructor takes back."""
        sd: Dict[str, torch.Tensor] = {}
        for name in STACKS:
            sd.update(getattr(self, name).reference_state_dict())
        sd.update(self.entropy.reference_state_dict())
        sd.update({f"entropy_bottleneck.{k}": v.detach() for k, v in self.entropy_bottleneck.state_dict().items()})
        sd.update({f"gaussian_conditional.{k}": v.detach() for k, v in self.gaussian_conditional.state_dict().items()})
        return sd

    def update(self, force: bool = False) -> bool:
        """compressai's update(): the coder tables of both entropy models (dcae.py:616-621)."""
        updated = self.gaussian_conditional.update_scale_table(self.gaussian_conditional.scale_table, force=force)
        updated |= self.entropy_bottleneck.update(force=force)
        return updated
