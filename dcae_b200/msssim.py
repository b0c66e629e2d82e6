"""MS-SSIM on the library (pytorch_msssim.ms_ssim v1.0 with its defaults), the distortion of the ms-ssim rate-distortion
loss (`training.dcae_rate_distortion_loss(..., metric="ms-ssim")`).

  MSSSIMStatsFunction   per-level means of the ssim and cs maps, [5, B, C], as one autograd node: forward
                        dcae_msssim_forward (which leaves the pooled pyramid in a scratch buffer kept for the backward),
                        backward dcae_msssim_backward.  Only the first image is differentiated.
  ms_ssim               pytorch_msssim's combination of those statistics in torch ops: prod(relu(cs_0..3) ** w_0..3) *
                        relu(ssim_4) ** w_4, averaged over channels (and over images with size_average)

Window, constants and levels are pytorch_msssim's defaults (11 taps, sigma 1.5, K = (0.01, 0.03), 5 levels); only
data_range and size_average are exposed.  Inputs are fp32 CUDA [B, C, H, W] with min(H, W) > 160.
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import DcaeError

WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)
LEVELS = len(WEIGHTS)


def _check(X: torch.Tensor, Y: torch.Tensor) -> None:
    if not (X.is_cuda and Y.is_cuda):
        raise DcaeError("ms_ssim: the library has no CPU path; move both images to the GPU")
    if X.device != Y.device:
        raise ValueError(f"ms_ssim: images on different devices ({X.device}, {Y.device})")
    if Y.requires_grad:
        raise DcaeError("ms_ssim: only the first argument is differentiated; pass the second one detached")
    if X.dim() != 4 or X.shape != Y.shape:
        raise ValueError(f"ms_ssim: need two [B, C, H, W] images of one shape, got {tuple(X.shape)} and {tuple(Y.shape)}")
    if min(X.shape[-2:]) <= 160:
        raise ValueError(f"ms_ssim: min(H, W) must exceed 160 for 5 levels of an 11-tap window, got {tuple(X.shape[-2:])}")
    if X.dtype != torch.float32 or Y.dtype != torch.float32:
        raise ValueError(f"ms_ssim: fp32 images only, got {X.dtype} and {Y.dtype}")


def _args(cls, X, Y, data_range, scratch):
    a = cls()
    a.x, a.y = X.data_ptr(), Y.data_ptr()
    a.B, a.C, a.H, a.W = X.shape
    a.data_range = data_range
    a.scratch, a.scratch_bytes = scratch.data_ptr(), scratch.numel()
    return a


class MSSSIMStatsFunction(torch.autograd.Function):
    """(ssim, cs) = the means of the ssim and cs maps of every (level, image, channel), each [5, B, C].  Y gets no
    gradient."""

    @staticmethod
    def forward(ctx, X, Y, data_range: float):
        _check(X, Y)
        lib = _lib.load()
        X, Y = X.contiguous(), Y.contiguous()
        B, C, H, W = X.shape
        scratch = torch.empty(lib.dcae_msssim_scratch_bytes(B, C, H, W), dtype=torch.uint8, device=X.device)
        ssim = torch.empty(LEVELS, B, C, dtype=torch.float32, device=X.device)
        cs = torch.empty_like(ssim)
        a = _args(_lib.MsssimArgs, X, Y, data_range, scratch)
        a.ssim, a.cs = ssim.data_ptr(), cs.data_ptr()
        _lib.check(lib.dcae_msssim_forward(a, _lib.current_stream(X.device)), "dcae_msssim_forward")
        ctx.save_for_backward(X, Y, scratch)
        ctx.data_range = data_range
        return ssim, cs

    @staticmethod
    def backward(ctx, g_ssim, g_cs):
        X, Y, scratch = ctx.saved_tensors
        g_ssim = torch.zeros(LEVELS, *X.shape[:2], device=X.device) if g_ssim is None else g_ssim.contiguous()
        g_cs = torch.zeros_like(g_ssim) if g_cs is None else g_cs.contiguous()
        dX = torch.empty_like(X)
        a = _args(_lib.MsssimBwdArgs, X, Y, ctx.data_range, scratch)
        a.grad_ssim, a.grad_cs, a.grad_x = g_ssim.data_ptr(), g_cs.data_ptr(), dX.data_ptr()
        _lib.check(_lib.load().dcae_msssim_backward(a, _lib.current_stream(X.device)), "dcae_msssim_backward")
        return dX, None, None


def ms_ssim(X: torch.Tensor, Y: torch.Tensor, data_range: float = 1.0, size_average: bool = True) -> torch.Tensor:
    """pytorch_msssim.ms_ssim(X, Y, data_range, size_average) with its default window, K and weights: a scalar, or [B]
    without size_average.  Differentiable in X."""
    _check(X, Y)
    ssim, cs = MSSSIMStatsFunction.apply(X, Y, float(data_range))
    # Python-float exponents and a chain of products rather than torch.prod: no host-to-device copy and no host sync
    # (torch.prod's backward reads its zero count on the host), so the loss can sit inside a captured training step.
    # A relu-clamped zero factor still gets gradient 0: relu's backward masks the pow's infinite slope at 0.
    v = torch.relu(ssim[-1]) ** WEIGHTS[-1]
    for c, w in zip(cs[:-1], WEIGHTS[:-1]):
        v = v * torch.relu(c) ** w
    return v.mean() if size_average else v.mean(1)
