"""CPU: the MS-SSIM oracle (oracle/msssim.py) against an independent direct implementation and closed forms, the
backward formulation the kernels implement against fp64 autograd of the oracle, the C ABI of dcae_msssim_* (struct
layout, argument checks before any launch) and the `metric` keyword of dcae_rate_distortion_loss."""
import math
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch
from scipy import ndimage

from oracle import msssim as oms

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = [(161, 161), (200, 333), (256, 256)]      # odd and even sizes at every level


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from dcae_b200 import _lib
    return _lib.load()


def _pair(B, C, H, W, seed, noise=0.1):
    g = torch.Generator().manual_seed(seed)
    X = torch.rand(B, C, H, W, dtype=torch.float64, generator=g)
    return X, (X + noise * torch.randn(B, C, H, W, dtype=torch.float64, generator=g)).clamp(0, 1)


def _direct_level_stats(X: np.ndarray, Y: np.ndarray, data_range: float):
    """MS-SSIM statistics of one plane from scratch: scipy's 2-D correlation with the 11 x 11 outer-product window,
    cropped to the valid region, and explicit zero-padded 2 x 2 means between levels."""
    k = np.arange(11) - 5.0
    g = np.exp(-k ** 2 / (2 * 1.5 ** 2))
    g /= g.sum()
    w2 = np.outer(g, g)
    C1, C2 = (0.01 * data_range) ** 2, (0.03 * data_range) ** 2

    def f(a):
        return ndimage.correlate(a, w2, mode="constant")[5:-5, 5:-5]

    def pool(a):
        h, w = a.shape
        p = np.zeros((h + h % 2, w + w % 2))
        p[h % 2:, w % 2:] = a
        return (p[0::2, 0::2] + p[0::2, 1::2] + p[1::2, 0::2] + p[1::2, 1::2]) / 4

    out = []
    for level in range(5):
        if level:
            X, Y = pool(X), pool(Y)
        mx, my = f(X), f(Y)
        sxx, syy, sxy = f(X * X) - mx ** 2, f(Y * Y) - my ** 2, f(X * Y) - mx * my
        cs = (2 * sxy + C2) / (sxx + syy + C2)
        ssim = (2 * mx * my + C1) / (mx ** 2 + my ** 2 + C1) * cs
        out.append((ssim.mean(), cs.mean(), X.shape))
    return out


@pytest.mark.parametrize("H,W", SIZES)
@pytest.mark.parametrize("data_range", [1.0, 255.0])
def test_oracle_against_direct_correlation(H, W, data_range):
    X, Y = _pair(1, 2, H, W, seed=H + W)
    X, Y = X * data_range, Y * data_range
    ssim, cs = oms.level_stats(X, Y, data_range)
    for c in range(2):
        direct = _direct_level_stats(X[0, c].numpy(), Y[0, c].numpy(), data_range)
        for level, (s, k, shape) in enumerate(direct):
            assert abs(float(ssim[level, 0, c]) - s) <= 1e-12 and abs(float(cs[level, 0, c]) - k) <= 1e-12, (level, c)
    # the pyramid really has odd and even sizes where the parameters say so
    shapes = [d[2] for d in direct]
    assert shapes[0] == (H, W) and all(shapes[i + 1] == ((h + 1) // 2, (w + 1) // 2) for i, (h, w) in enumerate(shapes[:-1]))


def test_constant_planes_closed_form():
    a, b = 0.3, 0.6
    X = torch.full((1, 1, 256, 256), a, dtype=torch.float64)
    Y = torch.full((1, 1, 256, 256), b, dtype=torch.float64)
    C1 = 0.01 ** 2
    got = float(oms.ms_ssim(X, Y, data_range=1.0))
    assert abs(got - ((2 * a * b + C1) / (a * a + b * b + C1)) ** 0.1333) <= 1e-12
    assert abs(got - 0.970700181) <= 5e-10


@pytest.mark.parametrize("H,W", SIZES)
def test_identical_images_give_exactly_one(H, W):
    X, _ = _pair(2, 3, H, W, seed=5)
    assert float(oms.ms_ssim(X, X.clone())) == 1.0
    assert torch.equal(oms.ms_ssim(X, X.clone(), size_average=False), torch.ones(2, dtype=torch.float64))


@pytest.mark.parametrize("H,W", SIZES)
@pytest.mark.parametrize("data_range", [1.0, 255.0])
def test_backward_formulation_against_autograd(H, W, data_range):
    """oracle.stats_backward (the kernels' per-level G maps, full correlations and 1/4-weighted coarser dX) against fp64
    autograd of the oracle's statistics, for arbitrary upstream gradients of every level."""
    X, Y = _pair(2, 3, H, W, seed=H * W)
    X, Y = X * data_range, Y * data_range
    g = torch.Generator().manual_seed(1)
    g_ssim = torch.randn(5, 2, 3, dtype=torch.float64, generator=g)
    g_cs = torch.randn(5, 2, 3, dtype=torch.float64, generator=g)
    Xr = X.clone().requires_grad_(True)
    s, c = oms.level_stats(Xr, Y, data_range)
    want, = torch.autograd.grad((s * g_ssim).sum() + (c * g_cs).sum(), [Xr])
    got = oms.stats_backward(X, Y, g_ssim, g_cs, data_range)
    assert float((got - want).norm() / want.norm()) <= 1e-12


def test_oracle_rejects_small_images():
    X = torch.rand(1, 1, 160, 300, dtype=torch.float64)
    with pytest.raises(ValueError):
        oms.ms_ssim(X, X)


def test_msssim_args_layout_matches_header(lib):
    import ctypes
    from dcae_b200 import _lib
    prog = ('#include <stdio.h>\n#include "dcae_b200.h"\nint main(){printf("%zu %zu\\n", sizeof(dcae_msssim_args), '
            'sizeof(dcae_msssim_bwd_args));return 0;}\n')
    with tempfile.TemporaryDirectory() as td:
        open(os.path.join(td, "t.c"), "w").write(prog)
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(td, "t"), os.path.join(td, "t.c")], check=True)
        sizes = [int(v) for v in subprocess.run([os.path.join(td, "t")], capture_output=True, text=True, check=True).stdout.split()]
    assert sizes == [ctypes.sizeof(_lib.MsssimArgs), ctypes.sizeof(_lib.MsssimBwdArgs)]


def test_scratch_bytes(lib):
    n = lib.dcae_msssim_scratch_bytes(2, 3, 256, 256)
    # pooled x, y and dx of levels 1..4 plus the fp64 partials: at least the pyramid, at most a full image more
    pyramid = 3 * 2 * 3 * 4 * sum((256 >> l) ** 2 for l in range(1, 5))
    assert pyramid <= n <= pyramid + 2 * 3 * 256 * 256 * 4
    assert lib.dcae_msssim_scratch_bytes(2, 3, 256, 512) > n
    for bad in ((-1, 3, 256, 256), (2, 0, 256, 256), (2, 3, 160, 256), (2, 3, 256, 160)):
        assert lib.dcae_msssim_scratch_bytes(*bad) == 0, bad
    assert lib.dcae_msssim_scratch_bytes(0, 3, 256, 256) == 0          # an empty batch needs none


def test_msssim_rejects_bad_arguments_before_any_launch(lib):
    """Each bad argument answers -1 with a message on dcae_last_error() and launches nothing (pointers are never
    dereferenced on the host, so this runs without a GPU)."""
    from dcae_b200 import _lib
    fake = 0x1000
    B, C, H, W = 2, 3, 256, 200
    need = lib.dcae_msssim_scratch_bytes(B, C, H, W)

    def fwd(**kw):
        a = _lib.MsssimArgs()
        a.x, a.y, a.scratch, a.ssim, a.cs = (fake,) * 5
        a.B, a.C, a.H, a.W, a.data_range, a.scratch_bytes = B, C, H, W, 1.0, need
        for k, v in kw.items():
            setattr(a, k, v)
        return a

    def bwd(**kw):
        a = _lib.MsssimBwdArgs()
        a.x, a.y, a.scratch, a.grad_ssim, a.grad_cs, a.grad_x = (fake,) * 6
        a.B, a.C, a.H, a.W, a.data_range, a.scratch_bytes = B, C, H, W, 1.0, need
        for k, v in kw.items():
            setattr(a, k, v)
        return a

    err = lambda: lib.dcae_last_error().decode()                 # noqa: E731
    before = lib.dcae_launch_count()
    for call, args in ((lib.dcae_msssim_forward, fwd), (lib.dcae_msssim_backward, bwd)):
        for field in ("x", "y"):
            assert call(args(**{field: None}), None) == -1 and "null input" in err(), field
        for shape in ({"B": -1}, {"C": 0}, {"C": -2}):
            assert call(args(**shape), None) == -1 and "bad shape" in err(), shape
        for shape in ({"H": 160}, {"W": 160}, {"H": 0}, {"W": -5}):
            assert call(args(**shape), None) == -1 and "exceed 160" in err(), shape
        assert call(args(H=65536, W=65536), None) == -1 and "bad shape" in err()
        for r in (0.0, -1.0, math.nan, math.inf):
            assert call(args(data_range=r), None) == -1 and "data_range" in err(), r
        assert call(args(scratch=None), None) == -1 and "scratch" in err()
        assert call(args(scratch=fake + 4), None) == -1 and "aligned" in err()
        assert call(args(scratch_bytes=need - 1), None) == -1 and "scratch too small" in err()
        assert call(args(W=W + 1), None) == -1 and "scratch too small" in err()
        assert call(None, None) == -1 and "null arguments" in err()
    for field in ("ssim", "cs"):
        assert lib.dcae_msssim_forward(fwd(**{field: None}), None) == -1 and "null output" in err(), field
    for field in ("grad_ssim", "grad_cs"):
        assert lib.dcae_msssim_backward(bwd(**{field: None}), None) == -1 and "null input" in err(), field
    assert lib.dcae_msssim_backward(bwd(grad_x=None), None) == -1 and "null output" in err()
    assert lib.dcae_launch_count() == before


def test_ms_ssim_refuses_cpu_tensors():
    from dcae_b200._lib import DcaeError
    from dcae_b200.msssim import ms_ssim
    X = torch.rand(1, 3, 200, 200)
    with pytest.raises(DcaeError):
        ms_ssim(X, X)


def _fake_out(seed):
    g = torch.Generator().manual_seed(seed)
    return {"x_hat": torch.rand(2, 3, 64, 64, generator=g),
            "likelihoods": {"y": torch.rand(2, 320, 4, 4, generator=g).clamp_min(1e-9),
                            "z": torch.rand(2, 192, 1, 1, generator=g).clamp_min(1e-9)}}


def test_rate_distortion_loss_default_metric_is_unchanged():
    """Without `metric` (and with metric="mse") the loss is the mse form, bit for bit as before the keyword existed."""
    import torch.nn.functional as F
    from dcae_b200.training import dcae_rate_distortion_loss
    out = _fake_out(0)
    target = torch.rand(2, 3, 64, 64, generator=torch.Generator().manual_seed(1))
    pixels = 2 * 64 * 64
    bpp = sum(torch.log(lik).sum() / (-math.log(2) * pixels) for lik in out["likelihoods"].values())
    mse = F.mse_loss(out["x_hat"], target)
    want = (0.013 * 255 ** 2 * mse + bpp, bpp, mse)
    for got in (dcae_rate_distortion_loss(out, target), dcae_rate_distortion_loss(out, target, metric="mse"),
                dcae_rate_distortion_loss(out, target, 0.013, "mse")):
        assert all(torch.equal(a, b) for a, b in zip(got, want))
    got = dcae_rate_distortion_loss(out, target, lmbda=0.0483)
    assert torch.equal(got[0], 0.0483 * 255 ** 2 * mse + bpp)


@pytest.mark.parametrize("metric", ["msssim", "MS-SSIM", "ssim", "", None])
def test_rate_distortion_loss_rejects_unknown_metric(metric):
    from dcae_b200.training import dcae_rate_distortion_loss
    with pytest.raises(ValueError):
        dcae_rate_distortion_loss(_fake_out(0), torch.rand(2, 3, 64, 64), metric=metric)
