"""TEST INFRASTRUCTURE ONLY -- torch restatement of `pytorch_msssim.ms_ssim` (v1.0, the package the reference's
train.py imports for its ms-ssim rate-distortion loss) with its defaults: 11-tap Gaussian window, sigma 1.5, applied
separably (W, then H) as a valid correlation; C1 = (0.01 R)^2, C2 = (0.03 R)^2; 5 levels joined by
avg_pool2d(2, 2, padding = (h % 2, w % 2)) with count_include_pad; weights (0.0448, 0.2856, 0.3001, 0.2363, 0.1333).

pytorch_msssim is not installed here, so this follows its published source.  Dtype-generic (grouped conv2d): the tests
run it in fp64 as the reference value of the library's fp32 kernels.  `stats_backward` restates, in the same ops, the
analytic backward those kernels implement (dcae_b200/csrc/msssim_kernel.cu)."""
from __future__ import annotations

import torch
import torch.nn.functional as F

WIN_SIZE = 11
WIN_SIGMA = 1.5
WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)
LEVELS = len(WEIGHTS)


def window(dtype=torch.float64, device=None) -> torch.Tensor:
    """The 1-D Gaussian window [11], normalised to sum 1 (computed in fp64)."""
    k = torch.arange(WIN_SIZE, dtype=torch.float64) - WIN_SIZE // 2
    g = torch.exp(-(k ** 2) / (2 * WIN_SIGMA ** 2))
    return (g / g.sum()).to(dtype=dtype, device=device)


def constants(data_range: float):
    return (0.01 * data_range) ** 2, (0.03 * data_range) ** 2


def filt(x: torch.Tensor) -> torch.Tensor:
    """Valid separable correlation of every plane of x [B, C, h, w] with the window: [B, C, h - 10, w - 10]."""
    C = x.shape[1]
    g = window(x.dtype, x.device)
    x = F.conv2d(x, g.reshape(1, 1, 1, -1).repeat(C, 1, 1, 1), groups=C)
    return F.conv2d(x, g.reshape(1, 1, -1, 1).repeat(C, 1, 1, 1), groups=C)


def full(g: torch.Tensor) -> torch.Tensor:
    """Transpose of `filt`: the map zero-padded by 10 on each side, correlated with the same symmetric window."""
    return filt(F.pad(g, (WIN_SIZE - 1,) * 4))


def pool(x: torch.Tensor) -> torch.Tensor:
    return F.avg_pool2d(x, kernel_size=2, stride=2, padding=(x.shape[2] % 2, x.shape[3] % 2))


def moments(X: torch.Tensor, Y: torch.Tensor):
    mx, my = filt(X), filt(Y)
    return mx, my, filt(X * X) - mx * mx, filt(Y * Y) - my * my, filt(X * Y) - mx * my


def level_stats(X: torch.Tensor, Y: torch.Tensor, data_range: float = 1.0):
    """(ssim, cs) means [5, B, C] of each level."""
    if min(X.shape[-2:]) <= 160:
        raise ValueError("min(H, W) must exceed 160")
    C1, C2 = constants(data_range)
    ssim, cs = [], []
    for level in range(LEVELS):
        if level > 0:
            X, Y = pool(X), pool(Y)
        mx, my, sxx, syy, sxy = moments(X, Y)
        cs_map = (2 * sxy + C2) / (sxx + syy + C2)
        ssim_map = (2 * mx * my + C1) / (mx * mx + my * my + C1) * cs_map
        ssim.append(ssim_map.flatten(2).mean(-1))
        cs.append(cs_map.flatten(2).mean(-1))
    return torch.stack(ssim), torch.stack(cs)


def combine(ssim: torch.Tensor, cs: torch.Tensor, size_average: bool = True) -> torch.Tensor:
    """pytorch_msssim's combination of the level statistics [5, B, C]."""
    w = torch.tensor(WEIGHTS, dtype=ssim.dtype, device=ssim.device)
    vals = torch.stack([torch.relu(c) for c in cs[:-1]] + [torch.relu(ssim[-1])])
    v = torch.prod(vals ** w.reshape(-1, 1, 1), dim=0)
    return v.mean() if size_average else v.mean(1)


def ms_ssim(X: torch.Tensor, Y: torch.Tensor, data_range: float = 1.0, size_average: bool = True) -> torch.Tensor:
    return combine(*level_stats(X, Y, data_range), size_average=size_average)


def stats_backward(X: torch.Tensor, Y: torch.Tensor, g_ssim: torch.Tensor, g_cs: torch.Tensor, data_range: float = 1.0):
    """dL/dX given dL/d(ssim means) and dL/d(cs means) [5, B, C], in the kernels' formulation: per level the maps
    G_mu, G_xx, G_xy on the valid positions, their full correlations, and 1/4 of the coarser level's dX, coarse to fine."""
    C1, C2 = constants(data_range)
    pyr = [(X, Y)]
    for _ in range(LEVELS - 1):
        pyr.append((pool(pyr[-1][0]), pool(pyr[-1][1])))
    d_next = None
    for level in reversed(range(LEVELS)):
        Xl, Yl = pyr[level]
        mx, my, sxx, syy, sxy = moments(Xl, Yl)
        n = mx.shape[2] * mx.shape[3]
        a = (g_ssim[level] / n)[..., None, None]
        b = (g_cs[level] / n)[..., None, None]
        n1, d1 = 2 * mx * my + C1, mx * mx + my * my + C1
        n2, d2 = 2 * sxy + C2, sxx + syy + C2
        lum, cs = n1 / d1, n2 / d2
        g_l, g_c = a * cs, b + a * lum
        dcs_xx, dcs_xy = -n2 / d2 ** 2, 2 / d2
        dl_mx = (2 * my * d1 - 2 * mx * n1) / d1 ** 2
        g_mu = g_l * dl_mx + g_c * (-2 * mx * dcs_xx - my * dcs_xy)
        dX = full(g_mu) + 2 * Xl * full(g_c * dcs_xx) + Yl * full(g_c * dcs_xy)
        if d_next is not None:
            h, w = Xl.shape[2:]
            ph, pw = h % 2, w % 2
            rows = (torch.arange(h, device=X.device) + ph) // 2
            cols = (torch.arange(w, device=X.device) + pw) // 2
            dX = dX + 0.25 * d_next[:, :, rows][:, :, :, cols]
        d_next = dX
    return d_next

