"""Drop-in for compressai's `EntropyBottleneck` as the reference uses it for the hyper-latent z (SURVEY 8f N3, first
part): `net.entropy_bottleneck` of a `DCAE` (dcae.py:513 `entropy_bottleneck_channels=192`) with the calls of
dcae.py:629-633 (`forward`, `_get_medians`), :705-706 (`compress`, `decompress`), :861 (`decompress`),
`update()` (through `CompressionModel.update`, dcae.py:621) and `loss()` (train.py:177 `aux_loss`).

Parameter names and shapes are compressai's (`_matrix{0..4}`, `_bias{0..4}`, `_factor{0..3}`, `quantiles`, buffers
`_offset`, `_quantized_cdf`, `_cdf_length`, `target`), so a reference checkpoint loads key for key.  Quantisation,
likelihood and symbols of a call run in ONE launch of `dcae_eb_fused`; the strings are produced by the native range
coder (`dcae_b200.ans`), one stream per image like compressai.  Forward-only on the device: `loss()` (three numbers per
channel) is plain torch, and a call under autograd raises (the hyper path's transforms are outside this library).
compressai's source is not in /root/reference: restated from its published version, parity unpinned (DESIGN.md).
"""
from __future__ import annotations

import math
from typing import List, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from .gaussian_conditional import _pmf_to_quantized_cdf

FILTERS = (3, 3, 3, 3)


class EntropyBottleneck(nn.Module):
    def __init__(self, channels: int, tail_mass: float = 1e-9, init_scale: float = 10, filters=FILTERS,
                 likelihood_bound: float = 1e-9, entropy_coder_precision: int = 16):
        super().__init__()
        if tuple(filters) != FILTERS:
            raise ValueError("dcae_b200.EntropyBottleneck supports compressai's default filters (3, 3, 3, 3) only")
        self.channels, self.filters = int(channels), tuple(filters)
        self.init_scale, self.tail_mass = float(init_scale), float(tail_mass)
        self.likelihood_bound, self.entropy_coder_precision = float(likelihood_bound), int(entropy_coder_precision)
        f = (1,) + self.filters + (1,)
        scale = self.init_scale ** (1 / (len(self.filters) + 1))
        for i in range(len(self.filters) + 1):
            init = math.log(math.expm1(1 / scale / f[i + 1]))
            self.register_parameter(f"_matrix{i}", nn.Parameter(torch.full((channels, f[i + 1], f[i]), init)))
            self.register_parameter(f"_bias{i}", nn.Parameter(torch.rand(channels, f[i + 1], 1) - 0.5))
            if i < len(self.filters):
                self.register_parameter(f"_factor{i}", nn.Parameter(torch.zeros(channels, f[i + 1], 1)))
        self.quantiles = nn.Parameter(torch.tensor([-self.init_scale, 0.0, self.init_scale]).repeat(channels, 1, 1))
        target = math.log(2 / self.tail_mass - 1)
        self.register_buffer("target", torch.tensor([-target, 0.0, target]))
        self.register_buffer("_offset", torch.IntTensor())
        self.register_buffer("_quantized_cdf", torch.IntTensor())
        self.register_buffer("_cdf_length", torch.IntTensor())
        self._packed = None

    offset = property(lambda self: self._offset)
    quantized_cdf = property(lambda self: self._quantized_cdf)
    cdf_length = property(lambda self: self._cdf_length)

    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        for name in ("_quantized_cdf", "_offset", "_cdf_length"):          # table sizes follow the checkpoint (dcae.py:84-150)
            src = state_dict.get(prefix + name)
            if src is not None and tuple(getattr(self, name).shape) != tuple(src.shape):
                setattr(self, name, torch.empty(src.shape, dtype=torch.int32, device=getattr(self, name).device))
        super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)

    # ---- the density (host side: tables, aux loss) ------------------------------------------------------------------
    def _get_medians(self) -> torch.Tensor:
        return self.quantiles[:, :, 1:2]

    def _logits_cumulative(self, inputs: torch.Tensor, stop_gradient: bool = False) -> torch.Tensor:
        """stop_gradient (compressai's keyword): the density parameters enter detached, so only `inputs` is differentiated."""
        def param(name):
            t = getattr(self, name)
            return t.detach() if stop_gradient else t
        logits = inputs
        for i in range(len(self.filters) + 1):
            logits = torch.matmul(F.softplus(param(f"_matrix{i}")), logits) + param(f"_bias{i}")
            if i < len(self.filters):
                logits = logits + torch.tanh(param(f"_factor{i}")) * torch.tanh(logits)
        return logits

    def loss(self) -> torch.Tensor:
        """aux loss (train.py:177): sum |logits_cumulative(quantiles) - target|; plain torch, differentiable."""
        return torch.abs(self._logits_cumulative(self.quantiles) - self.target).sum()

    @torch.no_grad()
    def update(self, force: bool = False) -> bool:
        """compressai EntropyBottleneck.update(): integer pmf of every channel between its outer quantiles -> 16-bit CDFs."""
        if self._offset.numel() > 0 and not force:
            return False
        dev = self.quantiles.device
        q = self.quantiles.detach().float().cpu()
        med = q[:, 0, 1]
        minima = torch.clamp(torch.ceil(med - q[:, 0, 0]).int(), min=0)
        maxima = torch.clamp(torch.ceil(q[:, 0, 2] - med).int(), min=0)
        pmf_start, pmf_length = med - minima, maxima + minima + 1
        max_length = int(pmf_length.max())
        samples = torch.arange(max_length)[None, :] + pmf_start[:, None, None]
        host = {k: v.detach().float().cpu() for k, v in self.named_parameters()}

        def logits(v):
            for i in range(len(self.filters) + 1):
                v = torch.matmul(F.softplus(host[f"_matrix{i}"]), v) + host[f"_bias{i}"]
                if i < len(self.filters):
                    v = v + torch.tanh(host[f"_factor{i}"]) * torch.tanh(v)
            return v

        lower, upper = logits(samples - 0.5), logits(samples + 0.5)
        pmf = (torch.sigmoid(upper) - torch.sigmoid(lower))[:, 0, :]
        tail = torch.sigmoid(lower[:, 0, :1]) + torch.sigmoid(-upper[:, 0, -1:])
        cdf = torch.zeros(self.channels, max_length + 2, dtype=torch.int32)
        for i in range(self.channels):
            n = int(pmf_length[i])
            row = _pmf_to_quantized_cdf(torch.cat((pmf[i, :n], tail[i])).tolist(), self.entropy_coder_precision)
            cdf[i, : len(row)] = torch.tensor(row, dtype=torch.int32)
        self._quantized_cdf, self._offset, self._cdf_length = cdf.to(dev), (-minima).to(dev), (pmf_length + 2).to(dev)
        return True

    # ---- the device pass ---------------------------------------------------------------------------------------------
    def _pack(self, device) -> tuple:
        """[C, 58] = softplus(matrices) | biases | tanh(factors), and the medians [C]; repacked when a parameter changes."""
        sig = tuple((p.data_ptr(), p._version) for p in self.parameters()) + (str(device),)
        if self._packed is None or self._packed[0] != sig:
            with torch.no_grad():
                parts = [F.softplus(getattr(self, f"_matrix{i}")).reshape(self.channels, -1) for i in range(5)]
                parts += [getattr(self, f"_bias{i}").reshape(self.channels, -1) for i in range(5)]
                parts += [torch.tanh(getattr(self, f"_factor{i}")).reshape(self.channels, -1) for i in range(4)]
                params = torch.cat(parts, dim=1).to(device, torch.float32).contiguous()
                med = self.quantiles[:, 0, 1].detach().to(device, torch.float32).contiguous()
            assert params.shape[1] == 58
            self._packed = (sig, params, med)
        return self._packed[1], self._packed[2]

    def _run(self, mode, x=None, noise=None, sym_in=None, want=("z_hat", "lik", "sym"), shape=None):
        ref = x if x is not None else sym_in
        if not ref.is_cuda:
            raise _lib.DcaeError("dcae_b200.EntropyBottleneck runs on CUDA tensors only (no CPU fallback)")
        shape = tuple(ref.shape)
        if len(shape) != 4 or shape[1] != self.channels:
            raise ValueError(f"expected [B, {self.channels}, h, w], got {shape}")
        params, med = self._pack(ref.device)
        a = _lib.EbArgs()
        keep = [params, med]
        if x is not None:
            x = x.contiguous().float()
            keep.append(x)
            a.z = x.data_ptr()
        if noise is not None:
            noise = noise.contiguous().float()
            keep.append(noise)
            a.noise = noise.data_ptr()
        if sym_in is not None:
            sym_in = sym_in.contiguous().to(torch.int32)
            keep.append(sym_in)
            a.sym_in = sym_in.data_ptr()
        a.params, a.medians, a.mode = params.data_ptr(), med.data_ptr(), mode
        a.B, a.C, a.HW, a.lik_bound = shape[0], shape[1], shape[2] * shape[3], self.likelihood_bound
        outs = {}
        for name, dt in (("z_hat", torch.float32), ("lik", torch.float32), ("sym", torch.int32)):
            if name in want:
                outs[name] = torch.empty(shape, dtype=dt, device=ref.device)
                setattr(a, name, outs[name].data_ptr())
        if ref.numel():
            with torch.cuda.device(ref.device):
                _lib.check(_lib.load().dcae_eb_fused(a, _lib.current_stream(ref.device)), "dcae_eb_fused")
        return outs

    def forward(self, x: torch.Tensor, training: Optional[bool] = None, noise: Optional[torch.Tensor] = None):
        """-> (outputs, likelihood) like compressai (dcae.py:630)."""
        if torch.is_grad_enabled() and x.requires_grad:
            raise _lib.DcaeError("dcae_b200.EntropyBottleneck is forward-only: call it under torch.no_grad() (the hyper path's "
                                 "transforms are outside this library; train it with compressai's module)")
        if training is None:
            training = self.training
        if training:
            if noise is None:
                noise = torch.empty_like(x).uniform_(-0.5, 0.5)
            o = self._run(_lib.GC_NOISE, x, noise=noise, want=("lik",))
            return x + noise, o["lik"]
        o = self._run(_lib.GC_EVAL, x, want=("z_hat", "lik"))
        return o["z_hat"], o["lik"]

    def _tables(self):
        if self._quantized_cdf.numel() == 0:
            raise _lib.DcaeError("EntropyBottleneck has no CDF tables: call net.update() first")
        key = (self._quantized_cdf.data_ptr(), self._quantized_cdf._version)
        if getattr(self, "_host_tables_key", None) != key:
            self._host_tables = (self._quantized_cdf.cpu().int().contiguous(), self._cdf_length.cpu().int().reshape(-1).contiguous(),
                                 self._offset.cpu().int().reshape(-1).contiguous())
            self._host_tables_key = key
        return self._host_tables

    def compress(self, x: torch.Tensor) -> List[bytes]:
        """dcae.py:705: one stream per image, symbols in (c, h, w) order with the channel as the CDF index."""
        from .ans import BufferedRansEncoder
        sym = self._run(_lib.GC_EVAL, x, want=("sym",))["sym"]
        B, Cc, h, w = sym.shape
        host = sym.cpu().reshape(B, -1).numpy()                          # one D2H for the batch
        idx = torch.arange(Cc, dtype=torch.int32).reshape(-1, 1).expand(Cc, h * w).reshape(-1).contiguous().numpy()
        strings = []
        for i in range(B):
            enc = BufferedRansEncoder()
            enc.encode_with_indexes(host[i], idx, *self._tables())
            strings.append(enc.flush())
        return strings

    def decompress(self, strings: List[bytes], size) -> torch.Tensor:
        """dcae.py:706, :861: -> z_hat [B, C, h, w] on the module's device."""
        from .ans import RansDecoder
        import numpy as np
        h, w = int(size[0]), int(size[1])
        Cc = self.channels
        idx = torch.arange(Cc, dtype=torch.int32).reshape(-1, 1).expand(Cc, h * w).reshape(-1).contiguous().numpy()
        out = np.empty((len(strings), Cc * h * w), dtype=np.int32)
        for i, s in enumerate(strings):
            dec = RansDecoder()
            dec.set_stream(s)
            out[i] = dec.decode_array(idx, *self._tables())
        sym = torch.from_numpy(out).reshape(len(strings), Cc, h, w).to(self.quantiles.device)
        return self._run(_lib.GC_DECODE, sym_in=sym, want=("z_hat",))["z_hat"]
