"""The whole reference model on libdcae_b200.so: `DCAE.forward / compress / decompress / update`
(/root/reference/models/dcae.py:616-677, 698-761, 859-910) with every sub-module on the library --

    g_a, h_a, h_z_s1, h_z_s2, g_s      dcae_b200.transforms.TransformStack      (SURVEY 8f N3 / N4)
    entropy_bottleneck                 dcae_b200.EntropyBottleneck              (8f N3)
    the channel-slice loop             dcae_b200.EntropySliceLoop               (8a: the hot path)
    gaussian_conditional + range coder dcae_b200.GaussianConditional, dcae_b200.ans  (8a G1-G6, 8f N1 / N2)

Built from a reference state dict alone (same keys; `DCAECodec(net.state_dict())` for a live model); the reference's
Python class is not needed.  Inference only.  To keep the reference's own class and text instead, use
`accelerate(net)` + `accelerate_transforms(net)`.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import _lib
from .entropy_bottleneck import EntropyBottleneck
from .entropy_model import EntropySliceLoop
from .gaussian_conditional import GaussianConditional
from .modules import HOT_PREFIXES
from .transforms import STACKS, TransformStack


class DCAECodec:
    def __init__(self, params: Dict[str, torch.Tensor], device="cuda:0", math: str = "f16x3", lanes: int = 2):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.DcaeError("dcae_b200 runs on CUDA devices only (no CPU fallback)")
        self.math = math
        self.stacks = {name: TransformStack(name, params, device=self.device, math=math) for name in STACKS}
        hot = {k: v.detach() for k, v in params.items() if k.split(".")[0] in HOT_PREFIXES}
        table = params.get("gaussian_conditional.scale_table")
        self.loop = EntropySliceLoop(hot, device=self.device, math=math, lanes=lanes,
                                     scale_table=table if table is not None and table.numel() else None)
        self.entropy_bottleneck = EntropyBottleneck(192).to(self.device)
        eb = {k[len("entropy_bottleneck."):]: v for k, v in params.items() if k.startswith("entropy_bottleneck.")}
        if eb:
            self.entropy_bottleneck.load_state_dict(eb, strict=False)
        self.entropy_bottleneck.eval()
        self.gaussian_conditional = GaussianConditional(None).to(self.device)
        gc = {k[len("gaussian_conditional."):]: v for k, v in params.items() if k.startswith("gaussian_conditional.")}
        if gc:
            self.gaussian_conditional.load_state_dict(gc, strict=False)
        if self.gaussian_conditional.scale_table.numel() == 0:
            self.gaussian_conditional.update_scale_table(self.loop.scale_table)
        self.gaussian_conditional.eval()

    # dcae.py:616-621
    def update(self, scale_table: Optional[torch.Tensor] = None, force: bool = False) -> bool:
        updated = self.gaussian_conditional.update_scale_table(scale_table if scale_table is not None else self.loop.scale_table, force=force)
        updated |= self.entropy_bottleneck.update(force=force)
        return updated

    def _latents(self, x: torch.Tensor):
        if torch.is_grad_enabled() and x.requires_grad:
            raise _lib.DcaeError("DCAECodec is forward-only: call it under torch.no_grad()")
        y = self.stacks["g_a"](x)
        z = self.stacks["h_a"](y)
        return y, z

    @torch.no_grad()
    def forward(self, x: torch.Tensor) -> dict:
        """dcae.py:623-677 -> {"x_hat", "likelihoods": {"y", "z"}, "para": {"means", "scales", "y"}}."""
        y, z = self._latents(x)
        z_hat, z_lik = self.entropy_bottleneck(z, training=False)         # round(z - median) + median, :630-633
        latent_scales, latent_means = self.stacks["h_z_s1"](z_hat), self.stacks["h_z_s2"](z_hat)
        o = self.loop.forward(y, latent_scales, latent_means)
        x_hat = self.stacks["g_s"](o["y_hat"])
        return {"x_hat": x_hat, "likelihoods": {"y": o["likelihoods"], "z": z_lik},
                "para": {"means": o["means"], "scales": o["scales"], "y": y}, "log2_lik_sum_y": o["log2_lik_sum"]}

    __call__ = forward

    def capture(self, x: torch.Tensor):
        """CUDA-graph form of `forward` for launch-bound shapes (one 768x512 image is 561 launches of 5 - 20 us enqueued
        through ctypes).  `x` is captured BY ADDRESS: refill it in place and call replay().
        -> (replay, out) with `out` the dict `forward` returns, overwritten by every replay."""
        for _ in range(2):                      # warm-up: plans, kernel attributes, the first-call range check, pooled buffers
            self.forward(x)
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = self.forward(x)
        self._graphs = getattr(self, "_graphs", []) + [graph]        # the graph owns the memory `out` lives in
        return graph.replay, out

    CODERS = ("reference", "interleaved")

    @classmethod
    def _check_coder(cls, coder):
        if coder not in cls.CODERS:
            raise ValueError(f"coder must be one of {cls.CODERS} (got {coder!r})")

    @torch.no_grad()
    def compress(self, x: torch.Tensor, coder: str = "reference", lanes: int = 32) -> dict:
        """dcae.py:698-761 -> {"strings": [y_strings, z_strings], "shape": z.shape[-2:]}, one z stream per image.
        coder="reference" (default): y_strings = [one y stream for the batch in the reference's coder order], coded on
        the host.  coder="interleaved": y_strings = one ilv1 string per image (include/dcae_rans.h), coded on the GPU
        on `lanes` interleaved states; it decodes only with decompress(..., coder="interleaved")."""
        self._check_coder(coder)
        y, z = self._latents(x)
        z_strings = self.entropy_bottleneck.compress(z)
        z_hat = self.entropy_bottleneck.decompress(z_strings, z.shape[-2:])
        latent_scales, latent_means = self.stacks["h_z_s1"](z_hat), self.stacks["h_z_s2"](z_hat)
        if coder == "interleaved":
            enc = self.loop.compress_to_strings_interleaved(y, latent_scales, latent_means, self.gaussian_conditional, lanes=lanes)
            return {"strings": [enc["y_strings"], z_strings], "shape": tuple(z.shape[-2:])}
        enc = self.loop.compress_to_string(y, latent_scales, latent_means, self.gaussian_conditional)
        return {"strings": [[enc["y_string"]], z_strings], "shape": tuple(z.shape[-2:])}

    @torch.no_grad()
    def decompress(self, strings, shape, coder: str = "reference") -> dict:
        """dcae.py:859-910 -> {"x_hat"} (clamped to [0, 1]).  `coder` names the format `compress` wrote."""
        self._check_coder(coder)
        z_hat = self.entropy_bottleneck.decompress(strings[1], shape)
        latent_scales, latent_means = self.stacks["h_z_s1"](z_hat), self.stacks["h_z_s2"](z_hat)
        if coder == "interleaved":
            dec = self.loop.decompress_from_strings_interleaved(strings[0], latent_scales, latent_means, self.gaussian_conditional)
        else:
            dec = self.loop.decompress_from_string(strings[0][0], latent_scales, latent_means, self.gaussian_conditional)
        return {"x_hat": self.stacks["g_s"](dec["y_hat"]).clamp_(0, 1)}

    # ---- image <-> container (compress_and_decompress.py:150-215: pad to multiples of 128, compress, save_bin / read_bin,
    # decompress, crop, clamp); one image per container like the reference
    def encode_image(self, x: torch.Tensor, coder: str = "reference") -> bytes:
        """x [1, 3, H, W] in [0, 1] (any H, W >= 1 whose padded size is >= 256) -> container bytes: the reference's .bin
        (coder="reference") or the DCI1 container of the ilv1 format (coder="interleaved", `container.pack_ilv`)."""
        from . import container
        self._check_coder(coder)
        if x.dim() != 4 or x.size(0) != 1:
            raise ValueError("the container holds one image: expected [1, 3, H, W]")
        xp, _ = container.pad(x.to(self.device, torch.float32))
        enc = self.compress(xp, coder=coder)
        pack = container.pack_ilv if coder == "interleaved" else container.pack_bin
        return pack(enc["strings"], x.shape[-2:])

    def decode_image(self, blob: bytes, coder: str = "reference") -> torch.Tensor:
        """-> x_hat [1, 3, H, W] in [0, 1], cropped back to the size stored in the container.  `coder` names the
        container's format; it is never guessed from the bytes."""
        from . import container
        self._check_coder(coder)
        unpack = container.unpack_ilv if coder == "interleaved" else container.unpack_bin
        strings, z_shape, padding, _ = unpack(blob)
        out = self.decompress(strings, z_shape, coder=coder)
        return container.crop(out["x_hat"], padding).clamp_(0, 1)


__all__ = ["DCAECodec"]
