"""Host-side mirror of the reference's channel-slice loop, running on libdcae_b200.so.

`EntropySliceLoop` is what `DCAE.forward` (dcae.py:638-670), `DCAE.compress` (:713-753) and
`DCAE.decompress` (:878-906) do between `(y, latent_scales, latent_means)` and
`(y_hat, means, scales, likelihoods)` / `(symbols, indexes)`.  Inputs and outputs are the
reference's NCHW fp32 CUDA tensors; everything in between is token-major inside the library.
There is no torch math on this path and no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import math as _math
from typing import Callable, Dict, Optional

import torch

from . import _lib
from .params import M_LATENT, NUM_SLICES, SLICE_CH
from .weights import PackedWeights

SCALES_MIN, SCALES_MAX, SCALES_LEVELS = 0.11, 256, 64


def get_scale_table(min=SCALES_MIN, max=SCALES_MAX, levels=SCALES_LEVELS) -> torch.Tensor:
    """dcae.py:54-55 (host-side constant table; the kernels always take the buffer, never recompute it)."""
    return torch.exp(torch.linspace(_math.log(min), _math.log(max), levels))


class _Plan:
    """One dcae_slice_loop plan + its workspace for a fixed (B, h, w)."""

    def __init__(self, eng: "EntropySliceLoop", B: int, h: int, w: int):
        lib = eng.lib
        nbytes = lib.dcae_slice_loop_workspace_bytes(B, h, w)
        self.workspace = torch.empty(nbytes + 256, dtype=torch.uint8, device=eng.device)
        base = (self.workspace.data_ptr() + 255) // 256 * 256
        self.handle = C.c_void_p()
        table = eng.scale_table.data_ptr() if eng.scale_table is not None else None
        n_table = int(eng.scale_table.numel()) if eng.scale_table is not None else 0
        _lib.check(lib.dcae_slice_loop_create(C.byref(self.handle), B, h, w, eng.weights.array, table, n_table, base,
                                              nbytes, _lib.MATH[eng.math]), "dcae_slice_loop_create")
        self.lib = lib
        _lib.check(lib.dcae_slice_loop_set_option(self.handle, _lib.OPT_LIK_MATH, _lib.GC_LIK[eng.likelihood_math]), "set_option")

    def __del__(self):
        try:
            if self.handle:
                self.lib.dcae_slice_loop_destroy(self.handle)
        except Exception:
            pass


class EntropySliceLoop:
    """params: reference state dict (hot-path keys).
    math: 'f16x3' (default: fp16 hi/lo planes, fp32-level accuracy) | 'tf32x3' | 'fp32' (FFMA) | 'tf32' (reduced).
    likelihood_math: 'fast' (default: cancellation-free evaluation of kernel 3's likelihood, <= 1e-5 of the exact value) |
    'reference' (the reference's op order with libdevice erfcf: bit-identical to torch-CUDA on dcae.py:839-857; test mode).
    lanes: images are independent (SURVEY 8e), so `forward` splits the batch into this many sub-batches, each with its
    own plan on its own stream.  Every kernel of the loop is a persistent grid with a partly filled last wave (960
    tiles on 148 SMs; 192 for the small conv layers) and the loop is one dependent chain, so a lone lane leaves SMs
    idle at every kernel boundary; with two lanes the other lane's kernels take those SMs.  Per-image results do not
    depend on the split (tests: batch invariance)."""

    def __init__(self, params: Dict[str, torch.Tensor], device="cuda:0", math: str = "f16x3",
                 scale_table: Optional[torch.Tensor] = None, lanes: int = 2, likelihood_math: str = "fast",
                 validate_f16_range: bool = True):
        if math not in _lib.MATH:
            raise ValueError(f"math must be one of {list(_lib.MATH)}")
        if likelihood_math not in _lib.GC_LIK:
            raise ValueError(f"likelihood_math must be one of {list(_lib.GC_LIK)}")
        self.likelihood_math = likelihood_math
        # f16x3 / f16: the first forward() of an engine (and the first after refresh()) also runs the fp16 range check on
        # its inputs (`check_f16_range`: one counting launch behind every producer, once), so a checkpoint whose
        # activations leave the fp16 range raises instead of being clamped silently
        self._range_checked = not (validate_f16_range and math in ("f16x3", "f16"))
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.DcaeError("dcae_b200 runs on CUDA devices only (no CPU fallback)")
        self.lib = _lib.load()
        self.math = math
        with torch.cuda.device(self.device):
            _lib.check(self.lib.dcae_device_check(), "dcae_device_check")
        self.weights = PackedWeights(params, self.device, split_tf32=True, math=math)
        self.dictionary = params["dt"].detach().to(self.device, torch.float32).clone()     # what K / V were packed from
        if scale_table is None:
            scale_table = get_scale_table()
        self.scale_table = scale_table.detach().to(self.device, torch.float32).contiguous().reshape(-1)
        if not 2 <= self.scale_table.numel() <= 256:
            raise ValueError(f"scale_table must have 2..256 entries (got {self.scale_table.numel()}): indexes travel as uint8")
        self._plans: Dict[tuple, _Plan] = {}
        self.last_launches = 0
        self.lanes = max(1, int(lanes))
        with torch.cuda.device(self.device):
            self._lane_streams = [torch.cuda.Stream(self.device) for _ in range(self.lanes)] if self.lanes > 1 else []

    def refresh(self, params: Dict[str, torch.Tensor]) -> None:
        """Repack the device weights from a new state dict (after `load_state_dict` or an optimizer step).  Plans are
        rebuilt on the next call; the previous packed tensors are released once no launch uses them any more."""
        torch.cuda.synchronize(self.device)
        self._plans.clear()
        self.weights = PackedWeights(params, self.device, split_tf32=True, math=self.math)
        self.dictionary = params["dt"].detach().to(self.device, torch.float32).clone()
        self._dt_checked = False

    # ---- plumbing -------------------------------------------------------------------------------
    def _plan(self, B, h, w, lane: int = -1) -> _Plan:
        key = (B, h, w, lane)
        if key not in self._plans:
            self._plans[key] = _Plan(self, B, h, w)
        return self._plans[key]

    LANE_MIN_TOKENS = 8192      # below this a step is launch- / latency-bound and a second lane only adds launches
                                # (measured B = 4 x 16 x 16: 2.76 ms with one lane, 2.99 ms with two)

    def _lane_split(self, B, tokens_per_image=None):
        """[(lane, first image, images)] of a batch of B images (one entry when lanes do not apply)."""
        n = min(self.lanes, B)
        if tokens_per_image is not None and B * tokens_per_image < self.LANE_MIN_TOKENS:
            n = 1
        if n <= 1:
            return [(-1, 0, B)]
        base, extra, out, b0 = B // n, B % n, [], 0
        for lane in range(n):
            nb = base + (1 if lane < extra else 0)
            out.append((lane, b0, nb))
            b0 += nb
        return out

    def _check_in(self, name, t, B=None, C_=M_LATENT):
        if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 and t.dim() == 4):
            raise ValueError(f"{name}: expected a 4-D float32 CUDA tensor")
        if t.device != self.device:
            raise ValueError(f"{name}: tensor is on {t.device}, engine on {self.device}")
        if t.shape[1] != C_:
            raise ValueError(f"{name}: expected {C_} channels, got {t.shape[1]}")
        return t.contiguous()

    def _stream(self):
        return _lib.current_stream(self.device)

    # ---- DCAE.forward slice loop (eval mode or training noise) ----------------------------------
    def forward(self, y, latent_scales, latent_means, noise: Optional[torch.Tensor] = None,
                want_symbols: bool = False, out: Optional[dict] = None):
        """-> dict(y_hat, means, scales, likelihoods [B,320,h,w], log2_lik_sum [1])
        (+ symbols, indexes int32 [5,B,64,h,w] if want_symbols).  `out`: a dict returned by an earlier call
        with the same shapes, to be overwritten in place (no allocation on the hot path)."""
        y = self._check_in("y", y)
        ls = self._check_in("latent_scales", latent_scales)
        lm = self._check_in("latent_means", latent_means)
        B, _, h, w = y.shape
        if ls.shape != y.shape or lm.shape != y.shape:
            raise ValueError("y, latent_scales and latent_means must have the same shape")
        if noise is not None:
            noise = self._check_in("noise", noise)
        lib, s = self.lib, self._stream()
        sym = idx = None
        if out is None:
            out = {k: torch.empty_like(y) for k in ("y_hat", "means", "scales", "likelihoods")}
            out["log2_lik_sum"] = torch.empty(1, device=self.device)
            if want_symbols:
                out["symbols"] = torch.empty(NUM_SLICES, B, SLICE_CH, h, w, dtype=torch.int32, device=self.device)
                out["indexes"] = torch.empty_like(out["symbols"])
        elif out["y_hat"].shape != y.shape or (want_symbols and "symbols" not in out):
            raise ValueError("out= does not match this call")
        if want_symbols:
            sym, idx = out["symbols"], out["indexes"]
        if B == 0 or h == 0 or w == 0:
            return out
        if not self._range_checked and not torch.cuda.is_current_stream_capturing():
            self._range_checked = True
            self.check_f16_range(y, ls, lm)
        split = self._lane_split(B, h * w)
        self._last_call_lanes = len(split) > 1
        if len(split) == 1:
            with torch.cuda.device(self.device):
                self._run_forward(self._plan(B, h, w), s, y, ls, lm, noise, out, sym, idx, out["log2_lik_sum"])
        else:
            cur = torch.cuda.current_stream(self.device)
            fork = torch.cuda.Event()
            fork.record(cur)
            sums = torch.empty(len(split), device=self.device)
            lane_sym = []
            with torch.cuda.device(self.device):
                for lane, b0, nb in split:
                    st = self._lane_streams[lane]
                    st.wait_event(fork)
                    sl = slice(b0, b0 + nb)
                    lo = {k: out[k][sl] for k in ("y_hat", "means", "scales", "likelihoods")}
                    ssym = sidx = None
                    if want_symbols:          # [5, nb, 64, h, w] per lane, copied into the coder-order tensor below
                        ssym = torch.empty(NUM_SLICES, nb, SLICE_CH, h, w, dtype=torch.int32, device=self.device)
                        sidx = torch.empty_like(ssym)
                        lane_sym.append((sl, ssym, sidx))
                    with torch.cuda.stream(st):
                        self._run_forward(self._plan(nb, h, w, lane), st.cuda_stream, y[sl], ls[sl], lm[sl],
                                          None if noise is None else noise[sl], lo, ssym, sidx, sums[lane:lane + 1])
                    done = torch.cuda.Event()
                    done.record(st)
                    cur.wait_event(done)
                for sl, ssym, sidx in lane_sym:
                    sym[:, sl].copy_(ssym)
                    idx[:, sl].copy_(sidx)
                _lib.check(lib.dcae_reduce_partials(sums.data_ptr(), len(split), out["log2_lik_sum"].data_ptr(), s),
                           "dcae_reduce_partials")
        self.last_launches = int(lib.dcae_launch_count())
        return out

    def check_f16_range(self, y, latent_scales, latent_means) -> int:
        """Validation of a checkpoint for the default `f16x3` mode: activations travel as fp16 hi/lo planes written with
        a saturating convert, so a magnitude above 65504 would be clamped without any signal.  Runs one forward with
        the library's range check on (one small counting launch behind every producer of operand planes) and returns
        the number of clamped elements; 0 means the 22-bit operand claim held for these inputs.  Raises if not 0 and
        `math` is f16x3 -- use `math="tf32x3"` (fp32 operands in HBM, no range limit) for such a checkpoint."""
        if self.math not in ("f16x3", "f16"):
            return 0
        y = self._check_in("y", y)
        B, _, h, w = y.shape
        plan = self._plan(B, h, w, lane=-2)            # its own plan: the production plans never pay for the check
        n = C.c_ulonglong(0)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.dcae_slice_loop_check_f16_range(plan.handle, 1, None), "check_f16_range")
            out = {k: torch.empty_like(y) for k in ("y_hat", "means", "scales", "likelihoods")}
            self._run_forward(plan, self._stream(), y, self._check_in("latent_scales", latent_scales),
                              self._check_in("latent_means", latent_means), None, out, None, None, torch.empty(1, device=self.device))
            _lib.check(self.lib.dcae_slice_loop_check_f16_range(plan.handle, 0, C.byref(n)), "check_f16_range")
        self._plans.pop((B, h, w, -2), None)           # its workspace is as large as a production plan's: do not keep it
        if n.value:
            raise _lib.DcaeError(f"f16x3: {n.value} activation elements exceed the fp16 range (|x| > 65504) and were clamped; "
                                 "run this checkpoint with math='tf32x3'")
        return int(n.value)

    def capture(self, y, latent_scales, latent_means, want_symbols: bool = False):
        """CUDA-graph form of `forward` for launch-bound shapes (a 256x256 image is 173 launches of a few microseconds:
        replay measured 2.43 ms against 2.71 ms of stream launches; at config #2 there is nothing to gain, the host
        enqueues a step in under 1.5 ms).  The three input tensors are captured BY ADDRESS: refill them in place and
        call replay().  -> (replay, out) with `out` the dict `forward` returns, overwritten by every replay."""
        out = self.forward(y, latent_scales, latent_means, want_symbols=want_symbols)       # warm-up: plans, attributes
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            self.forward(y, latent_scales, latent_means, want_symbols=want_symbols, out=out)
        return graph.replay, out

    def _run_forward(self, plan, s, y, ls, lm, noise, out, sym, idx, log2_sum):
        """One plan, one stream: the slice loop for the (sub-)batch whose NCHW tensors are given (contiguous views)."""
        lib = self.lib
        if noise is None:
            _lib.check(lib.dcae_slice_loop_forward(plan.handle, y.data_ptr(), ls.data_ptr(), lm.data_ptr(),
                                                   out["y_hat"].data_ptr(), out["means"].data_ptr(),
                                                   out["scales"].data_ptr(), out["likelihoods"].data_ptr(),
                                                   _lib.ptr(sym), _lib.ptr(idx), log2_sum.data_ptr(), s),
                       "dcae_slice_loop_forward")
        else:
            _lib.check(lib.dcae_slice_loop_set_option(plan.handle, _lib.OPT_WANT_SYMBOLS, int(sym is not None)), "set_option")
            _lib.check(lib.dcae_slice_loop_load(plan.handle, y.data_ptr(), ls.data_ptr(), lm.data_ptr(), s), "load")
            for i, nz in enumerate(noise.chunk(NUM_SLICES, 1)):
                nz = nz.contiguous()
                _lib.check(lib.dcae_slice_loop_params(plan.handle, i, s), "params")
                _lib.check(lib.dcae_slice_loop_encode(plan.handle, i, _lib.GC_NOISE, nz.data_ptr(), s), "encode")
            _lib.check(lib.dcae_slice_loop_store(plan.handle, out["y_hat"].data_ptr(), out["means"].data_ptr(),
                                                 out["scales"].data_ptr(), out["likelihoods"].data_ptr(),
                                                 _lib.ptr(sym), _lib.ptr(idx), log2_sum.data_ptr(), s), "store")

    # ---- DCAE.compress slice loop ---------------------------------------------------------------
    def compress(self, y, latent_scales, latent_means, with_likelihoods: bool = False):
        """-> dict(symbols, indexes int32 [5,B,64,h,w] in the reference's coder order (dcae.py:742-743),
        y_hat, means, scales [, likelihoods])."""
        out = self.forward(y, latent_scales, latent_means, want_symbols=True)
        if not with_likelihoods:
            out.pop("likelihoods", None)
        return out

    def compress_to_host(self, y, latent_scales, latent_means):
        """The GPU -> coder hand-off (SURVEY 8f N1): compress(), then ONE packed device->host copy instead of the
        reference's ten `.tolist()` round trips (dcae.py:742-743).  Returns dict(symbols, indexes: pinned host tensors
        in coder order, flat; int16 / uint8 unless a symbol left the int16 range, then int32 / uint8; overflow: int,
        y_hat: device tensor).  `symbols.numpy()` / `indexes.numpy()` are zero-copy views for the rANS coder."""
        out = self.compress(y, latent_scales, latent_means)
        sym, idx = out["symbols"], out["indexes"]
        n = sym.numel()
        s16 = torch.empty(n, dtype=torch.int16, device=self.device)
        i8 = torch.empty(n, dtype=torch.uint8, device=self.device)
        ovf = torch.zeros(1, dtype=torch.int64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.dcae_pack_symbols(sym.data_ptr(), idx.data_ptr(), n, s16.data_ptr(), i8.data_ptr(), ovf.data_ptr(),
                                                  self._stream()), "dcae_pack_symbols")
        h16 = torch.empty(n, dtype=torch.int16).pin_memory()
        h8 = torch.empty(n, dtype=torch.uint8).pin_memory()
        hov = torch.empty(1, dtype=torch.int64).pin_memory()
        h16.copy_(s16, non_blocking=True)
        h8.copy_(i8, non_blocking=True)
        hov.copy_(ovf, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()          # the one host sync of the hand-off
        overflow = int(hov[0])
        symbols = h16 if overflow == 0 else sym.flatten().cpu()
        return {"symbols": symbols, "indexes": h8, "overflow": overflow, "y_hat": out["y_hat"]}

    # ---- DCAE.compress / decompress with the native range coder (SURVEY 8f N1 + N2) -----------------------------
    def compress_to_string(self, y, latent_scales, latent_means, gc) -> dict:
        """dcae.py:713-761 between `(y, latent_scales, latent_means)` and `y_string`: the slice loop, ONE packed
        device->host copy (int16 symbols, uint8 indexes, coder order) and one call into the native coder
        (`dcae_b200.ans.BufferedRansEncoder`, libdcae_rans.so) -- instead of ten `.tolist()` syncs, 2 x 320 T Python
        ints and a 200 k-element table list per call.  `gc`: the model's GaussianConditional (tables: `quantized_cdf`,
        `cdf_length`, `offset`, dcae.py:718-720).  -> dict(y_string: bytes, y_hat: device tensor, overflow: int)."""
        from .ans import BufferedRansEncoder
        h = self.compress_to_host(y, latent_scales, latent_means)
        enc = BufferedRansEncoder()
        enc.encode_with_indexes(h["symbols"], h["indexes"], *self._coder_tables(gc))
        return {"y_string": enc.flush(), "y_hat": h["y_hat"], "overflow": h["overflow"]}

    def decompress_from_string(self, y_string: bytes, latent_scales, latent_means, gc) -> dict:
        """dcae.py:875-906: per slice, the indexes leave the device in one copy, the native decoder returns the
        symbols as one int32 array, and they go back in one copy (the reference: `.tolist()`, a Python list of ints,
        `torch.Tensor(rv)` on the CPU, batch hard-coded to 1 at :894).  -> dict(y_hat, indexes)."""
        from .ans import RansDecoder
        dec = RansDecoder()
        dec.set_stream(y_string)
        tables = self._coder_tables(gc)
        B, _, h, w = latent_scales.shape
        n = B * SLICE_CH * h * w
        host_idx = torch.empty(n, dtype=torch.int32).pin_memory()
        host_sym = torch.empty(n, dtype=torch.int32).pin_memory()
        stream = torch.cuda.current_stream(self.device)

        def decode_slice(i, idx):
            host_idx.copy_(idx.reshape(-1), non_blocking=True)
            stream.synchronize()                                  # the decoder needs the indexes: one sync per slice
            host_sym.numpy()[:] = dec.decode_array(host_idx.numpy(), *tables)
            return host_sym.to(self.device, non_blocking=True).reshape(B, SLICE_CH, h, w)

        return self.decompress(latent_scales, latent_means, decode_slice)

    def _coder_tables(self, gc):
        """Host copies of the three coder tables of a GaussianConditional, cached per (object, table version)."""
        key = (id(gc), gc._quantized_cdf.data_ptr(), gc._quantized_cdf._version)
        if getattr(self, "_tables_key", None) != key:
            if gc._quantized_cdf.numel() == 0:
                raise _lib.DcaeError("the GaussianConditional has no CDF tables: call net.update() / update_scale_table() first")
            self._tables = (gc.quantized_cdf.detach().cpu().int().contiguous(), gc.cdf_length.detach().cpu().int().reshape(-1).contiguous(),
                            gc.offset.detach().cpu().int().reshape(-1).contiguous())
            self._tables_key = key
        return self._tables

    # ---- the opt-in interleaved y format ilv1 coded on the GPU (include/dcae_rans.h, csrc/rans_gpu.cu) ------------
    def _device_tables(self, gc):
        """Device copies of the coder tables, uploaded once per table version (same key as `_coder_tables`)."""
        key = (id(gc), gc._quantized_cdf.data_ptr(), gc._quantized_cdf._version)
        if getattr(self, "_dev_tables_key", None) != key:
            q, ln, off = (t.to(self.device) for t in self._coder_tables(gc))
            self._dev_tables = (q, ln, off, _lib.CoderTables(q.data_ptr(), q.shape[1], ln.data_ptr(), off.data_ptr(), q.shape[0]))
            self._dev_tables_key = key
        return self._dev_tables[3]

    def compress_to_strings_interleaved(self, y, latent_scales, latent_means, gc, lanes: int = 32) -> dict:
        """Like `compress_to_string`, in the ilv1 format and with the coder on the GPU: one y string per image, its five
        slices coded on `lanes` interleaved rANS states (1, 2, 4, 8, 16 or 32) by `dcae_ilv_encode`, straight from the
        device symbols / indexes of `compress`.  One small copy of the segment sizes, then one copy of the strings.
        -> dict(y_strings: list of B bytes, y_hat: device tensor)."""
        out = self.compress(y, latent_scales, latent_means)
        return {"y_strings": self.encode_symbols_interleaved(out["symbols"], out["indexes"], gc, lanes), "y_hat": out["y_hat"]}

    def encode_symbols_interleaved(self, sym, idx, gc, lanes: int = 32) -> list:
        """The coder alone: device int32 symbols / indexes [5, B, 64, h, w] (coder order) -> B ilv1 strings."""
        if sym.dim() != 5 or sym.shape[0] != NUM_SLICES or sym.shape[2] != SLICE_CH or idx.shape != sym.shape:
            raise ValueError("symbols / indexes: expected int32 [5, B, 64, h, w]")
        sym, idx = sym.to(self.device, torch.int32).contiguous(), idx.to(self.device, torch.int32).contiguous()
        _, B, _, h, w = sym.shape
        lib, s = self.lib, self._stream()
        tables = self._device_tables(gc)
        cap = int(lib.dcae_ilv_encode_max_bytes(B, h, w, lanes))
        if cap < 0:
            raise ValueError(f"lanes must be 1, 2, 4, 8, 16 or 32 (got {lanes})")
        scratch = torch.empty(int(lib.dcae_ilv_encode_scratch_bytes(B, h, w, lanes)) + 8, dtype=torch.uint8, device=self.device)
        buf = torch.empty(max(cap, 4), dtype=torch.uint8, device=self.device)
        sizes = torch.empty(B, NUM_SLICES, dtype=torch.int32, device=self.device)
        status = torch.empty(B, dtype=torch.int32, device=self.device)
        a = _lib.IlvEncArgs(sym.data_ptr(), idx.data_ptr(), B, h, w, lanes, tables, (scratch.data_ptr() + 7) // 8 * 8,
                            scratch.numel() - 8, sizes.data_ptr(), buf.data_ptr(), buf.numel(), status.data_ptr())
        with torch.cuda.device(self.device):
            _lib.check(lib.dcae_ilv_encode(C.byref(a), s), "dcae_ilv_encode")
        host_sizes, host_status = sizes.cpu(), status.cpu()
        self._raise_on_status(host_status, "encode")
        lengths = (24 + host_sizes.to(torch.int64).sum(1)).tolist()
        data = buf[: sum(lengths)].cpu().numpy().tobytes()
        strings, pos = [], 0
        for n in lengths:
            strings.append(data[pos: pos + n])
            pos += n
        return strings

    def decompress_from_strings_interleaved(self, y_strings, latent_scales, latent_means, gc) -> dict:
        """Inverse of `compress_to_strings_interleaved`: the B strings go to the device in one copy, then every slice is
        decoded by `dcae_ilv_decode` on the stream, between `dcae_slice_loop_indexes` and `dcae_slice_loop_decode`,
        with no host sync until the per-image status words are read once at the end.  A malformed or corrupt string
        raises DcaeError.  -> dict(y_hat, indexes)."""
        B, _, h, w = latent_scales.shape
        decode_slice, finish = self._ilv_decoder(y_strings, B, h, w, gc)
        out = self.decompress(latent_scales, latent_means, decode_slice)
        finish()
        return out

    def decode_symbols_interleaved(self, y_strings, idx, gc) -> torch.Tensor:
        """The coder alone: B ilv1 strings + device int32 indexes [5, B, 64, h, w] -> symbols [5, B, 64, h, w]."""
        _, B, _, h, w = idx.shape
        decode_slice, finish = self._ilv_decoder(y_strings, B, h, w, gc)
        out = torch.stack([decode_slice(i, idx[i].to(self.device, torch.int32).contiguous()).clone() for i in range(NUM_SLICES)])
        finish()
        return out

    def _ilv_decoder(self, y_strings, B, h, w, gc):
        """(decode_slice(i, indexes [B, 64, h, w]) -> symbols, finish()) over the B strings, uploaded in one copy."""
        if len(y_strings) != B:
            raise ValueError(f"{len(y_strings)} y strings for a batch of {B}")
        bounds, chunks, pos = [], [], 0
        for st in y_strings:
            st = bytes(st)
            bounds += [pos, pos + len(st)]
            pad = -len(st) % 4                                     # every string starts 4-byte aligned
            chunks.append(st + b"\0" * pad)
            pos += len(st) + pad
        blob = torch.frombuffer(bytearray(b"".join(chunks) or b"\0\0\0\0"), dtype=torch.uint8)
        dev_blob = blob.to(self.device)
        dev_bounds = torch.tensor(bounds or [0], dtype=torch.int64).to(self.device)
        status = torch.zeros(B, dtype=torch.int32, device=self.device)
        sym = torch.empty(B, SLICE_CH, h, w, dtype=torch.int32, device=self.device)
        tables = self._device_tables(gc)

        def decode_slice(i, idx):
            a = _lib.IlvDecArgs(dev_blob.data_ptr(), dev_bounds.data_ptr(), idx.data_ptr(), i, B, h, w, tables,
                                sym.data_ptr(), status.data_ptr())
            with torch.cuda.device(self.device):
                _lib.check(self.lib.dcae_ilv_decode(C.byref(a), self._stream()), "dcae_ilv_decode")
            return sym

        return decode_slice, lambda: self._raise_on_status(status.cpu(), "decode")

    @staticmethod
    def _raise_on_status(status, what):
        bad = [(b, int(v)) for b, v in enumerate(status.tolist()) if v]
        if bad:
            b, v = bad[0]
            raise _lib.DcaeError(f"ilv1 {what}: image {b}: {_lib.ILV_STATUS.get(v, v)} ({len(bad)} of {len(status)} images failed)")

    # ---- DCAE.decompress slice loop -------------------------------------------------------------
    def decompress(self, latent_scales, latent_means,
                   decode_slice: Callable[[int, torch.Tensor], torch.Tensor]):
        """decode_slice(i, indexes int32 [B,64,h,w] on device) -> symbols (int tensor, same shape) plays
        the rANS decoder of dcae.py:893.  -> dict(y_hat, indexes [5,B,64,h,w])."""
        ls = self._check_in("latent_scales", latent_scales)
        lm = self._check_in("latent_means", latent_means)
        B, _, h, w = ls.shape
        plan, lib, s = self._plan(B, h, w), self.lib, self._stream()
        self._last_call_lanes = False
        y_hat = torch.empty_like(ls)
        idx_all = torch.empty(NUM_SLICES, B, SLICE_CH, h, w, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(lib.dcae_slice_loop_load(plan.handle, None, ls.data_ptr(), lm.data_ptr(), s), "load")
            launches = 0
            for i in range(NUM_SLICES):
                _lib.check(lib.dcae_slice_loop_params(plan.handle, i, s), "params")
                _lib.check(lib.dcae_slice_loop_indexes(plan.handle, i, idx_all[i].data_ptr(), s), "indexes")
                sym = decode_slice(i, idx_all[i])
                sym = torch.as_tensor(sym).to(self.device, torch.int32).reshape(B, SLICE_CH, h, w).contiguous()
                _lib.check(lib.dcae_slice_loop_decode(plan.handle, i, sym.data_ptr(), s), "decode")
            _lib.check(lib.dcae_slice_loop_store(plan.handle, y_hat.data_ptr(), None, None, None, None, None, None, s), "store")
        self.last_launches = int(lib.dcae_launch_count())
        return {"y_hat": y_hat, "indexes": idx_all}

    # ---- module-level calls (dcae_b200/modules.py: drop-ins for the reference's own sub-modules) -------
    def module_dca(self, i: int, x: torch.Tensor) -> torch.Tensor:
        """dt_cross_attention[i](x, dt): x [B, 640 + 64 i, h, w] -> dict_info [B, 320, h, w]  (dcae.py:479-509)."""
        x = self._check_in("x", x, C_=2 * M_LATENT + SLICE_CH * i)
        B, _, h, w = x.shape
        out = torch.empty(B, M_LATENT, h, w, device=self.device)
        self._last_call_lanes = False
        with torch.cuda.device(self.device):
            _lib.check(self.lib.dcae_slice_loop_module_dca(self._plan(B, h, w).handle, i, x.data_ptr(), out.data_ptr(),
                                                           self._stream()), "dcae_slice_loop_module_dca")
        self.last_launches = int(self.lib.dcae_launch_count())
        return out

    def module_conv(self, i: int, which: int, x: torch.Tensor) -> torch.Tensor:
        """which 0 / 1 / 2 = cc_mean_transforms[i] / cc_scale_transforms[i] / lrp_transforms[i] (raw conv stack):
        x [B, 960 + 64 i (+ 64 for lrp), h, w] -> [B, 64, h, w]  (dcae.py:584-611)."""
        x = self._check_in("x", x, C_=3 * M_LATENT + SLICE_CH * i + (SLICE_CH if which == 2 else 0))
        B, _, h, w = x.shape
        out = torch.empty(B, SLICE_CH, h, w, device=self.device)
        self._last_call_lanes = False
        with torch.cuda.device(self.device):
            _lib.check(self.lib.dcae_slice_loop_module_conv(self._plan(B, h, w).handle, i, which, x.data_ptr(), out.data_ptr(),
                                                            self._stream()), "dcae_slice_loop_module_conv")
        self.last_launches = int(self.lib.dcae_launch_count())
        return out

    # ---- debugging / stage-wise parity (the reference's debug_save pattern, dcae_5_fixed.py:29-34) ---
    def tap(self, name: str, B: int, h: int, w: int) -> torch.Tensor:
        """Copy of a named token-major intermediate [T, cols] of the most recent call (`forward` lanes concatenated)."""
        split = self._lane_split(B, h * w) if getattr(self, "_last_call_lanes", False) else [(-1, 0, B)]
        if len(split) > 1:
            return torch.cat([self._tap_plan(self._plan(nb, h, w, lane), name, nb, h, w) for lane, _, nb in split])
        return self._tap_plan(self._plan(B, h, w), name, B, h, w)

    def _tap_plan(self, plan, name, B, h, w):
        p, cols, ld = C.c_void_p(), C.c_int32(), C.c_int64()
        _lib.check(self.lib.dcae_slice_loop_tap(plan.handle, name.encode(), C.byref(p), C.byref(cols), C.byref(ld)), "tap")
        T = B * h * w
        base = (plan.workspace.data_ptr() + 255) // 256 * 256
        off = (p.value - base) // 4
        o = base - plan.workspace.data_ptr()
        n = (plan.workspace.numel() - o) // 4 * 4
        flat = plan.workspace[o: o + n].view(torch.float32)
        return flat[off: off + T * ld.value].view(T, ld.value)[:, : cols.value].clone()


def _tap16(self, name: str, B: int, h: int, w: int) -> torch.Tensor:
    """f16x3 mode: a planes-only intermediate [T, cols] reconstructed as fp32 (hi + lo)."""
    split = self._lane_split(B, h * w) if getattr(self, "_last_call_lanes", False) else [(-1, 0, B)]
    if len(split) > 1:
        return torch.cat([_tap16_plan(self, self._plan(nb, h, w, lane), name, nb, h, w) for lane, _, nb in split])
    return _tap16_plan(self, self._plan(B, h, w), name, B, h, w)


def _tap16_plan(self, plan, name, B, h, w):
    pl, cols = _lib.Planes(), C.c_int32()
    _lib.check(self.lib.dcae_slice_loop_tap16(plan.handle, name.encode(), C.byref(pl), C.byref(cols)), "tap16")
    T, ld = B * h * w, int(pl.ld)
    ws = plan.workspace

    def view(ptr):
        off = ptr - ws.data_ptr()
        return ws[off: off + T * ld * 2].view(torch.float16).view(T, ld)

    return (view(pl.hi).float() + view(pl.lo).float())[:, : cols.value].clone()


EntropySliceLoop.tap16 = _tap16


def bits_per_pixel(log2_lik_sum: torch.Tensor, num_pixels: int) -> torch.Tensor:
    """train.py:82-85 with the log2 sum the slice loop already reduced: bpp = -sum(log2 lik) / num_pixels."""
    return -log2_lik_sum / float(num_pixels)
