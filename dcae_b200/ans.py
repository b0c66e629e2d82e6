"""`compressai.ans` stand-in on libdcae_rans.so (SURVEY 8f N2): `BufferedRansEncoder` / `RansDecoder` with the method
names and argument order the reference uses (dcae.py:722, 755-756, 875-876, 893), accepting Python lists like the
original AND numpy / pinned torch arrays -- int32, or the packed int16 symbols / uint8 indexes that
`EntropySliceLoop.compress_to_host` brings back in one D2H copy -- without any per-element Python work.

The CDF tables may be given as the reference gives them (`quantized_cdf.tolist()`, `cdf_length.reshape(-1).int().tolist()`,
`offset.reshape(-1).int().tolist()`, dcae.py:718-720) or as the tensors themselves; they are converted once per object
and cached by identity.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdcae_rans.so")

I32, I16, U8 = 0, 1, 2
_DTYPES = {np.dtype(np.int32): I32, np.dtype(np.int16): I16, np.dtype(np.uint8): U8}


class RansTables(C.Structure):
    _fields_ = [("cdfs", C.c_void_p), ("cdf_stride", C.c_int32), ("cdf_sizes", C.c_void_p), ("offsets", C.c_void_p),
                ("n_cdfs", C.c_int32)]


_P, _I32, _I64 = C.c_void_p, C.c_int32, C.c_int64
SIGNATURES = {
    "dcae_rans_last_error": (C.c_char_p, []),
    "dcae_rans_encoder_create": (_P, []),
    "dcae_rans_encoder_destroy": (None, [_P]),
    "dcae_rans_encoder_encode_with_indexes": (C.c_int, [_P, _P, _I32, _P, _I32, _I64, C.POINTER(RansTables)]),
    "dcae_rans_encoder_flush": (_I64, [_P]),
    "dcae_rans_encoder_bytes": (_P, [_P]),
    "dcae_rans_decoder_create": (_P, []),
    "dcae_rans_decoder_destroy": (None, [_P]),
    "dcae_rans_decoder_set_stream": (C.c_int, [_P, C.c_char_p, _I64]),
    "dcae_rans_decoder_decode_stream": (C.c_int, [_P, _P, _I32, _I64, C.POINTER(RansTables), _P]),
    "dcae_pmf_to_quantized_cdf": (C.c_int, [_P, _I32, _I32, _P]),
    "dcae_rans_ilv_max_bytes": (_I64, [_I64, _I32]),
    "dcae_rans_ilv_encode": (_I64, [_P, _P, _I64, _I32, C.POINTER(RansTables), _P, _I64]),
    "dcae_rans_ilv_decode": (C.c_int, [C.c_char_p, _I64, _P, _I64, C.POINTER(RansTables), _P]),
}

_lib = None


class RansError(RuntimeError):
    pass


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RansError(f"{LIB_PATH} not found: run `python __graft_entry__.py` (build()) first")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def _check(rc: int, what: str) -> None:
    if rc < 0:
        raise RansError(f"{what} failed ({rc}): {load().dcae_rans_last_error().decode('utf-8', 'replace')}")


def _array(x, allow=(np.int32, np.int16, np.uint8)) -> np.ndarray:
    """Flat, contiguous host array of one of the coder's element types (zero-copy for numpy / CPU torch inputs)."""
    if hasattr(x, "detach"):                   # torch tensor
        if x.is_cuda:
            raise RansError("the range coder runs on the host: pass a CPU tensor (see EntropySliceLoop.compress_to_host)")
        x = x.detach().numpy()
    a = np.asarray(x)
    if a.dtype not in [np.dtype(t) for t in allow]:
        a = a.astype(np.int32)
    return np.ascontiguousarray(a).reshape(-1)


class _Tables:
    """(cdf, cdf_lengths, offsets) as C arrays, cached by the identity of the three arguments."""

    def __init__(self):
        self._key = None
        self.struct = None

    def get(self, cdf, cdf_lengths, offsets) -> RansTables:
        key = (id(cdf), id(cdf_lengths), id(offsets))
        if key != self._key:
            if hasattr(cdf, "detach"):
                q = np.ascontiguousarray(cdf.detach().cpu().numpy().astype(np.int32))
            elif isinstance(cdf, np.ndarray):
                q = np.ascontiguousarray(cdf.astype(np.int32))
            else:                                  # list of rows (possibly ragged)
                width = max(len(r) for r in cdf)
                q = np.zeros((len(cdf), width), dtype=np.int32)
                for i, r in enumerate(cdf):
                    q[i, : len(r)] = r
            ln = _array(cdf_lengths, allow=(np.int32,))
            off = _array(offsets, allow=(np.int32,))
            if not (q.ndim == 2 and len(ln) == q.shape[0] == len(off)):
                raise RansError("cdf / cdf_lengths / offsets shapes disagree")
            self._keep = (q, ln, off, cdf, cdf_lengths, offsets)        # pins the ids for the cache key
            self.struct = RansTables(q.ctypes.data, q.shape[1], ln.ctypes.data, off.ctypes.data, q.shape[0])
            self._key = key
        return self.struct


class BufferedRansEncoder:
    """compressai.ans.BufferedRansEncoder: encode_with_indexes(...)* then flush() -> bytes."""

    def __init__(self):
        self._lib = load()
        self._h = self._lib.dcae_rans_encoder_create()
        self._tables = _Tables()

    def __del__(self):
        if getattr(self, "_h", None):
            self._lib.dcae_rans_encoder_destroy(self._h)

    def encode_with_indexes(self, symbols, indexes, cdf, cdf_lengths, offsets) -> None:
        s, i = _array(symbols, allow=(np.int32, np.int16)), _array(indexes, allow=(np.int32, np.uint8))
        if s.size != i.size:
            raise RansError("symbols and indexes differ in length")
        t = self._tables.get(cdf, cdf_lengths, offsets)
        _check(self._lib.dcae_rans_encoder_encode_with_indexes(self._h, s.ctypes.data, _DTYPES[s.dtype], i.ctypes.data,
                                                               _DTYPES[i.dtype], s.size, C.byref(t)), "encode_with_indexes")

    def flush(self) -> bytes:
        n = self._lib.dcae_rans_encoder_flush(self._h)
        _check(int(n), "flush")
        return C.string_at(self._lib.dcae_rans_encoder_bytes(self._h), int(n))


class RansDecoder:
    """compressai.ans.RansDecoder: set_stream(bytes) then decode_stream(indexes, cdf, cdf_lengths, offsets)."""

    def __init__(self):
        self._lib = load()
        self._h = self._lib.dcae_rans_decoder_create()
        self._tables = _Tables()

    def __del__(self):
        if getattr(self, "_h", None):
            self._lib.dcae_rans_decoder_destroy(self._h)

    def set_stream(self, stream: bytes) -> None:
        _check(self._lib.dcae_rans_decoder_set_stream(self._h, stream, len(stream)), "set_stream")

    def decode_array(self, indexes, cdf, cdf_lengths, offsets) -> np.ndarray:
        """decode_stream into an int32 numpy array (no Python-int materialisation)."""
        i = _array(indexes, allow=(np.int32, np.uint8))
        out = np.empty(i.size, dtype=np.int32)
        t = self._tables.get(cdf, cdf_lengths, offsets)
        _check(self._lib.dcae_rans_decoder_decode_stream(self._h, i.ctypes.data, _DTYPES[i.dtype], i.size, C.byref(t),
                                                         out.ctypes.data), "decode_stream")
        return out

    def decode_stream(self, indexes, cdf, cdf_lengths, offsets) -> Sequence[int]:
        """The reference's call (dcae.py:893): returns a list, as compressai does."""
        return self.decode_array(indexes, cdf, cdf_lengths, offsets).tolist()


ILV_SLICES = 5
ILV_LANES = (1, 2, 4, 8, 16, 32)


def _slices(x, what) -> np.ndarray:
    a = _array(x, allow=(np.int32,))
    if a.size % ILV_SLICES:
        raise RansError(f"{what}: expected {ILV_SLICES} slices of equal length, got {a.size} values")
    return a


def encode_interleaved(symbols, indexes, cdf, cdf_lengths, offsets, lanes: int = 32) -> bytes:
    """The ilv1 string of one image (include/dcae_rans.h): symbols / indexes [5, n] (the image's five slices, each in
    coder order), coded on `lanes` interleaved rANS states.  The host reference of the sm_100a encoder."""
    s, i = _slices(symbols, "symbols"), _slices(indexes, "indexes")
    if s.size != i.size:
        raise RansError("symbols and indexes differ in length")
    n = s.size // ILV_SLICES
    tab = _Tables()                              # owns the arrays the struct points at until the call returns
    t = tab.get(cdf, cdf_lengths, offsets)
    cap = int(load().dcae_rans_ilv_max_bytes(n, lanes))
    _check(cap, "ilv_max_bytes")
    out = np.empty(cap, dtype=np.uint8)
    size = int(load().dcae_rans_ilv_encode(s.ctypes.data, i.ctypes.data, n, lanes, C.byref(t), out.ctypes.data, cap))
    _check(size, "ilv_encode")
    return out[:size].tobytes()


def decode_interleaved(data: bytes, indexes, cdf, cdf_lengths, offsets) -> np.ndarray:
    """ilv1 string + indexes [5, n] -> int32 symbols [5, n]; raises RansError on a malformed or corrupt string."""
    i = _slices(indexes, "indexes")
    out = np.empty(i.size, dtype=np.int32)
    tab = _Tables()
    t = tab.get(cdf, cdf_lengths, offsets)
    data = bytes(data)
    _check(load().dcae_rans_ilv_decode(data, len(data), i.ctypes.data, i.size // ILV_SLICES, C.byref(t), out.ctypes.data),
           "ilv_decode")
    return out.reshape(ILV_SLICES, -1)


def pmf_to_quantized_cdf(pmf, precision: int = 16):
    """compressai._CXX.pmf_to_quantized_cdf: list of floats -> list of ints (len + 1)."""
    p = np.ascontiguousarray(np.asarray(pmf, dtype=np.float32).reshape(-1))
    out = np.empty(p.size + 1, dtype=np.int32)
    _check(load().dcae_pmf_to_quantized_cdf(p.ctypes.data, p.size, precision, out.ctypes.data), "pmf_to_quantized_cdf")
    return out.tolist()
