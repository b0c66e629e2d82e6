"""The reference's bitstream container and image padding (data formats either side of the path, SURVEY 8f N2):
`/root/reference/compress_and_decompress.py` `save_bin` / `read_bin` (:110-148), `calculate_padding` (:125-134), `pad` /
`crop` (:48-71).  One image per file:

    >H height  >H width  >I len(y_string)  y_string  >I len(z_string)  z_string

(height / width = the UNPADDED image size; the decoder recomputes the centred zero padding to multiples of 128 and the
z grid = padded size / 64 from them).  Host-side byte shuffling only; files written here are read by the reference's
`read_bin` and the other way round.
"""
from __future__ import annotations

import struct
from typing import List, Sequence, Tuple

import torch
import torch.nn.functional as F

PAD_MULTIPLE = 128


def calculate_padding(h: int, w: int, p: int = PAD_MULTIPLE):
    """-> ((new_h, new_w), (left, right, top, bottom)): centred padding to multiples of p (compress_and_decompress.py:125-134)."""
    new_h, new_w = (h + p - 1) // p * p, (w + p - 1) // p * p
    left = (new_w - w) // 2
    top = (new_h - h) // 2
    return (new_h, new_w), (left, new_w - w - left, top, new_h - h - top)


def pad(x: torch.Tensor, p: int = PAD_MULTIPLE):
    """Zero-pad [B, C, H, W] to multiples of p, centred (:48-65).  -> (x_padded, padding)."""
    _, padding = calculate_padding(x.size(2), x.size(3), p)
    return F.pad(x, padding, mode="constant", value=0), padding


def crop(x: torch.Tensor, padding: Sequence[int]) -> torch.Tensor:
    """Undo `pad` (:67-71)."""
    return F.pad(x, (-padding[0], -padding[1], -padding[2], -padding[3]))


def pack_bin(strings: Sequence[Sequence[bytes]], size: Sequence[int]) -> bytes:
    """strings = [[y_string], [z_string]] as `DCAE.compress` returns them (dcae.py:761), size = (H, W) of the unpadded image."""
    y, z = strings[0][0], strings[1][0]
    if not (0 <= int(size[0]) < 65536 and 0 <= int(size[1]) < 65536):
        raise ValueError("image sides must fit in 16 bits (the container stores them as >H)")
    return b"".join((struct.pack(">H", int(size[0])), struct.pack(">H", int(size[1])), struct.pack(">I", len(y)), bytes(y),
                     struct.pack(">I", len(z)), bytes(z)))


def unpack_bin(blob: bytes):
    """-> (strings [[y], [z]], z_shape [h_pad / 64, w_pad / 64], padding, (H, W))   (read_bin, :136-148)."""
    if len(blob) < 12:
        raise ValueError("truncated container")
    h, w, ly = struct.unpack(">HHI", blob[:8])
    if len(blob) < 12 + ly:
        raise ValueError("truncated container (y stream)")
    y = blob[8:8 + ly]
    (lz,) = struct.unpack(">I", blob[8 + ly:12 + ly])
    z = blob[12 + ly:12 + ly + lz]
    if len(z) != lz:
        raise ValueError("truncated container (z stream)")
    padded, padding = calculate_padding(h, w)
    return [[y], [z]], [padded[0] // 64, padded[1] // 64], padding, (h, w)


ILV_MAGIC = b"DCI1"


def pack_ilv(strings: Sequence[Sequence[bytes]], size: Sequence[int]) -> bytes:
    """The container of the interleaved y format (`DCAECodec.compress(..., coder="interleaved")`), one image per file:

        b"DCI1"  >H height  >H width  >I len(y_string)  y_string  >I len(z_string)  z_string

    y_string is the image's ilv1 string (include/dcae_rans.h), z_string the same z stream as in `pack_bin`.  Its own
    magic keeps it apart from the reference's `.bin`, which the reference's `read_bin` cannot decode."""
    return ILV_MAGIC + pack_bin(strings, size)


def unpack_ilv(blob: bytes):
    """-> (strings [[y], [z]], z_shape, padding, (H, W)), like `unpack_bin`."""
    if blob[:4] != ILV_MAGIC:
        raise ValueError("not a DCI1 container")
    strings, z_shape, padding, size = unpack_bin(blob[4:])
    if 16 + len(strings[0][0]) + len(strings[1][0]) != len(blob):
        raise ValueError("DCI1 container: trailing bytes")
    return strings, z_shape, padding, size


def save_bin(strings, size, path: str) -> None:
    with open(path, "wb") as f:
        f.write(pack_bin(strings, size))


def read_bin(path: str):
    with open(path, "rb") as f:
        strings, z_shape, padding, _ = unpack_bin(f.read())
    return strings, z_shape, padding


__all__ = ["calculate_padding", "pad", "crop", "pack_bin", "unpack_bin", "pack_ilv", "unpack_ilv", "save_bin", "read_bin"]
