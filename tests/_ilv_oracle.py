"""TEST INFRASTRUCTURE ONLY -- pure-Python restatement of the interleaved y-stream format `ilv1`
(`dcae_b200.ans.encode_interleaved / decode_interleaved`, `csrc/rans_coder.cpp` dcae_rans_ilv_*, `csrc/rans_gpu.cu`) on
top of the restatement of the single-stream coder in oracle/rans.py: the same per-step arithmetic, only the assignment of
symbols to states and the order of the words are new.  Python ints, small cases only."""
from __future__ import annotations

import struct
from typing import List

from oracle.rans import BYPASS_BITS, BYPASS_MAX, PRECISION, RANS_L

# Same arithmetic as oracle.rans.encode / Decoder.  Symbol j of a slice goes to lane j % L at step j // L; one string holds a
# 24-byte header (u8 version 1, u8 L, u16 0, 5 x u32 segment bytes) and one segment per slice: the L final states
# (u64) then one shared stream of u32 words, in the order the decoder consumes them (step, sub-operation, lane).
ILV_VERSION = 1
ILV_SLICES = 5
ILV_LANES = (1, 2, 4, 8, 16, 32)


def _symbol_steps(sym, k, cdfs, cdf_sizes, offsets):
    """The coding steps of one symbol, in decode order: (start, freq, is_bypass)."""
    cdf, max_value = cdfs[k], cdf_sizes[k] - 2
    value, raw = sym - offsets[k], 0
    if value < 0:
        raw, value = -2 * value - 1, max_value
    elif value >= max_value:
        raw, value = 2 * (value - max_value), max_value
    steps = [(cdf[value], cdf[value + 1] - cdf[value], False)]
    if value == max_value:
        n_bypass = 0
        while (raw >> (n_bypass * BYPASS_BITS)) != 0:
            n_bypass += 1
        val = n_bypass
        while val >= BYPASS_MAX:
            steps.append((BYPASS_MAX, 1, True))
            val -= BYPASS_MAX
        steps.append((val, 1, True))
        for j in range(n_bypass):
            steps.append(((raw >> (j * BYPASS_BITS)) & BYPASS_MAX, 1, True))
    return steps


def _put(x, start, freq, bypass, words):
    if not bypass:
        if x >= ((RANS_L >> PRECISION) << 32) * freq:
            words.append(x & 0xFFFFFFFF)
            x >>= 32
        return ((x // freq) << PRECISION) + (x % freq) + start
    if x >= ((RANS_L >> 16) << 32) * (1 << (16 - BYPASS_BITS)):
        words.append(x & 0xFFFFFFFF)
        x >>= 32
    return (x << BYPASS_BITS) | start


def encode_interleaved_segment(symbols, indexes, lanes, cdfs, cdf_sizes, offsets) -> bytes:
    n = len(symbols)
    steps = [_symbol_steps(s, k, cdfs, cdf_sizes, offsets) for s, k in zip(symbols, indexes)]
    x, words = [RANS_L] * lanes, []                  # words in emission order = reverse of the decoder's order
    for t in reversed(range((n + lanes - 1) // lanes)):
        js = [(lane, t * lanes + lane) for lane in range(lanes) if t * lanes + lane < n]
        for k in reversed(range(max(len(steps[j]) for _, j in js))):
            for lane, j in reversed(js):
                if k < len(steps[j]):
                    x[lane] = _put(x[lane], *steps[j][k], words)
    return struct.pack("<%dQ" % lanes, *x) + struct.pack("<%dI" % len(words), *reversed(words))


def encode_interleaved(symbols, indexes, lanes, cdfs, cdf_sizes, offsets) -> bytes:
    """symbols / indexes: 5 sequences (the slices of one image, each in coder order) -> the ilv1 string."""
    assert lanes in ILV_LANES and len(symbols) == len(indexes) == ILV_SLICES
    segs = [encode_interleaved_segment(s, i, lanes, cdfs, cdf_sizes, offsets) for s, i in zip(symbols, indexes)]
    return struct.pack("<BBH5I", ILV_VERSION, lanes, 0, *map(len, segs)) + b"".join(segs)


class _IlvLane:
    """One lane's decoder state machine: phase 0 = symbol, 1 = bypass count, 2 = bypass digits, 3 = done."""

    def __init__(self, x):
        self.x, self.phase = x, 3


def decode_interleaved(data: bytes, indexes, cdfs, cdf_sizes, offsets) -> List[List[int]]:
    """-> 5 lists of symbols.  Raises ValueError on a malformed or corrupt string."""
    if len(data) < 24:
        raise ValueError("ilv1: truncated header")
    version, lanes, zero, *seg = struct.unpack("<BBH5I", data[:24])
    if version != ILV_VERSION or lanes not in ILV_LANES or zero != 0 or 24 + sum(seg) != len(data):
        raise ValueError("ilv1: bad header")
    out, pos = [], 24
    for nbytes, idx in zip(seg, indexes):
        if nbytes < 8 * lanes or (nbytes - 8 * lanes) % 4:
            raise ValueError("ilv1: bad segment size")
        body = data[pos:pos + nbytes]
        pos += nbytes
        st = [_IlvLane(x) for x in struct.unpack("<%dQ" % lanes, body[:8 * lanes])]
        words = struct.unpack("<%dI" % ((nbytes - 8 * lanes) // 4), body[8 * lanes:])
        w, n, sym = 0, len(idx), [0] * len(idx)
        for t in range((n + lanes - 1) // lanes):
            for lane in range(lanes):
                if t * lanes + lane < n:
                    st[lane].phase = 0
            while any(s.phase != 3 for s in st):          # one sub-operation k per pass, lanes ascending
                for lane, s in enumerate(st):
                    if s.phase == 3:
                        continue
                    j = t * lanes + lane
                    k = idx[j]
                    if s.phase == 0:
                        cdf, max_value = cdfs[k], cdf_sizes[k] - 2
                        cum = s.x & ((1 << PRECISION) - 1)
                        v = next(i for i in range(cdf_sizes[k]) if cdf[i] > cum) - 1
                        s.x = (cdf[v + 1] - cdf[v]) * (s.x >> PRECISION) + cum - cdf[v]
                        if v == max_value:
                            s.phase, s.count, s.raw, s.got = 1, 0, 0, 0
                        else:
                            sym[j], s.phase = v + offsets[k], 3
                    else:
                        d = s.x & BYPASS_MAX
                        s.x >>= BYPASS_BITS
                        if s.phase == 1:
                            s.count += d
                            if s.count > 16:
                                raise ValueError("ilv1: corrupt bypass length")
                            if d != BYPASS_MAX:
                                s.phase = 2
                        else:
                            s.raw |= d << (s.got * BYPASS_BITS)
                            s.got += 1
                        if s.phase == 2 and s.got == s.count:
                            v = s.raw >> 1
                            v = -v - 1 if s.raw & 1 else v + cdf_sizes[k] - 2
                            sym[j], s.phase = v + offsets[k], 3
                    if s.x < RANS_L:
                        if w >= len(words):
                            raise ValueError("ilv1: stream exhausted")
                        s.x = (s.x << 32) | words[w]
                        w += 1
        if w != len(words) or any(s.x != RANS_L for s in st):
            raise ValueError("ilv1: segment does not end where the encoder started")
        out.append(sym)
    return out
