"""CPU: the interleaved y-stream format ilv1 (include/dcae_rans.h) in the host coder (libdcae_rans.so,
`dcae_b200.ans.encode_interleaved / decode_interleaved`) against the pure-Python restatement (tests/_ilv_oracle.py), the
single-stream coder it reuses, and the DCI1 container."""
import struct

import numpy as np
import pytest

from dcae_b200 import ans, container
from dcae_b200.gaussian_conditional import GaussianConditional
from oracle import gaussian_conditional as ogc
import _ilv_oracle as oilv

LANES = (1, 2, 4, 8, 16, 32)


@pytest.fixture(scope="module")
def tables():
    import __graft_entry__ as ge
    ge.build()
    gc = GaussianConditional(None)
    gc.update_scale_table(ogc.get_scale_table())
    return gc.quantized_cdf, gc.cdf_length, gc.offset


def _lists(tables):
    q, ln, off = tables
    return q.tolist(), ln.reshape(-1).int().tolist(), off.reshape(-1).int().tolist()


def _draw(n, seed, outliers=0.03, extreme=False):
    """[5, n] symbols / indexes like the slice loop's, with bypass outliers on both sides (int32 extremes if asked)."""
    g = np.random.default_rng(seed)
    idx = g.integers(0, 64, (5, n)).astype(np.int32)
    sym = np.rint(g.standard_normal((5, n)) * ogc.get_scale_table().numpy()[idx]).astype(np.int32)
    far = g.random((5, n)) < outliers
    sym[far] = g.integers(-40000, 40000, far.sum()).astype(np.int32)
    if extreme and n >= 4:
        sym[:, :4] = [np.iinfo(np.int32).min, np.iinfo(np.int32).max, -(1 << 20), (1 << 24) + 5]
    return sym, idx


def _segments(data):
    version, lanes, zero, *seg = struct.unpack("<BBH5I", data[:24])
    out, pos = [], 24
    for nb in seg:
        out.append(data[pos:pos + nb])
        pos += nb
    return lanes, out


@pytest.mark.parametrize("lanes", LANES)
def test_native_bytes_equal_the_restatement(tables, lanes):
    """n < L, n not a multiple of L, an empty slice and bypass symbols up to int32 magnitudes, for every L."""
    cdf, ln, off = _lists(tables)
    for seed, n, extreme in ((0, 0, False), (1, 1, False), (2, 7, True), (3, 33, False), (4, 301, True)):
        sym, idx = _draw(n, seed + 10 * lanes, extreme=extreme)
        got = ans.encode_interleaved(sym, idx, *tables, lanes=lanes)
        want = oilv.encode_interleaved(sym.tolist(), idx.tolist(), lanes, cdf, ln, off)
        assert got == want, (lanes, n)
        assert np.array_equal(ans.decode_interleaved(got, idx, *tables), sym)
        assert oilv.decode_interleaved(got, idx.tolist(), cdf, ln, off) == sym.tolist()


def test_one_lane_segment_is_the_single_stream_coder(tables):
    """L = 1: each slice segment is byte for byte what BufferedRansEncoder writes for that slice's symbols."""
    sym, idx = _draw(2000, 5, extreme=True)
    lanes, segs = _segments(ans.encode_interleaved(sym, idx, *tables, lanes=1))
    assert lanes == 1
    for s in range(5):
        enc = ans.BufferedRansEncoder()
        enc.encode_with_indexes(sym[s], idx[s], *tables)
        assert segs[s] == enc.flush(), s


@pytest.mark.parametrize("lanes", (1, 32))
def test_round_trip_at_image_size(tables, lanes):
    sym, idx = _draw(64 * 48 * 32, 6)                      # one 768x512 image: 5 slices of 64 x 48 x 32
    data = ans.encode_interleaved(sym, idx, *tables, lanes=lanes)
    assert np.array_equal(ans.decode_interleaved(data, idx, *tables), sym)
    ref = ans.BufferedRansEncoder()
    for s in range(5):
        ref.encode_with_indexes(sym[s], idx[s], *tables)
    # the format costs 4 + 5 (4 + 8 L) bytes per image, the reference format 8; the words themselves differ by about one
    # per state and slice, where each state stops renormalising
    assert abs(len(data) - len(ref.flush()) - (4 + 5 * (4 + 8 * lanes) - 8)) <= 4 * 5 * (lanes + 1)


def test_bad_arguments_and_corrupt_strings_return_errors(tables):
    sym, idx = _draw(500, 7)
    data = ans.encode_interleaved(sym, idx, *tables, lanes=8)
    for lanes in (0, 3, 12, 64):
        with pytest.raises(ans.RansError, match="lanes"):
            ans.encode_interleaved(sym, idx, *tables, lanes=lanes)
    bad_idx = idx.copy()
    bad_idx[2, 10] = 64
    with pytest.raises(ans.RansError, match="index"):
        ans.encode_interleaved(sym, bad_idx, *tables, lanes=8)
    with pytest.raises(ans.RansError, match="index"):
        ans.decode_interleaved(data, bad_idx, *tables)
    broken = [data[:10], data[:-4], data[:-1], data + b"\0\0\0\0",
              b"\x02" + data[1:],                                   # version
              data[:1] + b"\x03" + data[2:],                        # L not a power of two
              data[:1] + b"\x40" + data[2:],                        # L > 32
              data[:2] + b"\x01" + data[3:]]                        # reserved field
    seg0 = struct.unpack("<I", data[4:8])[0]
    broken.append(data[:4] + struct.pack("<I", seg0 - 4) + data[8:])            # header sizes disagree with the string
    broken.append(data[:4] + struct.pack("<II", seg0 - 4, struct.unpack("<I", data[8:12])[0] + 4) + data[12:])  # words moved
    broken.append(data[:4] + struct.pack("<II", 4, seg0 + struct.unpack("<I", data[8:12])[0] - 4) + data[12:])  # < 8 L
    for b in broken:
        with pytest.raises(ans.RansError):
            ans.decode_interleaved(b, idx, *tables)
    g = np.random.default_rng(0)
    raised = 0
    for trial in range(40):                                     # flipped words in the body: an error or other symbols,
        b = bytearray(data)                                     # never a crash or a read outside the string
        pos = int(g.integers(24, len(b) - 4))
        b[pos:pos + 4] = g.integers(0, 256, 4, dtype=np.uint8).tobytes()
        try:
            out = ans.decode_interleaved(bytes(b), idx, *tables)
            assert out.shape == sym.shape
        except ans.RansError:
            raised += 1
    assert raised >= 30                                         # the end-state check catches nearly every corruption


def test_ilv_container_round_trip():
    strings = [[bytes(range(256)) * 3], [b"z-stream"]]
    blob = container.pack_ilv(strings, (513, 770))
    assert blob[:4] == b"DCI1"
    assert blob[4:12] == struct.pack(">HHI", 513, 770, 768)
    got, z_shape, padding, size = container.unpack_ilv(blob)
    assert got == strings and size == (513, 770)
    assert (z_shape, padding) == container.unpack_bin(container.pack_bin(strings, (513, 770)))[1:3]
    for cut in (3, 10, 20, len(blob) - 1):
        with pytest.raises(ValueError):
            container.unpack_ilv(blob[:cut])
    with pytest.raises(ValueError):
        container.unpack_ilv(b"DCA1" + blob[4:])
    with pytest.raises(ValueError):
        container.unpack_ilv(container.pack_bin(strings, (513, 770)))        # a .bin container is not sniffed as DCI1


def test_gpu_coder_abi_layout_and_argument_checks():
    """The ctypes mirrors of dcae_ilv_enc_args / dcae_ilv_dec_args match the C compiler, and bad arguments are rejected
    before any launch (testable without a device)."""
    import ctypes as C
    import os
    import subprocess
    import tempfile
    import __graft_entry__ as ge
    ge.build()
    from dcae_b200 import _lib
    lib = _lib.load()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    prog = ('#include <stdio.h>\n#include <stddef.h>\n#include "dcae_b200.h"\nint main(){printf("%zu %zu %zu %zu %zu\\n", '
            'sizeof(dcae_coder_tables), sizeof(dcae_ilv_enc_args), sizeof(dcae_ilv_dec_args), '
            'offsetof(dcae_ilv_enc_args, status), offsetof(dcae_ilv_dec_args, status));return 0;}\n')
    with tempfile.TemporaryDirectory() as td:
        open(os.path.join(td, "t.c"), "w").write(prog)
        subprocess.run(["gcc", "-I", os.path.join(root, "include"), "-o", os.path.join(td, "t"), os.path.join(td, "t.c")], check=True)
        sizes = [int(v) for v in subprocess.run([os.path.join(td, "t")], capture_output=True, text=True, check=True).stdout.split()]
    assert sizes == [C.sizeof(_lib.CoderTables), C.sizeof(_lib.IlvEncArgs), C.sizeof(_lib.IlvDecArgs),
                     _lib.IlvEncArgs.status.offset, _lib.IlvDecArgs.status.offset]
    t = _lib.CoderTables(8, 10, 8, 8, 64)                       # non-null placeholders: no launch happens below
    a = _lib.IlvEncArgs(8, 8, 1, 4, 4, 3, t)
    assert lib.dcae_ilv_encode(C.byref(a), None) == -1 and b"lanes" in lib.dcae_last_error()
    a.lanes = 32
    assert lib.dcae_ilv_encode(C.byref(a), None) == -1 and b"null pointer" in lib.dcae_last_error()
    a.B = 0
    assert lib.dcae_ilv_encode(C.byref(a), None) == 0           # an empty batch enqueues nothing
    d = _lib.IlvDecArgs(8, 8, 8, 5, 1, 4, 4, t, 8, 8)
    assert lib.dcae_ilv_decode(C.byref(d), None) == -1 and b"slice" in lib.dcae_last_error()
    d.slice, d.strings = 0, 10
    assert lib.dcae_ilv_decode(C.byref(d), None) == -1 and b"aligned" in lib.dcae_last_error()
    assert lib.dcae_ilv_encode_max_bytes(2, 3, 5, 32) == 2 * ans.load().dcae_rans_ilv_max_bytes(64 * 15, 32)
    assert lib.dcae_ilv_encode_max_bytes(1, 3, 5, 12) == -1
