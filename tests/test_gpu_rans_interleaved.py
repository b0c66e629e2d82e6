"""GPU: the ilv1 coder kernels (csrc/rans_gpu.cu: dcae_ilv_encode / dcae_ilv_decode) against the host coder's bytes
(libdcae_rans.so, itself pinned to the Python restatement by tests/test_rans_interleaved_host.py), and the opt-in
`coder="interleaved"` path through EntropySliceLoop, DCAECodec and the DCI1 container."""
import numpy as np
import pytest
import torch

from dcae_b200 import _lib, ans
from dcae_b200.gaussian_conditional import GaussianConditional
from dcae_b200.transforms import init_transform_params
from oracle import gaussian_conditional as ogc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
LANES = (1, 2, 4, 8, 16, 32)


@pytest.fixture(scope="module")
def eng(lively_params):
    import __graft_entry__ as ge
    ge.build()
    from dcae_b200.entropy_model import EntropySliceLoop
    return EntropySliceLoop(lively_params, device=DEV)


@pytest.fixture(scope="module")
def gc():
    g = GaussianConditional(None).to(DEV)
    g.update_scale_table(ogc.get_scale_table())
    return g


@pytest.fixture(scope="module")
def codec(lively_params):
    from dcae_b200 import DCAECodec
    P = dict(lively_params)
    P.update(init_transform_params(2))
    c = DCAECodec(P, device=DEV)
    c.update()
    return c


def _draw(B, h, w, seed, outliers=0.02):
    """[5, B, 64, h, w] symbols / indexes with bypass outliers on both sides, some outside int16 and at the int32 ends."""
    g = np.random.default_rng(seed)
    idx = g.integers(0, 64, (5, B, 64, h, w)).astype(np.int32)
    sym = np.rint(g.standard_normal(idx.shape) * ogc.get_scale_table().numpy()[idx]).astype(np.int32)
    far = g.random(idx.shape) < outliers
    sym[far] = g.integers(-70000, 70000, far.sum()).astype(np.int32)
    flat = sym.reshape(5, B, -1)
    flat[:, :, 0], flat[:, :, 1] = np.iinfo(np.int32).min, np.iinfo(np.int32).max
    return torch.from_numpy(sym), torch.from_numpy(idx)


def _host(gc):
    return gc.quantized_cdf.cpu(), gc.cdf_length.cpu(), gc.offset.cpu()


@pytest.mark.parametrize("B,h,w", [(1, 3, 5), (3, 7, 9), (3, 1, 1)])
def test_kernel_bytes_equal_the_host_coder(eng, gc, B, h, w):
    sym, idx = _draw(B, h, w, seed=B * 100 + h * 10 + w)
    tables = _host(gc)
    dsym, didx = sym.to(DEV), idx.to(DEV)
    for lanes in LANES:
        got = eng.encode_symbols_interleaved(dsym, didx, gc, lanes=lanes)
        want = [ans.encode_interleaved(sym[:, b].reshape(5, -1).numpy(), idx[:, b].reshape(5, -1).numpy(), *tables, lanes=lanes)
                for b in range(B)]
        assert got == want, lanes
        # the decode kernel returns the exact symbols, for kernel-encoded and host-encoded strings alike
        assert torch.equal(eng.decode_symbols_interleaved(got, didx, gc).cpu(), sym)
        assert torch.equal(eng.decode_symbols_interleaved(want, didx, gc).cpu(), sym)


def test_encoding_is_deterministic_and_batch_invariant(eng, gc):
    sym, idx = _draw(4, 12, 8, seed=5)
    dsym, didx = sym.to(DEV), idx.to(DEV)
    batch = eng.encode_symbols_interleaved(dsym, didx, gc)
    assert batch == eng.encode_symbols_interleaved(dsym, didx, gc)
    for b in range(4):
        assert eng.encode_symbols_interleaved(dsym[:, b:b + 1], didx[:, b:b + 1], gc) == [batch[b]]


@pytest.mark.parametrize("H,W", [(256, 256), (512, 768)])
def test_codec_round_trip_is_bit_identical(codec, H, W):
    x = torch.rand(2, 3, H, W, generator=torch.Generator().manual_seed(H + W)).to(DEV)
    want = codec.forward(x)["x_hat"].clamp(0, 1)
    ref = codec.decompress(**_args(codec.compress(x)))["x_hat"]
    enc = codec.compress(x, coder="interleaved")
    assert len(enc["strings"][0]) == 2 and len(enc["strings"][1]) == 2
    got = codec.decompress(enc["strings"], enc["shape"], coder="interleaved")["x_hat"]
    assert torch.equal(got, want) and torch.equal(got, ref)
    for lanes in (1, 8):
        enc = codec.compress(x, coder="interleaved", lanes=lanes)
        assert torch.equal(codec.decompress(enc["strings"], enc["shape"], coder="interleaved")["x_hat"], want)


def _args(enc):
    return {"strings": enc["strings"], "shape": enc["shape"]}


def test_image_container_round_trip(codec):
    from dcae_b200 import container
    x = torch.rand(1, 3, 300, 517, generator=torch.Generator().manual_seed(5)).to(DEV)
    blob = codec.encode_image(x, coder="interleaved")
    assert blob[:4] == b"DCI1"
    x_hat = codec.decode_image(blob, coder="interleaved")
    xp, padding = container.pad(x)
    assert torch.equal(x_hat, container.crop(codec.forward(xp)["x_hat"], padding).clamp(0, 1))
    assert torch.equal(x_hat, codec.decode_image(codec.encode_image(x)))
    with pytest.raises(ValueError):
        codec.decode_image(blob)                                  # a DCI1 container is not read as the reference's .bin


def test_corrupt_string_raises_and_the_codec_recovers(codec):
    x = torch.rand(2, 3, 256, 256, generator=torch.Generator().manual_seed(11)).to(DEV)
    enc = codec.compress(x, coder="interleaved")
    good = codec.decompress(enc["strings"], enc["shape"], coder="interleaved")["x_hat"]
    y = enc["strings"][0]
    cases = [[y[0], y[1][:-4]],                                        # truncated
             [y[0], b"\x07" + y[1][1:]],                               # bad header
             [y[0], y[1][:100] + bytes(b ^ 0x5A for b in y[1][100:140]) + y[1][140:]]]   # corrupt words
    for bad in cases:
        with pytest.raises(_lib.DcaeError, match="image 1"):
            codec.decompress([bad, enc["strings"][1]], enc["shape"], coder="interleaved")
        assert torch.equal(codec.decompress(enc["strings"], enc["shape"], coder="interleaved")["x_hat"], good)
