"""The REAL reference class on the GPU (SURVEY 8b): `/root/reference/models/dcae.py` `DCAE` (unmodified; staged into
oracle/_ref/ by build(), loaded with import stubs for the absent third-party packages), its hot-path sub-modules
redirected by `dcae_b200.accelerate(net)`, its `forward / compress / decompress` text running as written -- against
the same class left untouched on the same device, and through the native range coder."""
import os
import tempfile

import pytest
import torch

from _util import mismatch_rate, rel_err
from oracle.reference_loader import build_reference_net, load_reference_dcae_module, reference_available

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def nets(lively_params):
    if not reference_available():
        pytest.skip("reference models/dcae.py not available")
    # the reference's evaluation flags (eval.py:3182-3187, 3904): true fp32 matmul, no cuDNN
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cudnn.enabled = False
    from dcae_b200 import accelerate
    plain = build_reference_net(lively_params).cuda()
    fast = build_reference_net(lively_params).cuda()          # same seed: identical g_a / h_a / h_z_s / g_s weights
    handle = accelerate(fast, device="cuda:0", math="f16x3")
    yield plain, fast, handle
    torch.backends.cudnn.enabled = True


def _image(seed=1234, B=1, H=256, W=256):
    return torch.rand(B, 3, H, W, generator=torch.Generator().manual_seed(seed)).cuda()


def test_accelerated_dcae_forward_matches_the_untouched_class(nets):
    """DCAE.forward (dcae.py:623-677) on BASELINE config #1 (one 256x256 image).  Everything outside the slice loop runs
    the same torch kernels in both nets, so the loop sees bit-identical (y, latent_scales, latent_means)."""
    plain, fast, handle = nets
    x = _image()
    with torch.no_grad():
        want, got = plain(x), fast(x)
    assert torch.equal(want["para"]["y"], got["para"]["y"])
    # slice 0: nothing has cascaded yet
    for k in ("means", "scales"):
        assert rel_err(got["para"][k][:, :64], want["para"][k][:, :64]) < 1e-5, k
    y, mu_w, mu_g = want["para"]["y"], want["para"]["means"], got["para"]["means"]
    flips = mismatch_rate(torch.round(y - mu_g), torch.round(y - mu_w))
    print(f"\nsymbol flips vs the untouched reference on the same GPU: {flips:.2e}; "
          f"means {rel_err(mu_g, mu_w):.2e}, scales {rel_err(got['para']['scales'], want['para']['scales']):.2e}")
    assert flips <= 5e-4
    if flips == 0.0:
        for k in ("means", "scales"):
            assert rel_err(got["para"][k], want["para"][k]) < 1e-5, k
        lw, lg = want["likelihoods"]["y"].double(), got["likelihoods"]["y"].double()
        assert abs(float(torch.log2(lg).sum() - torch.log2(lw).sum())) <= 1e-4 * abs(float(torch.log2(lw).sum()))
    assert handle.loop.last_launches > 0
    # the hot-path parameters are still the reference's, under the reference's keys
    keys = set(fast.state_dict())
    assert "dt_cross_attention.0.x_trans.weight" in keys and "cc_mean_transforms.4.4.bias" in keys and "lrp_transforms.2.0.weight" in keys


def test_compress_decompress_text_with_the_native_coder(nets):
    """DCAE.compress (dcae.py:698-761) and DCAE.decompress (:859-910) as written, with `BufferedRansEncoder` /
    `RansDecoder` = dcae_b200.ans (the reference imports them from compressai.ans): the decoder regenerates the same
    indexes from its own scales, the stream decodes, and x_hat equals the forward pass's reconstruction."""
    from dcae_b200 import ans
    _, fast, _ = nets
    ref = load_reference_dcae_module()
    saved = ref.BufferedRansEncoder, ref.RansDecoder
    ref.BufferedRansEncoder, ref.RansDecoder = ans.BufferedRansEncoder, ans.RansDecoder
    x = _image(seed=77)
    cwd = os.getcwd()
    try:
        with tempfile.TemporaryDirectory() as td, torch.no_grad():
            os.makedirs(os.path.join(td, "output", "debug"))        # compress() writes debug dumps there (dcae.py:707, 758)
            os.chdir(td)
            enc = fast.compress(x)
            y_string = enc["strings"][0][0]
            assert isinstance(y_string, bytes) and len(y_string) > 8
            dec = fast.decompress(enc["strings"], enc["shape"])
            fwd = fast(x)
    finally:
        os.chdir(cwd)
        ref.BufferedRansEncoder, ref.RansDecoder = saved
    assert dec["x_hat"].shape == x.shape
    assert float((dec["x_hat"] - fwd["x_hat"].clamp(0, 1)).abs().max()) < 1e-5
    assert 0.2 < len(y_string) * 8 / float(-torch.log2(fwd["likelihoods"]["y"].double()).sum()) < 2.0     # same order as the rate estimate


def test_weights_follow_the_module_parameters(nets):
    """`load_state_dict` / an optimizer step change the reference modules' parameters in place; the packed device weights
    follow (tensor version counters), no new accelerate() call needed."""
    _, fast, handle = nets
    x = _image(seed=5)
    with torch.no_grad():
        before = fast(x)["para"]["means"][:, :64].clone()
        fast.cc_mean_transforms[0][4].bias.add_(1.0)
        after = fast(x)["para"]["means"][:, :64]
        assert float((after - before - 1.0).abs().max()) < 1e-4
        sd = {k: v.clone() for k, v in fast.state_dict().items()}
        sd["cc_mean_transforms.0.4.bias"] -= 1.0
        fast.load_state_dict(sd)
        again = fast(x)["para"]["means"][:, :64]
    assert torch.equal(again, before)


def test_a_different_dictionary_is_refused(nets):
    _, fast, handle = nets
    x = torch.randn(1, 640, 4, 4).cuda()
    with torch.no_grad():
        fast.dt_cross_attention[0](x, fast.dt.repeat([1, 1, 1]))
        handle.loop._dt_checked = False
        with pytest.raises(ValueError):
            fast.dt_cross_attention[0](x, fast.dt.repeat([1, 1, 1]) + 1.0)
    out = fast.dt_cross_attention[0](x.requires_grad_(), None)       # under autograd: a recompute node, never silent zero gradients
    assert out.grad_fn is not None


def test_f16_range_check(lively_params):
    """The range check of the slice loop accelerate() builds (same weights, one lane)."""
    from dcae_b200.entropy_model import EntropySliceLoop
    loop = EntropySliceLoop(lively_params, device="cuda:0", math="f16x3", lanes=1)
    gen = torch.Generator().manual_seed(3)
    y = (4 * torch.randn(1, 320, 8, 12, generator=gen)).cuda()
    ls, lm = torch.randn(1, 320, 8, 12, generator=gen).cuda(), torch.randn(1, 320, 8, 12, generator=gen).cuda()
    assert loop.check_f16_range(y, ls, lm) == 0
    from dcae_b200 import _lib
    with pytest.raises(_lib.DcaeError):
        loop.check_f16_range(y, ls * 1e6, lm)                         # latents beyond the fp16 range: counted, not ignored
