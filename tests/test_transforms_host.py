"""CPU checks of dcae_b200.transforms (SURVEY 8f N3 / N4): the host logic -- architecture table, weight re-indexing,
channel padding, block composition -- run over a torch restatement of the C-ABI operator contracts
(tests/_emul_kernels.py) and compared with the reference's REAL modules (`DCAE().g_a` ... of models/dcae.py, loaded by
oracle/reference_loader.py).  The CUDA kernels themselves are checked in tests/test_gpu_transforms.py."""
import pytest
import torch
import torch.nn.functional as F

from _emul_kernels import TorchKernels
from _util import rel_err
from dcae_b200 import _lib
from dcae_b200.transforms import (ARCH, STACKS, Act, TransformStack, conv_s2_to_gemm, deconv_s2_to_gemm, pad8, pad32,
                                  transform_param_shapes)
from oracle.reference_loader import load_reference_dcae_module, reference_available

needs_ref = pytest.mark.skipif(not reference_available(), reason="reference models/dcae.py not available")


def lively_transform_net(seed=3):
    """`DCAE()` of the reference with the parameters the default init leaves at trivial values (Scale = 1, relative
    position bias ~ 0.02, LayerNorm affine = identity) randomised, so that every term of the blocks is exercised."""
    ref = load_reference_dcae_module()
    torch.manual_seed(seed)
    net = ref.DCAE().eval()
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for name, p in net.named_parameters():
            if name.split(".")[0] not in STACKS:
                continue
            if name.endswith("res_scale_1.scale") or name.endswith("res_scale_2.scale"):
                p.copy_(0.5 + torch.rand(p.shape, generator=g))
            elif name.endswith("relative_position_params"):
                p.copy_(0.5 * torch.randn(p.shape, generator=g))
            elif ".ln1." in name or ".ln2." in name:
                p.add_(0.2 * torch.randn(p.shape, generator=g))
            elif name.endswith("bias"):
                p.add_(0.1 * torch.randn(p.shape, generator=g))
    return net


@pytest.fixture(scope="module")
def ref_net():
    return lively_transform_net()


@needs_ref
@pytest.mark.parametrize("stack", STACKS)
def test_param_table_matches_the_reference_state_dict(ref_net, stack):
    want = {k: tuple(v.shape) for k, v in getattr(ref_net, stack).state_dict().items()}
    assert transform_param_shapes(stack) == want


@pytest.mark.parametrize("k", [3, 5])
@pytest.mark.parametrize("hw", [(8, 12), (7, 9)])
def test_stride2_conv_is_a_3x3_conv_over_space_to_depth(k, hw):
    g = torch.Generator().manual_seed(k)
    cin, cout = 6, 16
    w, b = torch.randn(cout, cin, k, k, generator=g), torch.randn(cout, generator=g)
    x = torch.randn(2, cin, *hw, generator=g)
    want = F.conv2d(x, w, b, stride=2, padding=k // 2)
    K = TorchKernels()
    cs = pad8(cin)
    pg = K.pack_gemm(conv_s2_to_gemm(w, pad32(cout), cs), b, taps=9)
    a = K.gemm(K.space_to_depth(K.to_tokens(x, 8), cin, cs), pg)
    got = K.to_nchw(a, cout)
    assert got.shape == want.shape
    assert rel_err(got, want) < 1e-6
    assert float(a.buf[:, cout:].abs().max()) == 0.0          # padded output channels are exact zeros


@pytest.mark.parametrize("k", [3, 5])
def test_stride2_transposed_conv_is_a_3x3_conv_plus_depth_to_space(k):
    g = torch.Generator().manual_seed(10 + k)
    cin, cout = 32, 5
    w, b = torch.randn(cin, cout, k, k, generator=g), torch.randn(cout, generator=g)
    x = torch.randn(2, cin, 5, 7, generator=g)
    want = F.conv_transpose2d(x, w, b, stride=2, padding=k // 2, output_padding=1)
    K = TorchKernels()
    cs = pad8(cout)
    pg = K.pack_gemm(deconv_s2_to_gemm(w, cs, pad32(cin)), torch.cat([b, b.new_zeros(cs - cout)]).repeat(4), taps=9)
    a = K.depth_to_space(K.gemm(K.to_tokens(x, 32), pg), cs, cout, 8)
    got = K.to_nchw(a, cout)
    assert got.shape == want.shape
    assert rel_err(got, want) < 1e-6
    assert float(a.buf[:, cout:].abs().max()) == 0.0


SHAPES = {"g_a": (1, 3, 128, 192), "g_s": (1, 320, 8, 12), "h_a": (2, 320, 16, 24), "h_z_s1": (2, 192, 4, 6), "h_z_s2": (1, 192, 4, 4)}


@needs_ref
@pytest.mark.parametrize("stack", STACKS)
def test_stack_composition_matches_the_reference_module(ref_net, stack):
    """TransformStack over the emulated operators == the reference nn.Sequential (dcae.py:558-582), incl. SW windows,
    144 / 72 / 48-channel padding, non-square grids and B = 2."""
    mod = getattr(ref_net, stack)
    x = torch.randn(*SHAPES[stack], generator=torch.Generator().manual_seed(5))
    if stack == "g_a":
        x = torch.rand(*SHAPES[stack], generator=torch.Generator().manual_seed(5))
    with torch.no_grad():
        want = mod(x)
    ts = TransformStack(stack, mod.state_dict(), kernels=TorchKernels())
    got = ts.forward(x)
    assert got.shape == want.shape
    err = rel_err(got, want)
    print(f"\n{stack}: emulated-operator composition vs the reference module: {err:.2e}")
    assert err < 2e-5


def test_prefixed_keys_and_errors():
    from dcae_b200.transforms import init_transform_params
    sd = init_transform_params(0, ("h_a",))                       # keys prefixed "h_a." like a whole-model state dict
    ts = TransformStack("h_a", sd, kernels=TorchKernels())
    with pytest.raises(ValueError):
        ts.forward(torch.zeros(1, 3, 16, 16))
    with pytest.raises(_lib.DcaeError):
        ts.forward(torch.zeros(1, 320, 8, 8))                    # 4x4 tokens at the Swin block: not larger than the window
    bad = dict(sd)
    bad.pop("h_a.1.conv.bias")
    with pytest.raises(KeyError):
        TransformStack("h_a", bad, kernels=TorchKernels())
    with pytest.raises(ValueError):
        TransformStack("nope", sd, kernels=TorchKernels())


def test_product_has_no_cpu_backend():
    """The default backend is the CUDA library; without it the constructor raises (no silent CPU path)."""
    import dcae_b200.transforms as T
    src = open(T.__file__).read()
    assert "_emul" not in src and "oracle" not in src.replace("oracle restatement", "")
    if not torch.cuda.is_available():
        with pytest.raises(Exception):
            TransformStack("h_a", {k: torch.zeros(s) for k, s in transform_param_shapes("h_a").items()})


@pytest.mark.parametrize("stack", STACKS)
def test_golden_fixture_is_reproduced_by_the_emulated_composition(stack):
    """tests/golden/transforms.npz (outputs of the reference's own modules, generator make_golden_transforms.py) from the
    regenerated weights and inputs: pins init_transform_params / transform_golden_input on every machine."""
    import numpy as np
    import os
    sys_path_golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    import sys
    sys.path.insert(0, sys_path_golden)
    from make_golden_transforms import transform_golden_input
    from dcae_b200.transforms import init_transform_params
    want = torch.from_numpy(np.load(os.path.join(sys_path_golden, "transforms.npz"))[stack])
    ts = TransformStack(stack, init_transform_params(0, (stack,)), kernels=TorchKernels())
    got = ts.forward(transform_golden_input(stack))
    assert got.shape == want.shape and rel_err(got, want) < 2e-5


def test_large_batches_run_in_slices():
    """One call must stay below 2^32 elements per buffer (32-bit offsets in the element-wise kernels): bigger batches are cut
    into slices of independent images; the result is the same bits."""
    from dcae_b200.transforms import init_transform_params
    ts = TransformStack("h_a", init_transform_params(0, ("h_a",)), kernels=TorchKernels())
    x = torch.randn(3, 320, 16, 16, generator=torch.Generator().manual_seed(1))
    whole = ts.forward(x)
    ts._ELEMS_PER_INPUT_POSITION = dict(ts._ELEMS_PER_INPUT_POSITION, h_a=(1 << 31) / (16 * 16) / 2 + 1)      # forces slices of one image
    assert torch.equal(ts.forward(x), whole)
