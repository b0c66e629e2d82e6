"""CPU checks of dcae_b200.transform_graph, the differentiable restatement of the transform stacks that the training
backward recomputes: against the reference modules' golden outputs, the restated window-attention contract and (when
staged) the reference's own modules and their fp64 gradients.  Also the argument checks of
dcae_op_window_attention_backward, which answer before any launch."""
import os
import sys

import numpy as np
import pytest
import torch

from _emul_kernels import TorchKernels
from _util import rel_err
from dcae_b200 import transform_graph
from dcae_b200.transforms import STACKS, Act, init_transform_params, pad32
from oracle.reference_loader import load_reference_dcae_module, reference_available

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, GOLDEN)
needs_ref = pytest.mark.skipif(not reference_available(), reason="reference models/dcae.py not available")
ATTN_CASES = [(8, 8, 0), (8, 8, 4), (16, 8, 4), (32, 8, 0), (32, 8, 4), (32, 4, 0), (32, 4, 2), (16, 4, 2), (8, 4, 0)]


@pytest.mark.parametrize("stack", STACKS)
def test_graph_reproduces_the_reference_golden(stack):
    """tests/golden/transforms.npz = outputs of the reference's own modules on init_transform_params(0) and
    transform_golden_input; the same bar as the emulated operator composition."""
    from make_golden_transforms import transform_golden_input
    want = torch.from_numpy(np.load(os.path.join(GOLDEN, "transforms.npz"))[stack])
    with torch.no_grad():
        got = transform_graph.stack(stack, init_transform_params(0, (stack,), prefixed=False), transform_golden_input(stack))
    assert got.shape == want.shape and rel_err(got, want) < 2e-5


@pytest.mark.parametrize("hd,window,shift", ATTN_CASES)
def test_window_attention_equals_the_restated_contract(hd, window, shift):
    heads, B, h, w = 3, 2, 3 * window, 2 * window
    C = heads * hd
    cp = pad32(C)
    g = torch.Generator().manual_seed(hd * 100 + window * 10 + shift)
    qkv = torch.zeros(B * h * w, 3 * cp)
    for j in range(3):
        qkv[:, j * cp:j * cp + C] = 1.5 * torch.randn(B * h * w, C, generator=g)
    rel = torch.randn(heads, 2 * window - 1, 2 * window - 1, generator=g)
    want = TorchKernels().window_attention(Act(qkv, B, h, w), C, cp, hd, window, shift, rel).buf[:, :C]
    x = torch.cat([qkv[:, j * cp:j * cp + C] for j in range(3)], dim=1).reshape(B, h, w, 3 * C)
    got = transform_graph.window_attention(x, hd, window, shift, rel).reshape(B * h * w, C)
    assert rel_err(got, want) < 1e-6


def test_graph_refuses_grids_the_swin_block_does_not_take():
    with pytest.raises(ValueError):
        transform_graph.stack("h_a", init_transform_params(0, ("h_a",), prefixed=False), torch.zeros(1, 320, 8, 8))


SHAPES = {"g_a": (2, 3, 64, 96), "g_s": (2, 320, 8, 12), "h_a": (2, 320, 16, 24), "h_z_s1": (2, 192, 4, 6), "h_z_s2": (1, 192, 4, 4)}


@needs_ref
@pytest.mark.parametrize("stack", STACKS)
def test_graph_and_its_fp64_gradients_equal_the_reference_modules(stack):
    ref = load_reference_dcae_module()
    torch.manual_seed(0)
    net = ref.DCAE().double()
    P = {k: v.double() for k, v in init_transform_params(1, (stack,)).items()}
    torch.nn.Module.load_state_dict(net, P, strict=False)
    mod = getattr(net, stack)
    g = torch.Generator().manual_seed(3)
    x = (torch.rand(SHAPES[stack], generator=g) if stack == "g_a" else torch.randn(SHAPES[stack], generator=g)).double()
    xr, xg = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
    want = mod(xr)
    params = {k: v.detach().clone().requires_grad_(True) for k, v in mod.state_dict().items()}
    got = transform_graph.stack(stack, params, xg)
    assert rel_err(got.detach(), want.detach()) < 1e-12
    cot = torch.randn(want.shape, generator=g).double()
    names = list(params)
    gr = torch.autograd.grad(want, [xr] + [dict(mod.named_parameters())[k] for k in names], cot, allow_unused=True)
    gg = torch.autograd.grad(got, [xg] + [params[k] for k in names], cot, allow_unused=True)
    for n, a, b in zip(["x"] + names, gg, gr):
        if b is None:
            assert a is None or float(a.abs().max()) == 0.0, n
            continue
        assert float((a - b).abs().max()) <= 1e-10 * max(float(b.abs().max()), 1e-30), n


def test_backward_scratch_size_and_argument_checks():
    """dcae_window_attention_backward_scratch_bytes does not grow with the image beyond the block cap, and the backward
    answers DCAE_E_INVALID with a message, before any launch, for unsupported or inconsistent arguments."""
    import __graft_entry__ as ge
    ge.build()
    from dcae_b200 import _lib
    lib = _lib.load()
    sz = lib.dcae_window_attention_backward_scratch_bytes
    assert sz(1, 16, 16, 96, 8, 8) == 4 * 12 * 225 * 4
    assert sz(16, 128, 128, 96, 8, 8) == sz(64, 512, 512, 96, 8, 8) > 0
    assert sz(1, 16, 16, 192, 32, 4) == 16 * 6 * 49 * 4
    fake = 0x1000
    err = lambda: lib.dcae_last_error().decode()                                               # noqa: E731
    need = sz(1, 16, 16, 96, 8, 8)

    def call(ld=288, q=0, k=96, v=192, C=96, hd=8, win=8, shift=0, B=1, h=16, w=16, dout_ld=96, dq_ld=288, scratch=fake, nbytes=need, qkv=fake, dqkv=fake):
        return lib.dcae_op_window_attention_backward(qkv, ld, q, k, v, C, hd, win, shift, fake, B, h, w, fake, dout_ld, dqkv, dq_ld, fake,
                                                     scratch, nbytes, None)

    assert call(win=5) == -1 and "window" in err()
    assert call(hd=12) == -1 and "head_dim" in err()
    assert call(C=100, dout_ld=100) == -1 and "head_dim" in err()
    assert call(h=12) == -1 and "multiple of the window" in err()
    assert call(shift=3) == -1 and "shift" in err()
    assert call(ld=200) == -1 and "leading dimension" in err()
    assert call(dq_ld=200) == -1 and "leading dimension" in err()
    assert call(k=48) == -1 and "overlap" in err()
    assert call(qkv=fake + 4) == -1 and "aligned" in err()
    assert call(dqkv=fake + 8) == -1 and "aligned" in err()
    assert call(q=2, k=98, v=194, ld=292, dq_ld=292) == -1 and "multiples of 4" in err()
    assert call(nbytes=need - 4) == -1 and "scratch" in err()
    assert call(scratch=None) == -1 and "scratch" in err()
    assert call(B=0) == 0
