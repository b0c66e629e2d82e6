"""Training through the transform stacks: the window-attention backward kernel against fp64 autograd of the torch
restatement, its determinism, and the autograd node of each stack (`TransformModel`, `accelerate_transforms`) against
fp64 autograd of `transform_graph` -- gradient parity 1e-4 per tensor (max |a - b| / max |b|), the config #4 bar."""
import contextlib
import os
import sys

import pytest
import torch

from _util import rel_err
from dcae_b200 import _lib, transform_graph
from dcae_b200.transforms import STACKS, TransformStack, init_transform_params, pad32
from oracle.reference_loader import reference_available

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
DEV = "cuda:0"
GRAD_TOL = 1e-4
ATTN_CASES = [(8, 8, 0), (8, 8, 4), (16, 8, 4), (32, 8, 0), (32, 8, 4), (32, 4, 0), (32, 4, 2), (16, 4, 2), (8, 4, 0)]
SENTINEL = 7.0


@pytest.fixture(autouse=True)
def fp32_torch():
    """The torch sides (recompute and references) in true fp32: TF32 off for cuBLAS and cuDNN, restored afterwards."""
    saved = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved


def _attn_case(hd, window, B, seed, heads=3):
    """qkv [T, 3 cp + 4] with q / k / v in the column windows 0 / cp / 2 cp (padding and a tail column around them),
    rel_bias and an output cotangent; grid 3 x 2 windows: SW layers mask the last window row and column."""
    h, w = 3 * window, 2 * window
    C = heads * hd
    cp = pad32(C)
    g = torch.Generator().manual_seed(seed)
    qkv = torch.zeros(B * h * w, 3 * cp + 4)
    for j in range(3):
        qkv[:, j * cp:j * cp + C] = 1.5 * torch.randn(B * h * w, C, generator=g)
    rel = torch.randn(heads, 2 * window - 1, 2 * window - 1, generator=g)
    dout = torch.randn(B * h * w, C, generator=g)
    return qkv, rel, dout, (B, h, w, C, cp)


def _kernel_backward(qkv, rel, dout, dims, hd, window, shift):
    B, h, w, C, cp = dims
    lib = _lib.load()
    qkv, rel, dout = qkv.to(DEV).contiguous(), rel.to(DEV).contiguous(), dout.to(DEV).contiguous()
    dqkv = torch.full_like(qkv, SENTINEL)
    drel = torch.full_like(rel, SENTINEL)
    n = int(lib.dcae_window_attention_backward_scratch_bytes(B, h, w, C, hd, window))
    scratch = torch.empty(n, dtype=torch.uint8, device=DEV)
    _lib.check(lib.dcae_op_window_attention_backward(qkv.data_ptr(), qkv.shape[1], 0, cp, 2 * cp, C, hd, window, shift, rel.data_ptr(), B, h, w,
                                                     dout.data_ptr(), C, dqkv.data_ptr(), dqkv.shape[1], drel.data_ptr(), scratch.data_ptr(), n,
                                                     _lib.current_stream(torch.device(DEV))), "dcae_op_window_attention_backward")
    return dqkv.cpu(), drel.cpu()


@pytest.mark.parametrize("hd,window,shift", ATTN_CASES)
def test_window_attention_backward_against_fp64_autograd(hd, window, shift):
    qkv, rel, dout, dims = _attn_case(hd, window, 2, hd * 100 + window * 10 + shift)
    B, h, w, C, cp = dims
    x = torch.cat([qkv[:, j * cp:j * cp + C] for j in range(3)], dim=1).reshape(B, h, w, 3 * C).double().requires_grad_(True)
    r = rel.double().requires_grad_(True)
    out = transform_graph.window_attention(x, hd, window, shift, r)
    gx, gr = torch.autograd.grad(out, [x, r], dout.double().reshape(B, h, w, C))
    gx = gx.reshape(B * h * w, 3 * C)
    dqkv, drel = _kernel_backward(qkv, rel, dout, dims, hd, window, shift)
    errs = {name: rel_err(dqkv[:, j * cp:j * cp + C], gx[:, j * C:(j + 1) * C]) for j, name in enumerate(("dq", "dk", "dv"))}
    errs["drel"] = rel_err(drel, gr)
    print(f"\nwindow {window} head_dim {hd} shift {shift}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    assert max(errs.values()) <= 1e-5, errs
    outside = torch.ones(dqkv.shape[1], dtype=torch.bool)
    for j in range(3):
        outside[j * cp:j * cp + C] = False
    assert bool((dqkv[:, outside] == SENTINEL).all())          # columns outside the q / k / v windows are untouched


@pytest.mark.parametrize("hd,window,shift", [(16, 8, 4), (32, 4, 2)])
def test_window_attention_backward_is_deterministic_and_batch_invariant(hd, window, shift):
    qkv, rel, dout, dims = _attn_case(hd, window, 3, 5)
    B, h, w, C, cp = dims
    a = _kernel_backward(qkv, rel, dout, dims, hd, window, shift)
    b = _kernel_backward(qkv, rel, dout, dims, hd, window, shift)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    T = h * w
    one = _kernel_backward(qkv[T:2 * T], rel, dout[T:2 * T], (1, h, w, C, cp), hd, window, shift)
    assert torch.equal(one[0], a[0][T:2 * T])                   # image 1 alone: the same bits as inside B = 3


def test_window_attention_function_matches_the_torch_form():
    """WindowAttentionFunction (the recompute's attention core) forward and backward against torch autograd in fp64."""
    from dcae_b200.training import WindowAttentionFunction
    g = torch.Generator().manual_seed(2)
    x = torch.randn(2, 16, 24, 3 * 144, generator=g)
    rel = torch.randn(9, 15, 15, generator=g)
    cot = torch.randn(2, 16, 24, 144, generator=g)
    xd, rd = x.to(DEV).requires_grad_(True), rel.to(DEV).requires_grad_(True)
    out = WindowAttentionFunction.apply(xd, 16, 8, 4, rd)
    got = torch.autograd.grad(out, [xd, rd], cot.to(DEV))
    x64, r64 = x.double().requires_grad_(True), rel.double().requires_grad_(True)
    ref = transform_graph.window_attention(x64, 16, 8, 4, r64)
    want = torch.autograd.grad(ref, [x64, r64], cot.double())
    assert rel_err(out.detach().cpu(), ref.detach()) < 2e-6
    assert rel_err(got[0].cpu(), want[0]) < 1e-5 and rel_err(got[1].cpu(), want[1]) < 1e-5


def _input(stack, shape, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(shape, generator=g) if stack == "g_a" else torch.randn(shape, generator=g)


def _compare_grads(names, got, want):
    """Per-tensor relative errors; gradients that are zero in exact arithmetic (the k third of embedding_layer.bias:
    softmax ignores a shift common to all keys) are held against a floor of 1e-6 of the largest parameter gradient."""
    floor = 1e-6 * max(float(b.abs().max()) for n, b in zip(names, want) if n != "x")
    errs = {}
    for n, a, b in zip(names, got, want):
        errs[n] = float((a.double() - b.double()).abs().max()) / max(float(b.abs().max()), floor)
    return errs


GOLDEN_B2 = {"g_a": (2, 3, 128, 128), "g_s": (2, 320, 8, 8), "h_a": (2, 320, 16, 16), "h_z_s1": (2, 192, 4, 4), "h_z_s2": (2, 192, 4, 4)}


@contextlib.contextmanager
def _relu_branches(rec):
    """Record which branch every F.relu call takes (input > 0), in call order, while the block runs."""
    orig = torch.nn.functional.relu

    def relu(t, *args, **kwargs):
        rec.append(t.detach() > 0)
        return orig(t, *args, **kwargs)
    torch.nn.functional.relu = relu
    try:
        yield
    finally:
        torch.nn.functional.relu = orig


def _branch_flips(a, b):
    """Number of ReLU inputs on opposite sides of zero in two passes over the same graph."""
    assert len(a) == len(b) and len(a) > 0, (len(a), len(b))
    return sum(int((x != y.to(x.device)).sum()) for x, y in zip(a, b))


# ReLU's gradient jumps at 0: where a pre-activation within rounding of 0 lands on the other side in the two passes, the
# gradients differ by that position's whole term (one such input in 3.6 M moves a 3x3 weight gradient of g_s by 2e-2).
# Gradient parity is defined on inputs where both passes take the same branches -- checked, next seed otherwise (the
# quantisation flips of tests/test_gpu_training.py are handled the same way).
SEEDS = range(11, 27)


@pytest.mark.parametrize("stack,shape", list(GOLDEN_B2.items()) + [("g_a", (2, 3, 128, 192))])
def test_transform_model_gradients_against_fp64_autograd(stack, shape):
    from dcae_b200.training import TransformModel
    params = init_transform_params(0, (stack,))
    model = TransformModel(stack, params, device=DEV)
    P64 = {k[len(stack) + 1:]: v.to(DEV, torch.float64).requires_grad_(True) for k, v in params.items()}
    for seed in SEEDS:
        x = _input(stack, shape, seed)
        xd = x.to(DEV).requires_grad_(True)
        r32, r64 = [], []
        with _relu_branches(r32):
            y = model(xd)
            cot = torch.randn(y.shape, generator=torch.Generator().manual_seed(seed + 100)).to(DEV)
            got = torch.autograd.grad(y, [xd] + list(model.plist), cot)          # the backward recomputes the graph here
        x64 = x.to(DEV, torch.float64).requires_grad_(True)
        with _relu_branches(r64):
            y64 = transform_graph.stack(stack, P64, x64)
        flips = _branch_flips(r32, r64)
        print(f"\n{stack} seed {seed}: {flips} ReLU inputs take the other branch in the fp32 recompute than in fp64", end="")
        if flips == 0:
            break
    else:
        pytest.fail("no input with identical ReLU branches found")
    want = torch.autograd.grad(y64, [x64] + [P64[k[len(stack) + 1:]] for k in model.keys], cot.double())
    assert rel_err(y.detach(), y64.detach()) < 5e-5
    errs = _compare_grads(["x"] + model.keys, got, want)
    worst = max(errs, key=errs.get)
    print(f"\n{stack} {tuple(shape)}: {len(errs)} gradients (input + {len(model.keys)} parameters), worst per-tensor rel err "
          f"{errs[worst]:.2e} ({worst})")
    assert errs[worst] < GRAD_TOL


def test_transform_model_weights_follow_the_parameters():
    from dcae_b200.training import TransformModel
    params = init_transform_params(0, ("h_a",))
    model = TransformModel("h_a", params, device=DEV).eval()
    x = _input("h_a", (2, 320, 16, 16), 3).to(DEV)
    with torch.no_grad():
        before = model(x)
    assert torch.equal(before, TransformStack("h_a", params, device=DEV).forward(x))
    model.train()
    y = model(x)
    (y * torch.randn_like(y)).sum().backward()
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    opt.step()
    with torch.no_grad():
        after = model.eval()(x)
    assert float((after - before).abs().max()) > 1e-4
    assert torch.equal(after, TransformStack("h_a", model.reference_state_dict(), device=DEV).forward(x))


class _StandIn(torch.nn.Module):
    """A module tree with the state-dict keys of one reference stack; its own forward is the torch graph."""

    def __init__(self, stack, params):
        super().__init__()
        self.stack = stack
        for key, v in params.items():
            cur = self
            *path, leaf = key.split(".")
            for p in path:
                if p not in cur._modules:
                    cur.add_module(p, torch.nn.Module())
                cur = cur._modules[p]
            cur.register_parameter(leaf, torch.nn.Parameter(v.clone()))

    def forward(self, x):
        return transform_graph.stack(self.stack, dict(self.named_parameters()), x)


def _standin_net():
    net = torch.nn.Module()
    for s in STACKS:
        net.add_module(s, _StandIn(s, init_transform_params(2, (s,), prefixed=False)))
    return net


@pytest.mark.parametrize("which", ["stand-in", "reference"])
def test_accelerate_transforms_trains_through_the_modules_parameters(which, lively_params):
    """Per stack, the accelerated module and the untouched one on the same input and cotangent: gradients of the input and
    of every parameter land in the module's own parameters and agree (both sides fp32, same ReLU branches)."""
    from dcae_b200.transforms import accelerate_transforms
    if which == "reference":
        if not reference_available():
            pytest.skip("reference models/dcae.py not staged")
        from oracle.reference_loader import build_reference_net
        P = dict(lively_params)
        P.update(init_transform_params(2))
        plain, fast = build_reference_net(P).cuda().train(), build_reference_net(P).cuda().train()
    else:
        plain, fast = _standin_net().cuda(), _standin_net().cuda()
    stacks = accelerate_transforms(fast, device=DEV)
    for name in STACKS:
        mp, mf = getattr(plain, name), getattr(fast, name)
        shape = (1,) + GOLDEN_B2[name][1:]
        for seed in SEEDS:
            x = _input(name, shape, seed).to(DEV)
            xp, xf = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
            mp.zero_grad(set_to_none=True)
            mf.zero_grad(set_to_none=True)
            rp, rf = [], []
            with _relu_branches(rp):
                yp = mp(xp)
                cot = torch.randn(yp.shape, generator=torch.Generator().manual_seed(seed + 100)).to(DEV)
                yp.backward(cot)
            with _relu_branches(rf):
                yf = mf(xf)
                yf.backward(cot)
            if _branch_flips(rf, rp) == 0:
                break
        else:
            pytest.fail(f"{name}: no input with identical ReLU branches found")
        assert yf.grad_fn is not None and rel_err(yf.detach(), yp.detach()) < 5e-5
        gp = dict(mp.named_parameters())
        names = sorted(gp)
        got = [xf.grad] + [dict(mf.named_parameters())[k].grad for k in names]
        assert all(g is not None for g in got), name
        errs = _compare_grads(["x"] + names, got, [xp.grad] + [gp[k].grad for k in names])
        worst = max(errs, key=errs.get)
        print(f"\naccelerate_transforms under autograd ({which}) {name}: {len(names)} parameter gradients + input, worst per-tensor "
              f"rel err {errs[worst]:.2e} ({worst})")
        assert errs[worst] < GRAD_TOL, (name, worst)
    # calls without autograd run the packed kernels; an in-place parameter change is picked up (version counter)
    y = torch.randn(1, 320, 16, 16, generator=torch.Generator().manual_seed(23)).to(DEV)
    with torch.no_grad():
        assert torch.equal(fast.h_a(y), stacks["h_a"].forward(y))
        for p in fast.h_a.parameters():
            p.mul_(1.01)
        want = TransformStack("h_a", fast.h_a.state_dict(), device=DEV).forward(y)
        assert torch.equal(fast.h_a(y), want)
