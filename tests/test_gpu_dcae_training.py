"""Training the whole DCAE on the library: the entropy-bottleneck backward kernel (`dcae_eb_backward`) against fp64 autograd
of the oracle restatement, `EntropyBottleneckModel`, and `DCAEModel` -- whole-model gradient parity against fp64 autograd
of the same composition in torch, optimizer steps, and the trained weights in `DCAECodec`.  Gradient bar: 1e-4 per tensor
(max |a - b| / max |b|).  No staged reference source is needed."""
import contextlib
import math

import pytest
import torch
import torch.nn.functional as F

from _util import rel_err
from dcae_b200 import _lib, torch_graph, transform_graph
from dcae_b200.transforms import STACKS
from oracle import entropy_bottleneck as oeb
from oracle import gaussian_conditional as ogc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
C = 192
GRAD_TOL = 1e-4
BOUND = 1e-9
LAYOUT = [("_matrix0", 3), ("_matrix1", 9), ("_matrix2", 9), ("_matrix3", 9), ("_matrix4", 3), ("_bias0", 3), ("_bias1", 3),
          ("_bias2", 3), ("_bias3", 3), ("_bias4", 1), ("_factor0", 3), ("_factor1", 3), ("_factor2", 3), ("_factor3", 3)]


@pytest.fixture(autouse=True)
def fp32_torch():
    """The torch sides (recompute and references) in true fp32: TF32 off for cuBLAS and cuDNN, restored afterwards."""
    saved = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = saved


class LowerBound(torch.autograd.Function):
    """compressai's LowerBoundFunction: forward max(x, bound); the gradient passes where x >= bound or where it is < 0."""

    @staticmethod
    def forward(ctx, x, bound: float):
        ctx.save_for_backward(x)
        ctx.bound = bound
        return torch.clamp(x, min=bound)

    @staticmethod
    def backward(ctx, g):
        x, = ctx.saved_tensors
        return g * ((x >= ctx.bound) | (g < 0)), None


def _pack(p):
    """[C, 58] in dcae_eb_fused's layout from the oracle's parameter dict."""
    parts = [(F.softplus(p[n]) if n.startswith("_matrix") else torch.tanh(p[n]) if n.startswith("_factor") else p[n]).reshape(C, -1)
             for n, _ in LAYOUT]
    return torch.cat(parts, dim=1)


def _unpack_grad(gp, p):
    """Chain the kernel's gradient w.r.t. the packed values to the parameters (softplus' = sigmoid, tanh' = 1 - tanh^2), fp64."""
    out, col = {}, 0
    for n, k in LAYOUT:
        g = gp[:, col:col + k].double().reshape(p[n].shape)
        v = p[n].double()
        out[n] = g * torch.sigmoid(v) if n.startswith("_matrix") else g * (1 - torch.tanh(v) ** 2) if n.startswith("_factor") else g
        col += k
    return out


def _lik64(p, z, noise):
    """fp64 EntropyBottleneck likelihood of z [B, C, h, w] (oracle network, compressai LowerBound); medians detached."""
    B, _, h, w = z.shape
    med = oeb.medians(p).detach().reshape(1, C, 1, 1)
    out = z + noise if noise is not None else torch.round(z - med) + med
    lik, _, _ = oeb.likelihood(p, out.transpose(0, 1).reshape(C, 1, -1))
    return LowerBound.apply(lik, BOUND).reshape(C, B, h, w).transpose(0, 1)


def _eb_case(B, h, w, seed, p):
    """z around each channel's median at a channel-dependent spread, plus elements deep in both tails (the likelihood
    floor and LowerBound's pass rule) and at the edge of the quantiles."""
    g = torch.Generator().manual_seed(seed)
    med = oeb.medians(p).reshape(1, C, 1, 1)
    width = (p["quantiles"][:, 0, 2] - p["quantiles"][:, 0, 0]).reshape(1, C, 1, 1) / 2
    z = med + width * (0.1 + torch.rand(1, C, 1, 1, generator=g)) * torch.randn(B, C, h, w, generator=g)
    z[:, 0::5, 0, 0] = (med + 100.0 + 500.0 * torch.rand(1, C, 1, 1, generator=g))[:, 0::5, 0, 0]
    z[:, 1::5, -1, -1] = (med - 100.0 - 500.0 * torch.rand(1, C, 1, 1, generator=g))[:, 1::5, 0, 0]
    z[:, 2::5, 0, -1] = (med + 1.3 * width)[:, 2::5, 0, 0]
    z[:, 3::5, -1, 0] = (med - 1.3 * width)[:, 3::5, 0, 0]
    noise = torch.empty(B, C, h, w).uniform_(-0.5, 0.5, generator=g)
    return z, noise


def _kernel(z, noise, packed, med, grad_lik):
    lib = _lib.load()
    z, packed, med, grad_lik = (t.to(DEV, torch.float32).contiguous() for t in (z, packed, med, grad_lik))
    B, _, h, w = z.shape
    a = _lib.EbBwdArgs()
    a.z, a.params, a.medians, a.grad_lik = z.data_ptr(), packed.data_ptr(), med.data_ptr(), grad_lik.data_ptr()
    a.mode = _lib.GC_EVAL
    if noise is not None:
        noise = noise.to(DEV, torch.float32).contiguous()
        a.mode, a.noise = _lib.GC_NOISE, noise.data_ptr()
    a.B, a.C, a.HW, a.lik_bound = B, C, h * w, BOUND
    gz, gp = torch.full_like(z, 7.0), torch.full_like(packed, 7.0)
    a.grad_z, a.grad_params = gz.data_ptr(), gp.data_ptr()
    _lib.check(lib.dcae_eb_backward(a, _lib.current_stream(torch.device(DEV))), "dcae_eb_backward")
    return gz.cpu(), gp.cpu()


@pytest.fixture(scope="module")
def eb_params():
    return oeb.init_params(C, seed=5, trained_like=True)


@pytest.mark.parametrize("B,h,w", [(1, 5, 7), (3, 5, 7), (3, 4, 4)])
@pytest.mark.parametrize("noisy", [True, False])
@pytest.mark.parametrize("cot", ["random", "rate"])
def test_eb_backward_kernel_against_fp64_autograd(B, h, w, noisy, cot, eb_params):
    z, noise = _eb_case(B, h, w, 100 * B + h, eb_params)
    noise = noise if noisy else None
    p64 = {k: v.double().requires_grad_(k != "quantiles") for k, v in eb_params.items()}
    z64 = z.double().requires_grad_(True)
    lik = _lik64(p64, z64, noise.double() if noisy else None)
    if cot == "random":
        g = torch.randn(lik.shape, generator=torch.Generator().manual_seed(B + h), dtype=torch.float64)
    else:                                                          # d bpp / d lik of train.py:82-85
        g = -1.0 / (math.log(2) * lik.detach() * (B * h * w * 4096))
    names = [n for n, _ in LAYOUT]
    want = torch.autograd.grad(lik, [z64] + [p64[n] for n in names], g)
    at_floor = int((lik.detach() <= BOUND).sum())
    med = eb_params["quantiles"][:, 0, 1]
    gz, gp = _kernel(z, noise, _pack(eb_params), med, g.float())
    got = _unpack_grad(gp, eb_params)
    errs = {n: rel_err(got[n], w_) for n, w_ in zip(names, want[1:])}
    if noisy:
        errs["z"] = rel_err(gz, want[0])
    else:
        assert bool((gz == 0).all())                               # round() passes no gradient
    worst = max(errs, key=errs.get)
    print(f"\ndcae_eb_backward B={B} {h}x{w} {'noise' if noisy else 'eval'} {cot} cotangent ({at_floor} likelihoods at the floor): "
          f"worst per-tensor rel err {errs[worst]:.2e} ({worst})")
    assert at_floor > 0
    assert errs[worst] < GRAD_TOL, errs


def test_eb_backward_is_deterministic_and_batch_invariant(eb_params):
    z, noise = _eb_case(3, 5, 7, 77, eb_params)
    g = torch.randn(z.shape, generator=torch.Generator().manual_seed(4))
    packed, med = _pack(eb_params), eb_params["quantiles"][:, 0, 1]
    a = _kernel(z, noise, packed, med, g)
    b = _kernel(z, noise, packed, med, g)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    one = _kernel(z[1:2], noise[1:2], packed, med, g[1:2])
    assert torch.equal(one[0], a[0][1:2])                          # image 1 alone: the same bits as inside B = 3


def test_entropy_bottleneck_model_bits_and_gradients(eb_params):
    from dcae_b200.entropy_bottleneck import EntropyBottleneck
    from dcae_b200.training import EntropyBottleneckModel
    plain, model = EntropyBottleneck(C), EntropyBottleneckModel(C)
    for m in (plain, model):
        m.load_state_dict(eb_params, strict=False)
        m.to(DEV)
    z, noise = _eb_case(2, 6, 8, 3, eb_params)
    zd, nd = z.to(DEV), noise.to(DEV)
    with torch.no_grad():
        for training in (False, True):
            a = plain(zd, training=training, noise=nd)
            b = model(zd, training=training, noise=nd)
            assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), training
    # under autograd: the same likelihood bits, and gradients of every density parameter against the oracle in fp64
    for training in (False, True):
        model.zero_grad(set_to_none=True)
        x = zd.clone().requires_grad_(True)
        out, lik = model(x, training=training, noise=nd)
        assert torch.equal(lik.detach(), plain(zd, training=training, noise=nd)[1])
        cot = torch.randn(lik.shape, generator=torch.Generator().manual_seed(11)).to(DEV)
        (lik * cot).sum().backward()
        p64 = {k: v.double().requires_grad_(True) for k, v in eb_params.items()}
        z64 = z.double().requires_grad_(True)
        lik64 = _lik64(p64, z64, noise.double() if training else None)
        (lik64 * cot.cpu().double()).sum().backward()
        errs = {n: rel_err(dict(model.named_parameters())[n].grad.cpu(), p64[n].grad) for n, _ in LAYOUT}
        if training:
            errs["z"] = rel_err(x.grad.cpu(), z64.grad)
        else:
            assert float(x.grad.abs().max()) == 0.0
        assert model.quantiles.grad is None or float(model.quantiles.grad.abs().max()) == 0.0
        worst = max(errs, key=errs.get)
        print(f"\nEntropyBottleneckModel [{'train' if training else 'eval'}]: worst per-tensor rel err {errs[worst]:.2e} ({worst})")
        assert errs[worst] < GRAD_TOL, errs


# ---- the whole model ----------------------------------------------------------------------------------------------------

def _named_params(model):
    """(reference key, parameter) of every parameter of a DCAEModel."""
    out = []
    for s in STACKS:
        m = getattr(model, s)
        out += list(zip(m.keys, m.plist))
    out += list(zip(model.entropy.keys, model.entropy.plist))
    out += [(f"entropy_bottleneck.{n}", p) for n, p in model.entropy_bottleneck.named_parameters()]
    return out


@contextlib.contextmanager
def _relu_by_stack(rec):
    """Record, per transform stack, which branch every F.relu call takes (input > 0), in call order."""
    orig_stack, orig_relu, cur = transform_graph.stack, torch.nn.functional.relu, [None]

    def stack(name, p, x, attn=transform_graph.window_attention):
        cur[0] = name
        return orig_stack(name, p, x, attn=attn)

    def relu(t, *args, **kwargs):
        rec.setdefault(cur[0], []).append(t.detach() > 0)
        return orig_relu(t, *args, **kwargs)
    transform_graph.stack, torch.nn.functional.relu = stack, relu
    try:
        yield
    finally:
        transform_graph.stack, torch.nn.functional.relu = orig_stack, orig_relu


@contextlib.contextmanager
def _replayed_rounding(ints):
    """torch_graph.ste_round returning the recorded integers of each slice in turn, with the straight-through gradient."""
    orig, it = torch_graph.ste_round, iter(ints)
    torch_graph.ste_round = lambda t: t + (next(it) - t).detach()
    try:
        yield
    finally:
        torch_graph.ste_round = orig


def _forward64(P, x, y_noise, z_noise, z_int, y_int):
    """DCAE.forward (dcae.py:623-677) in fp64 torch: transform_graph stacks, the oracle bottleneck with LowerBound, the
    slice loop of torch_graph with an fp64 Gaussian likelihood; the rounding decisions of z and y replayed."""
    from dcae_b200.modules import HOT_PREFIXES

    def sub(pre):
        return {k[len(pre) + 1:]: v for k, v in P.items() if k.startswith(pre + ".")}
    y = transform_graph.stack("g_a", sub("g_a"), x)
    z = transform_graph.stack("h_a", sub("h_a"), y)
    ebp = sub("entropy_bottleneck")
    z_lik = _lik64(ebp, z, z_noise)
    med = ebp["quantiles"][:, 0, 1].detach().reshape(1, C, 1, 1)
    z_hat = z + (z_int + med - z).detach()
    ls, lm = transform_graph.stack("h_z_s1", sub("h_z_s1"), z_hat), transform_graph.stack("h_z_s2", sub("h_z_s2"), z_hat)
    hot = {k: v for k, v in P.items() if k.split(".")[0] in HOT_PREFIXES}
    gc = lambda ys, sc, mu, nz: ogc.lower_bound(ogc.likelihood(ys + nz, sc, mu), 1e-9)    # noqa: E731
    with _replayed_rounding(list(y_int.chunk(5, 1))):
        y_hat, mu, sc, y_lik = torch_graph.slice_loop(hot, y, ls, lm, gc, y_noise)
    x_hat = transform_graph.stack("g_s", sub("g_s"), y_hat)
    return {"x_hat": x_hat, "likelihoods": {"y": y_lik, "z": z_lik}, "para": {"means": mu, "scales": sc, "y": y}}


def _flips(a, b):
    assert set(a) == set(b) and len(a) > 0, (sorted(a), sorted(b))
    total = 0
    for name in a:
        assert len(a[name]) == len(b[name]) > 0, name
        total += sum(int((u != v.to(u.device)).sum()) for u, v in zip(a[name], b[name]))
    return total


def test_dcae_model_gradients_against_fp64_autograd():
    """One training-mode pass of DCAEModel against fp64 autograd of the same composition in torch: same noise, and each
    side differentiates dcae_rate_distortion_loss of its own forward pass.  The rate term's gradient is -(1 / lik) dlik/dθ
    = -d log(lik)/dθ; evaluated at one forward point the likelihood's own fp32 error cancels in it (driving the fp32
    backward by cotangents 1 / lik taken from the fp64 pass would not cancel it, and in a tail that is most of the error)."""
    from dcae_b200.training import DCAEModel, dcae_rate_distortion_loss
    model = DCAEModel(device=DEV, seed=0).train()
    named = _named_params(model)
    keys = [k for k, _ in named]
    B = 1
    for seed in range(11, 27):
        gen = torch.Generator().manual_seed(seed)
        x = torch.rand(B, 3, 256, 256, generator=gen)
        y_noise = torch.empty(B, 320, 16, 16).uniform_(-0.5, 0.5, generator=gen).to(DEV)
        z_noise = torch.empty(B, C, 4, 4).uniform_(-0.5, 0.5, generator=gen).to(DEV)
        x32 = x.to(DEV).requires_grad_(True)
        out = model(x32, y_noise=y_noise, z_noise=z_noise)
        with torch.no_grad():                                       # the fp32 pass's rounding decisions
            z32 = model.h_a(out["para"]["y"])
            med = model.entropy_bottleneck.quantiles[:, 0, 1].reshape(1, C, 1, 1)
            z_int = torch.round(z32 - med).double()
            y_int = torch.round(out["para"]["y"] - out["para"]["means"]).double()
        loss32, _, _ = dcae_rate_distortion_loss(out, x32.detach())
        r32, r64 = {}, {}
        with _relu_by_stack(r32):                                   # the backward recomputes the stacks here
            got = torch.autograd.grad(loss32, [x32] + [p for _, p in named], allow_unused=True)
        P = {k: p.detach().double().requires_grad_(True) for k, p in named}
        x64 = x.to(DEV, torch.float64).requires_grad_(True)
        with _relu_by_stack(r64):
            out64 = _forward64(P, x64, y_noise.double(), z_noise.double(), z_int, y_int)
        flips = _flips(r32, r64)
        print(f"\nseed {seed}: {flips} ReLU inputs take the other branch in the fp32 recompute than in fp64", end="")
        if flips == 0:
            break
    else:
        pytest.fail("no input with identical ReLU branches found")
    loss64, _, _ = dcae_rate_distortion_loss(out64, x64.detach())
    want = torch.autograd.grad(loss64, [x64] + [P[k] for k in keys], allow_unused=True)
    print(f"\nloss fp32 {float(loss32.detach()):.6f} fp64 {float(loss64.detach()):.6f}")
    assert abs(float(loss32.detach()) - float(loss64.detach())) <= 1e-4 * abs(float(loss64.detach()))
    # quantiles: no gradient from the main loss (the medians are detached)
    q = keys.index("entropy_bottleneck.quantiles")
    assert want[1 + q] is None and (got[1 + q] is None or float(got[1 + q].abs().max()) == 0.0)
    floor = 1e-6 * max(float(w.abs().max()) for w in want[1:] if w is not None)
    errs = {"x": rel_err(got[0], want[0])}
    for k, a, b in zip(keys, got[1:], want[1:]):
        if b is None:
            continue
        assert a is not None, k
        if k.endswith(".k.bias"):              # zero in exact arithmetic (softmax ignores a shift common to all keys)
            assert float(a.abs().max()) < 1e3 * floor and float(b.abs().max()) < 1e3 * floor, k
            continue
        errs[k] = float((a.double() - b).abs().max()) / max(float(b.abs().max()), floor)
    worst = max(errs, key=errs.get)
    print(f"DCAEModel vs fp64 autograd: {len(errs) - 1} parameter tensors + input, worst per-tensor rel err {errs[worst]:.2e} ({worst})")
    eb = [k for k in errs if k.startswith("entropy_bottleneck.")]
    print("entropy bottleneck: " + ", ".join(f"{k[19:]} {errs[k]:.1e}" for k in eb))
    assert len(eb) == 14
    assert errs[worst] < GRAD_TOL, (worst, errs[worst])


def test_dcae_model_trains_and_the_codec_follows():
    from dcae_b200.codec import DCAECodec
    from dcae_b200.entropy_bottleneck import EntropyBottleneck
    from dcae_b200.gaussian_conditional import GaussianConditional
    from dcae_b200.params import entropy_param_shapes
    from dcae_b200.training import DCAEModel, dcae_rate_distortion_loss
    from dcae_b200.transforms import transform_param_shapes
    model = DCAEModel(device=DEV, seed=1).train()
    gen = torch.Generator().manual_seed(3)
    x = torch.rand(2, 3, 256, 256, generator=gen).to(DEV)
    y_noise = torch.empty(2, 320, 16, 16).uniform_(-0.5, 0.5, generator=gen).to(DEV)
    z_noise = torch.empty(2, C, 4, 4).uniform_(-0.5, 0.5, generator=gen).to(DEV)
    main, aux = model.parameter_groups()
    assert len(aux) == 1 and aux[0] is model.entropy_bottleneck.quantiles
    assert len(main) + len(aux) == len(list(model.parameters()))
    opt, aux_opt = torch.optim.Adam(main, lr=1e-4), torch.optim.Adam(aux, lr=1e-3)
    losses, aux_losses = [], []
    for _ in range(5):                                        # train.py:165-179
        opt.zero_grad()
        aux_opt.zero_grad()
        loss, bpp, mse = dcae_rate_distortion_loss(model(x, y_noise=y_noise, z_noise=z_noise), x)
        loss.backward()
        opt.step()
        a = model.aux_loss()
        a.backward()
        aux_opt.step()
        losses.append(float(loss.detach()))
        aux_losses.append(float(a.detach()))
    with torch.no_grad():
        losses.append(float(dcae_rate_distortion_loss(model(x, y_noise=y_noise, z_noise=z_noise), x)[0]))
        aux_losses.append(float(model.aux_loss()))
    print(f"\nrate-distortion loss {' '.join(f'{v:.4f}' for v in losses)}; aux loss {' '.join(f'{v:.2f}' for v in aux_losses)}")
    assert losses[-1] < losses[0] and aux_losses[-1] < aux_losses[0]
    # the trained weights: DCAEModel in eval() equals DCAECodec built from reference_state_dict(), bit for bit
    sd = model.reference_state_dict()
    want_keys = {f"{s}.{k}" for s in STACKS for k in transform_param_shapes(s)} | set(entropy_param_shapes())
    want_keys |= {f"entropy_bottleneck.{k}" for k in EntropyBottleneck(C).state_dict()}
    want_keys |= {f"gaussian_conditional.{k}" for k in GaussianConditional(None).state_dict()}
    assert set(sd) == want_keys
    model.eval()
    codec = DCAECodec(sd, device=DEV)
    with torch.no_grad():
        a = model(x)
        b = codec.forward(x)
        c = DCAEModel(sd, device=DEV).eval()(x)
    for got in (a, c):
        assert torch.equal(got["x_hat"], b["x_hat"])
        for k in ("y", "z"):
            assert torch.equal(got["likelihoods"][k], b["likelihoods"][k]), k
        for k in ("means", "scales", "y"):
            assert torch.equal(got["para"][k], b["para"][k]), k
    # compress -> decompress and the image container with the trained weights
    codec.update()
    enc = codec.compress(x)
    dec = codec.decompress(enc["strings"], enc["shape"])
    diff = float((dec["x_hat"] - b["x_hat"].clamp(0, 1)).abs().max())
    blob = codec.encode_image(x[:1])
    img = codec.decode_image(blob)
    diff_img = float((img - b["x_hat"][:1].clamp(0, 1)).abs().max())
    print(f"compress -> decompress vs forward x_hat: {diff:.2e}; encode_image -> decode_image: {diff_img:.2e} ({len(blob)} bytes)")
    assert diff < 1e-5 and diff_img < 1e-5 and img.shape == x[:1].shape
