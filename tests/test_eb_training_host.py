"""CPU: the entropy-bottleneck backward's C ABI (struct layout, argument checks before any launch) and the aux loss of the
trainable bottleneck (`EntropyBottleneckModel.loss`: compressai's stop_gradient) against `EntropyBottleneck.loss` and the
oracle restatement."""
import os
import subprocess
import tempfile

import pytest
import torch

from oracle import entropy_bottleneck as oeb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
C = 192


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from dcae_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module")
def params():
    return oeb.init_params(C, seed=3, trained_like=True)


def test_eb_bwd_args_layout_matches_header(lib):
    import ctypes
    from dcae_b200 import _lib
    prog = '#include <stdio.h>\n#include "dcae_b200.h"\nint main(){printf("%zu %zu\\n", sizeof(dcae_eb_bwd_args), sizeof(dcae_eb_args));return 0;}\n'
    with tempfile.TemporaryDirectory() as td:
        open(os.path.join(td, "t.c"), "w").write(prog)
        subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", os.path.join(td, "t"), os.path.join(td, "t.c")], check=True)
        sizes = [int(v) for v in subprocess.run([os.path.join(td, "t")], capture_output=True, text=True, check=True).stdout.split()]
    assert sizes == [ctypes.sizeof(_lib.EbBwdArgs), ctypes.sizeof(_lib.EbArgs)]


def test_eb_backward_rejects_bad_arguments_before_any_launch(lib):
    """Each bad argument answers -1 with a message on dcae_last_error() and launches nothing (pointers are never
    dereferenced on the host, so this runs without a GPU)."""
    from dcae_b200 import _lib
    fake = 0x1000

    def args(**kw):
        a = _lib.EbBwdArgs()
        a.z, a.noise, a.params, a.medians, a.grad_lik, a.grad_z, a.grad_params = (fake,) * 7
        a.mode, a.B, a.C, a.HW, a.lik_bound = _lib.GC_NOISE, 2, C, 35, 1e-9
        for k, v in kw.items():
            setattr(a, k, v)
        return a

    err = lambda: lib.dcae_last_error().decode()                 # noqa: E731
    before = lib.dcae_launch_count()
    for field in ("z", "params", "medians", "grad_lik"):
        assert lib.dcae_eb_backward(args(**{field: None}), None) == -1 and "null input" in err(), field
    for field in ("grad_z", "grad_params"):
        assert lib.dcae_eb_backward(args(**{field: None}), None) == -1 and "null output" in err(), field
    assert lib.dcae_eb_backward(args(noise=None), None) == -1 and "noise" in err()
    assert lib.dcae_eb_backward(args(mode=_lib.GC_DECODE), None) == -1 and "bad mode" in err()
    assert lib.dcae_eb_backward(args(mode=7), None) == -1 and "bad mode" in err()
    assert lib.dcae_eb_backward(args(mode=-1), None) == -1 and "bad mode" in err()
    for shape in ({"B": -1}, {"C": 0}, {"C": -3}, {"HW": -1}):
        assert lib.dcae_eb_backward(args(**shape), None) == -1 and "bad shape" in err(), shape
    assert lib.dcae_eb_backward(None, None) == -1
    assert lib.dcae_launch_count() == before


def _modules(params):
    from dcae_b200.entropy_bottleneck import EntropyBottleneck
    from dcae_b200.training import EntropyBottleneckModel
    mods = []
    for cls in (EntropyBottleneck, EntropyBottleneckModel):
        m = cls(C)
        missing, unexpected = m.load_state_dict(params, strict=False)
        assert not unexpected and set(missing) <= {"target", "_offset", "_quantized_cdf", "_cdf_length"}
        mods.append(m)
    return mods


def test_aux_loss_stops_the_gradient_at_the_density(params):
    """compressai's aux loss: the same value as EntropyBottleneck.loss() and the oracle's aux_loss; its gradient reaches
    `quantiles` only, and there equals autograd of the oracle."""
    plain, model = _modules(params)
    want = oeb.aux_loss(params)
    got = model.loss()
    assert torch.equal(got.detach(), plain.loss().detach())
    assert abs(float(got.detach()) - float(want)) <= 1e-6 * float(want)
    got.backward()
    for name, p in model.named_parameters():
        if name == "quantiles":
            assert p.grad is not None and float(p.grad.abs().max()) > 0
        else:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, name
    q = params["quantiles"].clone().double().requires_grad_(True)
    p64 = {k: (q if k == "quantiles" else v.double()) for k, v in params.items()}
    g64, = torch.autograd.grad(oeb.aux_loss(p64), [q])
    assert torch.equal(model.quantiles.grad.sign(), g64.float().sign())        # d|.| / d. is the sign of each term


def test_logits_cumulative_keeps_its_graph_without_the_keyword(params):
    """EntropyBottleneck.loss() (no keyword) still differentiates into every density parameter, as before."""
    plain, _ = _modules(params)
    names = [n for n, _ in plain.named_parameters()]
    grads = torch.autograd.grad(plain.loss(), list(plain.parameters()))
    p64 = {k: v.double().requires_grad_(True) for k, v in params.items()}
    want = torch.autograd.grad(oeb.aux_loss(p64), [p64[n] for n in names])
    for n, g, w in zip(names, grads, want):
        assert float((g.double() - w).abs().max()) <= 1e-4 * max(float(w.abs().max()), 1e-3), n
    assert all(float(g.abs().max()) > 0 for g in grads)
    v = torch.linspace(-5, 5, 11).reshape(1, 1, -1).repeat(C, 1, 1)
    assert torch.equal(plain._logits_cumulative(v), plain._logits_cumulative(v, stop_gradient=False))
    assert torch.equal(plain._logits_cumulative(v).detach(), plain._logits_cumulative(v, stop_gradient=True))
