"""CPU: pin the oracle against the reference's own code (the tests marked `needs_ref` skip where the reference's
models/dcae.py is not available), and the index search against torch.searchsorted."""
import pytest
import torch

from _reference_loader import reference_available, load_reference_dcae_module
from _util import rel_err
from dcae_b200 import params as P
from oracle import entropy_model as om
from oracle import gaussian_conditional as gc

needs_ref = pytest.mark.skipif(not reference_available(), reason="reference models/dcae.py not available")


@needs_ref
def test_scale_table_and_ste_round_match_reference():
    ref = load_reference_dcae_module()
    assert torch.equal(ref.get_scale_table(), gc.get_scale_table())
    x = torch.randn(1000) * 3
    assert torch.equal(ref.ste_round(x), gc.ste_round(x))


@needs_ref
def test_likelihood_bit_exact_vs_in_tree_copy():
    """dcae.py:839-857 is the reference's in-tree copy of compressai's _likelihood."""
    ref = load_reference_dcae_module()
    g = torch.Generator().manual_seed(4321)
    y = 4 * torch.randn(2, 64, 16, 16, generator=g)
    mu = 2 * torch.randn(2, 64, 16, 16, generator=g)
    scale = torch.exp(torch.empty(2, 64, 16, 16).uniform_(-3.0, 5.7, generator=g))
    out = gc.quantize(y, "dequantize", mu)
    class _Self:   # _likelihood only needs self._standardized_cumulative
        _standardized_cumulative = lambda self, x: ref.DCAE._standardized_cumulative(self, x)
    want = ref.DCAE._likelihood(_Self(), out, scale, mu)
    got = gc.likelihood(out, scale, mu)
    assert torch.equal(want, got)


def test_build_indexes_equals_searchsorted():
    table = gc.get_scale_table()
    g = torch.Generator().manual_seed(1)
    s = torch.exp(torch.empty(100000).uniform_(-3.0, 5.7, generator=g))
    s = torch.cat([s, table, torch.nextafter(table, torch.tensor(0.0)), torch.nextafter(table, torch.tensor(1e9)),
                   torch.tensor([-1.0, 0.0, 0.11, 1e4, float("inf")])])
    idx = gc.build_indexes(s, table)
    want = torch.searchsorted(table[:-1].contiguous(), s.clamp_min(0.11), right=False).int()
    assert torch.equal(idx, want)


@needs_ref
@pytest.mark.parametrize("i", [0, 3])
def test_dictionary_cross_attention_vs_reference_module(i, lively_params):
    ref = load_reference_dcae_module()
    m = ref.MutiScaleDictionaryCrossAttentionGLU(input_dim=P.cq(i), output_dim=320, head_num=20)
    sd = {k[len(f"dt_cross_attention.{i}."):]: v for k, v in lively_params.items()
          if k.startswith(f"dt_cross_attention.{i}.")}
    m.load_state_dict(sd)
    m.eval()
    g = torch.Generator().manual_seed(5)
    x = torch.randn(2, P.cq(i), 5, 7, generator=g)
    dt = lively_params["dt"]
    with torch.no_grad():
        want = m(x, dt.repeat([2, 1, 1]))
        got = om.dictionary_cross_attention(x, dt, sd)
    assert rel_err(got, want) < 2e-6


@needs_ref
def test_conv_stack_vs_reference_sequential(lively_params):
    ref = load_reference_dcae_module()
    i = 2
    seq = torch.nn.Sequential(ref.conv(P.cs(i), 224, stride=1, kernel_size=3), torch.nn.GELU(),
                              ref.conv(224, 128, stride=1, kernel_size=3), torch.nn.GELU(),
                              ref.conv(128, 64, stride=1, kernel_size=3))
    sd = {k[len(f"cc_scale_transforms.{i}."):]: v for k, v in lively_params.items()
          if k.startswith(f"cc_scale_transforms.{i}.")}
    seq.load_state_dict(sd)
    x = torch.randn(1, P.cs(i), 6, 5)
    with torch.no_grad():
        assert rel_err(om.conv_stack(x, sd), seq(x)) < 1e-6


@needs_ref
def test_param_spec_covers_reference_hot_path_keys():
    ref = load_reference_dcae_module()
    net = ref.DCAE()
    hot = ("dt", "dt_cross_attention", "cc_mean_transforms", "cc_scale_transforms", "lrp_transforms")
    want = {k: tuple(v.shape) for k, v in net.state_dict().items() if k.split(".")[0] in hot}
    got = dict(P.entropy_param_shapes())
    assert want == got


@needs_ref
def test_accelerate_swaps_exactly_the_attributes_the_reference_loop_calls():
    """dcae_b200.modules.accelerate() replaces ModuleList entries and `gaussian_conditional` of a DCAE instance: the real
    reference class must have them with the shapes the drop-ins assume (the swap itself needs a GPU: test_gpu_modules)."""
    import inspect
    ref = load_reference_dcae_module()
    net = ref.DCAE()
    for name in ("dt_cross_attention", "cc_mean_transforms", "cc_scale_transforms", "lrp_transforms"):
        ml = getattr(net, name)
        assert isinstance(ml, torch.nn.ModuleList) and len(ml) == 5, name
    assert hasattr(net, "gaussian_conditional") and tuple(net.dt.shape) == (128, 640)
    src = inspect.getsource(ref.DCAE.forward)
    for call in ("self.dt_cross_attention[slice_index](query, dt)", "self.cc_mean_transforms[slice_index](support)",
                 "self.cc_scale_transforms[slice_index](support)", "self.lrp_transforms[slice_index](lrp_support)",
                 "self.gaussian_conditional(y_slice, scale, mu)"):
        assert call in src, call
    sig = inspect.signature(type(net.dt_cross_attention[0]).forward)
    assert list(sig.parameters)[:3] == ["self", "x", "dt"]
