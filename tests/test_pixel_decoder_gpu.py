"""Pixel-decoder input assembly (weed_instance_segmentation_b200/pixel_decoder.py, csrc/input_assembly.cu) against the
reference's own code: ``Mask2FormerPixelDecoder.forward`` (M2F:1287-1385) on the same weights and features."""
import copy

import pytest
import torch

pytestmark = pytest.mark.gpu


def _rel(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30)).item()


@pytest.fixture(scope="module")
def wis():
    import weed_instance_segmentation_b200 as w
    from weed_instance_segmentation_b200 import _cabi, build
    build.build()
    _cabi.load()
    pytest.importorskip("transformers")
    return w


def _group_inputs(kind, B, C, G, h, w):
    if kind == "spread":
        return 2.0 * torch.randn(B, C, h, w, device="cuda") + 0.5
    if kind == "offset":  # every (image, group) at its own mean around 100, std 1
        mean = 100.0 + 10.0 * torch.randn(B, G, 1, 1, 1, device="cuda")
        return (mean + torch.randn(B, G, C // G, h, w, device="cuda")).view(B, C, h, w)
    return 3.0 + 1e-3 * torch.randn(B, C, h, w, device="cuda")  # near-constant groups


def _groupnorm_chain(xs, norms, go, dtype):
    """M2F:1303, :1312 in torch at `dtype`: rows, input gradients, weight and bias gradients."""
    xr = [x.detach().to(dtype).requires_grad_(True) for x in xs]
    nr = [copy.deepcopy(n).to(dtype) for n in norms]
    y = torch.cat([n(x).flatten(2).transpose(1, 2) for n, x in zip(nr, xr)], 1)
    y.backward(go.to(dtype))
    return [y.detach()], [x.grad for x in xr], [n.weight.grad for n in nr], [n.bias.grad for n in nr]


GN_SHAPES = {"pyramid": [(4, 6), (8, 12), (16, 24)], "odd": [(31, 41), (61, 81)], "tiny": [(1, 1), (3, 5), (7, 2)]}
# (shapes, inputs): 2 randn + 0.5 everywhere, then per-group offsets and near-constant groups
GN_CASES = [(k, "spread") for k in GN_SHAPES] + [(k, kind) for kind in ("offset", "near_constant") for k in GN_SHAPES]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("shapes,inputs", [(GN_SHAPES[k], kind) for k, kind in GN_CASES],
                         ids=[k if kind == "spread" else f"{k}-{kind}" for k, kind in GN_CASES])
def test_groupnorm_to_rows_matches_torch(wis, shapes, dtype, inputs):
    """GroupNorm(32, 256) + flatten/transpose/cat: values, input gradients, weight and bias gradients against float64.
    Groups whose mean is far above their spread ("offset": mean ~100, std 1; "near_constant": mean 3, std 1e-3) are
    where statistics of the form E[x^2] - mean^2 cancel. Bar: the fixed one, or twice the error of torch's float32
    GroupNorm on the same inputs where that is larger (for those two)."""
    torch.manual_seed(0)
    B, C, G = 3, 256, 32
    xs = [_group_inputs(inputs, B, C, G, h, w).to(dtype) for h, w in shapes]
    norms = [torch.nn.GroupNorm(G, C).cuda() for _ in shapes]
    for n in norms:
        torch.nn.init.normal_(n.weight, 1.0, 0.3)
        torch.nn.init.normal_(n.bias, 0.0, 0.3)
    go = torch.randn(B, sum(h * w for h, w in shapes), C, device="cuda")
    want = _groupnorm_chain(xs, norms, go, torch.float64)
    torch32 = _groupnorm_chain(xs, norms, go, torch.float32)
    got_x = [x.detach().requires_grad_(True) for x in xs]
    got = wis.groupnorm_to_rows(got_x, norms)
    got.backward(go)
    assert got.dtype == torch.float32 and got.shape == want[0][0].shape
    got = [got.detach()], [x.grad for x in got_x], [n.weight.grad for n in norms], [n.bias.grad for n in norms]
    bars = (2e-5, 2e-5 if dtype == torch.float32 else 1e-2, 2e-5, 2e-5)  # bf16: the input gradient is rounded to bf16
    for name, gs, ts, ws, bar in zip(("y", "grad_x", "grad_gamma", "grad_beta"), got, torch32, want, bars):
        for a, t, w in zip(gs, ts, ws):
            limit = bar if inputs == "spread" else max(bar, 2 * _rel(t, w))
            assert _rel(a, w) <= limit, f"{name}: rel err {_rel(a, w):.3e} > {limit:.3e}"


@pytest.mark.parametrize("size", [(128, 160), (97, 130)])
def test_pixel_decoder_forward_and_gradients_match_reference(wis, size):
    """The whole pixel decoder (assembly + encoder + FPN tail) of a small model: outputs and every parameter gradient of
    the stock module vs the module with ``convert_pixel_decoder_inputs`` (encoder layers left stock in both)."""
    from weed_instance_segmentation_b200 import train
    model = train.build_model("swin_tiny_test", num_labels=3, seed=0, decoder_layers=2, num_queries=10).cuda()
    model.eval()  # the Swin backbone's stochastic depth would make two calls differ; gradients flow in eval mode too
    ref = model.model.pixel_level_module
    new = copy.deepcopy(ref)
    assert wis.convert_pixel_decoder_inputs(new) == 1
    torch.manual_seed(3)
    pixel_values = torch.randn(2, 3, *size, device="cuda")
    outs = []
    for m in (ref, new):
        m.zero_grad(set_to_none=True)
        o = m(pixel_values)
        feats = (o.decoder_last_hidden_state,) + tuple(o.decoder_hidden_states)
        loss = sum((f.float() ** 2).mean() for f in feats)
        loss.backward()
        outs.append((feats, {k: p.grad for k, p in m.named_parameters() if p.grad is not None}))
    for a, b in zip(outs[1][0], outs[0][0]):
        assert a.shape == b.shape and _rel(a, b) <= 1e-3  # six encoder layers and TF32 convolutions downstream of the assembly
    assert outs[0][1].keys() == outs[1][1].keys()
    for k in outs[0][1]:
        a, b = outs[1][1][k].float(), outs[0][1][k].float()
        # (the attention key biases have a mathematically zero gradient -- softmax shift invariance -- hence the floor)
        assert (a - b).abs().max().item() <= 1e-2 * b.abs().max().item() + 1e-7, k
    # second call: the cached constants are reused and give the same result
    o2 = new(pixel_values)
    assert torch.equal(o2.decoder_last_hidden_state, outs[1][0][0])
