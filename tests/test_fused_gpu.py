"""Fused-prologue operator (softmax + ref + off/(W,H) inside the kernels) against the reference chain.

Reference chain = the module code M2F:955-971 in torch followed by the reference op (M2F:798-837) through the
CPU oracle wrapper (`oracle.hf_reference`), differentiated by autograd in fp64 on the CPU.
"""
import numpy as np
import pytest
import torch

from conftest import rel_err

pytestmark = pytest.mark.gpu


def _inputs(B, shapes, H, D, P, Q, seed, dist="init"):
    from weed_instance_segmentation_b200 import synth
    L = len(shapes)
    S = sum(h * w for h, w in shapes)
    Q = S if Q is None else Q
    g = torch.Generator().manual_seed(seed)
    value = torch.randn(B, S, H, D, generator=g)
    if Q == S:
        ref = synth.reference_points(shapes)[None].expand(B, -1, -1, -1).contiguous()
    else:
        ref = torch.rand(B, Q, 1, 2, generator=g).expand(-1, -1, L, -1).contiguous()
    if dist == "init":
        off = synth.init_offsets(H, L, P)[None, None] + 0.5 * torch.randn(B, Q, H, L, P, 2, generator=g)
    else:
        off = 3.0 * torch.randn(B, Q, H, L, P, 2, generator=g)
    logits = 2.0 * torch.randn(B, Q, H, L * P, generator=g)
    go = torch.randn(B, Q, H * D, generator=g)
    return value, off.contiguous(), logits, ref, go


def _reference_chain(value, off, logits, ref, go, shapes, dtype=torch.float64):
    """M2F:955-971 + M2F:798-837 in torch on the CPU, autograd gradients."""
    from oracle.hf_reference import hf_forward_torch
    B, Q, H, L, P, _ = off.shape
    v = value.to(dtype).requires_grad_(True)
    o = off.to(dtype).requires_grad_(True)
    lg = logits.to(dtype).requires_grad_(True)
    attn = torch.softmax(lg, -1).view(B, Q, H, L, P)
    normalizer = torch.tensor([[w, h] for h, w in shapes], dtype=dtype)
    loc = ref.to(dtype)[:, :, None, :, None, :] + o / normalizer[None, None, None, :, None, :]
    out = hf_forward_torch(v, shapes, loc, attn)
    out.backward(go.to(dtype))
    return [t.detach().numpy() for t in (out, v.grad, o.grad, lg.grad, attn)]


def _run_fused(wis, value, off, logits, ref, go, shapes, want_attn=False):
    v = value.cuda().requires_grad_(True)
    o = off.cuda().requires_grad_(True)
    lg = logits.cuda().requires_grad_(True)
    res = wis.ms_deform_attn_fused(v, shapes, None, o, lg, ref.cuda(), return_attention_weights=want_attn)
    out, attn = res if want_attn else (res, None)
    out.backward(go.cuda().to(out.dtype))
    torch.cuda.synchronize()
    outs = [t.detach().float().cpu().numpy() for t in (out, v.grad, o.grad, lg.grad)]
    return outs + [attn.cpu().numpy() if attn is not None else None]


def _kink_mask(off, ref, shapes, eps=1e-3):
    wh = torch.tensor([[w, h] for h, w in shapes], dtype=torch.float64)[None, None, None, :, None, :]
    pix = (ref.double()[:, :, None, :, None, :] + off.double() / wh) * wh - 0.5
    return ((pix - pix.round()).abs() > eps).all(-1).numpy()


FIVE_LEVELS = [(3, 3), (5, 5), (9, 9), (17, 17), (33, 33)]
EIGHT_LEVELS = [(2, 2), (3, 3), (4, 4), (5, 5), (6, 7), (8, 8), (11, 9), (16, 16)]

CASES = [
    # (tag, B, shapes, H, D, P, Q)  -- D=32 & P=4 in bf16 takes the group-sorted backward, the rest v1
    ("m2f", 2, [(8, 8), (16, 16), (32, 32)], 8, 32, 4, None),
    ("odd", 1, [(7, 9), (13, 18), (25, 35)], 8, 32, 4, None),
    ("ragged_p3", 2, [(5, 7), (9, 4)], 4, 32, 3, 77),
    ("d64", 1, [(6, 6), (12, 12)], 4, 64, 2, 50),
    # L*P > 16: the forward's three-pass softmax; L >= 5 levels in the group-sorted backward's closing loop
    ("l5p4", 1, FIVE_LEVELS, 4, 32, 4, None),
    ("l8p4", 1, EIGHT_LEVELS, 2, 32, 4, None),
    ("l8p8", 1, EIGHT_LEVELS, 2, 32, 8, 90),  # L*P = 64, the most validate() takes
    ("d16", 2, [(6, 6), (12, 12)], 8, 16, 4, None),
    ("d128", 1, [(6, 6), (12, 12)], 2, 128, 4, 50),
]
BF16_CASES = CASES[:3] + [c for c in CASES if c[0] in ("d64", "l5p4", "l8p4", "l8p8", "d128")]


@pytest.fixture(scope="module")
def wis():
    import weed_instance_segmentation_b200 as w
    from weed_instance_segmentation_b200 import _cabi, build
    build.build()  # no-op when libmsda_b200.so is current; the product itself never builds or falls back
    _cabi.load()
    return w


@pytest.mark.parametrize("dist", ["init", "wide"])
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_fused_fp32(wis, case, dist):
    tag, B, shapes, H, D, P, Q = case
    value, off, logits, ref, go = _inputs(B, shapes, H, D, P, Q, seed=3, dist=dist)
    want = _reference_chain(value, off, logits, ref, go, shapes)
    got = _run_fused(wis, value, off, logits, ref, go, shapes, want_attn=True)
    safe = _kink_mask(off, ref, shapes)[..., None]
    for name, g, w in zip(("out", "grad_value", "grad_offsets", "grad_logits", "attn"), got, want):
        if name == "grad_offsets":
            g, w = g * safe, w * safe
        if name == "attn":
            g = g.reshape(w.shape)
        e = rel_err(g.reshape(w.shape), w)
        assert e <= 4e-5, f"{tag}/{dist}: {name} rel err {e:.3e}"


@pytest.mark.parametrize("case", BF16_CASES, ids=[c[0] for c in BF16_CASES])
def test_fused_bf16(wis, case):
    tag, B, shapes, H, D, P, Q = case
    value, off, logits, ref, go = _inputs(B, shapes, H, D, P, Q, seed=4)
    vb, ob, lb, gb = value.bfloat16(), off.bfloat16(), logits.bfloat16(), go.bfloat16()
    want = _reference_chain(vb.float(), ob.float(), lb.float(), ref, gb.float(), shapes)
    got = _run_fused(wis, vb, ob, lb, ref, gb, shapes)
    safe = _kink_mask(ob.float(), ref, shapes)[..., None]
    for name, g, w in zip(("out", "grad_value", "grad_offsets", "grad_logits"), got, want):
        if name == "grad_offsets":
            g, w = g * safe, w * safe
        e = rel_err(g.reshape(w.shape), w)
        assert e <= 2e-2, f"{tag}: {name} rel err {e:.3e}"


# bf16, D = 32, P = 4: the group-sorted backward by default; three and five levels
COMMON_MODE_GEOMS = [
    ("l3", 1, [(8, 8), (16, 16), (32, 32)], 8, 32, 4, None),
    ("l5", 1, FIVE_LEVELS, 4, 32, 4, None),
]
COMMON_MODE_PARAMS = [(g, mu, peaked, torch.bfloat16) for g in COMMON_MODE_GEOMS for mu in (0.0, 3.0, 10.0)
                      for peaked in (False, True)] + [(COMMON_MODE_GEOMS[1], 10.0, True, torch.float32)]


def _common_mode_inputs(case, mu, peaked, seed=17):
    """value = mu + randn; with `peaked`, one logit of every (query, head) row raised by 8 (its weight close to 1)."""
    tag, B, shapes, H, D, P, Q = case
    value, off, logits, ref, go = _inputs(B, shapes, H, D, P, Q, seed=seed)
    if peaked:
        j = torch.randint(0, logits.shape[-1], logits.shape[:-1] + (1,), generator=torch.Generator().manual_seed(seed))
        logits = logits.scatter_add(-1, j, torch.full(j.shape, 8.0))
    return value + mu, off, logits, ref, go


@pytest.mark.parametrize("case,mu,peaked,dtype", COMMON_MODE_PARAMS,
                         ids=[f"{g[0]}-mu{mu:g}-{'peaked' if pk else 'spread'}-{'fp32' if dt == torch.float32 else 'bf16'}"
                              for g, mu, pk, dt in COMMON_MODE_PARAMS])
def test_fused_softmax_backward_common_mode(wis, monkeypatch, case, mu, peaked, dtype):
    """grad_logits = a_j * (ga_j - sum_k a_k ga_k) cancels whenever the L*P attention gradients ga of a row share a
    common part: value rows with a non-zero mean (ga ~ mu * <grad_out, 1>) or one dominant logit. The result must come
    from fp32 ga (one rounding to the logits' dtype) in every backward the fused entry point runs: the default (the
    group-sorted kernel in bf16), the per-corner kernel and the deterministic one."""
    from weed_instance_segmentation_b200 import functional as F
    tag, B, shapes, H, D, P, Q = case
    value, off, logits, ref, go = _common_mode_inputs(case, mu, peaked)
    value, off, logits, go = (t.to(dtype) for t in (value, off, logits, go))  # reference points stay fp32
    want = _reference_chain(value.float(), off.float(), logits.float(), ref, go.float(), shapes)
    safe = _kink_mask(off.float(), ref, shapes)[..., None]
    bars = {"grad_logits": 1e-2} if dtype == torch.bfloat16 else {}
    for mode in ("default", "per_corner", "deterministic"):
        monkeypatch.setattr(F, "_BWD_V1", mode == "per_corner")
        prev = torch.are_deterministic_algorithms_enabled()
        torch.use_deterministic_algorithms(mode == "deterministic")
        try:
            got = _run_fused(wis, value, off, logits, ref, go, shapes)
        finally:
            torch.use_deterministic_algorithms(prev)
        for name, g, w in zip(("out", "grad_value", "grad_offsets", "grad_logits"), got, want):
            if name == "grad_offsets":
                g, w = g * safe, w * safe
            e = rel_err(g.reshape(w.shape), w)
            bar = bars.get(name, 2e-2 if dtype == torch.bfloat16 else 4e-5)
            assert e <= bar, f"{mode}: {name} rel err {e:.3e} > {bar:g}"


def test_fused_softmax_backward_common_mode_full_size(wis, monkeypatch):
    """BASELINE config 2 geometry (B = 2) in bf16 with value = 10 + randn: grad_logits of the default (group-sorted)
    backward against the per-corner one, which keeps ga in fp32; each carries one bf16 rounding of the result."""
    from weed_instance_segmentation_b200 import functional as F
    shapes = [(32, 32), (64, 64), (128, 128)]
    value, off, logits, ref, go = _inputs(2, shapes, 8, 32, 4, None, seed=23)
    args = ((value + 10.0).bfloat16(), off.bfloat16(), logits.bfloat16(), ref, go.bfloat16(), shapes)
    grad_logits = []
    for per_corner in (False, True):
        monkeypatch.setattr(F, "_BWD_V1", per_corner)
        grad_logits.append(_run_fused(wis, *args)[3])
    e = rel_err(grad_logits[0], grad_logits[1])
    assert e <= 1e-2, f"grad_logits: group-sorted vs per-corner rel err {e:.3e}"


def test_fused_matches_unfused_bitwise_forward(wis):
    """Same kernels, same arithmetic order: the fused forward equals the unfused one fed with torch's
    softmax / locations up to the softmax's last bit."""
    shapes = [(8, 8), (16, 16), (32, 32)]
    value, off, logits, ref, go = _inputs(2, shapes, 8, 32, 4, None, seed=9)
    B, Q, H, L, P, _ = off.shape
    v, o, lg, r = value.cuda(), off.cuda(), logits.cuda(), ref.cuda()
    attn = torch.softmax(lg, -1).view(B, Q, H, L, P)
    wh = torch.tensor([[w, h] for h, w in shapes], dtype=torch.float32, device="cuda")
    loc = r[:, :, None, :, None, :] + o / wh[None, None, None, :, None, :]
    a = wis.ms_deform_attn(v, shapes, None, loc, attn)
    b = wis.ms_deform_attn_fused(v, shapes, None, o, lg, r)
    assert rel_err(b.cpu().numpy(), a.cpu().numpy()) < 1e-6


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("shapes", [[(8, 8), (16, 16), (32, 32)], [(31, 41), (61, 81), (121, 162)], [(1, 1), (1, 9), (7, 1)]],
                         ids=["pyramid", "config3", "one_pixel"])
def test_implicit_reference_points_equal_the_reference_ones_bitwise(wis, shapes, dtype):
    """reference_points=None (Q == S): the kernels derive each query's reference point from its index. The result
    must be bit-identical to passing the tensor the reference's own get_reference_points (M2F:1095-1125) builds for
    un-padded inputs -- forward and all three gradients."""
    from transformers.models.mask2former.modeling_mask2former import Mask2FormerPixelDecoderEncoderOnly as Enc
    value, off, logits, _, go = _inputs(2, shapes, 8, 32, 4, None, seed=12)
    L = len(shapes)
    ref = Enc.get_reference_points(shapes, torch.ones(2, L, 2, device="cuda"), "cuda")
    res = []
    for r in (ref, None):
        v = value.cuda().to(dtype).requires_grad_(True)
        o = off.cuda().to(dtype).requires_grad_(True)
        lg = logits.cuda().to(dtype).requires_grad_(True)
        out = wis.ms_deform_attn_fused(v, shapes, None, o, lg, r)
        out.backward(go.cuda().to(dtype))
        res.append((out.detach(), v.grad, o.grad, lg.grad))
    assert torch.equal(res[0][0], res[1][0])
    for a, b in zip(res[0][1:], res[1][1:]):
        # gradients: same arithmetic, but the accumulation into grad_value uses atomics (summation order)
        assert rel_err(b.float().cpu().numpy(), a.float().cpu().numpy()) <= (2e-6 if dtype == torch.float32 else 1e-2)
    with pytest.raises(ValueError):  # implicit reference points need Q == S
        wis.ms_deform_attn_fused(value.cuda(), shapes, None, off.cuda()[:, :5], logits.cuda()[:, :5], None)


def test_fused_errors(wis):
    v = torch.zeros(1, 16, 8, 32, device="cuda")
    off = torch.zeros(1, 16, 8, 1, 4, 2, device="cuda")
    lg = torch.zeros(1, 16, 8, 4, device="cuda")
    ref = torch.zeros(1, 16, 1, 2, device="cuda")
    with pytest.raises(ValueError):
        wis.ms_deform_attn_fused(v, [(4, 4)], None, off, lg, torch.zeros(1, 16, 1, 4, device="cuda"))
    with pytest.raises(ValueError):
        wis.ms_deform_attn_fused(v, [(4, 4)], None, off, lg[..., :3], ref)
    with pytest.raises(RuntimeError):
        wis.ms_deform_attn_fused(v.cpu(), [(4, 4)], None, off.cpu(), lg.cpu(), ref.cpu())
