"""Parity of the CUDA path against the oracle, through the C ABI (ctypes -> libmsda_b200.so).

Bars (BASELINE.json north_star): fp32 within 1e-5 relative, bf16 within 2e-2 relative, where
"relative" is max|a-b| / max|b| over the tensor (``conftest.rel_err``).
Nothing here reads /root/reference; the oracle is oracle/ (C restatement) plus tests/golden/.
"""
import numpy as np
import pytest
import torch

import oracle
from conftest import rel_err

pytestmark = pytest.mark.gpu

FP32_BAR = 1e-5
BF16_BAR = 2e-2


@pytest.fixture(scope="module")
def wis():
    import weed_instance_segmentation_b200 as w
    from weed_instance_segmentation_b200 import _cabi, build
    build.build()  # no-op when libmsda_b200.so is current; the product itself never builds or falls back
    _cabi.load()  # fail loudly if the extension is missing
    assert torch.cuda.is_available()
    return w


def _run(wis, value, shapes, loc, attn, grad_out, level_start=None):
    dev = "cuda"
    v = value.to(dev).requires_grad_(True)
    lo = loc.to(dev).requires_grad_(True)
    a = attn.to(dev).requires_grad_(True)
    out = wis.ms_deform_attn(v, shapes, level_start, lo, a)
    out.backward(grad_out.to(dev).reshape(out.shape))
    torch.cuda.synchronize()
    return [t.detach().float().cpu().numpy() for t in (out, v.grad, lo.grad, a.grad)]


def _oracle(value, shapes, loc, attn, grad_out, level_start=None, dtype=np.float64):
    """C oracle. fp32 parity is judged against the oracle evaluated in fp32 like the reference
    (pixel coordinates up to ~160 carry 1e-5 px of fp32 rounding, which any fp32 implementation --
    the reference included -- shows against an fp64 evaluation); bf16 parity against fp64."""
    v, lo, a, go = (t.float().numpy() for t in (value, loc, attn, grad_out))
    out = oracle.c_forward(v, shapes, lo, a, level_start=level_start, dtype=dtype)
    gv, gl, ga = oracle.c_backward(v, shapes, lo, a, go, level_start=level_start, dtype=dtype)
    return out, gv, gl, ga


def _kink_safe(loc, shapes, eps=1e-3):
    """Samples whose pixel coordinates are at least `eps` px away from a grid line.

    Bilinear sampling is continuous but not differentiable where px or py is an integer, so d/d(loc)
    jumps there and which side a sample falls on depends on the last bit of the coordinate arithmetic
    (fp32 in the kernel and in the reference, fp64 in the high-precision oracle). grad_loc is compared
    on the other samples when the two sides evaluate coordinates in different precision; out,
    grad_value and grad_attn are continuous and always compared everywhere."""
    loc = np.asarray(loc, dtype=np.float64)
    wh = np.asarray([[w, h] for h, w in shapes], dtype=np.float64)[None, None, None, :, None, :]
    pix = loc * wh - 0.5
    with np.errstate(invalid="ignore"):
        d = np.abs(pix - np.round(pix))
    return (np.nan_to_num(d, nan=1.0) > eps).all(-1)


def _assert_close(got, want, bar, tag, safe=None, min_safe=0.98):
    for name, g, w in zip(("out", "grad_value", "grad_loc", "grad_attn"), got, want):
        assert g.shape == w.shape, (tag, name)
        if name == "grad_loc" and safe is not None:
            assert safe.mean() > min_safe, "kink mask should only drop a sliver of the samples"
            g, w = g * safe[..., None], w * safe[..., None]
        e = rel_err(g, w)
        assert e <= bar, f"{tag}: {name} rel err {e:.3e} > {bar:g}"


# ---------------------------------------------------------------------------- golden fixtures
def test_golden_fp32(wis, golden):
    name, g = golden
    shapes = [tuple(int(v) for v in r) for r in g["shapes"]]
    D = g["value"].shape[-1]
    if D not in (8, 16, 32, 64, 128):
        pytest.skip(f"head dim {D} has no kernel (documented: 8/16/32/64/128)")
    got = _run(wis, *(torch.from_numpy(g[k]) for k in ("value",)), shapes,
               torch.from_numpy(g["loc"]), torch.from_numpy(g["attn"]), torch.from_numpy(g["grad_out"]))
    want = (g["out_f64"], g["grad_value_f64"], g["grad_loc_f64"], g["grad_attn_f64"])
    _assert_close(got, want, FP32_BAR, name)


def test_golden_bf16(wis, golden):
    name, g = golden
    shapes = [tuple(int(v) for v in r) for r in g["shapes"]]
    if g["value"].shape[-1] not in (8, 16, 32, 64, 128):
        pytest.skip("head dim without a kernel")
    value = torch.from_numpy(g["value"]).bfloat16()
    attn = torch.from_numpy(g["attn"]).bfloat16()
    go = torch.from_numpy(g["grad_out"]).bfloat16()
    loc = torch.from_numpy(g["loc"])
    got = _run(wis, value, shapes, loc, attn, go)
    want = _oracle(value, shapes, loc, attn, go)  # oracle on the bf16-rounded inputs, fp64 arithmetic
    _assert_close(got, want, BF16_BAR, name, safe=_kink_safe(loc.numpy(), shapes),
                  min_safe=0.5)  # the edge-case fixture puts many samples exactly on grid lines


# ---------------------------------------------------------------------------- seeded random cases
CASES = [
    # (tag, B, shapes, H, D, P, Q)
    ("c1_512", 1, [(16, 16), (32, 32), (64, 64)], 8, 32, 4, None),
    ("c3_odd", 1, [(31, 41), (61, 81), (121, 162)], 8, 32, 4, None),
    ("ragged_q", 3, [(5, 7), (9, 4)], 4, 32, 3, 77),
    ("d16", 2, [(6, 6), (12, 12)], 8, 16, 4, None),
    ("d64", 2, [(6, 6), (12, 12)], 4, 64, 2, 50),
    ("one_pixel_levels", 2, [(1, 1), (1, 9), (7, 1), (4, 4)], 2, 32, 2, 33),
    ("many_points", 1, [(8, 8)], 2, 32, 16, None),
    ("d128", 1, [(6, 6), (12, 12)], 2, 128, 4, 40),
    ("d8", 2, [(6, 6), (12, 12)], 4, 8, 4, None),
]
# bf16: the model's geometry, and every head dim besides 32 (the per-corner backward at D = 8, 16, 64, 128)
BF16_CASES = CASES[:4] + [c for c in CASES if c[0] in ("d64", "d128", "d8")]


@pytest.mark.parametrize("dist", ["init", "trained", "adversarial"])
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_random_fp32(wis, case, dist):
    from weed_instance_segmentation_b200.synth import msda_inputs
    tag, B, shapes, H, D, P, Q = case
    x = msda_inputs(B, shapes, num_heads=H, head_dim=D, num_points=P, dist=dist, seed=7, num_queries=Q)
    args = (x["value"], shapes, x["sampling_locations"], x["attention_weights"], x["grad_out"])
    got = _run(wis, *args)
    _assert_close(got, _oracle(*args, dtype=np.float32), FP32_BAR, f"{tag}/{dist}")
    _assert_close(got, _oracle(*args), 4 * FP32_BAR, f"{tag}/{dist} vs fp64",
                  safe=_kink_safe(x["sampling_locations"].numpy(), shapes))


@pytest.mark.parametrize("attn_dtype", [torch.bfloat16, torch.float32], ids=["attn_bf16", "attn_f32"])
@pytest.mark.parametrize("dist", ["init", "trained", "adversarial"])
@pytest.mark.parametrize("case", BF16_CASES, ids=[c[0] for c in BF16_CASES])
def test_random_bf16(wis, case, dist, attn_dtype):
    from weed_instance_segmentation_b200.synth import msda_inputs
    tag, B, shapes, H, D, P, Q = case
    x = msda_inputs(B, shapes, num_heads=H, head_dim=D, num_points=P, dist=dist, seed=8, num_queries=Q,
                    value_dtype=torch.bfloat16, attn_dtype=attn_dtype)
    args = (x["value"], shapes, x["sampling_locations"], x["attention_weights"], x["grad_out"])
    _assert_close(_run(wis, *args), _oracle(*args), BF16_BAR, f"{tag}/{dist}",
                  safe=_kink_safe(x["sampling_locations"].numpy(), shapes))


# Geometries that stress the group-sorted backward's window logic (D=32, P=4, bf16 -> msda_bwd_mma_kernel): levels
# wider than the window's 64 groups (256 pixels), bounding boxes far larger than its 256 4x2-pixel groups (everything
# outside takes the fallback route), Q != S so queries arrive in no spatial order, one and five levels.
SORTED_CASES = [
    ("wide_levels", 1, [(12, 300), (256, 20)], 8, 32, 4, 500),
    ("c5_like", 1, [(64, 64), (128, 128), (256, 256)], 2, 32, 4, 3000),
    ("one_level", 2, [(40, 40)], 8, 32, 4, None),
    ("five_levels", 1, [(3, 3), (5, 5), (9, 9), (17, 17), (33, 33)], 4, 32, 4, None),
]


@pytest.mark.parametrize("dist", ["init", "trained", "adversarial"])
@pytest.mark.parametrize("case", SORTED_CASES, ids=[c[0] for c in SORTED_CASES])
def test_sorted_backward_windows(wis, case, dist):
    from weed_instance_segmentation_b200.synth import msda_inputs
    tag, B, shapes, H, D, P, Q = case
    x = msda_inputs(B, shapes, num_heads=H, head_dim=D, num_points=P, dist=dist, seed=21, num_queries=Q,
                    value_dtype=torch.bfloat16)
    args = (x["value"], shapes, x["sampling_locations"], x["attention_weights"], x["grad_out"])
    _assert_close(_run(wis, *args), _oracle(*args), BF16_BAR, f"{tag}/{dist}",
                  safe=_kink_safe(x["sampling_locations"].numpy(), shapes))


VARIANT_CASES = SORTED_CASES[:2] + [CASES[1]] + [c for c in CASES if c[0] in ("d64", "d128")]


@pytest.mark.parametrize("variant", ["v1", "v3"])
@pytest.mark.parametrize("case", VARIANT_CASES, ids=[c[0] for c in VARIANT_CASES])
def test_every_backward_variant_matches_oracle(wis, monkeypatch, case, variant):
    """Both bf16 backward kernels -- v1 per-corner reductions (MSDA_B200_FLAG_BWD_V1) and v3 group-sorted mma.sync
    (default) -- each against the oracle. At D = 64 and 128 the default is the per-corner kernel as well."""
    from weed_instance_segmentation_b200 import functional as F
    from weed_instance_segmentation_b200.synth import msda_inputs
    tag, B, shapes, H, D, P, Q = case
    monkeypatch.setattr(F, "_BWD_V1", variant == "v1")
    for dist in ("init", "adversarial"):
        x = msda_inputs(B, shapes, num_heads=H, head_dim=D, num_points=P, dist=dist, seed=31, num_queries=Q,
                        value_dtype=torch.bfloat16)
        args = (x["value"], shapes, x["sampling_locations"], x["attention_weights"], x["grad_out"])
        _assert_close(_run(wis, *args), _oracle(*args), BF16_BAR, f"{variant}/{tag}/{dist}",
                      safe=_kink_safe(x["sampling_locations"].numpy(), shapes))


def test_sorted_and_per_corner_backward_agree(wis, monkeypatch):
    """The default v3 (group-sorted) and v1 (per-corner reductions) differ only in fp32 summation order."""
    from weed_instance_segmentation_b200 import functional as F
    from weed_instance_segmentation_b200.synth import msda_inputs
    shapes = [(16, 16), (32, 32), (64, 64)]
    x = msda_inputs(2, shapes, dist="trained", seed=13, value_dtype=torch.bfloat16)
    args = (x["value"], shapes, x["sampling_locations"], x["attention_weights"], x["grad_out"])
    v3 = _run(wis, *args)
    monkeypatch.setattr(F, "_BWD_V1", True)
    v1 = _run(wis, *args)
    assert np.array_equal(v1[0], v3[0])
    for name, a, b in zip(("grad_value", "grad_loc", "grad_attn"), v1[1:], v3[1:]):
        assert rel_err(a, b) <= 1e-2, name  # both carry one bf16 rounding of the output


def test_query_order_does_not_change_results(wis, monkeypatch):
    from weed_instance_segmentation_b200 import functional as F
    from weed_instance_segmentation_b200.synth import msda_inputs
    shapes = [(7, 9), (13, 18)]
    x = msda_inputs(2, shapes, dist="trained", seed=5)
    args = (x["value"], shapes, x["sampling_locations"], x["attention_weights"], x["grad_out"])
    monkeypatch.setattr(F, "_USE_ORDER", True)
    with_order = _run(wis, *args)
    monkeypatch.setattr(F, "_USE_ORDER", False)
    without = _run(wis, *args)
    assert np.array_equal(with_order[0], without[0])  # forward is bit-identical
    _assert_close(with_order, without, 1e-6, "order")  # backward differs only by atomic ordering


def test_custom_level_start_and_padded_rows(wis):
    """S larger than the sum of the levels, levels not packed: level_start_index is honoured."""
    from weed_instance_segmentation_b200.synth import msda_inputs
    shapes = [(3, 4), (5, 6)]
    x = msda_inputs(2, shapes, dist="adversarial", seed=9, num_queries=21)
    S_pad = 60
    value = torch.randn(2, S_pad, 8, 32)
    lsi = [7, 25]
    args = (value, shapes, x["sampling_locations"], x["attention_weights"], x["grad_out"])
    got = _run(wis, *args, level_start=lsi)
    want = _oracle(*args, level_start=np.asarray(lsi), dtype=np.float32)
    _assert_close(got, want, FP32_BAR, "padded")
    assert not got[1][:, :7].any() and not got[1][:, 55:].any()  # untouched rows get zero gradient


def test_empty_and_noncontiguous(wis):
    from weed_instance_segmentation_b200.synth import msda_inputs
    shapes = [(4, 4)]
    v = torch.randn(2, 16, 8, 32, device="cuda")
    out = wis.ms_deform_attn(v, shapes, None, torch.zeros(2, 0, 8, 1, 4, 2, device="cuda"),
                             torch.zeros(2, 0, 8, 1, 4, device="cuda"))
    assert out.shape == (2, 0, 256)
    out = wis.ms_deform_attn(v[:0], shapes, None, torch.zeros(0, 5, 8, 1, 4, 2, device="cuda"),
                             torch.zeros(0, 5, 8, 1, 4, device="cuda"))
    assert out.shape == (0, 5, 256)
    # non-contiguous views are accepted (made contiguous on the host side)
    x = msda_inputs(2, shapes, dist="trained", seed=2)
    vt = x["value"].permute(0, 2, 1, 3).contiguous().permute(0, 2, 1, 3)
    assert not vt.is_contiguous()
    a = _run(wis, vt, shapes, x["sampling_locations"], x["attention_weights"], x["grad_out"])
    b = _run(wis, x["value"], shapes, x["sampling_locations"], x["attention_weights"], x["grad_out"])
    assert np.array_equal(a[0], b[0])


def test_error_behaviour(wis):
    v = torch.zeros(1, 16, 8, 32, device="cuda")
    loc = torch.zeros(1, 3, 8, 1, 4, 2, device="cuda")
    attn = torch.zeros(1, 3, 8, 1, 4, device="cuda")
    with pytest.raises(ValueError):  # shapes do not fit S (M2F:942-945)
        wis.ms_deform_attn(v, [(5, 5)], None, loc, attn)
    with pytest.raises(ValueError):
        wis.ms_deform_attn(v, [(4, 4)], None, loc[..., :1], attn)
    with pytest.raises(ValueError):
        wis.ms_deform_attn(v, [(4, 4)], None, loc, attn[:, :2])
    with pytest.raises(TypeError):
        wis.ms_deform_attn(v.half(), [(4, 4)], None, loc, attn)
    with pytest.raises(wis.MSDAError):  # head dim without a kernel: reported by the library, not swallowed
        wis.ms_deform_attn(torch.zeros(1, 16, 8, 24, device="cuda"), [(4, 4)], None, loc, attn)


def test_refused_backward_does_not_fail_the_next_calls(wis):
    """bf16 values with D = 8 take L*P <= 32 in the backward (shared memory; include/msda_b200.h), while the forward
    takes 64: at L*P = 33 the forward runs and the backward is refused as unsupported. The refusal is an argument
    error and must not resurface as an error of the next, valid, forward and backward on the same thread."""
    from weed_instance_segmentation_b200.synth import msda_inputs
    shapes = [(4, 4), (2, 3), (3, 2)]
    x = msda_inputs(1, shapes, num_heads=2, head_dim=8, num_points=11, dist="init", seed=3, num_queries=10,
                    value_dtype=torch.bfloat16)
    v = x["value"].cuda().requires_grad_(True)
    out = wis.ms_deform_attn(v, shapes, None, x["sampling_locations"].cuda(), x["attention_weights"].cuda())
    with pytest.raises(RuntimeError, match="shared memory") as refused:
        out.backward(x["grad_out"].cuda().reshape(out.shape))
    x = msda_inputs(1, [(6, 6), (12, 12)], num_heads=4, head_dim=8, num_points=4, dist="init", seed=3)
    args = (x["value"], [(6, 6), (12, 12)], x["sampling_locations"], x["attention_weights"], x["grad_out"])
    _assert_close(_run(wis, *args), _oracle(*args, dtype=np.float32), FP32_BAR, "after a refused backward")
    assert "error 2" in str(refused.value) and "227 KB" in str(refused.value)


def test_nan_and_far_locations_are_safe(wis):
    """NaN / huge coordinates contribute zero (as in the oracle) and never fault."""
    from weed_instance_segmentation_b200.synth import msda_inputs
    shapes = [(4, 5), (8, 9)]
    x = msda_inputs(1, shapes, dist="adversarial", seed=4, num_queries=32)
    loc = x["sampling_locations"].clone()
    loc.view(-1, 2)[::7] = float("nan")
    loc.view(-1, 2)[1::7] = 1e30
    loc.view(-1, 2)[2::7] = -1e30
    loc.view(-1, 2)[3::7] = float("inf")
    args = (x["value"], shapes, loc, x["attention_weights"], x["grad_out"])
    got, want = _run(wis, *args), _oracle(*args, dtype=np.float32)
    assert all(np.isfinite(g).all() for g in got)
    _assert_close(got, want, FP32_BAR, "nan")


# bf16 values, D = 32, even H: the head-pair forward. L = 3, P = 4 takes its constant-index descriptor path; the odd
# two-level geometry with three points per level takes the generic one.
PAIR_CASES = [
    ("c1_pyramid", 2, [(16, 16), (32, 32), (64, 64)], 8, 4),
    ("odd_two_levels", 2, [(8, 9), (10, 6)], 2, 3),
]


@pytest.mark.parametrize("attn_dtype", [torch.bfloat16, torch.float32], ids=["attn_bf16", "attn_f32"])
@pytest.mark.parametrize("case", PAIR_CASES, ids=[c[0] for c in PAIR_CASES])
def test_head_pair_forward_matches_one_head_kernel(wis, case, attn_dtype):
    """The head-pair forward (msda_fwd_pair_kernel) against the one-head kernel, which MSDA_B200_FLAG_STRICT_PADDING
    routes the same problem to: plain, fused, and fused with implicit reference points (ref_points = NULL). With finite
    inputs the results are bit-identical: strict mode only skips FMAs whose weight is exactly 0, which add +-0."""
    from weed_instance_segmentation_b200 import _cabi, functional, synth
    tag, B, shapes, H, P = case
    D, L = 32, len(shapes)
    lib = _cabi.load()
    acode = _cabi.BF16 if attn_dtype == torch.bfloat16 else _cabi.F32
    order = functional.query_order_2d(shapes, functional._TILE, "cuda")
    ref = synth.reference_points(shapes, device="cuda")[None].expand(B, -1, -1, -1).contiguous()
    stream = torch.cuda.current_stream().cuda_stream
    for dist in ("init", "adversarial"):
        x = synth.msda_inputs(B, shapes, num_heads=H, head_dim=D, num_points=P, dist=dist, seed=5, device="cuda",
                              value_dtype=torch.bfloat16, attn_dtype=attn_dtype, with_grad_out=False)
        value, loc, attn = x["value"], x["sampling_locations"], x["attention_weights"]
        S = value.shape[1]
        g = torch.Generator(device="cuda").manual_seed(1)
        off = (synth.init_offsets(H, L, P).to("cuda")[None, None]
               + 0.5 * torch.randn(B, S, H, L, P, 2, device="cuda", generator=g)).to(attn_dtype).contiguous()
        logits = torch.randn(B, S, H, L * P, device="cuda", generator=g).to(attn_dtype)

        def run(flags):
            desc, keep = _cabi.make_desc(B, S, S, H, D, L, P, _cabi.BF16, acode, shapes, synth.level_start_index(shapes),
                                         flags)
            outs = [torch.empty(B, S, H * D, dtype=torch.bfloat16, device="cuda") for _ in range(3)]
            _cabi.check(lib.msda_b200_forward(desc, value.data_ptr(), loc.data_ptr(), attn.data_ptr(), outs[0].data_ptr(),
                                              order.data_ptr(), stream))
            for out, r in ((outs[1], ref.data_ptr()), (outs[2], None)):
                _cabi.check(lib.msda_b200_forward_fused(desc, value.data_ptr(), off.data_ptr(), logits.data_ptr(), r,
                                                        out.data_ptr(), None, order.data_ptr(), stream))
            torch.cuda.synchronize()
            return outs

        for name, pair, one in zip(("plain", "fused", "fused, implicit ref"), run(0), run(_cabi.FLAG_STRICT_PADDING)):
            assert pair.abs().max() > 0, f"{tag}/{dist}: {name}"
            assert torch.equal(pair, one), f"{tag}/{dist}: {name}"


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_non_finite_values_outside_the_footprint_do_not_leak(wis, dtype, monkeypatch):
    """grid_sample's zeros padding never reads a pixel outside the level, and a sample only reads the (up to four)
    in-bounds pixels of its own footprint (M2F:823). Every pixel NO sample reads is filled with NaN / Inf here --
    in particular the clamped neighbours the kernels could load for a border sample -- and the results must still
    equal the oracle's, finite everywhere except the gradient of the planted pixels (which is exactly zero).
    Forward: under MSDA_B200_FLAG_STRICT_PADDING (the default forward trades this for speed, see the header);
    backward: always."""
    from weed_instance_segmentation_b200 import functional as F
    from weed_instance_segmentation_b200.synth import msda_inputs
    monkeypatch.setattr(F, "_STRICT_PADDING", True)
    shapes = [(8, 9), (10, 6), (1, 12)]
    H, D, P = 2, 32, 4
    x = msda_inputs(1, shapes, num_heads=H, head_dim=D, num_points=P, dist="adversarial", seed=11, num_queries=4,
                    value_dtype=dtype)
    loc = x["sampling_locations"].clone()
    loc.view(-1, 2)[::5] = torch.tensor([0.02, 0.97])   # footprints hanging over two borders
    loc.view(-1, 2)[1::5] = torch.tensor([-0.06, 0.5])  # px in (-1, -0.5): only the right-hand pixels are in bounds
    value = x["value"].clone()
    touched = torch.zeros(value.shape[:3], dtype=torch.bool)  # (B, S, H)
    start = 0
    for l, (hh, ww) in enumerate(shapes):
        px = loc[0, :, :, l, :, 0].double() * ww - 0.5  # (Q, H, P)
        py = loc[0, :, :, l, :, 1].double() * hh - 0.5
        x0, y0 = torch.floor(px).long(), torch.floor(py).long()
        for dy in (0, 1):
            for dx in (0, 1):
                xx, yy = x0 + dx, y0 + dy
                ok = (xx >= 0) & (xx < ww) & (yy >= 0) & (yy < hh)
                for h in range(H):
                    idx = (start + yy[:, h] * ww + xx[:, h])[ok[:, h]]
                    touched[0, idx, h] = True
        start += hh * ww
    assert (~touched).sum() > 10
    bad = torch.tensor([float("nan"), float("inf"), float("-inf")]).to(dtype)
    planted = value.clone()
    planted[~touched] = bad[torch.arange((~touched).sum()) % 3][:, None].expand(-1, D)
    args = (planted, shapes, loc, x["attention_weights"], x["grad_out"])
    got = _run(wis, *args)
    want = _oracle(value, shapes, loc, x["attention_weights"], x["grad_out"],
                   dtype=np.float32 if dtype == torch.float32 else np.float64)  # the oracle on the clean values
    assert all(np.isfinite(g).all() for g in got), "a non-finite value leaked out of a pixel the reference never reads"
    bar = FP32_BAR if dtype == torch.float32 else BF16_BAR
    _assert_close(got, want, bar, "planted", safe=_kink_safe(loc.numpy(), shapes), min_safe=0.5)
    assert not got[1][~touched.numpy()].any()  # no gradient reaches a pixel nobody reads


# ---------------------------------------------------------------------------- full-size properties
def _c2_inputs(dist, dtype):
    from weed_instance_segmentation_b200.synth import msda_inputs
    shapes = [(32, 32), (64, 64), (128, 128)]
    return shapes, msda_inputs(8, shapes, dist=dist, seed=1, device="cuda", value_dtype=dtype)


@pytest.mark.parametrize("dist", ["init", "adversarial"])
def test_full_size_linearity_and_adjoint_fp32(wis, dist):
    """At BASELINE config 2 (B=8, 1024^2): f is linear in value and in attn, and the backward is
    its adjoint:  <go, f(v,a)> == <grad_value, v> == <grad_attn, a>."""
    shapes, x = _c2_inputs(dist, torch.float32)
    v = x["value"].requires_grad_(True)
    lo = x["sampling_locations"].requires_grad_(True)
    a = x["attention_weights"].requires_grad_(True)
    go = x["grad_out"]
    out = wis.ms_deform_attn(v, shapes, x["level_start_index"], lo, a)
    out.backward(go)
    lhs = (go.double() * out.detach().double()).sum().item()
    assert abs((v.grad.double() * v.detach().double()).sum().item() - lhs) <= 1e-5 * max(abs(lhs), 1.0) * 10
    assert abs((a.grad.double() * a.detach().double()).sum().item() - lhs) <= 1e-5 * max(abs(lhs), 1.0) * 10
    # linearity in value
    v2 = torch.randn_like(v)
    with torch.no_grad():
        o2 = wis.ms_deform_attn(v2, shapes, None, lo, a)
        o3 = wis.ms_deform_attn(v.detach() * 0.5 + v2, shapes, None, lo, a)
    assert rel_err((0.5 * out.detach() + o2).cpu().numpy(), o3.cpu().numpy()) <= 1e-5
    # a slice against the oracle (first 64 queries of the last batch element)
    sl = slice(0, 64)
    want = oracle.c_forward(v.detach()[-1:].cpu().numpy(), shapes, lo.detach()[-1:, sl].cpu().numpy(),
                            a.detach()[-1:, sl].cpu().numpy(), dtype=np.float32)
    assert rel_err(out.detach()[-1:, sl].cpu().numpy(), want) <= FP32_BAR


def test_full_size_matches_reference_on_gpu_bf16(wis):
    """BASELINE config 2 in the bf16 contract against the reference's own function (M2F:798-837)
    run in fp32 on the same GPU, two batch elements at a time to bound its 2 GB temporary."""
    pytest.importorskip("transformers")
    from oracle.hf_reference import hf_forward_torch
    shapes, x = _c2_inputs("trained", torch.bfloat16)
    v = x["value"].requires_grad_(True)
    lo = x["sampling_locations"].requires_grad_(True)
    a = x["attention_weights"].requires_grad_(True)
    out = wis.ms_deform_attn(v, shapes, x["level_start_index"], lo, a)
    out.backward(x["grad_out"])
    for b0 in range(0, 8, 2):
        sl = slice(b0, b0 + 2)
        rv = v.detach()[sl].float().requires_grad_(True)
        rl = lo.detach()[sl].clone().requires_grad_(True)
        ra = a.detach()[sl].float().requires_grad_(True)
        ro = hf_forward_torch(rv, shapes, rl, ra)
        ro.backward(x["grad_out"][sl].float())
        wh = torch.tensor([[w, h] for h, w in shapes], dtype=torch.float64, device="cuda")[None, None, None, :, None, :]
        pix = lo.detach()[sl].double() * wh - 0.5
        safe = ((pix - pix.round()).abs() > 1e-3).all(-1, keepdim=True).float()  # see _kink_safe
        for name, got, want in (("out", out.detach()[sl], ro.detach()), ("grad_value", v.grad[sl], rv.grad),
                                ("grad_loc", lo.grad[sl] * safe, rl.grad * safe), ("grad_attn", a.grad[sl], ra.grad)):
            e = ((got.float() - want).abs().max() / want.abs().max()).item()
            assert e <= BF16_BAR, f"batch {b0}: {name} rel err {e:.3e}"
        del rv, rl, ra, ro


def test_sorted_backward_fuzz(wis):
    """40 random geometries / location patterns (tools/fuzz_sorted_backward.py): the default v3 and v1 agree to
    summation order."""
    import importlib.util
    import os
    from weed_instance_segmentation_b200 import functional as F
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools", "fuzz_sorted_backward.py")
    spec = importlib.util.spec_from_file_location("fuzz_sorted_backward", path)
    fz = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(fz)
    rng = np.random.default_rng(123)
    try:
        for i in range(40):
            B, shapes, H, Q, dist = fz.random_case(rng)
            value, loc, attn, go = fz.make_inputs(B, shapes, H, Q, dist, rng)
            F._BWD_V1 = False
            v3 = fz.run(value, shapes, loc, attn, go)
            F._BWD_V1 = True
            v1 = fz.run(value, shapes, loc, attn, go)
            assert torch.equal(v1[0], v3[0])
            assert fz.rel(v3[1], v1[1]) <= 1.6e-2 and fz.rel(v3[3], v1[3]) <= 1.6e-2, (i, shapes, dist)
            assert fz.rel(v3[2], v1[2]) <= 1e-4, (i, shapes, dist)
    finally:
        F._BWD_V1 = False
