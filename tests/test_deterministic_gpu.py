"""Deterministic backward (MSDA_B200_FLAG_DETERMINISTIC; torch.use_deterministic_algorithms(True) in Python).

Reproducibility is judged bit for bit: three backward calls on the same inputs -- plain, with another query order,
on a side stream -- must return byte-equal gradients. Accuracy keeps the bars of the default backward: fp32 1e-5
against the fp32 oracle (4e-5 against fp64), bf16 2e-2 against fp64.
"""
import contextlib
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import oracle
from conftest import load_golden, golden_names, rel_err

pytestmark = pytest.mark.gpu

FP32_BAR = 1e-5
BF16_BAR = 2e-2
C2 = [(32, 32), (64, 64), (128, 128)]
C3 = [(31, 41), (61, 81), (121, 162)]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def wis():
    import weed_instance_segmentation_b200 as w
    from weed_instance_segmentation_b200 import _cabi, build
    build.build()
    _cabi.load()
    assert torch.cuda.is_available()
    return w


@contextlib.contextmanager
def deterministic_mode():
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev)


def _bits(t):
    return t.detach().contiguous().view(torch.uint8)


def _assert_same_bits(a, b, tag):
    for name, x, y in zip(("grad_value", "grad_loc", "grad_attn"), a, b):
        assert torch.equal(_bits(x), _bits(y)), f"{tag}: {name} differs"


def _code(dtype):
    from weed_instance_segmentation_b200 import _cabi
    return _cabi.BF16 if dtype == torch.bfloat16 else _cabi.F32


def _flag():
    from weed_instance_segmentation_b200 import _cabi
    return _cabi.FLAG_DETERMINISTIC


def _workspace(lib, desc):
    n = int(lib.msda_b200_backward_workspace_bytes(desc))
    return (torch.empty(n, dtype=torch.uint8, device="cuda") if n else None), n


def _abi_backward(x, shapes, flags, order=None, stream=None, level_start=None):
    """msda_b200_backward on device tensors x = (value, loc, attn, grad_out); returns (grad_value, grad_loc, grad_attn)."""
    from weed_instance_segmentation_b200 import _cabi, synth
    lib = _cabi.load()
    value, loc, attn, go = x
    B, S, H, D = value.shape
    _, Q, _, L, P, _ = loc.shape
    lsi = synth.level_start_index(shapes) if level_start is None else level_start
    desc, keep = _cabi.make_desc(B, S, Q, H, D, L, P, _code(value.dtype), _code(attn.dtype), shapes, lsi, flags)
    ws, n = _workspace(lib, desc)
    # NaN-filled outputs: every element the call should write is checked to be written
    gv, gl, ga = (torch.full_like(t, float("nan")) for t in (value, loc, attn))
    st = stream or torch.cuda.current_stream()
    st.wait_stream(torch.cuda.current_stream())  # the NaN fill above runs on the current stream
    with torch.cuda.stream(st):
        _cabi.check(lib.msda_b200_backward(desc, value.data_ptr(), loc.data_ptr(), attn.data_ptr(), go.data_ptr(),
                                           gv.data_ptr(), gl.data_ptr(), ga.data_ptr(), ws.data_ptr() if ws is not None
                                           else None, n, order.data_ptr() if order is not None else None,
                                           st.cuda_stream))
    torch.cuda.synchronize()
    return gv, gl, ga


def _abi_backward_fused(x, shapes, flags, order=None, stream=None):
    """msda_b200_backward_fused on x = (value, offsets, logits, ref or None, grad_out)."""
    from weed_instance_segmentation_b200 import _cabi, synth
    lib = _cabi.load()
    value, off, logits, ref, go = x
    B, S, H, D = value.shape
    _, Q, _, L, P, _ = off.shape
    desc, keep = _cabi.make_desc(B, S, Q, H, D, L, P, _code(value.dtype), _code(off.dtype), shapes,
                                 synth.level_start_index(shapes), flags)
    ws, n = _workspace(lib, desc)
    gv, go_, gl = (torch.full_like(t, float("nan")) for t in (value, off, logits))
    st = stream or torch.cuda.current_stream()
    st.wait_stream(torch.cuda.current_stream())  # the NaN fill above runs on the current stream
    with torch.cuda.stream(st):
        _cabi.check(lib.msda_b200_backward_fused(desc, value.data_ptr(), off.data_ptr(), logits.data_ptr(),
                                                 ref.data_ptr() if ref is not None else None, go.data_ptr(),
                                                 gv.data_ptr(), go_.data_ptr(), gl.data_ptr(),
                                                 ws.data_ptr() if ws is not None else None, n,
                                                 order.data_ptr() if order is not None else None, st.cuda_stream))
    torch.cuda.synchronize()
    return gv, go_, gl


def _three_calls(run, Q, tag):
    """plain, another query order, side stream: byte-equal; returns the first result."""
    from weed_instance_segmentation_b200 import _cabi
    flags = _cabi.FLAG_DETERMINISTIC
    g = torch.Generator().manual_seed(Q)
    perm = torch.randperm(Q, generator=g).to(torch.int32).cuda()
    a = run(flags, None, None)
    b = run(flags, perm, None)
    side = torch.cuda.Stream()
    c = run(flags, None, side)
    for t in a:
        assert not torch.isnan(t.float()).any(), f"{tag}: an element was not written"
    _assert_same_bits(a, b, f"{tag} query order")
    _assert_same_bits(a, c, f"{tag} side stream")
    return a


def _device(x):
    return tuple(x[k].cuda() for k in ("value", "sampling_locations", "attention_weights", "grad_out"))


# ---------------------------------------------------------------------------- 1. reproducibility
DTYPES = [(torch.bfloat16, torch.bfloat16), (torch.bfloat16, torch.float32), (torch.float32, torch.float32)]


@pytest.mark.parametrize("D", [8, 32, 128])
@pytest.mark.parametrize("dtypes", DTYPES, ids=["bf16", "bf16_attn_f32", "f32"])
def test_reproducible(wis, dtypes, D):
    from weed_instance_segmentation_b200.synth import msda_inputs
    vd, ad = dtypes
    shapes = [(9, 11), (5, 6), (1, 3)]
    x = _device(msda_inputs(2, shapes, num_heads=4, head_dim=D, num_points=4, dist="trained", seed=D,
                            value_dtype=vd, attn_dtype=ad))
    Q = x[1].shape[1]
    _three_calls(lambda f, o, s: _abi_backward(x, shapes, f, o, s), Q, f"D={D}")


@pytest.mark.parametrize("dist", ["init", "trained", "adversarial"])
def test_reproducible_config2(wis, dist):
    from weed_instance_segmentation_b200 import functional
    from weed_instance_segmentation_b200.synth import msda_inputs
    x = _device(msda_inputs(8, C2, dist=dist, seed=1, device="cuda", value_dtype=torch.bfloat16))
    order = functional.query_order_2d(C2, functional._TILE, "cuda")
    a = _three_calls(lambda f, o, s: _abi_backward(x, C2, f, o, s), x[1].shape[1], f"config 2 {dist}")
    _assert_same_bits(a, _abi_backward(x, C2, _flag(), order), f"config 2 {dist} 2-D order")


# ---------------------------------------------------------------------------- 2. parity with the oracle
def _run_torch(wis, value, shapes, loc, attn, grad_out, level_start=None):
    v = value.cuda().requires_grad_(True)
    lo = loc.cuda().requires_grad_(True)
    a = attn.cuda().requires_grad_(True)
    with deterministic_mode():
        out = wis.ms_deform_attn(v, shapes, level_start, lo, a)
        out.backward(grad_out.cuda().reshape(out.shape))
    torch.cuda.synchronize()
    return [t.detach().float().cpu().numpy() for t in (out, v.grad, lo.grad, a.grad)]


def _oracle(value, shapes, loc, attn, grad_out, level_start=None, dtype=np.float64):
    v, lo, a, go = (t.float().numpy() for t in (value, loc, attn, grad_out))
    out = oracle.c_forward(v, shapes, lo, a, level_start=level_start, dtype=dtype)
    return (out,) + tuple(oracle.c_backward(v, shapes, lo, a, go, level_start=level_start, dtype=dtype))


def _kink_safe(loc, shapes, eps=1e-3):
    loc = np.asarray(loc, dtype=np.float64)
    wh = np.asarray([[w, h] for h, w in shapes], dtype=np.float64)[None, None, None, :, None, :]
    pix = loc * wh - 0.5
    with np.errstate(invalid="ignore"):
        d = np.abs(pix - np.round(pix))
    return (np.nan_to_num(d, nan=1.0) > eps).all(-1)


def _assert_close(got, want, bar, tag, safe=None):
    for name, g, w in zip(("out", "grad_value", "grad_loc", "grad_attn"), got, want):
        assert g.shape == w.shape, (tag, name)
        if name == "grad_loc" and safe is not None:
            g, w = g * safe[..., None], w * safe[..., None]
        e = rel_err(g, w)
        assert e <= bar, f"{tag}: {name} rel err {e:.3e} > {bar:g}"


@pytest.mark.parametrize("name", golden_names())
def test_golden(wis, name):
    g = load_golden(name)
    shapes = [tuple(int(v) for v in r) for r in g["shapes"]]
    if g["value"].shape[-1] not in (8, 16, 32, 64, 128):
        pytest.skip("head dim without a kernel")
    value, loc, attn, go = (torch.from_numpy(g[k]) for k in ("value", "loc", "attn", "grad_out"))
    got = _run_torch(wis, value, shapes, loc, attn, go)
    _assert_close(got, (g["out_f64"], g["grad_value_f64"], g["grad_loc_f64"], g["grad_attn_f64"]), FP32_BAR, name)
    args = (value.bfloat16(), shapes, loc, attn.bfloat16(), go.bfloat16())
    _assert_close(_run_torch(wis, *args), _oracle(*args), BF16_BAR, f"{name} bf16",
                  safe=_kink_safe(loc.numpy(), shapes))


CASES = [
    # (tag, B, shapes, H, D, P, Q)
    ("c3_odd", 1, C3, 8, 32, 4, None),
    ("ragged_q", 3, [(5, 7), (9, 4)], 4, 32, 3, 77),
    ("d16", 2, [(6, 6), (12, 12)], 8, 16, 4, None),
    ("d64", 2, [(6, 6), (12, 12)], 4, 64, 2, 50),
    ("one_pixel_levels", 2, [(1, 1), (1, 9), (7, 1), (4, 4)], 2, 32, 2, 33),
    ("lp64", 1, [(6, 7), (3, 4), (9, 5), (2, 2)], 2, 32, 16, 40),
]


@pytest.mark.parametrize("dist", ["init", "trained", "adversarial"])
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_random_matches_oracle(wis, case, dist):
    from weed_instance_segmentation_b200.synth import msda_inputs
    tag, B, shapes, H, D, P, Q = case
    x = msda_inputs(B, shapes, num_heads=H, head_dim=D, num_points=P, dist=dist, seed=7, num_queries=Q)
    args = (x["value"], shapes, x["sampling_locations"], x["attention_weights"], x["grad_out"])
    got = _run_torch(wis, *args)
    _assert_close(got, _oracle(*args, dtype=np.float32), FP32_BAR, f"{tag}/{dist}")
    _assert_close(got, _oracle(*args), 4 * FP32_BAR, f"{tag}/{dist} vs fp64",
                  safe=_kink_safe(x["sampling_locations"].numpy(), shapes))
    for ad in (torch.bfloat16, torch.float32):
        xb = msda_inputs(B, shapes, num_heads=H, head_dim=D, num_points=P, dist=dist, seed=8, num_queries=Q,
                         value_dtype=torch.bfloat16, attn_dtype=ad)
        args = (xb["value"], shapes, xb["sampling_locations"], xb["attention_weights"], xb["grad_out"])
        _assert_close(_run_torch(wis, *args), _oracle(*args), BF16_BAR, f"{tag}/{dist}/bf16 {ad}",
                      safe=_kink_safe(xb["sampling_locations"].numpy(), shapes))


def test_padded_rows_are_exactly_zero(wis):
    from weed_instance_segmentation_b200.synth import msda_inputs
    shapes = [(3, 4), (5, 6)]
    x = msda_inputs(2, shapes, dist="adversarial", seed=9, num_queries=21)
    value = torch.randn(2, 60, 8, 32)
    lsi = [7, 25]
    args = (value, shapes, x["sampling_locations"], x["attention_weights"], x["grad_out"])
    got = _run_torch(wis, *args, level_start=lsi)
    _assert_close(got, _oracle(*args, level_start=np.asarray(lsi), dtype=np.float32), FP32_BAR, "padded")
    assert not got[1][:, :7].any() and not got[1][:, 55:].any() and not got[1][:, 19:25].any()


def test_nan_and_far_locations_are_safe(wis):
    from weed_instance_segmentation_b200.synth import msda_inputs
    shapes = [(4, 5), (8, 9)]
    x = msda_inputs(1, shapes, dist="adversarial", seed=4, num_queries=32)
    loc = x["sampling_locations"].clone()
    loc.view(-1, 2)[::7] = float("nan")
    loc.view(-1, 2)[1::7] = 1e30
    loc.view(-1, 2)[2::7] = -1e30
    loc.view(-1, 2)[3::7] = float("inf")
    args = (x["value"], shapes, loc, x["attention_weights"], x["grad_out"])
    got = _run_torch(wis, *args)
    assert all(np.isfinite(g).all() for g in got)
    _assert_close(got, _oracle(*args, dtype=np.float32), FP32_BAR, "nan")


def test_non_finite_grad_out_propagates_like_the_default(wis):
    from weed_instance_segmentation_b200.synth import msda_inputs
    shapes = [(6, 7), (3, 4)]
    x = msda_inputs(1, shapes, dist="trained", seed=3)
    go = x["grad_out"].clone()
    go[0, 5, :8] = float("nan")
    go[0, 9, 40:48] = float("inf")
    xs = _device(dict(x, grad_out=go))
    det = _abi_backward(xs, shapes, _flag())
    ref = _abi_backward(xs, shapes, 0)
    for a, b in zip(det, ref):
        assert torch.equal(torch.isnan(a), torch.isnan(b)) and torch.equal(torch.isinf(a), torch.isinf(b))


# ---------------------------------------------------------------------------- 3. agreement with the default backward
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
@pytest.mark.parametrize("config", ["config2", "config3"])
def test_agrees_with_default_backward(wis, config, dtype):
    from weed_instance_segmentation_b200.synth import msda_inputs
    shapes, B = (C2, 8) if config == "config2" else (C3, 16)
    x = _device(msda_inputs(B, shapes, dist="trained", seed=2, device="cuda", value_dtype=dtype))
    det = _abi_backward(x, shapes, _flag())
    ref = _abi_backward(x, shapes, 0)
    safe = torch.from_numpy(_kink_safe(x[1].cpu().numpy(), shapes)).cuda()[..., None]
    bar = BF16_BAR if dtype == torch.bfloat16 else FP32_BAR
    for name, a, b in zip(("grad_value", "grad_loc", "grad_attn"), det, ref):
        if name == "grad_loc":
            a, b = a * safe, b * safe
        e = ((a.float() - b.float()).abs().max() / b.float().abs().max()).item()
        assert e <= bar, f"{config} {name}: {e:.3e}"


# ---------------------------------------------------------------------------- 4. fused variant
def _fused_inputs(B, shapes, dtype, seed, device="cuda"):
    from weed_instance_segmentation_b200 import synth
    H, P, D, L = 8, 4, 32, len(shapes)
    S = sum(h * w for h, w in shapes)
    g = torch.Generator(device=device).manual_seed(seed)
    value = torch.randn(B, S, H, D, generator=g, device=device).to(dtype)
    off = (synth.init_offsets(H, L, P).to(device)[None, None]
           + 0.5 * torch.randn(B, S, H, L, P, 2, generator=g, device=device)).to(dtype).contiguous()
    logits = (2.0 * torch.randn(B, S, H, L * P, generator=g, device=device)).to(dtype)
    ref = synth.reference_points(shapes, device=device)[None].expand(B, -1, -1, -1).contiguous()
    go = torch.randn(B, S, H * D, generator=g, device=device).to(dtype)
    return value, off, logits, ref, go


@pytest.mark.parametrize("implicit", [False, True], ids=["explicit_ref", "implicit_ref"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_fused_reproducible_and_close_to_default(wis, dtype, implicit):
    shapes = [(8, 8), (16, 16), (32, 32)]
    value, off, logits, ref, go = _fused_inputs(2, shapes, dtype, seed=9)
    x = (value, off, logits, None if implicit else ref, go)
    det = _three_calls(lambda f, o, s: _abi_backward_fused(x, shapes, f, o, s), value.shape[1], "fused")
    default = _abi_backward_fused(x, shapes, 0)
    bar = 2e-6 if dtype == torch.float32 else 1e-2  # test_fused_gpu: default fused backward against itself
    for name, a, b in zip(("grad_value", "grad_offsets", "grad_logits"), det, default):
        e = rel_err(a.float().cpu().numpy(), b.float().cpu().numpy())
        assert e <= bar, f"fused {name}: {e:.3e}"


# ---------------------------------------------------------------------------- 5. batch independence
def test_image_alone_equals_image_in_batch(wis):
    from weed_instance_segmentation_b200.synth import msda_inputs
    shapes = [(16, 16), (8, 8), (4, 4)]
    x = _device(msda_inputs(8, shapes, dist="trained", seed=6, value_dtype=torch.bfloat16))
    whole = _abi_backward(x, shapes, _flag())
    for b in (0, 5):
        alone = _abi_backward(tuple(t[b:b + 1].contiguous() for t in x), shapes, _flag())
        _assert_same_bits([t[b:b + 1] for t in whole], alone, f"image {b}")


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_host_pipeline_chunks_equal_device_call(wis, dtype):
    from weed_instance_segmentation_b200.synth import msda_inputs
    shapes = [(8, 8), (16, 16), (32, 32)]
    B = 8
    x = msda_inputs(B, shapes, dist="trained", seed=12, value_dtype=dtype)
    order = None
    from weed_instance_segmentation_b200 import functional
    if functional._USE_ORDER:
        order = functional.query_order_2d(shapes, functional._TILE, "cuda")
    want = _abi_backward(_device(x), shapes, _flag(), order)
    host = [x[k].contiguous().pin_memory() for k in ("value", "sampling_locations", "attention_weights", "grad_out")]
    for chunk in (1, 4):
        with wis.HostPipeline(B, shapes, 8, 32, 4, value_dtype=dtype, chunk_images=chunk, deterministic=True) as pipe:
            res = pipe.empty_outputs()
            pipe.step(*host, **res)
            pipe.synchronize()
        got = [res[k].cuda().view(w.shape) for k, w in
               zip(("grad_value", "grad_sampling_locations", "grad_attention_weights"), want)]
        _assert_same_bits(got, want, f"pipeline chunk {chunk}")


def test_host_pipeline_follows_the_torch_switch(wis):
    shapes = [(4, 4)]
    with wis.HostPipeline(1, shapes, 8, 32, 4) as pipe:
        assert pipe.deterministic == torch.are_deterministic_algorithms_enabled()
    with deterministic_mode():
        with wis.HostPipeline(1, shapes, 8, 32, 4) as pipe:
            assert pipe.deterministic
        with wis.HostPipeline(1, shapes, 8, 32, 4, deterministic=False) as pipe:
            assert not pipe.deterministic


# ---------------------------------------------------------------------------- 6. the torch switch
def test_torch_switch_makes_the_python_entry_points_deterministic(wis):
    from weed_instance_segmentation_b200 import functional
    from weed_instance_segmentation_b200.synth import msda_inputs
    shapes = [(16, 16), (8, 8), (4, 4)]
    x = msda_inputs(2, shapes, dist="trained", seed=14, value_dtype=torch.bfloat16)
    xd = _device(x)

    def plain(fn):
        v, lo, a = (t.clone().requires_grad_(True) for t in xd[:3])
        with deterministic_mode():
            fn(v, lo, a).backward(xd[3])
        torch.cuda.synchronize()
        return v.grad, lo.grad, a.grad

    five = plain(lambda v, lo, a: wis.ms_deform_attn(v, shapes, None, lo, a))
    _assert_same_bits(five, plain(lambda v, lo, a: wis.ms_deform_attn(v, shapes, None, lo, a)), "ms_deform_attn")
    four = plain(lambda v, lo, a: wis.multi_scale_deformable_attention(v, shapes, lo, a))
    _assert_same_bits(five, four, "multi_scale_deformable_attention")
    order = functional.query_order_2d(shapes, functional._TILE, "cuda") if functional._USE_ORDER else None
    _assert_same_bits(five, _abi_backward(xd, shapes, _flag(), order), "the C ABI with the flag")
    assert not torch.are_deterministic_algorithms_enabled()

    value, off, logits, ref, go = _fused_inputs(2, shapes, torch.bfloat16, seed=15)

    def fused(r):
        v, o, lg = (t.clone().requires_grad_(True) for t in (value, off, logits))
        with deterministic_mode():
            wis.ms_deform_attn_fused(v, shapes, None, o, lg, r).backward(go)
        torch.cuda.synchronize()
        return v.grad, o.grad, lg.grad

    for r in (ref, None):
        _assert_same_bits(fused(r), fused(r), "ms_deform_attn_fused")
        order = functional.query_order_2d(shapes, functional._TILE, "cuda") if functional._USE_ORDER else None
        _assert_same_bits(fused(r), _abi_backward_fused((value, off, logits, r, go), shapes, _flag(), order),
                          "fused: the C ABI with the flag")


# ---------------------------------------------------------------------------- 7. model level
_MODEL_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
import weed_instance_segmentation_b200 as wis
from weed_instance_segmentation_b200 import modules, pixel_decoder, synth, train

model = train.build_model("swin_tiny_test", num_labels=3, seed=0, decoder_layers=4, encoder_layers=6, num_queries=20,
                          train_num_points=256).cuda().train()
g = torch.Generator(device="cuda").manual_seed(1)
with torch.no_grad():
    for name, p in model.named_parameters():
        if name.endswith("self_attn.sampling_offsets.bias"):
            p.add_(0.1 + 0.3 * torch.rand(p.shape, generator=g, device="cuda"))
modules.convert_pixel_decoder(model)
pixel_decoder.convert_pixel_decoder_inputs(model)
decoder = model.model.pixel_level_module.decoder
batch = synth.collate_batch(2, 128, 160, num_classes=3, max_instances=4, seed=3, device="cuda")
with torch.no_grad():
    features = model.model.pixel_level_module.encoder(batch["pixel_values"]).feature_maps
weights = None


def grads(deterministic):
    global weights
    torch.use_deterministic_algorithms(deterministic)
    try:
        model.zero_grad(set_to_none=True)
        out = decoder([f.detach() for f in features])
        # the encoder outputs only: the FPN tail's bilinear upsampling has no deterministic backward in torch
        feats = out.multi_scale_features
        if weights is None:
            gw = torch.Generator(device="cuda").manual_seed(7)
            weights = [torch.randn(f.shape, generator=gw, device="cuda") for f in feats]
        loss = sum((f * w).sum() for f, w in zip(feats, weights))
        loss.backward()
        torch.cuda.synchronize()
        return {k: p.grad.clone() for k, p in decoder.named_parameters() if p.grad is not None}
    finally:
        torch.use_deterministic_algorithms(False)


a, b, c = grads(True), grads(True), grads(False)
assert set(a) == set(b) == set(c) and len(a) > 20, (len(a), len(b), len(c))
for k in a:
    assert torch.equal(a[k].view(torch.uint8), b[k].view(torch.uint8)), f"not reproducible: {k}"
    rel = ((a[k] - c[k]).abs().max() / c[k].abs().max().clamp_min(1e-30)).item()
    assert rel < 1e-2 or c[k].abs().max() <= 1e-6, (k, rel)
print("model ok", len(a))
"""


def test_model_pixel_decoder_gradients_reproducible(wis):
    pytest.importorskip("transformers")
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    res = subprocess.run([sys.executable, "-s", "-c", _MODEL_SCRIPT, ROOT], env=env, capture_output=True, text=True,
                         timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "model ok" in res.stdout
