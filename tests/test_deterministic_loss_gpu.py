"""Deterministic backwards of the loss path's point sampling and of the pixel decoder's bilinear upsampling on a B200,
and a whole converted training step under ``torch.use_deterministic_algorithms(True)``.

Bars: 1e-5 (fp32) / 8e-3 (bf16) relative against fp64 ``grid_sample`` as in ``test_point_sample_matches_grid_sample``;
1e-5 relative against fp64 autograd through ``F.interpolate``; the criterion and model bars of the existing tests.
"""
import contextlib
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_err

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@contextlib.contextmanager
def deterministic_mode(on=True):
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(on)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev)


@pytest.fixture(scope="module")
def lib():
    from weed_instance_segmentation_b200 import _cabi, build
    build.build()
    return _cabi.load()


def _same_bits(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.contiguous().view(torch.uint8),
                                                                     b.contiguous().view(torch.uint8))


# ---------------------------------------------------------------------------- 1. point_sample
# rows 0/5 and 2/7 share a plane; rows 8-10 put 3 x 3001 points on one 1x1 plane; source 2 is a uint8 mask
_SRC = np.array([0, 0, 1, 2, 1, 0, 2, 1, 3, 3, 3, 3])
_PLANE = np.array([4, 0, 2, 1, 0, 4, 0, 2, 0, 0, 0, 1])
_CROW = np.array([0, 1, 2, 3, 0, 2, 3, 2, 0, 1, 2, 3])


def _ps_problem(dtype):
    g = torch.Generator(device="cuda").manual_seed(0)
    a = torch.randn(5, 17, 23, device="cuda", generator=g).to(dtype)
    b = torch.randn(3, 64, 40, device="cuda", generator=g).to(dtype)
    c = (torch.rand(2, 9, 9, device="cuda", generator=g) > 0.5).to(torch.uint8)
    d = torch.randn(2, 1, 1, device="cuda", generator=g).to(dtype)
    coords = torch.rand(4, 3001, 2, device="cuda", generator=g) * 1.3 - 0.15      # some points outside
    coords[0, :3] = torch.tensor([[0.0, 0.0], [1.0, 1.0], [0.5, float("nan")]], device="cuda")
    go = torch.randn(len(_SRC), coords.shape[1], device="cuda", generator=g)
    return [a, b, c, d], coords, go


def _ps_grads(sources, coords, go, perm=None, stream=None, det=True):
    from weed_instance_segmentation_b200.point_sample import point_sample
    perm = np.arange(len(_SRC)) if perm is None else perm
    leaves = [s.clone().requires_grad_(s.dtype != torch.uint8) for s in sources]
    ctx = torch.cuda.stream(stream) if stream is not None else contextlib.nullcontext()
    with deterministic_mode(det), ctx:
        out = point_sample(leaves, _SRC[perm], _PLANE[perm], coords, _CROW[perm])
        out.backward(go[torch.from_numpy(perm).cuda()])
    torch.cuda.synchronize()
    return [s.grad for s in leaves if s.requires_grad]


def _ps_reference(sources, coords, go):
    safe = coords.double().clone()
    safe[0, 2] = 2.0  # grid_sample propagates NaN; the kernel treats it as "outside" (zero), like the MSDA op
    leaves = [s.detach().double().requires_grad_(s.dtype != torch.uint8) for s in sources]
    rows = []
    for s, p, r in zip(_SRC, _PLANE, _CROW):
        pts = safe[int(r)][None, :, None, :]
        rows.append(F.grid_sample(leaves[s][int(p)][None, None], 2.0 * pts - 1.0, align_corners=False)[0, 0, :, 0])
    with deterministic_mode(False):
        torch.stack(rows).backward(go.double())
    return [s.grad for s in leaves if s.requires_grad]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_point_sample_backward_reproducible_under_the_switch(lib, dtype):
    sources, coords, go = _ps_problem(dtype)
    plain = _ps_grads(sources, coords, go)
    # rows reordered among different planes (the rows of one plane keep their order): (source, plane) descending
    perm = np.lexsort((-_PLANE, -_SRC))
    assert not np.array_equal(perm, np.arange(len(_SRC)))
    permuted = _ps_grads(sources, coords, go, perm=perm)
    side = _ps_grads(sources, coords, go, stream=torch.cuda.Stream())
    for name, got in (("permuted rows", permuted), ("side stream", side)):
        for x, y in zip(plain, got):
            assert _same_bits(x, y), name
    assert all(g.dtype == dtype for g in plain)
    tol = 1e-5 if dtype == torch.float32 else 8e-3   # bf16: the gradient is rounded once on the way out
    want = _ps_reference(sources, coords, go)
    atomic = _ps_grads(sources, coords, go, det=False)
    for x, w, at in zip(plain, want, atomic):
        assert rel_err(x.float().cpu().numpy(), w.cpu().numpy()) <= tol
        assert rel_err(x.float().cpu().numpy(), at.float().cpu().numpy()) <= tol
    assert float(plain[2].abs().max()) > 0  # the 1x1 plane received its ~9000 points


# ---------------------------------------------------------------------------- 2. resize_bilinear
_RESIZE = [((2, 3, 121, 162), (242, 324)),   # exact 2x: the config-3 FPN step (at reduced batch x channels)
           ((1, 4, 7, 5), (16, 9)),          # non-integer up
           ((2, 2, 33, 10), (10, 33)),       # down in one axis, up in the other
           ((1, 3, 1, 1), (5, 4)),           # a 1-pixel input
           ((0, 3, 7, 5), (16, 9))]          # NC = 0


@pytest.mark.parametrize("shape,size", _RESIZE)
def test_resize_bilinear_backward(lib, shape, size):
    from weed_instance_segmentation_b200.pixel_decoder import resize_bilinear
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(shape, device="cuda", generator=g)
    go = torch.randn(shape[:2] + size, device="cuda", generator=g)

    def grad():
        xl = x.clone().requires_grad_(True)
        with deterministic_mode():
            y = resize_bilinear(xl, size)
            y.backward(go)
        torch.cuda.synchronize()
        assert torch.equal(y, F.interpolate(x, size=size, mode="bilinear", align_corners=False))
        return xl.grad

    first, second = grad(), grad()
    assert _same_bits(first, second)
    xd = x.double().requires_grad_(True)
    up = F.interpolate(xd, size=size, mode="bilinear", align_corners=False)
    up.backward(go.double())
    assert rel_err(first.cpu().numpy(), xd.grad.cpu().numpy()) <= 1e-5
    # adjoint identity <go, up(x)> = <grad_x, x>, in fp64
    lhs = float((go.double() * up.detach()).sum())
    rhs = float((first.double() * x.double()).sum())
    scale = float((go.double().abs() * up.detach().abs()).sum())
    assert abs(lhs - rhs) <= 1e-6 * max(scale, 1e-30)


def test_resize_bilinear_keeps_the_input_dtype(lib):
    from weed_instance_segmentation_b200.pixel_decoder import resize_bilinear
    x = torch.randn(2, 4, 9, 11, device="cuda").to(torch.bfloat16).requires_grad_(True)
    go = torch.randn(2, 4, 18, 22, device="cuda")
    with deterministic_mode():
        resize_bilinear(x, (18, 22)).float().backward(go)
    xf = x.detach().float().requires_grad_(True)
    F.interpolate(xf, size=(18, 22), mode="bilinear", align_corners=False).backward(go)
    assert x.grad.dtype == torch.bfloat16
    assert rel_err(x.grad.float().cpu().numpy(), xf.grad.cpu().numpy()) <= 8e-3


# ---------------------------------------------------------------------------- 3. the converted criterion
_CRITERION_SCRIPT = r"""
import copy, sys, torch
sys.path.insert(0, sys.argv[1])
sys.path.insert(0, sys.argv[2])
import numpy as np
from test_criterion_host import make_problem
from weed_instance_segmentation_b200.criterion import convert_criterion


def rel_err(a, b):
    a, b = a.double(), b.double()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def run(loss, masks, classes, mask_labels, class_labels, seed, det):
    torch.use_deterministic_algorithms(det)
    try:
        masks = [m.clone().requires_grad_(True) for m in masks]
        classes = [c.clone().requires_grad_(True) for c in classes]
        aux = [{"masks_queries_logits": m, "class_queries_logits": c} for m, c in zip(masks[:-1], classes[:-1])]
        torch.manual_seed(seed)
        out = loss(masks[-1], classes[-1], mask_labels, class_labels, aux)
        sum(v * (i + 1) for i, v in enumerate(out.values())).backward()
        torch.cuda.synchronize()
        return out, [m.grad for m in masks], [c.grad for c in classes]
    finally:
        torch.use_deterministic_algorithms(False)


# BASELINE config 4 geometry of the loss: 10 layers, batch 8, 100 queries, 256x256 logits, 1024x1024 targets
loss, masks, classes, mask_labels, class_labels = make_problem(
    1, B=8, Q=100, C=5, L=10, h=256, w=256, H=1024, W=1024, n_tgt=(3, 9, 14, 1, 20, 7, 5, 11), num_points=12544)
loss = loss.cuda()
masks, classes = [m.cuda() for m in masks], [c.cuda() for c in classes]
mask_labels, class_labels = [m.cuda() for m in mask_labels], [c.cuda() for c in class_labels]
want, gm_want, gc_want = run(loss, masks, classes, mask_labels, class_labels, 3, det=False)
mine = convert_criterion(copy.deepcopy(loss))
runs = [run(mine, masks, classes, mask_labels, class_labels, 3, det=True) for _ in range(2)]
for (o1, gm1, gc1), (o2, gm2, gc2) in zip(runs, runs[1:]):
    for a, b in zip(gm1 + gc1, gm2 + gc2):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), "gradients differ between runs"
got, gm_got, gc_got = runs[0]
for k in want:
    assert torch.allclose(got[k], want[k], rtol=1e-4, atol=1e-6), (k, float(got[k]), float(want[k]))
for a, b in zip(gm_got, gm_want):
    assert rel_err(a, b) <= 1e-3, rel_err(a, b)
for a, b in zip(gc_got, gc_want):
    assert rel_err(a, b) <= 1e-3, rel_err(a, b)
print("criterion ok")
"""


def _run_script(script, *args):
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    res = subprocess.run([sys.executable, "-s", "-c", script, ROOT, *args], env=env, capture_output=True, text=True,
                         timeout=1200)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    return res.stdout


def test_converted_criterion_reproducible_under_the_switch(lib):
    pytest.importorskip("transformers")
    assert "criterion ok" in _run_script(_CRITERION_SCRIPT, os.path.join(ROOT, "tests"))


# ---------------------------------------------------------------------------- 4. a whole training step
_STEP_SCRIPT = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
from weed_instance_segmentation_b200 import synth, train

model = train.build_model("swin_tiny_test", num_labels=3, seed=0, decoder_layers=4, encoder_layers=6, num_queries=20,
                          train_num_points=256).cuda().train()
train.use_b200_path(model)
batch = synth.collate_batch(2, 128, 160, num_classes=3, max_instances=4, seed=3, device="cuda")


def step(deterministic, amp):
    torch.use_deterministic_algorithms(deterministic)
    try:
        model.zero_grad(set_to_none=True)
        torch.manual_seed(11)
        ctx = torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp)
        with ctx:
            out = model(pixel_values=batch["pixel_values"], mask_labels=batch["mask_labels"],
                        class_labels=batch["class_labels"])
        out.loss.backward()
        torch.cuda.synchronize()
        return float(out.loss.detach()), {k: p.grad.clone() for k, p in model.named_parameters() if p.grad is not None}
    finally:
        torch.use_deterministic_algorithms(False)


# Against the switch-off step the gradients agree as a whole, not element by element: the loss's importance sampling
# (top-k of |logit|) and the Hungarian matching are discontinuous in the logits, so the last-bit differences between
# the two settings' kernels move a few sampled points (in fp32 one decoder weight's gradient differs by 2.3e-2 of its
# maximum, the whole gradient by 5e-4 of its norm, on a B200). Under bf16 autocast the two settings also round to bf16
# in different kernels, and the discontinuities amplify that (0.24 of the norm on this random-init model), so there
# only the losses are compared.
for amp in (False, True):
    (la, a), (lb, b), (lc, c) = step(True, amp), step(True, amp), step(False, amp)
    assert set(a) == set(b) == set(c) and len(a) > 100, (len(a), len(b), len(c))
    for k in a:
        assert torch.equal(a[k].view(torch.uint8), b[k].view(torch.uint8)), f"not reproducible ({amp}): {k}"
    assert la == lb and abs(la - lc) <= 1e-2 * abs(lc), (amp, la, lc)
    diff = sum(float((a[k].double() - c[k].double()).pow(2).sum()) for k in a) ** 0.5
    ref = sum(float(c[k].double().pow(2).sum()) for k in a) ** 0.5
    assert amp or diff <= 1e-2 * ref, (amp, diff / ref)
    print("step ok", amp, len(a), la, lc, diff / ref)
"""


def test_whole_training_step_reproducible_under_the_switch(lib):
    pytest.importorskip("transformers")
    out = _run_script(_STEP_SCRIPT)
    assert "step ok False" in out and "step ok True" in out
