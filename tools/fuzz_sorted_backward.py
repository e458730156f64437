"""Fuzz the group-sorted backward (v3, the default) against the per-corner backward (v1) on random geometries.

Both kernels compute the same sums in a different order, so bf16 outputs must agree to a couple of ulps
and the fp32 grad_loc to ~1e-5. Run on a GPU box:  python tools/fuzz_sorted_backward.py [n_cases] [seed]
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import weed_instance_segmentation_b200 as wis  # noqa: E402
from weed_instance_segmentation_b200 import functional as F  # noqa: E402


def random_case(rng):
    L = int(rng.integers(1, 5))
    kind = rng.choice(["tiny", "square", "wide", "tall", "mixed"])
    shapes = []
    for _ in range(L):
        if kind == "tiny":
            h, w = rng.integers(1, 6, 2)
        elif kind == "square":
            h = w = int(rng.integers(2, 90))
        elif kind == "wide":
            h, w = int(rng.integers(1, 12)), int(rng.integers(200, 700))
        elif kind == "tall":
            h, w = int(rng.integers(200, 700)), int(rng.integers(1, 12))
        else:
            h, w = rng.integers(1, 200, 2)
        shapes.append((int(h), int(w)))
    S = sum(h * w for h, w in shapes)
    B = int(rng.integers(1, 3))
    H = int(rng.choice([1, 2, 8]))
    Q = S if rng.random() < 0.4 else int(rng.integers(1, 700))
    dist = rng.choice(["uniform", "cluster", "outliers", "edges"])
    return B, shapes, H, Q, dist


def make_inputs(B, shapes, H, Q, dist, rng):
    L, P, D = len(shapes), 4, 32
    S = sum(h * w for h, w in shapes)
    value = torch.from_numpy(rng.standard_normal((B, S, H, D)).astype(np.float32)).bfloat16()
    if dist == "uniform":
        loc = rng.uniform(-0.2, 1.2, (B, Q, H, L, P, 2))
    elif dist == "cluster":
        c = rng.uniform(0, 1, (B, 1, H, L, 1, 2))
        loc = c + rng.normal(0, 0.02, (B, Q, H, L, P, 2))
    elif dist == "outliers":
        c = rng.uniform(0.3, 0.7, (B, 1, 1, L, 1, 2))
        loc = c + rng.normal(0, 0.01, (B, Q, H, L, P, 2))
        mask = rng.random((B, Q, H, L, P, 1)) < 0.02
        loc = np.where(mask, rng.uniform(-0.5, 1.5, loc.shape), loc)
    else:  # exact edges / centres / just outside
        loc = rng.choice([0.0, 1.0, 0.5, -1e-6, 1 + 1e-6, 0.25, 0.999999], (B, Q, H, L, P, 2))
    loc = torch.from_numpy(loc.astype(np.float32))
    attn = torch.softmax(torch.from_numpy(rng.standard_normal((B, Q, H, L * P)).astype(np.float32)), -1)
    attn = attn.view(B, Q, H, L, P).bfloat16()
    go = torch.from_numpy(rng.standard_normal((B, Q, H * D)).astype(np.float32)).bfloat16()
    return value, loc, attn, go


def run(value, shapes, loc, attn, go):
    v = value.cuda().requires_grad_(True)
    lo = loc.cuda().requires_grad_(True)
    a = attn.cuda().requires_grad_(True)
    out = wis.ms_deform_attn(v, shapes, None, lo, a)
    out.backward(go.cuda())
    torch.cuda.synchronize()
    return [t.detach().float().cpu() for t in (out, v.grad, lo.grad, a.grad)]


def rel(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-20)).item()


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 200
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 0
    rng = np.random.default_rng(seed)
    worst = {}
    for i in range(n):
        B, shapes, H, Q, dist = random_case(rng)
        value, loc, attn, go = make_inputs(B, shapes, H, Q, dist, rng)
        F._BWD_V1 = False
        v3 = run(value, shapes, loc, attn, go)
        F._BWD_V1 = True
        v1 = run(value, shapes, loc, attn, go)
        F._BWD_V1 = False
        assert torch.equal(v1[0], v3[0])
        errs = {"grad_value": rel(v3[1], v1[1]), "grad_loc": rel(v3[2], v1[2]), "grad_attn": rel(v3[3], v1[3])}
        bars = {"grad_value": 1.6e-2, "grad_loc": 1e-4, "grad_attn": 1.6e-2}
        for k, e in errs.items():
            worst[k] = max(worst.get(k, 0.0), e)
            if not (e <= bars[k]) or not all(torch.isfinite(t).all() for t in v3):
                print(f"MISMATCH case {i}: B={B} shapes={shapes} H={H} Q={Q} dist={dist}: {k} rel err {e:.3e}")
                sys.exit(1)
    print(f"fuzz ok: {n} cases, worst relative differences v3 vs v1: " + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))


if __name__ == "__main__":
    main()
