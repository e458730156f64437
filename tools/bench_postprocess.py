"""Instance post-processing on one GPU: Mask2FormerImageProcessor.post_process_instance_segmentation (transformers
5.5.0, "M2FIP") against weed_instance_segmentation_b200.post_process_instance_segmentation on the same inputs.

Workloads (Q = 100 queries, C = 3 classes, seeded random logits as in tests/test_postprocess_gpu.py):
  config3  evaluation shape of BASELINE config 3: batch 16, mask logits 242 x 324, targets 966 x 1296
  config5  BASELINE config 5: batch 4, mask logits 512 x 512, targets 2048 x 2048
each at threshold 0.5 and at 0.0 (every non-empty selection kept: M2FIP's worst case, up to 100 host paints per image).

M2FIP's cost is host synchronisation, so each call is timed by the host clock from a synchronised start to its return
(both functions return host maps, so the device is idle by then), and by CUDA events on the current stream. Means over
--iters calls after --warmup. The card's name and power limit are printed with the numbers.

    python tools/bench_postprocess.py [--iters 10] [--warmup 3] [--dtype float32] [--out results.json]
"""
import argparse
import json
import os
import sys
import time
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
from bench_deterministic import card  # noqa: E402
import weed_instance_segmentation_b200 as wis  # noqa: E402

WORKLOADS = {"config3": (16, (242, 324), (966, 1296)), "config5": (4, (512, 512), (2048, 2048))}


def inputs(B, hw, dtype, Q=100, C=3, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    cls = 2 * torch.randn(B, Q, C + 1, generator=g, device="cuda")
    cls.scatter_add_(2, torch.randint(0, C + 1, (B, Q, 1), generator=g, device="cuda"),
                     10 * torch.rand(B, Q, 1, generator=g, device="cuda"))
    masks = torch.randn(B, Q, *hw, generator=g, device="cuda") + 0.3 * torch.randn(B, Q, 1, 1, generator=g, device="cuda")
    return types.SimpleNamespace(class_queries_logits=cls.to(dtype), masks_queries_logits=masks.to(dtype))


def timed(fn, iters, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    wall, dev, out = [], [], None
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e0.record()
        out = fn()
        e1.record()
        wall.append((time.perf_counter() - t0) * 1e3)
        torch.cuda.synchronize()
        dev.append(e0.elapsed_time(e1))
    return sum(wall) / iters, sum(dev) / iters, out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dtype", default="float32", choices=("float32", "bfloat16"))
    ap.add_argument("--out", default=None, help="also write the results to this JSON file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_postprocess needs a CUDA device")
    from transformers import Mask2FormerImageProcessor
    m2fip = Mask2FormerImageProcessor().post_process_instance_segmentation
    dtype = getattr(torch, args.dtype)
    results = {"card": card(), "dtype": args.dtype, "iters": args.iters, "workloads": []}
    print(json.dumps(results["card"]))
    for name, (B, hw, target) in WORKLOADS.items():
        out = inputs(B, hw, dtype)
        kw0 = dict(target_sizes=[target] * B)
        for threshold in (0.5, 0.0):
            kw = dict(kw0, threshold=threshold)
            row = {"workload": name, "batch": B, "logits": list(hw), "target": list(target), "threshold": threshold}
            for arm, fn in (("m2fip", m2fip), ("b200", wis.post_process_instance_segmentation)):
                wall, dev, res = timed(lambda: fn(out, **kw), args.iters, args.warmup)
                row[arm] = {"ms_per_batch": round(wall, 3), "event_ms": round(dev, 3),
                            "images_per_s": round(B / wall * 1e3, 2),
                            "instances": sum(len(r["segments_info"]) for r in res)}
            row["speedup"] = round(row["m2fip"]["ms_per_batch"] / row["b200"]["ms_per_batch"], 1)
            results["workloads"].append(row)
            print(json.dumps(row), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
