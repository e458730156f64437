"""Cost of the loss path's and the FPN tail's deterministic backwards, and of a whole deterministic training step, on
one GPU: each item with torch.use_deterministic_algorithms on and off.

  point_sample  one backward of the converted criterion's point sampling at BASELINE config 4's loss geometry: 10
                layers of (800, 256, 256) fp32 mask logits, 700 gradient rows (70 matched masks x 10 layers) and 700
                uint8 target rows (1024 x 1024) without gradient, 12 544 points each. Includes the zero-filled
                gradient planes both modes allocate (2.1 GB).
  resize        the FPN tail's upsampling backward at config 3 (16 x 256 x 121 x 162 -> 242 x 324, fp32):
                pixel_decoder.resize_bilinear's gather (on) against torch's atomic upsample_bilinear2d_backward (off),
                and against what F.interpolate records under the switch (torch's decomposition, index_put backward).
  train_step    Trainer.step at config 3 (Swin-T, 966 x 1296, batch 16, fp32, the full B200 path), images/s; the
                switch also makes torch fill every torch.empty (torch.utils.deterministic.fill_uninitialized_memory),
                so a third arm runs it with that fill off.

Times are CUDA-event means after warm-up; a separate torch.profiler pass lists the kernels of each "on" arm. The card's
name and power limit are printed with the numbers.

    python tools/bench_deterministic_step.py [--iters 20] [--steps 6] [--out results.json]
"""
import argparse
import json
import os
import sys

os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")  # before cuBLAS is first used: the step's GEMMs need it

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)
from bench_deterministic import card, kernel_breakdown, time_ms  # noqa: E402
from weed_instance_segmentation_b200 import pixel_decoder, synth, train  # noqa: E402
from weed_instance_segmentation_b200.point_sample import point_sample  # noqa: E402


def switched(on, fn):
    def run():
        prev = torch.are_deterministic_algorithms_enabled()
        torch.use_deterministic_algorithms(on)
        try:
            fn()
        finally:
            torch.use_deterministic_algorithms(prev)
    return run


def point_sample_problem():
    g = torch.Generator(device="cuda").manual_seed(0)
    L, BQ, M, K = 10, 800, 70, 12544
    logits = [torch.randn(BQ, 256, 256, device="cuda", generator=g).requires_grad_(True) for _ in range(L)]
    n_tgt = (3, 9, 14, 1, 20, 7, 5, 11)
    targets = [(torch.rand(n, 1024, 1024, device="cuda", generator=g) > 0.6).to(torch.uint8) for n in n_tgt]
    rng = np.random.default_rng(0)
    pred_plane = np.concatenate([rng.choice(BQ, M, replace=False) for _ in range(L)])
    img = rng.integers(0, len(n_tgt), M)
    tgt_plane = np.array([rng.integers(0, n_tgt[i]) for i in img])
    src = np.concatenate([np.repeat(np.arange(L), M), np.tile(L + img, L)])
    plane = np.concatenate([pred_plane, np.tile(tgt_plane, L)])
    crow = np.concatenate([np.arange(L * M)] * 2)
    coords = torch.rand(L * M, K, 2, device="cuda", generator=g)
    out = point_sample(logits + targets, src, plane, coords, crow)
    go = torch.randn(out.shape, device="cuda", generator=g)
    return lambda: torch.autograd.grad(out, logits, go, retain_graph=True)


def resize_problem():
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(16, 256, 121, 162, device="cuda", generator=g).requires_grad_(True)
    go = torch.randn(16, 256, 242, 324, device="cuda", generator=g)
    y_det = pixel_decoder.resize_bilinear(x, (242, 324))
    y_ref = F.interpolate(x, size=(242, 324), mode="bilinear", align_corners=False)
    torch.use_deterministic_algorithms(True)
    try:  # what F.interpolate records under the switch: torch's decomposition, with an index_put backward
        y_decomp = F.interpolate(x, size=(242, 324), mode="bilinear", align_corners=False)
    finally:
        torch.use_deterministic_algorithms(False)
    det = lambda: torch.autograd.grad(y_det, x, go, retain_graph=True)
    ref = lambda: torch.autograd.grad(y_ref, x, go, retain_graph=True)
    decomp = lambda: torch.autograd.grad(y_decomp, x, go, retain_graph=True)
    return det, ref, decomp


def train_images_per_s(trainer, batches, on, fill, steps, warmup):
    prev = torch.are_deterministic_algorithms_enabled(), torch.utils.deterministic.fill_uninitialized_memory
    torch.use_deterministic_algorithms(on)
    torch.utils.deterministic.fill_uninitialized_memory = fill
    try:
        secs = train.throughput(trainer, batches, steps, warmup, prefetch=True)
    finally:
        torch.use_deterministic_algorithms(prev[0])
        torch.utils.deterministic.fill_uninitialized_memory = prev[1]
    return batches[0]["pixel_values"].shape[0] * steps / secs


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--steps", type=int, default=6, help="timed training steps per arm")
    ap.add_argument("--out", default=None, help="also write the results to this JSON file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_deterministic_step.py needs a CUDA device")
    result = {**card(), "iters": args.iters}
    print(f"{result['gpu']}, power limit {result['power_limit']}", flush=True)

    bwd = point_sample_problem()
    on, off = switched(True, bwd), switched(False, bwd)
    result["point_sample_backward"] = {"on_ms": time_ms(on, args.iters, args.warmup),
                                       "off_ms": time_ms(off, args.iters, args.warmup),
                                       "on_kernels_ms": kernel_breakdown(on, 3)}
    del bwd, on, off
    torch.cuda.empty_cache()

    det, ref, decomp = resize_problem()
    on, off, torch_on = switched(True, det), switched(False, ref), switched(True, decomp)
    result["resize_backward"] = {"on_ms": time_ms(on, args.iters, args.warmup),
                                 "off_ms": time_ms(off, args.iters, args.warmup),
                                 "torch_on_ms": time_ms(torch_on, args.iters, args.warmup),
                                 "on_kernels_ms": kernel_breakdown(on, 3), "off_kernels_ms": kernel_breakdown(off, 3)}
    del det, ref, decomp, on, off, torch_on
    torch.cuda.empty_cache()

    model = train.build_model("swin_t", num_labels=3, seed=0)
    train.use_b200_path(model, "modules")
    trainer = train.Trainer(model, "cuda")
    batches = [synth.collate_batch(16, 966, 1296, num_classes=3, seed=i, mask_dtype=torch.uint8, pin_memory=True)
               for i in range(2)]
    result["train_step_images_per_s"] = {
        "off": train_images_per_s(trainer, batches, False, True, args.steps, args.warmup),
        "on": train_images_per_s(trainer, batches, True, True, args.steps, args.warmup),
        "on_without_fill": train_images_per_s(trainer, batches, True, False, args.steps, args.warmup),
        "off_again": train_images_per_s(trainer, batches, False, True, args.steps, args.warmup),
    }
    for k in ("point_sample_backward", "resize_backward"):
        r = result[k]
        print(f"{k:24s} on {r['on_ms']:8.3f} ms   off {r['off_ms']:8.3f} ms"
              + (f"   torch's own under the switch {r['torch_on_ms']:8.3f} ms" if "torch_on_ms" in r else ""))
        for name, ms in r["on_kernels_ms"].items():
            print(f"    on  {ms:8.4f} ms  {name}")
        for name, ms in r.get("off_kernels_ms", {}).items():
            print(f"    off {ms:8.4f} ms  {name}")
    print("train step images/s:", {k: round(v, 2) for k, v in result["train_step_images_per_s"].items()}, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
