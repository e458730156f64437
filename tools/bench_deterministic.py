"""Cost of the deterministic backward (MSDA_B200_FLAG_DETERMINISTIC) next to the default one, on one GPU.

For each workload: device time of one msda_b200_backward call from CUDA events (mean over --iters calls after
--warmup), the workspace each mode asks for, and -- from a separate torch.profiler pass -- the device time of every
kernel of the deterministic call, so it is visible where the time goes. Workloads: BASELINE config 2 (B = 8,
1024^2 input, bf16) with init, trained and adversarial locations, config 3 (B = 16, 966 x 1296, bf16) and config 2
in the fp32 contract. The card's name and power limit are printed with the numbers.

    python tools/bench_deterministic.py [--iters 20] [--warmup 5] [--out results.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from weed_instance_segmentation_b200 import _cabi, functional  # noqa: E402
from weed_instance_segmentation_b200.synth import msda_inputs  # noqa: E402

C2 = [(32, 32), (64, 64), (128, 128)]
C3 = [(31, 41), (61, 81), (121, 162)]
WORKLOADS = [
    ("config2/init/bf16", 8, C2, "init", torch.bfloat16),
    ("config2/trained/bf16", 8, C2, "trained", torch.bfloat16),
    ("config2/adversarial/bf16", 8, C2, "adversarial", torch.bfloat16),
    ("config3/trained/bf16", 16, C3, "trained", torch.bfloat16),
    ("config2/trained/fp32", 8, C2, "trained", torch.float32),
]


class Problem:
    def __init__(self, batch, shapes, dist, dtype):
        self.lib = _cabi.load()
        x = msda_inputs(batch, shapes, dist=dist, seed=1, device="cuda", value_dtype=dtype)
        self.value, self.loc, self.attn, self.go = (x[k] for k in ("value", "sampling_locations", "attention_weights",
                                                                    "grad_out"))
        self.shapes, self.code = shapes, _cabi.BF16 if dtype == torch.bfloat16 else _cabi.F32
        self.order = functional.query_order_2d(shapes, functional._TILE, "cuda") if functional._USE_ORDER else None
        self.gv, self.gl, self.ga = (torch.empty_like(t) for t in (self.value, self.loc, self.attn))

    def desc(self, flags):
        B, S, H, D = self.value.shape
        _, Q, _, L, P, _ = self.loc.shape
        return _cabi.make_desc(B, S, Q, H, D, L, P, self.code, self.code, self.shapes,
                               functional._level_start(self.shapes, None), flags)

    def call(self, flags):
        """A closure that enqueues one backward (workspace allocated once), and the workspace size."""
        desc, keep = self.desc(flags)
        n = int(self.lib.msda_b200_backward_workspace_bytes(desc))
        ws = torch.empty(n, dtype=torch.uint8, device="cuda") if n else None
        order = self.order.data_ptr() if self.order is not None else None
        stream = torch.cuda.current_stream().cuda_stream

        def run():
            _cabi.check(self.lib.msda_b200_backward(desc, self.value.data_ptr(), self.loc.data_ptr(), self.attn.data_ptr(),
                                                    self.go.data_ptr(), self.gv.data_ptr(), self.gl.data_ptr(),
                                                    self.ga.data_ptr(), ws.data_ptr() if ws is not None else None, n,
                                                    order, stream))
            return keep
        return run, n


def time_ms(run, iters, warmup):
    for _ in range(warmup):
        run()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        run()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / iters


def kernel_breakdown(run, iters):
    """Device time per kernel name (ms per call), from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    run()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            run()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            out[e.key[:120]] = round(t / 1e3 / iters, 4)
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in q.split(","))
    except (OSError, IndexError, ValueError, subprocess.SubprocessError):
        name, power = torch.cuda.get_device_name(), "unknown"
    return {"gpu": name, "power_limit": power}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the results to this JSON file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_deterministic.py needs a CUDA device")
    result = {**card(), "iters": args.iters, "workloads": {}}
    print(f"{result['gpu']}, power limit {result['power_limit']}")
    for tag, B, shapes, dist, dtype in WORKLOADS:
        prob = Problem(B, shapes, dist, dtype)
        default, ws_default = prob.call(0)
        det, ws_det = prob.call(_cabi.FLAG_DETERMINISTIC)
        t_default = time_ms(default, args.iters, args.warmup)
        t_det = time_ms(det, args.iters, args.warmup)
        row = {"default_ms": round(t_default, 4), "deterministic_ms": round(t_det, 4),
               "ratio": round(t_det / t_default, 2), "default_workspace_bytes": ws_default,
               "deterministic_workspace_bytes": ws_det, "deterministic_kernels_ms": kernel_breakdown(det, 5)}
        result["workloads"][tag] = row
        print(f"{tag:28s} default {t_default:7.3f} ms ({ws_default / 2**20:7.1f} MiB)   deterministic {t_det:7.3f} ms "
              f"({ws_det / 2**20:7.1f} MiB)   x{t_det / t_default:.2f}")
        for k, v in row["deterministic_kernels_ms"].items():
            print(f"    {v:8.4f} ms  {k}")
        del prob, default, det
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
