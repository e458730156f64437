#!/usr/bin/env python
"""Benchmark of the MSDeformAttn hot path (BASELINE.json config 2) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dist init|trained|adversarial]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one forward + one backward of the op on one batch of synthetic input:
B = 8 images of 1024x1024 per GPU (levels 32^2 / 64^2 / 128^2, S = Q = 21504, H = 8, D = 32, L = 3,
P = 4), bf16 values/weights, fp32 locations -- the configuration BASELINE.json's metric is quoted on.
Ranks work on independent batches (the path shards by image; no data-path collective), so scaling
is weak and `value` = images all ranks processed / max-over-ranks device time.

Output: ONE JSON line on rank 0 (see DESIGN.md "Measurement" for every key).
`--impl reference` times the reference's own implementation (HF `multi_scale_deformable_attention`,
M2F:798-837, fp32, autograd backward) on the host CPU with all threads, on a bounded sample.
`--dump-outputs DIR` writes what the last timed step computed (the op's output and the three input gradients) as
DIR/<name>.npy in float32 (rank 0's batch; a fixed seeded sample of an array larger than DUMP_SAMPLE elements); the
inputs are seeded, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SHAPES_C2 = [(32, 32), (64, 64), (128, 128)]
B_PER_GPU = 8
H, D, L, P = 8, 32, 3, 4
METRIC = "msda_fwd_bwd_throughput"
UNIT = "images/s"
OUTPUT_NAMES = ("output", "grad_value", "grad_sampling_locations", "grad_attention_weights")
DUMP_SAMPLE = 1 << 21  # elements kept of a larger output: four float32 arrays of 8 MB, 32 MB in all


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--dist", choices=["init", "trained", "adversarial"], default="init")
    ap.add_argument("--dtype", choices=["bf16", "fp32"], default="bf16")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the other location distributions and fp32")
    ap.add_argument("--no-train", action="store_true", help="skip the `train` block (config 3 DDP fine-tune step)")
    ap.add_argument("--no-gpu-reference", action="store_true", help="skip timing the reference function on the GPU")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


def dump_outputs(directory, tensors):
    """Save each tensor as ``directory/<name>.npy`` in float32: whole when it has at most DUMP_SAMPLE elements, else
    the same DUMP_SAMPLE elements of its flattened form on every run (seeded, ascending indices)."""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    for name, t in tensors.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_SAMPLE, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(directory, f"{name}.npy"), t.float().cpu().numpy())


def algorithmic_bytes(B, S, dtype):
    """SURVEY.md section 8(d): compulsory traffic, Q == S, H=8 D=32 L=3 P=4."""
    fwd, bwd = (1984, 3456) if dtype == "bf16" else (3200, 5376)
    return fwd * B * S, bwd * B * S


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def library_source_hash():
    """sha256 over the CUDA sources the library is built from (what an ncu capture has to be taken on)."""
    import hashlib
    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "weed_instance_segmentation_b200", "csrc")
    for name in sorted(os.listdir(csrc)):
        if name.endswith((".cu", ".cuh")):
            with open(os.path.join(csrc, name), "rb") as f:
                h.update(name.encode() + b"\0" + f.read())
    return h.hexdigest()[:16]


def recorded_traffic(kernel):
    """dram bytes per launch from the committed ncu capture (profiles/traffic.json) -- only if that capture was taken
    on the library built from today's sources (the file carries their hash); a stale capture reads as null."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            rec = json.load(f)
        if rec.get("source_hash") != library_source_hash():
            return None
        return rec.get(kernel)
    except Exception:
        return None


class ClockSampler:
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.stop = [], set(), threading.Event()
        self.max_mhz, self.thread = None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4),
        }
        while not self.stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.005)

    def __enter__(self):
        if self.nv is not None:
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
        return self

    def __exit__(self, *exc):
        self.stop.set()
        if self.thread is not None:
            self.thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------- reference arm
def reference_step_fn(n_images, q_fraction=1.0):
    """One fwd+bwd of the reference implementation on the CPU (fp32, autograd), as a closure."""
    import torch
    from oracle.hf_reference import hf_forward_torch
    from weed_instance_segmentation_b200.synth import msda_inputs
    x = msda_inputs(n_images, SHAPES_C2, num_heads=H, head_dim=D, num_points=P, dist="init", seed=0)
    nq = max(1, int(round(x["sampling_locations"].shape[1] * q_fraction)))
    v = x["value"].requires_grad_(True)
    lo = x["sampling_locations"][:, :nq].contiguous().requires_grad_(True)
    a = x["attention_weights"][:, :nq].contiguous().requires_grad_(True)
    go = x["grad_out"][:, :nq].contiguous()

    def step():
        v.grad = lo.grad = a.grad = None
        out = hf_forward_torch(v, SHAPES_C2, lo, a)
        out.backward(go)
        return out, v.grad, lo.grad, a.grad

    return step, nq


def run_reference(args, rank, world):
    import torch
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    # one image (B=1 of the B=8 batch) with ALL its queries per step: the same per-image work as the b200 arm, fp32
    step, nq = reference_step_fn(1)
    step()  # cold call (imports, allocator) -- never timed
    warmup, steps = args.warmup, args.steps
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        res = step()
    dt = (time.perf_counter() - t0) / steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(OUTPUT_NAMES, res)))
    S = sum(h * w for h, w in SHAPES_C2)
    value = 1.0 / dt
    sample = (f"{steps} steps of 1 image each (B=1 of the B=8 batch, all {nq} of {S} queries), reference HF function "
              f"M2F:798-837 in fp32 with autograd backward, {dt * 1e3:.0f} ms per image")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config("init", "fp32"),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def workload_config(dist, dtype):
    return {
        "workload": "BASELINE.json configs[1]: MSDeformAttn fwd+bwd op microbench, batch 8 per GPU, 1024x1024 input "
                    "(levels 32^2/64^2/128^2, S=Q=21504), H=8 D=32 L=3 P=4",
        "batch_per_gpu": B_PER_GPU, "spatial_shapes": SHAPES_C2, "locations": dist,
        "contract": "value/out/grads bf16, sampling_locations fp32, attention_weights bf16, fp32 accumulate"
        if dtype == "bf16" else "all fp32",
        "l2": "no flush: each step touches ~0.9 GB (> 126 MB L2), inputs 341 MB",
    }


# --------------------------------------------------------------------------------------------- b200 arm
class Problem:
    """Device buffers + descriptor for direct C-ABI calls (no autograd in the timed region)."""

    def __init__(self, dist, dtype, device, seed, shapes=None, batch=None):
        import torch
        from weed_instance_segmentation_b200 import _cabi, functional
        from weed_instance_segmentation_b200.synth import msda_inputs
        self.torch, self.cabi = torch, _cabi
        self.lib = _cabi.load()
        tdt = torch.bfloat16 if dtype == "bf16" else torch.float32
        shapes = SHAPES_C2 if shapes is None else shapes
        batch = B_PER_GPU if batch is None else batch
        self.shapes, self.batch = shapes, batch
        x = msda_inputs(batch, shapes, num_heads=H, head_dim=D, num_points=P, dist=dist, seed=seed,
                        device=device, value_dtype=tdt)
        self.x = x
        self.value, self.loc, self.attn, self.go = (x["value"], x["sampling_locations"], x["attention_weights"],
                                                    x["grad_out"])
        self.S = self.value.shape[1]
        self.out = torch.empty_like(self.go)
        self.gv, self.gl, self.ga = torch.empty_like(self.value), torch.empty_like(self.loc), torch.empty_like(self.attn)
        code = _cabi.BF16 if dtype == "bf16" else _cabi.F32
        lsi = x["level_start_index"].tolist()
        self.order = functional.query_order_2d(shapes, functional._TILE, device) if functional._USE_ORDER else None
        self.flags = _cabi.FLAG_BF16_ATOMICS if (functional._BF16_ATOMICS and dtype == "bf16") else 0
        if functional._BWD_V1:
            self.flags |= _cabi.FLAG_BWD_V1
        if functional._BWD_V2:
            self.flags |= _cabi.FLAG_BWD_V2
        self.desc, self._keep = _cabi.make_desc(batch, self.S, self.S, H, D, L, P, code, code, shapes, lsi, self.flags)
        self.pdesc, self._keep2 = _cabi.make_desc(batch, self.S, self.S, H, D, L, P, code, code, shapes, lsi,
                                                  self.flags | _cabi.FLAG_PROFILE)
        nws = int(self.lib.msda_b200_backward_workspace_bytes(self.desc))
        self.ws = torch.empty(nws, dtype=torch.uint8, device=device) if nws else None
        self.nws = nws
        self.stream = torch.cuda.current_stream().cuda_stream

    def _p(self, t):
        return t.data_ptr() if t is not None else None

    def fwd(self, desc=None):
        self.cabi.check(self.lib.msda_b200_forward(desc or self.desc, self._p(self.value), self._p(self.loc),
                                                   self._p(self.attn), self._p(self.out), self._p(self.order), self.stream))

    def bwd(self, desc=None):
        self.cabi.check(self.lib.msda_b200_backward(desc or self.desc, self._p(self.value), self._p(self.loc),
                                                    self._p(self.attn), self._p(self.go), self._p(self.gv), self._p(self.gl),
                                                    self._p(self.ga), self._p(self.ws), self.nws, self._p(self.order),
                                                    self.stream))

    def step(self):
        self.fwd()
        self.bwd()


def time_steps(torch, fn, steps, warmup, barrier, finish=None):
    """W untimed + exactly K timed steps, barrier + synchronize on both sides, CUDA events.
    `finish` (optional) joins work `fn` enqueued on other streams back into the timed stream."""
    for _ in range(warmup):
        fn()
    if finish:
        finish()
    torch.cuda.synchronize()
    barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    if finish:
        finish()
    e1.record()
    torch.cuda.synchronize()
    barrier()
    return e0.elapsed_time(e1) / 1e3  # seconds for K steps


def profile_kernels(prob, iters):
    """Per-kernel device time from events the library records around each launch."""
    c = prob.cabi
    acc = {"fwd": [], "bwd_zero": [], "bwd_main": [], "bwd_convert": []}
    for _ in range(iters):
        prob.fwd(prob.pdesc)
        prob.bwd(prob.pdesc)
        prob.torch.cuda.synchronize()
        acc["fwd"].append(c.profile_ms(c.PROF_FWD))
        acc["bwd_zero"].append(c.profile_ms(c.PROF_BWD_ZERO))
        acc["bwd_main"].append(c.profile_ms(c.PROF_BWD_MAIN))
        if prob.nws:
            acc["bwd_convert"].append(c.profile_ms(c.PROF_BWD_CONVERT))
    return {k: (sum(v) / len(v) if v else 0.0) for k, v in acc.items()}


def e2e_steps(torch, wis, prob, steps, warmup, barrier):
    """The op over HOST (pinned) buffers through the package's host-buffer API (`HostPipeline`, the
    msda_b200_host_pipeline_* entry points): every step copies its inputs H2D and its results D2H inside the timed
    region; the pipeline overlaps the two copy directions with the kernels, image by image."""
    host_in = [t.detach().cpu().pin_memory() for t in (prob.value, prob.loc, prob.attn, prob.go)]
    pipe = wis.HostPipeline(prob.batch, prob.shapes, H, D, P, value_dtype=prob.value.dtype, chunk_images=2, slots=3)
    res = pipe.empty_outputs()
    secs = time_steps(torch, lambda: pipe.step(*host_in, **res), steps, warmup, barrier, finish=pipe.join)
    h2d, d2h = pipe.h2d_bytes_per_step, pipe.d2h_bytes_per_step
    # spot-check: the host results equal the device-buffer results of the same inputs
    prob.fwd()
    torch.cuda.synchronize()
    if not torch.equal(res["output"].view(prob.out.shape), prob.out.cpu()):
        raise SystemExit("e2e: host-pipeline output differs from the device-buffer call")
    pipe.close()
    return secs, h2d, d2h


def e2e_autograd_steps(torch, wis, prob, steps, warmup, barrier):
    """Un-pipelined comparison: torch copies + `ms_deform_attn` + autograd backward on one stream."""
    host_in = [t.detach().cpu().pin_memory() for t in (prob.value, prob.loc, prob.attn, prob.go)]
    host_out = None
    lsi = prob.x["level_start_index"]

    def step():
        nonlocal host_out
        v, lo, a, go = (t.to("cuda", non_blocking=True) for t in host_in)
        v.requires_grad_(True), lo.requires_grad_(True), a.requires_grad_(True)
        out = wis.ms_deform_attn(v, prob.shapes, lsi, lo, a)
        out.backward(go)
        res = (out.detach(), v.grad, lo.grad, a.grad)
        if host_out is None:
            host_out = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in res]
        for h, t in zip(host_out, res):
            h.copy_(t, non_blocking=True)

    return time_steps(torch, step, steps, warmup, barrier)


def gpu_reference_ms(torch, prob, autocast_bf16, iters=3):
    """The reference's own function (M2F:798-837) + autograd on THIS GPU: ms per fwd+bwd of the whole B=8 batch, run in
    slices of 2 images to bound its (B*H, D, Q, L*P) temporary (2 GB at B=8, M2F:833). fp32, or under autocast(bf16)."""
    from oracle.hf_reference import hf_forward_torch
    dt = torch.bfloat16 if autocast_bf16 else torch.float32
    v = prob.value.detach().to(dt)
    lo, a, go = prob.loc.detach(), prob.attn.detach().to(dt), prob.go.detach().to(dt)

    def step():
        for b0 in range(0, prob.batch, 2):
            sl = slice(b0, b0 + 2)
            rv, rl, ra = (t[sl].clone().requires_grad_(True) for t in (v, lo, a))
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast_bf16):
                out = hf_forward_torch(rv, prob.shapes, rl, ra)
            out.backward(go[sl].to(out.dtype))

    step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def copy_ceiling(torch, prob, steps, barrier):
    """Bare duplex copy of one step's e2e bytes (pinned H2D of the inputs on one stream, D2H of the results on another),
    every rank at once: the host-side ceiling the pipelined e2e leg can at best reach on this box."""
    host_in = [t.detach().cpu().pin_memory() for t in (prob.value, prob.loc, prob.attn, prob.go)]
    dev_out = [prob.out, prob.gv, prob.gl, prob.ga]
    host_out = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in dev_out]
    dev_in = [torch.empty_like(t, device="cuda") for t in host_in]
    s_in, s_out = torch.cuda.Stream(), torch.cuda.Stream()

    def step():
        with torch.cuda.stream(s_in):
            for d, h in zip(dev_in, host_in):
                d.copy_(h, non_blocking=True)
        with torch.cuda.stream(s_out):
            for h, d in zip(host_out, dev_out):
                h.copy_(d, non_blocking=True)

    def finish():
        torch.cuda.current_stream().wait_stream(s_in)
        torch.cuda.current_stream().wait_stream(s_out)

    def fork():
        s_in.wait_stream(torch.cuda.current_stream())
        s_out.wait_stream(torch.cuda.current_stream())

    def stepf():
        fork()
        step()

    secs = time_steps(torch, stepf, steps, 2, barrier, finish=finish)
    nbytes = sum(t.numel() * t.element_size() for t in host_in)
    return secs / steps, nbytes


def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import weed_instance_segmentation_b200 as wis
    from weed_instance_segmentation_b200 import _cabi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
    if local_rank == 0:
        from weed_instance_segmentation_b200 import build as _build
        _build.build()  # no-op when the in-tree library is current
    if world > 1:
        dist.barrier()
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)

    def barrier():
        if world > 1:
            dist.barrier()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    prob = Problem(args.dist, args.dtype, device, seed=rank)
    S = prob.S
    _cabi.launch_count(reset=True)
    with ClockSampler(local_rank) as clocks:
        secs = max_over_ranks(time_steps(torch, prob.step, args.steps, args.warmup, barrier))
    launches = _cabi.launch_count() // max(args.steps + args.warmup, 1)
    ms_step = secs / args.steps * 1e3
    value = world * B_PER_GPU * args.steps / secs
    if args.dump_outputs and rank == 0:  # before anything else reuses the problem's buffers
        dump_outputs(args.dump_outputs, dict(zip(OUTPUT_NAMES, (prob.out, prob.gv, prob.gl, prob.ga))))

    # per-kernel times (library-recorded events), fwd-only and bwd-only call times
    kern = profile_kernels(prob, min(args.steps, 20))
    fwd_ms = time_steps(torch, prob.fwd, args.steps, 3, barrier) / args.steps * 1e3
    bwd_ms = time_steps(torch, prob.bwd, args.steps, 3, barrier) / args.steps * 1e3

    peak, peak_src = measured_peak_gbs()
    ab_fwd, ab_bwd = algorithmic_bytes(B_PER_GPU, S, args.dtype)
    dominant = "bwd_main" if kern["bwd_main"] >= kern["fwd"] else "fwd"
    dom_bytes = ab_bwd if dominant == "bwd_main" else ab_fwd
    dom_ms = kern[dominant]
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    roofline = {
        "bound": "hbm",
        "kernel": (("msda_bwd_kernel" if (args.dtype != "bf16" or (prob.flags & _cabi.FLAG_BWD_V1)) else
                    "msda_bwd_sorted_kernel" if (prob.flags & (_cabi.FLAG_BWD_V2 | _cabi.FLAG_BF16_ATOMICS)) else
                    "msda_bwd_mma_kernel") if dominant == "bwd_main" else "msda_fwd_pair_kernel"),
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
        "algorithmic_bytes": dom_bytes, "kernel_ms": dom_ms, "traffic": recorded_traffic(dominant),
    }
    step_achieved = (ab_fwd + ab_bwd) / (ms_step * 1e-3) / 1e9
    roofline_step = {
        "what": "whole fwd+bwd step (forward kernel + zero-fill + backward kernel + bf16 convert)",
        "achieved": step_achieved, "peak": peak, "unit": "GB/s", "frac": step_achieved / peak,
        "algorithmic_bytes": ab_fwd + ab_bwd,
        "fwd": {"ms": fwd_ms, "frac": ab_fwd / (fwd_ms * 1e-3) / 1e9 / peak},
        "bwd": {"ms": bwd_ms, "frac": ab_bwd / (bwd_ms * 1e-3) / 1e9 / peak},
        "kernels_ms": kern,
        # dram bytes per launch of each kernel from the committed ncu capture (null when it predates today's sources);
        # the zero-fill is a memset of the fp32 accumulator
        "kernels_traffic": {k: recorded_traffic(k) for k in ("fwd", "bwd_main", "bwd_convert")},
    }

    # end to end through the public API with host buffers
    e2e_k = max(3, min(args.steps, 10))
    e2e_secs, h2d, d2h = e2e_steps(torch, wis, prob, e2e_k, 3, barrier)
    e2e_secs = max_over_ranks(e2e_secs)
    e2e = {"value": world * B_PER_GPU * e2e_k / e2e_secs, "unit": UNIT, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h, "steps": e2e_k, "ms_per_step": e2e_secs / e2e_k * 1e3,
           "api": "weed_instance_segmentation_b200.HostPipeline.step (msda_b200_host_pipeline_step), pinned host "
                  "buffers, 2 images per chunk, 3 staging slots"}
    ceil_secs, ceil_bytes = copy_ceiling(torch, prob, e2e_k, barrier)
    ceil_secs = max_over_ranks(ceil_secs)
    e2e["copy_ceiling"] = {
        "what": "bare duplex pinned copy of one step's bytes (H2D inputs + D2H results on two streams), all ranks at once",
        "ms_per_step": ceil_secs * 1e3, "images_per_s": world * B_PER_GPU / ceil_secs,
        "gbs_per_direction_per_rank": ceil_bytes / ceil_secs / 1e9, "fraction_reached": ceil_secs / (e2e_secs / e2e_k)}
    ag_secs = max_over_ranks(e2e_autograd_steps(torch, wis, prob, 3, 3, barrier))
    e2e["unpipelined"] = {"value": world * B_PER_GPU * 3 / ag_secs, "ms_per_step": ag_secs / 3 * 1e3,
                          "api": "torch copies + ms_deform_attn + autograd backward on one stream"}

    extras = {}
    if not args.no_extras and world == 1:
        for dname, dt in (("init", "bf16"), ("trained", "bf16"), ("adversarial", "bf16"), ("init", "fp32")):
            if (dname, dt) == (args.dist, args.dtype):
                continue
            p2 = Problem(dname, dt, device, seed=rank)
            s2 = time_steps(torch, p2.step, max(10, args.steps // 4), 3, barrier) / max(10, args.steps // 4)
            f2, b2 = algorithmic_bytes(B_PER_GPU, S, dt)
            extras[f"{dname}/{dt}"] = {"ms_per_step": s2 * 1e3, "images_per_s": B_PER_GPU / s2,
                                       "frac_of_hbm_peak": (f2 + b2) / s2 / 1e9 / peak}
            del p2
            torch.cuda.empty_cache()
        # the other BASELINE.json geometries the op sees (per layer): config 3 (966x1296, batch 16) fwd+bwd and
        # config 5 (2048x2048 inference, batch 4) forward only
        from weed_instance_segmentation_b200.synth import pixel_decoder_shapes
        n = max(10, args.steps // 4)
        p3 = Problem("init", "bf16", device, seed=rank, shapes=pixel_decoder_shapes(966, 1296), batch=16)
        s3 = time_steps(torch, p3.step, n, 3, barrier) / n
        extras["config3 966x1296 B=16 bf16 fwd+bwd"] = {
            "ms_per_step": s3 * 1e3, "images_per_s": 16 / s3,
            "frac_of_hbm_peak": sum(algorithmic_bytes(16, p3.S, "bf16")) / s3 / 1e9 / peak}
        del p3
        torch.cuda.empty_cache()
        p5 = Problem("init", "bf16", device, seed=rank, shapes=pixel_decoder_shapes(2048, 2048), batch=4)
        s5 = time_steps(torch, p5.fwd, n, 3, barrier) / n
        extras["config5 2048x2048 B=4 bf16 fwd only"] = {
            "ms_per_step": s5 * 1e3, "images_per_s": 4 / s5,
            "frac_of_hbm_peak": algorithmic_bytes(4, p5.S, "bf16")[0] / s5 / 1e9 / peak}
        del p5
        torch.cuda.empty_cache()

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        step, nq = reference_step_fn(1)
        step()  # warm-up
        n, t0 = 0, time.perf_counter()
        while n < 2 or (time.perf_counter() - t0 < 10.0 and n < 20):
            step()
            n += 1
        dt = (time.perf_counter() - t0) / n
        cpu_baseline = {"value": 1.0 / dt, "unit": UNIT, "cores": cores, "kind": "reference",
                        "sample": f"{n} fwd+bwd steps of 1 image (B=1 of the B=8 batch, all {nq} queries), reference "
                                  f"HF function M2F:798-837 in fp32 with autograd, {dt * 1e3:.0f} ms per image"}

    gpu_reference = None
    if rank == 0 and world == 1 and not args.no_gpu_reference:
        ref32 = gpu_reference_ms(torch, prob, False)
        ref16 = gpu_reference_ms(torch, prob, True)
        gpu_reference = {
            "what": "the reference's function (transformers M2F:798-837) + autograd on the same B200, same B=8 batch in "
                    "slices of 2 images (bounds its 2 GB temporary), CUDA events",
            "fp32_ms_per_step": ref32, "autocast_bf16_ms_per_step": ref16,
            "fp32_images_per_s": B_PER_GPU / ref32 * 1e3, "autocast_bf16_images_per_s": B_PER_GPU / ref16 * 1e3,
            "speedup_vs_fp32": ref32 / ms_step, "speedup_vs_autocast_bf16": ref16 / ms_step}
        torch.cuda.empty_cache()

    train_block = None
    if not args.no_train:
        # every rank takes part (DDP gradient all-reduce over NCCL); the op buffers are released first
        del prob
        torch.cuda.empty_cache()
        from weed_instance_segmentation_b200 import train as wtrain
        train_block = wtrain.bench_block(device, world, rank)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16" if args.dtype == "bf16" else "f32", "data": "synthetic",
            "config": workload_config(args.dist, args.dtype),
            "roofline": roofline, "roofline_step": roofline_step, "cpu_baseline": cpu_baseline, "e2e": e2e,
            "gpu_launches": launches * args.steps, "gpu_launches_per_step": launches,
            "clocks": clocks.summary(), "other_workloads": extras, "gpu_reference": gpu_reference, "train": train_block,
        }
        print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
