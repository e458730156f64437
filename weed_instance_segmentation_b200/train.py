"""Data-parallel training step around the B200 MSDeformAttn path.

Re-hosts the reference's training step (``/root/reference/models/mask2former/train.py:191-205``:
forward, ``loss / GRADIENT_ACCUMULATION``, backward, ``AdamW`` step every
``GRADIENT_ACCUMULATION`` micro-batches) as one process per GPU with
``torch.distributed`` (NCCL over NVLink). The path shards by image, so the only collective is
the bucketed gradient all-reduce that ``DistributedDataParallel`` overlaps with backward, plus a
4-byte all-reduce of ``num_masks`` (M2F:785-793) so that the DDP loss equals the single-process
loss on the same global batch.

Differences from the reference step that do not change results:
* ``loss.item()`` (train.py:204, a device->host sync every micro-batch) is replaced by an on-device
  running sum read once per logging interval;
* the first micro-batch of each accumulation window runs under ``no_sync()``.

There is no network here, so models are random-init from a config (the reference loads
``facebook/mask2former-swin-large-coco-instance``, ``/root/reference/config.py:4``) and batches are
synthetic (``synth.collate_batch``).
"""
from __future__ import annotations

import contextlib
import os
import time

import torch
import torch.distributed as dist

from . import hf_patch, modules, synth
from .linear import f32_gemm_available as _f32_gemm_available

# /root/reference/config.py:5-8
LEARNING_RATE = 5e-5
GRADIENT_ACCUMULATION = 2

BACKBONES = {
    # Swin-T / Swin-B / Swin-L shapes (the pixel-decoder MSDA dimensions do not depend on the backbone)
    "swin_t": dict(embed_dim=96, depths=[2, 2, 6, 2], num_heads=[3, 6, 12, 24], window_size=7),
    "swin_b": dict(embed_dim=128, depths=[2, 2, 18, 2], num_heads=[4, 8, 16, 32], window_size=12),
    "swin_l": dict(embed_dim=192, depths=[2, 2, 18, 2], num_heads=[6, 12, 24, 48], window_size=12),
    "swin_tiny_test": dict(embed_dim=24, depths=[1, 1, 1, 1], num_heads=[1, 2, 4, 8], window_size=4),
}


def build_model(backbone: str = "swin_t", num_labels: int = 3, seed: int = 0, **config_overrides):
    """Random-init ``Mask2FormerForUniversalSegmentation`` of the reference's architecture."""
    from transformers import Mask2FormerConfig, Mask2FormerForUniversalSegmentation, SwinConfig

    torch.manual_seed(seed)
    bb = SwinConfig(out_features=["stage1", "stage2", "stage3", "stage4"], **BACKBONES[backbone])
    cfg = Mask2FormerConfig(backbone_config=bb, num_labels=num_labels, **config_overrides)
    return Mask2FormerForUniversalSegmentation(cfg)


def use_b200_path(model, mode: str = "modules", criterion: bool = True) -> None:
    """Route the model's pixel-decoder MSDeformAttn through libmsda_b200.so.

    ``mode="function"`` rebinds the module-global function only (M2F:980); ``mode="modules"`` also
    swaps the encoder layers for the mirrors in ``modules.py`` (drops the per-layer isfinite sync) and, with
    ``criterion=True``, switches the loss / matcher to the batched path (``criterion.convert_criterion``).
    """
    hf_patch.install()
    if mode == "modules":
        modules.convert_pixel_decoder(model)
        from .pixel_decoder import convert_pixel_decoder_inputs
        convert_pixel_decoder_inputs(model)  # input assembly: GroupNorm + transpose + concat kernels, cached embeddings
        if criterion and hasattr(model, "criterion"):
            from .criterion import convert_criterion
            convert_criterion(model)


def install_distributed_num_masks() -> None:
    """All-reduce ``num_masks`` over the process group (what M2F:787-793 does through ``accelerate``)."""
    from transformers.models.mask2former import modeling_mask2former as m2f

    if getattr(m2f.Mask2FormerLoss.get_num_masks, "_b200_dist", False):
        return

    def get_num_masks(self, class_labels, device):
        num_masks = sum(len(classes) for classes in class_labels)
        num_masks = torch.as_tensor(num_masks, dtype=torch.float, device=device)
        world = 1
        if dist.is_available() and dist.is_initialized():
            dist.all_reduce(num_masks)
            world = dist.get_world_size()
        return torch.clamp(num_masks / world, min=1)

    get_num_masks._b200_dist = True
    m2f.Mask2FormerLoss.get_num_masks = get_num_masks


class Trainer:
    """The reference's step loop, one process per GPU."""

    def __init__(self, model, device, lr: float = LEARNING_RATE, grad_accum: int = GRADIENT_ACCUMULATION,
                 amp_dtype: torch.dtype | None = None, ddp: bool | None = None):
        self.device = torch.device(device)
        self.model = model.to(self.device)
        self.model.train()
        self.grad_accum = grad_accum
        self.amp_dtype = amp_dtype
        ddp = (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1) if ddp is None else ddp
        if ddp:
            install_distributed_num_masks()
            kw = dict(device_ids=[self.device.index]) if self.device.type == "cuda" else {}
            self.net = torch.nn.parallel.DistributedDataParallel(
                self.model, gradient_as_bucket_view=True, find_unused_parameters=False, **kw)
        else:
            self.net = self.model
        self.optimizer = torch.optim.AdamW(self.model.parameters(), lr=lr)  # train.py:174
        self.micro = 0
        self.loss_sum = torch.zeros((), device=self.device)
        self.loss_count = 0
        self._copy_stream = None

    def prefetch(self, batch: dict) -> dict:
        """Start copying a host batch to the device on a side stream; pass the result to ``step``.

        With page-locked host tensors (``synth.collate_batch(pin_memory=True)``, or a ``DataLoader`` with
        ``pin_memory=True``) the copy runs under the previous micro-batch's kernels; pageable tensors still work
        but block the host while they are staged (what the reference's ``.to(device)`` at train.py:193-195 does).
        """
        if self.device.type != "cuda":
            return batch
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=self.device)
        with torch.cuda.stream(self._copy_stream):
            out = {
                "pixel_values": batch["pixel_values"].to(self.device, non_blocking=True),
                "mask_labels": [m.to(self.device, non_blocking=True) for m in batch["mask_labels"]],
                "class_labels": [c.to(self.device, non_blocking=True) for c in batch["class_labels"]],
            }
            ready = torch.cuda.Event()
            ready.record()
        out["_ready"] = ready
        return out

    def step(self, batch: dict) -> torch.Tensor:
        """One micro-batch: train.py:192-202. Returns the (undivided) loss tensor, still on device."""
        pixel_values = batch["pixel_values"].to(self.device, non_blocking=True)
        mask_labels = [m.to(self.device, non_blocking=True) for m in batch["mask_labels"]]
        class_labels = [c.to(self.device, non_blocking=True) for c in batch["class_labels"]]
        if batch.get("_ready") is not None:  # came through prefetch(): order after the side-stream copies
            cur = torch.cuda.current_stream(self.device)
            cur.wait_event(batch["_ready"])
            for t in (pixel_values, *mask_labels, *class_labels):
                t.record_stream(cur)
        last = (self.micro + 1) % self.grad_accum == 0
        sync_ctx = contextlib.nullcontext() if (last or self.net is self.model) else self.net.no_sync()
        amp = (torch.autocast(self.device.type, dtype=self.amp_dtype) if self.amp_dtype is not None
               else contextlib.nullcontext())
        with sync_ctx:
            with amp:
                outputs = self.net(pixel_values=pixel_values, mask_labels=mask_labels, class_labels=class_labels)
            (outputs.loss / self.grad_accum).backward()
        if last:
            self.optimizer.step()
            self.optimizer.zero_grad(set_to_none=True)
        self.micro += 1
        loss = outputs.loss.detach().reshape(())
        self.loss_sum += loss
        self.loss_count += 1
        return loss

    def mean_loss(self) -> float:
        """Average loss since the last call (one device->host sync)."""
        v = float(self.loss_sum.item()) / max(self.loss_count, 1)
        self.loss_sum.zero_()
        self.loss_count = 0
        return v


def throughput(trainer: Trainer, batches: list, steps: int, warmup: int, prefetch: bool = False) -> float:
    """Seconds for ``steps`` micro-batches after ``warmup`` (device-timed on CUDA, barrier on both sides).
    Every micro-batch starts from HOST tensors; ``prefetch`` copies batch i+1 while batch i computes."""
    cuda = trainer.device.type == "cuda"
    multi = dist.is_available() and dist.is_initialized()
    if prefetch and cuda:
        def run(n):
            nxt = trainer.prefetch(batches[0])
            for i in range(n):
                cur, nxt = nxt, (trainer.prefetch(batches[(i + 1) % len(batches)]) if i + 1 < n else None)
                trainer.step(cur)
    else:
        def run(n):
            for i in range(n):
                trainer.step(batches[i % len(batches)])
    run(warmup)
    if cuda:
        torch.cuda.synchronize()
    if multi:
        dist.barrier()
    if cuda:
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    t0 = time.perf_counter()
    run(steps)
    if cuda:
        e1.record()
        torch.cuda.synchronize()
        secs = e0.elapsed_time(e1) / 1e3
    else:
        secs = time.perf_counter() - t0
    if multi:
        dist.barrier()
        t = torch.tensor([secs], dtype=torch.float64, device=trainer.device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        secs = float(t.item())
    return secs


def bench_block(device, world: int, rank: int, batch: int = 16, height: int = 966, width: int = 1296, classes: int = 3,
                steps: int = 4, warmup: int = 6, with_stock: bool = True) -> dict:
    """The ``train`` block of ``bench.py``'s JSON line: BASELINE config 3 (Swin-T fine-tune on 966x1296 synthetic
    crop_weed-shaped images, ``batch`` per GPU, fp32, AdamW, gradient accumulation 2 with ``no_sync`` on the first
    micro-batch) through :class:`Trainer` under the caller's process group -- the step of
    ``/root/reference/models/mask2former/train.py:191-205`` with the DDP gradient all-reduce over NCCL.

    Every rank calls this (DDP is collective). At ``world == 1`` the stock HF model is timed as well.
    Returns images/s over all ranks (max-over-ranks device time), ms per micro-batch and the all-reduce payload.
    """

    def run(impl: str, n_steps: int, n_warm: int) -> tuple[float, float, int]:
        torch.manual_seed(0)
        model = build_model("swin_t", classes)
        pinned = impl == "b200"
        if impl == "b200":
            use_b200_path(model, "modules", criterion=True)
        else:
            hf_patch.uninstall()  # the stock arm must run the reference's own function (M2F:798-837)
        model.to(device)
        if world > 1:
            install_distributed_num_masks()
        nparam = sum(p.numel() for p in model.parameters() if p.requires_grad)
        trainer = Trainer(model, device, ddp=world > 1)
        kw = dict(mask_dtype=torch.uint8, pin_memory=True) if pinned else {}
        batches = [synth.collate_batch(batch, height, width, classes, seed=rank * 1000 + i, **kw) for i in range(2)]
        secs = throughput(trainer, batches, n_steps, n_warm, prefetch=pinned)  # device time, max over ranks
        loss = trainer.mean_loss()
        del trainer, model, batches
        torch.cuda.empty_cache()
        return secs, loss, nparam

    secs, loss, nparam = run("b200", steps, warmup)
    out = {
        "config": f"BASELINE.json configs[2]: Mask2Former Swin-T fine-tune, synthetic {height}x{width}, {classes} classes, "
                  f"batch {batch} per GPU, fp32, AdamW, gradient accumulation {GRADIENT_ACCUMULATION}",
        "impl": "weed_instance_segmentation_b200.train.Trainer (MSDeformAttn modules + batched loss + pinned uint8 input)",
        "images_per_s": world * batch * steps / secs, "ms_per_step": secs / steps * 1e3, "micro_batches_timed": steps,
        "warmup": warmup, "n_gpus": world, "loss": loss,
        # one bucketed all-reduce of every gradient per optimizer step (every GRADIENT_ACCUMULATION micro-batches)
        "allreduce_bytes": nparam * 4 if world > 1 else 0, "allreduce_every_micro_batches": GRADIENT_ACCUMULATION,
        "params": nparam, "backend": "nccl" if world > 1 else None,
        # which GEMM the encoder layers' float32 projections ran on (csrc/gemm_f32.cu; falls back when the toolkit's
        # cuBLASLt >= 12.9 cannot be opened)
        "f32_projections": ("cuBLASLt CUBLAS_COMPUTE_32F_EMULATED_16BFX9 (bf16 tensor cores)" if _f32_gemm_available()
                            else "torch SGEMM"),
    }
    if with_stock and world == 1:
        s2, l2, _ = run("reference", steps, 3)
        out["stock_hf"] = {"images_per_s": batch * steps / s2, "ms_per_step": s2 / steps * 1e3, "loss": l2,
                           "what": "unmodified transformers Mask2FormerForUniversalSegmentation, same batches and step"}
    return out


def inference_throughput(model, device, args, rank: int) -> float:
    """Seconds for ``args.steps`` forward passes on one replica (max over ranks when run under torchrun)."""
    model = model.to(device).eval()
    g = torch.Generator().manual_seed(rank)
    pixel_values = torch.randn(args.batch, 3, args.height, args.width, generator=g).to(device)
    amp = (torch.autocast(device.type, dtype=torch.bfloat16) if args.amp == "bf16" else contextlib.nullcontext())
    multi = dist.is_available() and dist.is_initialized()

    def step():
        with torch.no_grad(), amp:
            return model(pixel_values=pixel_values)

    cuda = device.type == "cuda"
    for _ in range(args.warmup):
        step()
    if cuda:
        torch.cuda.synchronize()
    if multi:
        dist.barrier()
    if cuda:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    if cuda:
        e1.record()
        torch.cuda.synchronize()
        secs = e0.elapsed_time(e1) / 1e3
    else:
        secs = time.perf_counter() - t0  # the reference's CPU-runnable case (BASELINE config 1)
    if multi:
        dist.barrier()
        t = torch.tensor([secs], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        secs = float(t.item())
    return secs


def main(argv=None):
    import argparse
    import json

    ap = argparse.ArgumentParser(description="Synthetic Mask2Former fine-tune step benchmark (BASELINE config 3/4)")
    ap.add_argument("--backbone", default="swin_t", choices=sorted(BACKBONES))
    ap.add_argument("--height", type=int, default=966)
    ap.add_argument("--width", type=int, default=1296)
    ap.add_argument("--batch", type=int, default=16, help="images per GPU per micro-batch")
    ap.add_argument("--classes", type=int, default=3)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=6)
    ap.add_argument("--impl", choices=["b200", "b200-stock-loss", "b200-function", "reference"], default="b200")
    ap.add_argument("--amp", choices=["none", "bf16"], default="none")
    ap.add_argument("--input", choices=["auto", "reference", "b200"], default="auto",
                    help="host batch layout: reference = pageable float32 masks copied inside the step; b200 = pinned "
                         "uint8 masks prefetched on a side stream (needs the batched criterion); auto = b200 for "
                         "--impl b200, reference otherwise")
    ap.add_argument("--infer", action="store_true",
                    help="inference replicas instead of training (the reference's run_inference call shape, "
                         "/root/reference/models/mask2former/inference.py:25-30): eval(), no_grad, no collective")
    ap.add_argument("--deterministic", action="store_true",
                    help="torch.use_deterministic_algorithms(True): bit-identical gradients run to run (with --impl b200, "
                         "which converts the criterion); sets CUBLAS_WORKSPACE_CONFIG=:4096:8 unless it is set")
    args = ap.parse_args(argv)
    if args.deterministic:
        os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")  # read by cuBLAS when its first handle is made
        torch.use_deterministic_algorithms(True)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    device = torch.device("cuda", local) if torch.cuda.is_available() else torch.device("cpu")
    if device.type == "cuda":
        torch.cuda.set_device(device)
    if world > 1:
        dist.init_process_group("nccl" if device.type == "cuda" else "gloo",
                                **({"device_id": device} if device.type == "cuda" else {}))
    model = build_model(args.backbone, num_labels=args.classes, seed=0)
    if args.impl == "b200":
        use_b200_path(model, "modules")
    elif args.impl == "b200-stock-loss":
        use_b200_path(model, "modules", criterion=False)
    elif args.impl == "b200-function":
        use_b200_path(model, "function")
    if args.infer:
        secs = inference_throughput(model, device, args, rank)
        if rank == 0:
            print(json.dumps({
                "metric": "mask2former_inference_throughput", "value": world * args.batch * args.steps / secs,
                "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": secs / args.steps * 1e3, "impl": args.impl, "scaling": "weak (independent replicas)",
                "data": "synthetic", "dtype": "bf16 autocast" if args.amp == "bf16" else "f32",
                "config": {"workload": f"Mask2Former {args.backbone} inference, {args.height}x{args.width}, "
                                       f"batch {args.batch}/GPU"},
            }), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    trainer = Trainer(model, device, amp_dtype=torch.bfloat16 if args.amp == "bf16" else None)
    # Input path: the reference hands pageable float32 masks to `.to(device)` inside the step (train.py:193-195, a
    # DataLoader without pin_memory); the full B200 path keeps the binary masks at one byte per pixel in page-locked
    # memory and copies batch i+1 under batch i (`--input reference` forces the reference's layout for either arm).
    native_input = args.input == "b200" or (args.input == "auto" and args.impl == "b200")
    cuda = device.type == "cuda"
    batches = [synth.collate_batch(args.batch, args.height, args.width, num_classes=args.classes, seed=1000 * rank + i,
                                   mask_dtype=torch.uint8 if native_input else torch.float32,
                                   pin_memory=native_input and cuda)
               for i in range(2)]
    secs = throughput(trainer, batches, args.steps, args.warmup, prefetch=native_input)
    loss = trainer.mean_loss()
    if rank == 0:
        print(json.dumps({
            "metric": "mask2former_train_throughput", "value": world * args.batch * args.steps / secs, "unit": "images/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs / args.steps * 1e3,
            "impl": args.impl, "loss": loss, "scaling": "weak", "data": "synthetic",
            "dtype": "bf16 autocast" if args.amp == "bf16" else "f32",
            "config": {"workload": f"Mask2Former {args.backbone} fine-tune step, {args.height}x{args.width}, "
                                   f"{args.classes} classes, batch {args.batch}/GPU, AdamW lr {LEARNING_RATE}, "
                                   f"grad accumulation {GRADIENT_ACCUMULATION}",
                       "input": ("pinned uint8 masks, prefetched" if native_input
                                 else "pageable float32 masks copied inside the step (as the reference)")},
        }), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
