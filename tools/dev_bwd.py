"""Development check of the backward kernels on a GPU box: v3 (group-sorted, mma.sync) against v1 (per-corner
reductions) on a set of geometries, then their kernel times at BASELINE configs 2 and 3.

    python tools/dev_bwd.py [--quick]
"""
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from weed_instance_segmentation_b200 import _cabi, functional  # noqa: E402
from weed_instance_segmentation_b200.synth import msda_inputs  # noqa: E402

H, D, P = 8, 32, 4


class Prob:
    def __init__(self, batch, shapes, dist, heads=H, queries=None, seed=3, attn_dtype=torch.bfloat16):
        self.lib = _cabi.load()
        x = msda_inputs(batch, shapes, num_heads=heads, head_dim=D, num_points=P, dist=dist, seed=seed, device="cuda",
                        value_dtype=torch.bfloat16, num_queries=queries)
        self.value, self.loc, self.go = x["value"], x["sampling_locations"], x["grad_out"]
        self.attn = x["attention_weights"].to(attn_dtype)
        self.B, self.S, self.Q, self.heads, self.shapes = batch, self.value.shape[1], self.loc.shape[1], heads, shapes
        self.lsi = x["level_start_index"].tolist()
        self.order = (functional.query_order_2d(shapes, functional._TILE, "cuda") if self.Q == self.S else None)
        self.acode = _cabi.BF16 if attn_dtype == torch.bfloat16 else _cabi.F32
        self.stream = torch.cuda.current_stream().cuda_stream

    def run(self, flags, profile=False):
        desc, keep = _cabi.make_desc(self.B, self.S, self.Q, self.heads, D, len(self.shapes), P, _cabi.BF16, self.acode,
                                     self.shapes, self.lsi, flags | (_cabi.FLAG_PROFILE if profile else 0))
        gv, gl, ga = torch.empty_like(self.value), torch.empty_like(self.loc), torch.empty_like(self.attn)
        nws = int(self.lib.msda_b200_backward_workspace_bytes(desc))
        ws = torch.empty(nws, dtype=torch.uint8, device="cuda")
        p = lambda t: t.data_ptr() if t is not None and t.numel() else None  # noqa: E731
        _cabi.check(self.lib.msda_b200_backward(desc, p(self.value), p(self.loc), p(self.attn), p(self.go), p(gv), p(gl),
                                                p(ga), p(ws), nws, p(self.order), self.stream))
        torch.cuda.synchronize()
        ms = _cabi.profile_ms(_cabi.PROF_BWD_MAIN) if profile else None
        return (gv.float(), gl.float(), ga.float()), ms


def rel(a, b):
    return ((a.double() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30)).item()


def main():
    quick = "--quick" in sys.argv
    cases = [
        ("tiny", 1, [(8, 8), (16, 16), (32, 32)], "init", 2, None),
        ("odd", 2, [(8, 9), (10, 6), (1, 12)], "adversarial", 2, 37),
        ("onepx", 1, [(1, 1), (2, 3)], "adversarial", 1, 50),
        ("wide", 1, [(12, 300), (256, 20)], "trained", 8, 500),
        ("c2b1/init", 1, [(32, 32), (64, 64), (128, 128)], "init", 8, None),
        ("c2b1/trained", 1, [(32, 32), (64, 64), (128, 128)], "trained", 8, None),
        ("c2b1/adv", 1, [(32, 32), (64, 64), (128, 128)], "adversarial", 8, None),
        ("c3b1/init", 1, [(31, 41), (61, 81), (121, 162)], "init", 8, None),
    ]
    ok = True
    for tag, B, shapes, dist, heads, Q in cases:
        for adt in (torch.bfloat16, torch.float32):
            pr = Prob(B, shapes, dist, heads=heads, queries=Q, attn_dtype=adt)
            ref, _ = pr.run(_cabi.FLAG_BWD_V1)
            line = f"{tag:14s} attn={'bf16' if adt == torch.bfloat16 else 'f32 '}"
            got, _ = pr.run(0)
            errs = [rel(g, r) for g, r in zip(got, ref)]
            finite = all(torch.isfinite(g).all().item() for g in got)
            bad = (not finite) or max(errs) > 1e-2
            ok &= not bad
            line += f" | v3 gv={errs[0]:.2e} gl={errs[1]:.2e} ga={errs[2]:.2e}{' BAD' if bad else ''}"
            print(line, flush=True)
    if not quick:
        for tag, B, shapes in (("config2", 8, [(32, 32), (64, 64), (128, 128)]), ("config3", 16, [(31, 41), (61, 81), (121, 162)])):
            for dist in ("init", "trained", "adversarial"):
                pr = Prob(B, shapes, dist)
                line = f"{tag}/{dist:12s}"
                for name, flags in (("v1", _cabi.FLAG_BWD_V1), ("v3", 0)):
                    ts = []
                    for _ in range(8):
                        _, ms = pr.run(flags, profile=True)
                        ts.append(ms)
                    ts.sort()
                    line += f" | {name} {ts[len(ts) // 2]:.3f} ms"
                print(line, flush=True)
    print("OK" if ok else "FAILED")
    return 0 if ok else 1


if __name__ == "__main__":
    t0 = time.time()
    rc = main()
    print(f"{time.time() - t0:.1f} s")
    sys.exit(rc)
