"""Three backward launches at BASELINE config 2 (bf16, one location distribution) for an ncu capture of one kernel:

    python tools/ncu_bwd_one.py [init|trained|adversarial] [v1|v3]
    ncu --set full --import-source on --clock-control none -k regex:msda_bwd -s 2 -c 1 -o gpurun_out/x python tools/ncu_bwd_one.py
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from dev_bwd import Prob  # noqa: E402
from weed_instance_segmentation_b200 import _cabi  # noqa: E402

dist = sys.argv[1] if len(sys.argv) > 1 else "init"
ver = sys.argv[2] if len(sys.argv) > 2 else "v3"
flags = {"v1": _cabi.FLAG_BWD_V1, "v3": 0}[ver]
pr = Prob(8, [(32, 32), (64, 64), (128, 128)], dist)
for _ in range(3):
    _, ms = pr.run(flags, profile=True)
print(f"{dist} {ver}: {ms:.3f} ms")
