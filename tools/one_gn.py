"""One GroupNorm shape, a few launches (for ncu --set full): python tools/one_gn.py H C"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ctrlora_b200 import ops  # noqa: E402
from tools.profile_kernels import rnd  # noqa: E402

h, c = (int(v) for v in sys.argv[1:3]) if len(sys.argv) >= 3 else (64, 640)
x = rnd(8, h, h, c)
g, b = torch.randn(c, device="cuda"), torch.randn(c, device="cuda")
for _ in range(3):
    ops.groupnorm(x, g, b, 1e-5, True)
torch.cuda.synchronize()
