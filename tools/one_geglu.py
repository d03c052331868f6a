"""GEGLU projection of the 64x64 level, a few launches (for ncu --set full)."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ctrlora_b200 import ops  # noqa: E402
from tools.profile_kernels import rnd  # noqa: E402

m, k, n = 32768, 320, 1280
a, wt = rnd(m, k), rnd(2 * n, 1, k, scale=k ** -0.5)
bias = torch.randn(2 * n, device="cuda")
out = torch.empty(m, n, device="cuda", dtype=torch.float16)
for _ in range(3):
    ops.gemm(a, wt, bias=bias, out=out, geglu=True)
torch.cuda.synchronize()
