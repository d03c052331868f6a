"""One GEMM shape, a few launches (for ncu --set full): python tools/one_gemm.py B H W C N ksize [residual]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ctrlora_b200 import ops  # noqa: E402
from tools.profile_kernels import rnd  # noqa: E402

b, h, w, c, n, ks = (int(v) for v in sys.argv[1:7]) if len(sys.argv) >= 7 else (8, 64, 64, 320, 320, 1)
res = len(sys.argv) < 8 or sys.argv[7] != "0"
a, wt = rnd(b, h, w, c), rnd(n, ks * ks, c, scale=(ks * ks * c) ** -0.5)
bias = torch.randn(n, device="cuda")
r = rnd(b * h * w, n) if res else None
out = torch.empty(b, h, w, n, device="cuda", dtype=torch.float16)
for _ in range(3):
    ops.gemm(a, wt, ksize=ks, bias=bias, residual=r, out=out)
torch.cuda.synchronize()
