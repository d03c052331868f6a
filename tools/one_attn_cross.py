"""One cross-attention shape (77 context tokens, 64x64 level), a few launches (for ncu --set full)."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ctrlora_b200 import ops  # noqa: E402
from tools.profile_kernels import rnd  # noqa: E402

B, H, nq, nk, d = 8, 8, 4096, 77, 40
q, k, v = rnd(B * nq, H * d), rnd(B * nk, H * d), rnd(B * nk, H * d)
vt = torch.zeros(B, H, d, 80, device="cuda", dtype=torch.float16)
vt[..., :nk] = v.view(B, nk, H, d).permute(0, 2, 3, 1)
out = torch.empty(B * nq, H * d, device="cuda", dtype=torch.float16)
for _ in range(3):
    ops.attention(q, k, vt, B, H, nq, nk, d, out=out)
torch.cuda.synchronize()
