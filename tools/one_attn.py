"""One attention shape (forward, or backward with 'bwd'), a few launches (for ncu --set full)."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ctrlora_b200 import ops  # noqa: E402
from tools.profile_kernels import rnd  # noqa: E402

B, H, nq, nk, d = 8, 8, 4096, 4096, 40
q, k, v = rnd(B * nq, H * d), rnd(B * nk, H * d), rnd(B * nk, H * d)
vt = v.view(B, nk, H, d).permute(0, 2, 3, 1).contiguous()
out = torch.empty(B * nq, H * d, device="cuda", dtype=torch.float16)
lse = torch.empty(B, H, nq, device="cuda", dtype=torch.float32)
for _ in range(3):
    ops.attention(q, k, vt, B, H, nq, nk, d, out=out, lse=lse)
if len(sys.argv) > 1 and sys.argv[1] == "bwd":
    do = rnd(B * nq, H * d)
    for _ in range(3):
        ops.attention_bwd(q, k, v, out, do, lse, B, H, nq, nk, d)
torch.cuda.synchronize()
