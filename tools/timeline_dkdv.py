"""Debug: per-phase clock64 timeline of one dK/dV CTA (library built with -DCTRLORA_TIMELINE)."""
import ctypes
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ctrlora_b200 import _lib, ops  # noqa: E402
from tools.profile_kernels import rnd  # noqa: E402

B, H, nq, nk, d = 8, 8, 4096, 4096, 40
q, k, v = rnd(B * nq, H * d), rnd(B * nk, H * d), rnd(B * nk, H * d)
o, do = rnd(B * nq, H * d), rnd(B * nq, H * d)
lse = torch.randn(B, H, nq, device="cuda") + 8.0
for _ in range(2):
    ops.attention_bwd(q, k, v, o, do, lse, B, H, nq, nk, d)
torch.cuda.synchronize()
buf = (ctypes.c_longlong * 4096)()
lib = _lib.load()
lib.ctrlora_debug_timeline.argtypes = [ctypes.c_void_p, ctypes.c_int]
assert lib.ctrlora_debug_timeline(buf, 4096) == 0
t = list(buf)
base = t[0]
print("row warp 0 (cycles rel.): tile: start, s_full, ld0, qfree0, ld1, (x), pre-fence, arrived | MMA: p_full, sdp issued, acc issued")
for i in range(2, 14):
    r = [t[i * 8 + j] - base for j in range(8)]
    m = [t[2048 + i * 4 + j] - base for j in range(3)]
    print(i, r, m, " tile period", t[i * 8 + 7] - t[(i - 1) * 8 + 7])
