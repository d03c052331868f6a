"""Per-launch cost of small GEMMs inside a CUDA graph (PDL chains, warm L2): the fixed overhead of one launch."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ctrlora_b200 import ops  # noqa: E402
from tools.profile_kernels import rnd  # noqa: E402

SHAPES = [(128, 64, 32), (128, 320, 320), (2048, 1280, 1280), (8192, 640, 640), (32768, 320, 320), (512, 1280, 1280),
          (2048, 320, 320), (2048, 64, 320)]
for (m, k, n) in SHAPES:
    a, w = rnd(m, k), rnd(n, 1, k, scale=k ** -0.5)
    bias = torch.randn(n, device="cuda")
    outs = [torch.empty(m, n, device="cuda", dtype=torch.float16) for _ in range(2)]
    reps = 40

    def body():
        for i in range(reps):
            ops.gemm(a if i == 0 else a, w, bias=bias, out=outs[i & 1])
    body()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            body()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    print(f"M={m:6d} K={k:5d} N={n:5d}: {e0.elapsed_time(e1) / 5 / reps * 1e3:7.2f} us per launch in-graph")
