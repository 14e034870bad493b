"""Device time of kernels.gemm_tn against torch.mm(a.t(), b) on the weight-gradient shapes of the TGCN cell (config 4)."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stgraph_b200 import kernels  # noqa: E402

dev = torch.device("cuda")


def timed(fn, reps=20):
    for _ in range(3):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


res = []
for m, k, nc in ((1000000, 64, 64), (1000000, 64, 128), (1000000, 32, 192), (1000000, 64, 32), (200000, 100, 100), (1068, 16, 16)):
    A = torch.randn(m, k, device=dev)
    B = torch.randn(m, nc, device=dev)
    t_ours = timed(lambda: kernels.gemm_tn(A, B, colsum=True))
    t_torch = timed(lambda: (torch.mm(A.t(), B), B.sum(0)))
    t_mm = timed(lambda: torch.mm(A.t(), B))
    gb = 4.0 * m * (k + nc) / 1e6
    res.append({"M": m, "K": k, "Nc": nc, "ours_ms": round(t_ours, 4), "torch_mm_plus_colsum_ms": round(t_torch, 4),
                "torch_mm_ms": round(t_mm, 4), "ours_gbs": round(gb / t_ours, 1), "ours_tflops": round(2e-9 * m * k * nc / t_ours, 2)})
    print(res[-1], flush=True)
print(json.dumps(res))
