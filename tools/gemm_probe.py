#!/usr/bin/env python
"""A few GEMM launches at the update's shapes for an `ncu --set full` capture (tools/gpu_ncu.sh)."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rorl_b200.kernels as K  # noqa: E402

dev = torch.device("cuda:0")
M = 32 * 1019
shapes = {"efc2": (256, 256, 8), "efc1": (256, 384, 8), "fc": (256, 256, 1), "inproj": (512, 256, 1)}
which = (sys.argv[1] if len(sys.argv) > 1 else "efc2,fc").split(",")
passes = [int(x) for x in (sys.argv[2] if len(sys.argv) > 2 else "2,4").split(",")]
for name in which:
    n, k, g = shapes[name]
    a = torch.randn(M, k, device=dev) if (g == 1 or name == "efc1") else torch.randn(g, M, k, device=dev)
    b = torch.randn(n, k, device=dev) if g == 1 else torch.randn(g, n, k, device=dev)
    bias = torch.randn(n, device=dev) if g == 1 else torch.randn(g, n, device=dev)
    for p in passes:
        for _ in range(2):
            K.gemm_tn(a, b, bias, 1, passes=p)
torch.cuda.synchronize()
print("done")
