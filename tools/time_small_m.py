"""GEMM timing at the EgoMCQ question shape (5 clips x 4 frames: M = 5125 rows; another M as the first argument).
  python tools/time_small_m.py [M]"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from helping_hand_for_egocentric_videos_b200 import ops  # noqa: E402

M = int(sys.argv[1]) if len(sys.argv) > 1 else 5125
res = {}
for name, N, K, epi in (("qkv", 3072, 1024, 0), ("proj", 1024, 1024, 0), ("fc1", 4096, 1024, 1), ("fc2", 1024, 4096, 0)):
    a = torch.randn(M, K, device="cuda").bfloat16()
    w = (torch.randn(N, K, device="cuda") / 32).bfloat16()
    b = torch.randn(N, device="cuda")
    out = torch.empty(M, N, device="cuda", dtype=torch.bfloat16)
    for _ in range(5):
        ops.gemm_bf16(a, w, b, epilogue=epi, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(50):
        ops.gemm_bf16(a, w, b, epilogue=epi, out=out)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / 50
    res[name] = (round(us, 1), round(2.0 * M * N * K / us / 1e6))
print("M", M, res, "(us, TFLOP/s)")
