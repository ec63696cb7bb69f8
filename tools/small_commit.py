#!/usr/bin/env python3
"""Device-resident commit latency of one small shape, median of 20:
    python tools/small_commit.py n_log k"""
import os
import statistics
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from intmax_zkp_core_b200 import device as D

ctx = D.torch_context(0)
n_log, k = int(sys.argv[1]), int(sys.argv[2])
v = torch.randint(0, 2**62, (k, 1 << n_log), dtype=torch.int64, device="cuda")
out = D.DeviceCommitment(n_log, k, 3, 4, v.device)
ts = []
for it in range(25):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    D.commit_device(ctx, v, 3, 4, out=out)
    e1.record()
    torch.cuda.synchronize()
    if it >= 5:
        ts.append(e0.elapsed_time(e1))
print(f"2^{n_log} x {k}: {statistics.median(ts):.4f} ms")
ctx.close()
