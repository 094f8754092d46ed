"""Device time of the weight-gradient entry points at the loss step's shapes (batch 8 x 9 s): python scripts/time_wgrad.py"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench
from timbre_trap_b200.framework import layer_grads as LG

dev = torch.device('cuda')
B, T = 8, 3072
for C, H in ((4, 540), (8, 269), (16, 133), (32, 65)):
    Cp = max(8, C)
    x = torch.randn((B, Cp // 8, H, T, 8), device=dev).to(torch.bfloat16)
    dz = torch.randn((B, Cp // 8, H, T, 8), device=dev).to(torch.bfloat16)
    for k, d in ((1, 1), (3, 1), (3, 3)):
        ms = sorted(bench.time_kernel(lambda: LG._wgrad_same(x, dz, C, C, k, d), iters=10) for _ in range(3))[1]
        print(f'wgrad_same C={C:2d} H={H:3d} k={k} d={d}: {ms * 1e3:7.1f} us')
for (cf, hf), (cc, hc) in (((4, 540), (8, 269)), ((8, 269), (16, 133)), ((16, 133), (32, 65)), ((32, 65), (64, 31))):
    fine = torch.randn((B, max(8, cf) // 8, hf, T, 8), device=dev).to(torch.bfloat16)
    coarse = torch.randn((B, cc // 8, hc, T, 8), device=dev).to(torch.bfloat16)
    for tr in (False, True):
        ms = sorted(bench.time_kernel(lambda: LG._wgrad_updown(fine, coarse, cf, cc, tr), iters=10) for _ in range(3))[1]
        print(f'wgrad_updown fine {cf:2d} x {hf:3d} coarse {cc:2d} x {hc:3d} transposed={int(tr)}: {ms * 1e3:7.1f} us')
