#!/usr/bin/env python
"""Parity tests of the cross kernels, then CUDA-event timing of dir_cross_fwd / dir_cross_bwd at the cfg3 shape
(d = 624, L = 6: the backward takes the per-warp rings), in one process:
    python tools/time_cross.py [--no-tests]
"""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
rc = 0 if "--no-tests" in sys.argv else pytest.main(["-q", "-x", "-m", "gpu", os.path.join(ROOT, "tests", "test_gpu_cross.py")])
import dir_b200                                                          # noqa: E402
from dir_b200._lib import check, lib, ptr                                # noqa: E402

B, d, L = 65536, 624, 6
L_ = lib()
st = torch.cuda.current_stream().cuda_stream
x0 = [torch.randn((B, d), device="cuda") * 0.5 for _ in range(3)]
dy = [torch.randn((B, d), device="cuda") for _ in range(3)]
w, b = torch.randn((L, d), device="cuda") * 0.1, torch.randn((L, d), device="cuda") * 0.1
xL, s, dx0 = torch.empty_like(x0[0]), torch.empty((B, L), device="cuda"), torch.empty_like(x0[0])
dw, db = torch.empty_like(w), torch.empty_like(b)
ws = torch.empty(int(L_.dir_cross_bwd_workspace_bytes(B, d, L)), dtype=torch.uint8, device="cuda")
ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
tf = tb = 0.0
for it in range(23):
    r = it % 3
    ev[0].record()
    check(L_.dir_cross_fwd(ptr(x0[r]), ptr(w), ptr(b), B, d, L, ptr(xL), ptr(s), st), "fwd")
    ev[1].record()
    check(L_.dir_cross_bwd(ptr(x0[r]), ptr(w), ptr(b), ptr(dy[r]), ptr(s), B, d, L, ptr(dx0), ptr(dw), ptr(db),
                           ptr(ws), ws.numel(), st), "bwd")
    ev[2].record()
    torch.cuda.synchronize()
    if it >= 3:
        tf += ev[0].elapsed_time(ev[1])
        tb += ev[1].elapsed_time(ev[2])
print("tests rc=%d  cross_fwd %.1f us  cross_bwd %.1f us" % (rc, tf / 20 * 1e3, tb / 20 * 1e3))
