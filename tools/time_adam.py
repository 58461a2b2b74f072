#!/usr/bin/env python
"""Parity tests of TF's Adam on the tables, then CUDA-event timing at the cfg2 shape (B = 65 536, F = 39,
10 000 003 rows, K = 16, 4 rotating batches, DCN-style: no first-order weights, upstream gradient u), in one process:
    python tools/time_adam.py [--no-tests]
It prints one JSON line: the Adagrad fused backward (the reference point), the Adam backward (emit + apply sweep),
and the apply sweep alone with its algorithmic bytes (roofline.adam_apply_bytes) and its share of
roofline.measured_peaks(); 'fresh' is the sweep while most rows still have m = v = 0 (their stores are skipped),
'live' once every row's moments are nonzero (every row written).  The device name and its power limit come from
the same run.
"""
import ctypes
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
rc = 0 if "--no-tests" in sys.argv else pytest.main(["-q", "-x", "-m", "gpu", os.path.join(ROOT, "tests", "test_gpu_adam.py")])
import dir_b200                                                          # noqa: E402
from dir_b200 import roofline                                            # noqa: E402
from dir_b200._lib import AdamOpt, check, lib, ptr                       # noqa: E402

w = dir_b200.synth.cfg("cfg2")
B, F, K, N = w.batch, w.field_size, w.embedding_size, w.n_rows
R, ITERS = 4, 20
batches = []
for r in range(R):
    i, v, _ = dir_b200.synth.make_inputs(w, seed_shift=r)
    batches.append((torch.as_tensor(i).cuda(), torch.as_tensor(v).cuda()))
gen = torch.Generator(device="cuda").manual_seed(dir_b200.synth.SEED_UPSTREAM)
g_fm = torch.randn(B, device="cuda", generator=gen) * 0.5
u = torch.randn((B, F * K), device="cuda", generator=gen) * 0.01
ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]


def time_backward(layer):
    """mean backward time (µs) over ITERS steps after 4 warm-up steps, each forward outside the timed window"""
    total = 0.0
    for it in range(ITERS + 4):
        idx, val = batches[it % R]
        first, fm, emb = layer(idx, val)
        torch.cuda.synchronize()
        ev[0].record()
        torch.autograd.backward((fm, emb), (g_fm[:, None], u))
        ev[1].record()
        torch.cuda.synchronize()
        if it >= 4:
            total += ev[0].elapsed_time(ev[1])
    return total / ITERS * 1e3


out = {"workload": "cfg2", "B": B, "F": F, "K": K, "n_rows": N, "rotating_batches": R, "tests_rc": rc}
adagrad = dir_b200.EmbeddingFM(F, K, list(w.rows_per_field), optimizer="adagrad", lr=0.05, first_order=False).train()
out["adagrad_backward_us"] = time_backward(adagrad)
del adagrad
torch.cuda.empty_cache()

adam = dir_b200.EmbeddingFM(F, K, list(w.rows_per_field), optimizer="adam", lr=1e-3, optimizer_epsilon=1e-4,
                            first_order=False).train()
L = lib()
st = torch.cuda.current_stream().cuda_stream


def time_apply():
    """the sweep alone, on the distinct rows and gradients the last backward left in the layer's buffers"""
    c = adam._clip_bufs
    n = B * adam.n_sorted_fields
    opt = AdamOpt(adam.lr, adam.optimizer_beta1, adam.optimizer_beta2, adam.optimizer_epsilon, adam.beta_power.data_ptr())
    total = 0.0
    for it in range(ITERS + 3):
        ev[0].record()
        check(L.dir_rows_apply_adam(ptr(adam.rows), adam.row_stride, N, K, None, None, 1, None, ptr(c["gu"]), K + 4,
                                    ptr(c["urows"]), c["count"].data_ptr() + 8, n, ptr(adam.field_offset), F, None,
                                    0.0, ctypes.byref(opt), None, st), "dir_rows_apply_adam")
        ev[1].record()
        torch.cuda.synchronize()
        if it >= 3:
            total += ev[0].elapsed_time(ev[1])
    return total / ITERS * 1e3


idx, val = batches[0]
first, fm, emb = adam(idx, val)
torch.autograd.backward((fm, emb), (g_fm[:, None], u))
torch.cuda.synchronize()
U = int(adam.last_n_unique.item())
out["distinct_rows"] = U
out["adam_apply_fresh_us"] = time_apply()
with torch.no_grad():                     # every row live: nonzero moments, so the sweep writes all of them
    adam.adam_m.fill_(1e-4)
    adam.adam_v.fill_(1e-6)
out["adam_backward_us"] = time_backward(adam)
out["adam_apply_live_us"] = time_apply()
nbytes = roofline.adam_apply_bytes(N, K, U)
peak, src = roofline.measured_peaks()
out["adam_apply_bytes"] = nbytes
out["adam_apply_live_gbs"] = nbytes / (out["adam_apply_live_us"] * 1e-6) / 1e9
out["adam_apply_live_frac_of_peak"] = out["adam_apply_live_gbs"] / peak
out["peak_gbs"], out["peak_source"] = peak, src
out["device"] = torch.cuda.get_device_name(0)
try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30)
    out["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"
except (OSError, subprocess.SubprocessError, IndexError):
    out["power_limit_and_max_sm_clock"] = "unknown"
print(json.dumps({k: (round(v, 3) if isinstance(v, float) else v) for k, v in out.items()}))
