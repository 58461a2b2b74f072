#!/usr/bin/env python
"""Cost of TF's Adam on the row-sharded tables at the cfg2 shape (B = 65 536 per rank, F = 39, 10 000 003 rows,
K = 16, first-order weights trained with Adagrad, 4 rotating batches):
    python tools/time_sharded_adam.py                        (one process, N = 1)
    torchrun --nproc-per-node N tools/time_sharded_adam.py   (N ranks, each with its own B samples)
Two layers on the same inputs: optimizer='adam' (each owner sweeps its ceil(N_rows / N) rows) and the Adagrad
baseline (the owner updates the rows that arrived):
  owner half  grads barrier -> owner sweep (Adam) or owner update (Adagrad): `_owner_step` on the last step's exchange
              buffer, captured into one CUDA graph per layer and replayed alternately, CUDA events around each replay
  step        forward + backward of a whole step, eager, alternating the layers; samples/s over all ranks
Every row of the Adam layer is live (nonzero m and v, so the sweep stores every row, as in tools/time_adam.py's
'live' case).  The sweep's algorithmic bytes (roofline.shard_adam_apply_bytes) over the Adam owner half give its
rate, against the measured HBM peak.  Rank 0 prints one JSON line, with the device name, power limit and clock.
"""
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import dir_b200                                                          # noqa: E402

R, ITERS = 4, 30


def main():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
    w = dir_b200.synth.cfg("cfg2")
    B, F, K, N = w.batch, w.field_size, w.embedding_size, w.n_rows
    batches = []
    for r in range(R):
        i, v, _ = dir_b200.synth.make_inputs(w, seed_shift=r + 8 * rank)
        batches.append((torch.as_tensor(i).cuda(), torch.as_tensor(v).cuda()))
    gen = torch.Generator(device="cuda").manual_seed(dir_b200.synth.SEED_UPSTREAM + rank)
    g_first = torch.randn(B, device="cuda", generator=gen)
    g_fm = torch.randn(B, device="cuda", generator=gen) * 0.5
    u = torch.randn((B, F * K), device="cuda", generator=gen) * 0.01
    layers = {
        "adam": dir_b200.ShardedEmbeddingFM(F, K, list(w.rows_per_field), optimizer="adam", lr=0.001,
                                            optimizer_epsilon=1e-4, linear_optimizer="adagrad", linear_lr=0.05,
                                            max_batch=B, init="counter").train(),
        "adagrad": dir_b200.ShardedEmbeddingFM(F, K, list(w.rows_per_field), optimizer="adagrad", lr=0.05,
                                               max_batch=B, init="counter").train(),
    }
    names = list(layers)
    with torch.no_grad():                 # every row live: nonzero moments, so the sweep writes all of them
        layers["adam"].adam_m.fill_(1e-4)
        layers["adam"].adam_v.fill_(1e-6)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def step(it, name):
        idx, val = batches[it % R]
        first, fm, emb = layers[name](idx, val)
        torch.autograd.backward((first, fm, emb), (g_first[:, None], g_fm[:, None], u))

    # whole steps, eager, alternating
    tot = dict.fromkeys(names, 0.0)
    for it in range(2 * ITERS + 8):
        name = names[it % 2]
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev[0].record()
        step(it // 2, name)
        ev[1].record()
        torch.cuda.synchronize()
        if it >= 8:
            tot[name] += ev[0].elapsed_time(ev[1])
    for layer in layers.values():
        layer.check_errors()
    step_ms = {k: v / ITERS for k, v in tot.items()}
    n_unique = int(layers["adam"].last_n_unique.item())        # (the replays below add to the counter)
    # the owner half of each layer's last step, replayed from CUDA graphs
    graphs = {}
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for name, layer in layers.items():
            h = layer._last_handle
            layer._owner_step([h])                              # warm (eager) once, then capture
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s, capture_error_mode="thread_local"):
                layer._owner_step([h])
            graphs[name] = g
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    own = {k: [] for k in names}
    for it in range(4 * ITERS + 8):
        name = names[it % 2]
        ev[0].record()
        graphs[name].replay()
        ev[1].record()
        torch.cuda.synchronize()
        if it >= 8:
            own[name].append(ev[0].elapsed_time(ev[1]) * 1e3)
    for layer in layers.values():
        layer.check_errors()
    # arrivals at this owner: sum of the headers' counts of the Adam layer's last exchange buffer
    la = layers["adam"]
    h = la._last_handle
    lay = la.px.layouts[h.buf]
    hdr = la.px.bufs[h.buf][lay.off_hdr: lay.off_hdr + world * 32].view(torch.int64).view(world, 4)
    arr_in = int(hdr[:, 0].sum())
    n_local = la.n_rows
    nbytes = dir_b200.roofline.shard_adam_apply_bytes(n_local, K, arr_in, world, U=n_unique, first_order=True,
                                                      linear_optimizer="adagrad")
    peak, peak_src = dir_b200.roofline.measured_peaks()
    med = {k: sorted(v)[len(v) // 2] for k, v in own.items()}
    gbs = nbytes / med["adam"] / 1e3
    out = {"workload": "cfg2", "world": world, "B_per_rank": B, "F": F, "K": K, "n_rows": N, "n_local_rows": n_local,
           "first_order": True, "linear_optimizer": "adagrad", "rotating_batches": R, "adam_rows": "live (m, v != 0)",
           "owner_half_us_adam_median": round(med["adam"], 2), "owner_half_us_adagrad_median": round(med["adagrad"], 2),
           "owner_half_us_adam_mean": round(sum(own["adam"]) / len(own["adam"]), 2),
           "owner_half_us_adagrad_mean": round(sum(own["adagrad"]) / len(own["adagrad"]), 2),
           "step_ms_adam": round(step_ms["adam"], 4), "step_ms_adagrad": round(step_ms["adagrad"], 4),
           "samples_per_s_adam": round(B * world / step_ms["adam"] * 1e3),
           "samples_per_s_adagrad": round(B * world / step_ms["adagrad"] * 1e3),
           "arrivals_at_owner": arr_in, "rows_with_gradient": n_unique,
           "sweep_algorithmic_bytes": nbytes, "sweep_gbs_at_owner_half": round(gbs, 1),
           "hbm_peak_gbs": peak, "hbm_peak_source": peak_src, "sweep_fraction_of_peak": round(gbs / peak, 3),
           "step_timing": "eager, alternating", "owner_half_timing": "CUDA graph replays, alternating, median"}
    if rank == 0:
        out["device"] = torch.cuda.get_device_name()
        try:
            q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm,clocks.sm",
                                "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
            out["power_limit_max_sm_clock_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"
        except (OSError, subprocess.SubprocessError):
            out["power_limit_max_sm_clock_sm_clock"] = "unknown"
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
