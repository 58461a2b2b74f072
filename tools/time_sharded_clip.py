#!/usr/bin/env python
"""Cost of tf.clip_by_norm per column on the row-sharded tables at the cfg2 shape (B = 65 536 per rank, F = 39,
10 000 003 rows, K = 16, Adagrad, first-order weights trained, 4 rotating batches):
    python tools/time_sharded_clip.py                        (one process, N = 1)
    torchrun --nproc-per-node N tools/time_sharded_clip.py   (N ranks, each with its own B samples)
One layer built with clip_norm, switched per step between clipped and unclipped (`layer.clip_norm = None` takes the
unclipped owner step), so both run on the same tables and buffers:
  owner half  grads barrier -> (norm pass -> barrier ->) owner update -> dense apply: `_owner_step` on the last step's
              exchange buffer, captured into one CUDA graph per variant and replayed alternately, CUDA events around
              each replay
  step        forward + backward of a whole step, eager, alternating the variants; samples/s over all ranks
The norm pass's algorithmic bytes (arrivals x (4 + 4G + 4K + 16) read, 16 x arrivals written, G x F x 256 peer stores)
are printed beside its measured cost.  Rank 0 prints one JSON line, with the device name, power limit and clock.
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

R, ITERS, CLIP = 4, 30, 1.0


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
    layer = dir_b200.ShardedEmbeddingFM(F, K, list(w.rows_per_field), optimizer="adagrad", lr=0.05, clip_norm=CLIP,
                                        max_batch=B, init="counter").train()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def step(it, clip):
        layer.clip_norm = clip
        idx, val = batches[it % R]
        first, fm, emb = layer(idx, val)
        torch.autograd.backward((first, fm, emb), (g_first[:, None], g_fm[:, None], u))

    # whole steps, eager, alternating
    tot = {CLIP: 0.0, None: 0.0}
    for it in range(2 * ITERS + 8):
        clip = CLIP if it % 2 == 0 else None
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev[0].record()
        step(it, clip)
        ev[1].record()
        torch.cuda.synchronize()
        if it >= 8:
            tot[clip] += ev[0].elapsed_time(ev[1])
    layer.check_errors()
    step_ms = {k: v / ITERS for k, v in tot.items()}
    arrivals = int(layer.last_exchange["unique_sent"])          # this rank's sends; every rank's sends arrive somewhere
    # the owner half of the last step, replayed from CUDA graphs
    h = layer._last_handle
    graphs = {}
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for clip in (CLIP, None):
            layer.clip_norm = clip
            layer._owner_step([h])                              # warm (eager) once, then capture
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s, capture_error_mode="thread_local"):
                layer._owner_step([h])
            graphs[clip] = g
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    own = {CLIP: [], None: []}
    for it in range(4 * ITERS + 8):
        clip = CLIP if it % 2 == 0 else None
        ev[0].record()
        graphs[clip].replay()
        ev[1].record()
        torch.cuda.synchronize()
        if it >= 8:
            own[clip].append(ev[0].elapsed_time(ev[1]) * 1e3)
    layer.check_errors()
    # arrivals at this owner (the norm pass's work): sum of the headers' counts
    lay = layer.px.layouts[h.buf]
    hdr = layer.px.bufs[h.buf][lay.off_hdr: lay.off_hdr + world * 32].view(torch.int64).view(world, 4)
    arr_in = int(hdr[:, 0].sum())
    G = world
    rd, wr, peer = arr_in * (4 + 4 * G + 4 * K + 16), 16 * arr_in, G * F * 256
    med = {k: sorted(v)[len(v) // 2] for k, v in own.items()}
    out = {"workload": "cfg2", "world": world, "B_per_rank": B, "F": F, "K": K, "n_rows": N, "optimizer": "adagrad",
           "first_order": True, "rotating_batches": R, "clip_norm": CLIP,
           "owner_half_us_clipped_median": round(med[CLIP], 2), "owner_half_us_unclipped_median": round(med[None], 2),
           "owner_half_us_clipped_mean": round(sum(own[CLIP]) / len(own[CLIP]), 2),
           "owner_half_us_unclipped_mean": round(sum(own[None]) / len(own[None]), 2),
           "clip_cost_us": round(med[CLIP] - med[None], 2),
           "step_ms_clipped": round(step_ms[CLIP], 4), "step_ms_unclipped": round(step_ms[None], 4),
           "samples_per_s_clipped": round(B * world / step_ms[CLIP] * 1e3),
           "samples_per_s_unclipped": round(B * world / step_ms[None] * 1e3),
           "arrivals_at_owner": arr_in, "distinct_rows_sent": arrivals,
           "norm_pass_bytes_read": rd, "norm_pass_bytes_written": wr, "norm_pass_peer_store_bytes": peer,
           "norm_pass_gbs_at_clip_cost": round((rd + wr + peer) / max(med[CLIP] - med[None], 1e-3) / 1e3, 1),
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
