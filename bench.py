#!/usr/bin/env python
"""bench.py -- samples/sec of fwd + bwd (+ fused Adagrad update) of the embedding + FM / cross layer.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2|cfg3|cfg5] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic Criteo-shaped input
(BASELINE.json configs[1] by default: 26 sparse + 13 dense fields, 10 M rows, K = 16, B = 65 536,
embeddings emitted to / upstream gradients consumed from the DNN side):
    dir_shard_keys_sort (next batch) | dir_embed_fm_fwd -> g = sigmoid(first + fm) - y -> dir_embed_bwd_reduce_update
(cfg3 adds dir_cross_fwd / dir_cross_bwd between the two halves).  Prints ONE JSON line.

  value     device-resident inputs, CUDA-event timed, max over ranks
  e2e       the same step fed from pinned HOST buffers through `HostFeeder` (H2D of ids / values /
            labels and D2H of the logits inside the timed region, copies overlapped with compute)
  roofline  the dominant C-ABI call, algorithmic bytes (details-in-recommendation_b200/roofline.py)
            / its CUDA-event time, against MEASURED_PEAKS.json
  cpu_baseline / --impl reference
            the PyTorch-CPU op-by-op restatement of the reference's TF graph
            (oracle/torch_restatement.py; TF 1.x itself cannot be installed here) on the host cores.

--dump-outputs DIR writes, after the timed steps, what the last timed step handed its caller (logits, first-order
and FM terms, embeddings, the cross output) and a sample of the table state it left behind, one DIR/<name>.npy
per array (see dump_outputs).  Inputs and initial tables depend on the arguments only, so two builds run with
the same arguments can be compared array for array.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

DEFAULT_MICRO = 1          # micro-batches of the sharded step (see --micro)
METRIC = "samples/sec fwd+bwd embedding+FM/cross layer"
UNIT = "samples/s"
LR = 0.05


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=200, help="timed steps (each timed loop runs exactly this many)")
    p.add_argument("--warmup", type=int, default=10)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5"],
                   help="cfg4 = Terabyte-sized tables (880 M rows, 113 GB with accumulators): meant for --gpus >= 2")
    p.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the workload's)")
    p.add_argument("--strong", action="store_true",
                   help="strong scaling: the workload's batch is the GLOBAL batch, split over the ranks "
                        "(default: weak, the batch is per GPU)")
    p.add_argument("--rotate", type=int, default=4, help="distinct input sets cycled through")
    p.add_argument("--no-graph", action="store_true", help="launch eagerly instead of CUDA graphs")
    p.add_argument("--no-emit", action="store_true", help="FM only: no embeddings out / upstream in")
    p.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--profile", default="",
                   help="after the timed regions, trace 6 steps with torch.profiler (CUPTI kernel timeline) and "
                        "write the chrome trace of rank 0 to this path: a diagnostic, never a bench value")
    p.add_argument("--micro", type=int, default=0, choices=[0, 1, 2],
                   help="sharded layer: exchange a batch as this many micro-batches (2: the second half's row exchange "
                        "runs underneath the first half's forward; one owner update per batch either way); 0 = the default")
    p.add_argument("--sharded", action="store_true",
                   help="run the row-sharded layer even on one GPU (every exchange kernel, local buffers): a diagnostic")
    p.add_argument("--feed", default="columns", choices=["columns", "resolved"],
                   help="e2e host format: one column per feature (the reference's input_fn form) or the [B,F] pair")
    p.add_argument("--cpu-seconds", type=float, default=12.0)
    p.add_argument("--dump-outputs", default="", metavar="DIR",
                   help="after the timed steps, write the last timed step's outputs as DIR/<name>.npy "
                        "(float32, at most 64 MB in all; large arrays as a fixed-seed sample), replacing "
                        "any .npy files DIR held")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        p.error("--dump-outputs writes what the B200 path computed: it needs --impl b200")
    if args.strong:                        # per-GPU batch = global batch / ranks; everything below sees a per-GPU batch
        full = args.batch or dir_synth_batch(args.workload)
        if full % max(args.gpus, 1):
            p.error("--strong needs the batch to divide by --gpus")
        args.batch = full // max(args.gpus, 1)
    return args


def dir_synth_batch(name):
    import dir_b200
    return dir_b200.synth.cfg(name).batch


def workload_config(w, args, n_gpus):
    B = args.batch or w.batch
    return {
        "workload": "%s: DeepFM embedding + first-order + FM%s, fwd + bwd + fused Adagrad row update" % (
            w.name, " + %d-layer DCN cross" % w.cross_layer_num if w.cross_layer_num else ""),
        "batch_per_gpu": B, "global_batch": B * n_gpus, "field_size": w.field_size,
        "sparse_fields": w.field_size - w.n_dense, "dense_fields": w.n_dense,
        "embedding_size": w.embedding_size, "table_rows": w.n_rows, "ids": w.ids,
        "cross_layer_num": w.cross_layer_num, "optimizer": "adagrad",
        "emit_embeddings_and_upstream_grad": not args.no_emit,
        "parallelism": "single GPU" if n_gpus == 1 else "row-sharded tables (row mod %d), all-to-all, dp%d" % (n_gpus, n_gpus),
    }


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the PyTorch-CPU restatement of the reference graph on host cores
# ------------------------------------------------------------------------------------------------
def cpu_model_name():
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.lower().startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_cfg1(budget_s=6.0):
    """BASELINE.json configs[0] -- the reference's own CPU-runnable case (B = 1 024, 39 fields, K = 8) -- on the
    restatement: 20 warm-up steps, then timed steps for about `budget_s` (at most 200); median step time."""
    import torch
    from oracle import torch_restatement as TR
    import dir_b200
    w = dir_b200.synth.cfg("cfg1")
    torch.set_num_threads(os.cpu_count() or 1)
    model = TR.DeepFMLayerCPU(w.rows_per_field, w.embedding_size, lr=LR)
    i, v, y = dir_b200.synth.make_inputs(w)
    b = (torch.as_tensor(i), torch.as_tensor(v), torch.as_tensor(y),
         torch.randn((w.batch, w.field_size * w.embedding_size)) * 1e-2)
    for _ in range(20):
        model.step(*b)
    times, t_end = [], time.perf_counter() + budget_s
    while len(times) < 200 and time.perf_counter() < t_end:
        t0 = time.perf_counter()
        model.step(*b)
        times.append(time.perf_counter() - t0)
    times.sort()
    med = times[len(times) // 2]
    return {"value": w.batch / med, "unit": UNIT, "ms_per_step": med * 1e3,
            "p10_ms": times[len(times) // 10] * 1e3, "p90_ms": times[(len(times) * 9) // 10] * 1e3,
            "sample": "cfg1: B=1024, F=39, K=8, 26 x 10 000 + 13 x 1 rows; %d timed steps, median" % len(times)}


def cpu_restatement(w, steps, warmup, budget_s, full_batch):
    """Times oracle/torch_restatement.DeepFMLayerCPU (one variable per column, separate materialising
    ops, sparse Adagrad) on a bounded sample: the per-step batch is cut so that (steps + warmup)
    steps fit in `budget_s`.  Returns dict(value, ms_per_step, cores, sample, batch)."""
    import torch
    from oracle import torch_restatement as TR
    import dir_b200

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    K, F = w.embedding_size, w.field_size
    model = TR.DeepFMLayerCPU(w.rows_per_field, K, lr=LR)

    def batch_of(B, shift):
        i, v, y = dir_b200.synth.make_inputs(w, batch=B, seed_shift=shift)
        U = torch.randn((B, F * K)) * 1e-2
        return torch.as_tensor(i), torch.as_tensor(v), torch.as_tensor(y), U

    # calibrate on a small batch, then size the sample
    probe = min(4096, full_batch)
    b = batch_of(probe, 100)
    model.step(*b)
    t0 = time.perf_counter()
    model.step(*b)
    per_sample = (time.perf_counter() - t0) / probe
    B = int(min(full_batch, max(256, budget_s / max(1, steps + warmup) / per_sample)))
    sets = [batch_of(B, 200 + r) for r in range(2)]
    for s in range(warmup):
        model.step(*sets[s % 2])
    t0 = time.perf_counter()
    for s in range(steps):
        model.step(*sets[s % 2])
    dt = time.perf_counter() - t0
    return {"value": B * steps / dt, "ms_per_step": dt / steps * 1e3, "cores": cores, "batch": B,
            "sample": "%d steps of B=%d (of the workload's %d) %s rows, torch %d threads" % (
                steps, B, full_batch, w.name, cores)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import dir_b200
    # cfg3's lookup is cfg2's; cfg4's 880 M-row tables (56 GB of fp32 per copy) are not a bounded host sample
    w = dir_b200.synth.cfg("cfg2" if args.workload in ("cfg3", "cfg4") else args.workload)
    full = args.batch or w.batch
    r = cpu_restatement(w, args.steps, args.warmup, 150.0, full)
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(w, args, 1),
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
                         "sample": r["sample"] + "; PyTorch-CPU restatement of the TF 1.x graph (TF not installable)",
                         "cpu_model": cpu_model_name()},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = [("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
               ("sw_power_cap", 0x4), ("hw_power_brake_slowdown", 0x80)]

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz, self.h = [], set(), None, None
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.h = None

    def sample(self):
        if self.h is None:
            return
        try:
            self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            for name, bit in self.REASONS:
                if mask & bit:
                    self.reasons.add(name)
        except Exception:
            pass

    def _loop(self):
        while not self._stop.wait(0.02):
            self.sample()

    def __enter__(self):
        self.t = threading.Thread(target=self._loop, daemon=True)
        self.t.start()
        return self

    def __exit__(self, *a):
        self.sample()               # at least one sample while the queue is still draining
        self._stop.set()
        self.t.join()

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# ------------------------------------------------------------------------------------------------
# the B200 arm
# ------------------------------------------------------------------------------------------------
def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    import dir_b200
    from dir_b200 import roofline as RL

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this path has no CPU fallback "
                         "(use --impl reference for the CPU restatement)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if "NCCL_DEBUG" in os.environ:                          # keep NCCL's banner: it goes to stderr, the JSON line
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")     # owns stdout
        dist.init_process_group("nccl", device_id=dev)
    if world != args.gpus and rank == 0:
        print("bench.py: --gpus %d but WORLD_SIZE=%d; using WORLD_SIZE" % (args.gpus, world), file=sys.stderr)
    dir_b200._lib.lib()                    # raises if libdir_b200.so is missing

    w = dir_b200.synth.cfg(args.workload)
    B, F, K = args.batch or w.batch, w.field_size, w.embedding_size
    L, d = w.cross_layer_num, w.field_size * w.embedding_size
    emit = (not args.no_emit) or L > 0
    R = max(1, args.rotate)
    torch.manual_seed(dir_b200.synth.SEED_TABLES + rank)

    sharded = world > 1 or args.sharded
    micro = 1
    if not sharded:
        layer = dir_b200.EmbeddingFM(F, K, list(w.rows_per_field), optimizer="adagrad", lr=LR,
                                     emit_embeddings=emit, device=dev).train()
    else:
        # cfg4's 880 M rows are filled on the device from a counter hash (no 56 GB host table, no fp32 temporaries)
        micro = args.micro or DEFAULT_MICRO
        layer = dir_b200.ShardedEmbeddingFM(F, K, list(w.rows_per_field), optimizer="adagrad", lr=LR,
                                            emit_embeddings=emit, max_batch=B, device=dev, micro_batches=micro,
                                            init="counter" if w.name == "cfg4" else "trunc_normal").train()
    layer.w1.normal_(0.0, 0.01)            # TF's zero init would make the first-order path trivial
    if getattr(layer, "n_dense", 0):
        layer._sync_dense_replicas()
    cross = dir_b200.CrossNetwork(d, L, device=dev).train() if L else None

    # R rotating input sets: pinned host copies (for e2e) and device-resident copies (for value)
    host, devs, ups = [], [], []
    for r in range(R):
        i, v, y = dir_b200.synth.make_inputs(w, batch=B, seed_shift=r + 16 * rank)
        hs = [torch.as_tensor(a).pin_memory() for a in (i, v, y)]
        host.append(hs)
        devs.append([t.to(dev) for t in hs])
        ups.append(torch.randn((B, d), device=dev) * 1e-2 if emit else None)
    n_rows_touched = []

    # The id-only work of a batch (keys, sort; sharded: distinct-row numbering and the id exchange) needs its ids
    # only, so the work for batch i+1 is issued at the start of step i and runs underneath it on the side stream:
    # every step still performs exactly one sort.  A running cursor keeps the rotation (and, sharded, the
    # one-batch-ahead id phase) consistent across the warm-up, timed, e2e and trace loops.
    ready_events = {}          # e2e: slot -> event of its H2D copy (the id work of that batch waits for it)
    handles = [dir_b200.SortedLookups() if not sharded else dir_b200.ShardedLookups() for _ in range(R)]
    if micro == 2:
        if B % 2:
            raise SystemExit("--micro 2 needs an even batch")
        handles = [[dir_b200.ShardedLookups(), dir_b200.ShardedLookups()] for _ in range(R)]
    Bh = B // 2
    cursor = [0]
    side = layer.side_stream(dev)

    def half(slot, x):
        """views of micro-batch x of a slot: ids, values, labels, upstream gradient"""
        lo, hi = x * Bh, (x + 1) * Bh
        return devs[slot][0][lo:hi], devs[slot][1][lo:hi], devs[slot][2][lo:hi], (ups[slot][lo:hi] if emit else None)

    def id_work(nxt, phase="both", inline=False):
        if not sharded:
            layer.presort(devs[nxt][0], devs[nxt][1], handle=handles[nxt], record_event=not inline)
        elif micro == 2:
            for x in range(2):
                idx_, val_, _, _ = half(nxt, x)
                if inline:
                    layer.presort(idx_, val_, handle=handles[nxt][x], inline=True, phase=phase, half=x)
                else:
                    layer.presort(idx_, val_, handle=handles[nxt][x], fork=False, after=ready_events.get(nxt), half=x)
        elif inline:
            layer.presort(devs[nxt][0], devs[nxt][1], handle=handles[nxt], inline=True, phase=phase)
        else:
            layer.presort(devs[nxt][0], devs[nxt][1], handle=handles[nxt], fork=False, after=ready_events.get(nxt))

    # --dump-outputs: the outputs of the latest step of each (captured?, slot, micro-batch).  A graph replay rewrites
    # the tensors its capture produced, so those are kept apart from the ones an eager step of the same slot makes.
    # They are kept detached: holding a step's autograd graph would keep its AccumulateGrad nodes, bound to the
    # stream they were created on, alive into the next capture and invalidate it.
    produced = {} if args.dump_outputs else None

    def model(slot, x=None):
        if x is None:
            idx, val, y = devs[slot]
            up = ups[slot]
            first, fm, emb = layer(idx, val, presorted=handles[slot])
        else:
            idx, val, y, up = half(slot, x)
            first, fm, emb = layer(idx, val, presorted=handles[slot][x], defer_update=True)
        with torch.no_grad():
            logits = first + fm
            g = torch.sigmoid(logits).sub_(y.unsqueeze(1))          # SUM-reduced CE: no 1/B (deepFM.py:72)
        if produced is not None:
            produced[(getattr(layer, "capturing", False), slot, x)] = {
                "logits": logits, "first_order": first.detach(), "fm": fm.detach(), "embeddings": emb.detach()}
        return first, fm, emb, g, up, logits

    def backward(first, fm, emb, g, up):
        if cross is not None:
            xL = cross(emb)
            if produced is not None:
                for out in produced.values():        # the step whose embeddings these are (same storage)
                    if out["embeddings"].data_ptr() == emb.data_ptr():
                        out["cross_out"] = xL.detach()
            torch.autograd.backward((first, fm, xL), (g, g, up))
        elif emit:
            torch.autograd.backward((first, fm, emb), (g, g, up))
        else:
            torch.autograd.backward((first, fm), (g, g))

    def step_micro(slot, captured):
        """The sharded step as two micro-batches: half 1 runs on a second stream and starts its row exchange when
        half 0's rows have been sent, so its NVLink-bound gather + send runs underneath half 0's forward, and its
        forward underneath half 0's segmented reduce.  One owner update per batch (finish_step)."""
        nxt = (slot + 1) % R
        main, sb = torch.cuda.current_stream(), layer.micro_stream(dev)
        ha, hb = handles[slot]
        if captured:
            side.wait_stream(main)
            with torch.cuda.stream(side):
                id_work(nxt, phase="local", inline=True)
        a = model(slot, 0)
        sb.wait_event(ha.gs_done)
        with torch.cuda.stream(sb):
            b = model(slot, 1)
        if captured:
            side.wait_stream(main)
            side.wait_stream(sb)
            with torch.cuda.stream(side):
                id_work(nxt, phase="exchange", inline=True)
        backward(*a[:5])
        with torch.cuda.stream(sb):
            backward(*b[:5])
        main.wait_stream(sb)
        layer.finish_step(ha, hb)
        if captured:
            main.wait_stream(side)
        else:
            id_work(nxt)
        return torch.cat([a[5], b[5]])

    def step(slot, captured=False):
        """One step on resident inputs of `slot` plus the id-only work of the next slot."""
        nxt = (slot + 1) % R
        main = torch.cuda.current_stream()
        if not sharded:
            id_work(nxt, inline=captured)          # forks onto the side stream itself
            first, fm, emb, g, up, logits = model(slot)
            backward(first, fm, emb, g, up)
            if captured:                           # join the side branch inside the graph
                main.wait_stream(side)
            return logits
        if micro == 2:
            return step_micro(slot, captured)
        if not captured:
            first, fm, emb, g, up, logits = model(slot)
            backward(first, fm, emb, g, up)
            # issued AFTER this step's kernels are queued; it waits (on the device) for this step's rows barrier
            id_work(nxt)
            return logits
        # captured, sharded: the id phase of the next batch is a branch of the same graph.  Its local half (keys,
        # sort, numbering) starts with the step; its exchange half starts once this step's rows barrier has
        # passed -- every rank is then done with the previous step, whose buffers the exchange overwrites.
        side.wait_stream(main)
        with torch.cuda.stream(side):
            id_work(nxt, phase="local", inline=True)
        first, fm, emb, g, up, logits = model(slot)
        side.wait_stream(main)
        with torch.cuda.stream(side):
            id_work(nxt, phase="exchange", inline=True)
        backward(first, fm, emb, g, up)
        main.wait_stream(side)
        return logits

    # warm every slot eagerly (allocates workspaces), note U per slot
    id_work(0)
    if sharded:
        torch.cuda.current_stream().wait_stream(side)
    for r in range(R):
        step(r)
        n_rows_touched.append(int(layer.last_n_unique.item()))
    torch.cuda.synchronize()
    if sharded:
        layer.check_errors()
    cursor[0] = 0                                  # the last step left slot 0's id work ready

    graphs, graph_out = [None] * R, [None] * R
    use_graph = not args.no_graph and (not sharded or (layer.px is not None and R % 2 == 0))
    if use_graph:
        try:
            if sharded:
                # one more eager round so that every slot has run with exactly the parity it is captured with
                for r in range(R):
                    step(r)
                torch.cuda.synchronize()
                flat = [hs if isinstance(hs, list) else [hs] for hs in handles]
                assert all(h.parity == r % 2 for r, hs in enumerate(flat) for h in hs), "parity drifted"
                if world > 1:
                    dist.barrier()
            torch.cuda.synchronize()
            for hs_ in handles:                    # a captured stream may not wait for an event recorded outside the
                for h_ in (hs_ if isinstance(hs_, list) else [hs_]):     # capture; everything those events ordered
                    h_.event = None                                      # has completed
            cap_stream = torch.cuda.Stream()
            cap_stream.wait_stream(torch.cuda.current_stream())
            layer.capturing = True
            pool = None
            with torch.cuda.stream(cap_stream):
                for r in range(R):
                    g_ = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g_, pool=pool, stream=cap_stream, capture_error_mode="thread_local"):
                        graph_out[r] = step(r, captured=True)
                    pool = g_.pool()
                    graphs[r] = g_
            layer.capturing = False
            torch.cuda.current_stream().wait_stream(cap_stream)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
        except Exception as e:                                       # eager launches are still our kernels
            layer.capturing = False
            if rank == 0:
                print("bench.py: CUDA graph capture failed (%s); launching eagerly" % e, file=sys.stderr)
            use_graph = False
            torch.cuda.synchronize()
    if not sharded:
        id_work(0)                                 # slot 0's list for the first step
        torch.cuda.synchronize()

    def run():
        slot = cursor[0] % R
        cursor[0] += 1
        if use_graph:
            if sharded:
                ev = ready_events.get((slot + 1) % R)
                if ev is not None:                 # e2e: the graph's id branch reads the next batch
                    torch.cuda.current_stream().wait_event(ev)
            graphs[slot].replay()
            return slot, graph_out[slot]
        return slot, step(slot)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    lib = dir_b200._lib.lib()
    # per-step launch count of OUR kernels (graph replays do not pass through the library's counter)
    n0 = lib.dir_launch_count()
    s0 = cursor[0] % R
    step(s0)
    cursor[0] += 1
    launches_per_step = int(lib.dir_launch_count() - n0)
    torch.cuda.synchronize()

    # ---------------- value: device-resident inputs -------------------------------------------
    for s in range(max(3, args.warmup)):           # never fewer than three untimed steps, whatever --warmup says
        run()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        ev0.record()
        for s in range(args.steps):
            run()
        ev1.record()
        clocks.sample()
        torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    barrier()
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    value = B * world * args.steps / (ms * 1e-3)
    if args.dump_outputs:
        if rank == 0:
            last = (cursor[0] - 1) % R             # the slot the last timed step ran on
            halves = [None] if micro == 1 else [0, 1]
            dump_outputs(args.dump_outputs, [produced[(use_graph, last, x)] for x in halves], layer, cross)
        barrier()                                  # the other ranks' next steps hold the device-side rows barrier

    # ---------------- e2e: pinned host inputs, H2D + D2H inside the timed region ---------------
    e2e = None
    if not args.no_e2e and R >= 3:
        # R device slots form a ring: while step s computes on its slot, the id work of batch s+1 (already on
        # the device) runs on the side stream and batch s+2 lands through the copy stream.
        # The host ships what the reference's input_fn yields -- one column per feature: int32 ids of the
        # categorical fields, floats of the numeric ones, labels -- and dir_expand_features widens them into
        # feature_index / feature_value on the copy stream (--feed resolved ships the [B,F] pair instead).
        if args.feed == "columns":
            sp_f = [f for f, n in enumerate(w.rows_per_field) if n > 1]
            de_f = [f for f, n in enumerate(w.rows_per_field) if n == 1]
            feeder = dir_b200.ColumnFeeder(sp_f, de_f, *devs, index_dtype=torch.int32)
            host = [[hs[0][:, sp_f].to(torch.int32).contiguous().pin_memory(),
                     hs[1][:, de_f].contiguous().pin_memory(), hs[2]] for hs in host]
        else:
            feeder = dir_b200.HostFeeder(*devs)
        out_host = [torch.empty((B, 1), dtype=torch.float32).pin_memory() for _ in range(2)]
        h2d = sum(t.numel() * t.element_size() for t in host[0])
        d2h = out_host[0].numel() * 4
        ahead = 2
        d2h_stream = torch.cuda.Stream()

        def e2e_loop(n):
            # Slot cursor % R holds the batch whose id work the previous step already did from the RESIDENT copy
            # of that slot; the feeder ships the same batch again, so the first step stays consistent.
            c0 = cursor[0]
            for s in range(min(ahead, n)):
                feeder.prefetch((c0 + s) % R, host[(c0 + s) % R])
            for s in range(n):
                cur = (c0 + s) % R
                if s + ahead < n:
                    feeder.prefetch((c0 + s + ahead) % R, host[(c0 + s + ahead) % R])
                feeder.wait(cur)
                if s + 1 < n:
                    if not sharded and not use_graph:
                        feeder.wait((c0 + s + 1) % R)        # this step presorts the next batch
                    else:
                        ready_events[(c0 + s + 1) % R] = feeder.ready[(c0 + s + 1) % R]
                else:
                    ready_events.pop((c0 + s + 1) % R, None)   # the batch after the last one is the resident copy
                if not sharded and use_graph and s + 1 < n:
                    torch.cuda.current_stream().wait_event(feeder.ready[(c0 + s + 1) % R])
                _, o = run()
                feeder.release(cur)
                # the logits go home on a stream of their own: on the compute stream the 0.26 MB copy (and its
                # latency) would sit between two steps; `o` is the slot's static output, rewritten R steps later
                done = torch.cuda.Event()
                done.record()
                d2h_stream.wait_event(done)
                o.record_stream(d2h_stream)
                with torch.cuda.stream(d2h_stream):
                    out_host[s & 1].copy_(o, non_blocking=True)
            torch.cuda.current_stream().wait_stream(d2h_stream)
            torch.cuda.current_stream().synchronize()
            ready_events.clear()

        e2e_loop(max(4, args.warmup))
        barrier()
        ev0.record()
        e2e_loop(args.steps)
        ev1.record()
        torch.cuda.synchronize()
        t = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e = {"value": B * world * args.steps / (float(t.item()) * 1e-3), "unit": UNIT,
               "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "feed": "columns: int32 ids [B,%d] + fp32 values [B,%d] + labels [B], widened on the device by "
                       "dir_expand_features" % (len(sp_f), len(de_f)) if args.feed == "columns"
                       else "resolved: feature_index [B,F] int64 + feature_value [B,F] fp32 + labels [B]",
               "how": "%s.presort/forward/backward fed by %s from pinned host memory "
                      "(ring of %d device slots, H2D on a copy stream), logits read back each step on a third stream" % (
                          type(layer).__name__, type(feeder).__name__, R)}
        torch.cuda.synchronize()

    if args.profile:
        from torch.profiler import ProfilerActivity, profile
        barrier()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for s in range(6):
                run()
            torch.cuda.synchronize()
        barrier()
        if rank == 0:
            prof.export_chrome_trace(args.profile)

    # ---------------- roofline: each C-ABI call timed on its own (rank 0's GPU) ---------------
    roof, kernels = None, []
    if not sharded:
        roof, kernels = time_calls(dir_b200, RL, layer, cross, devs, ups, w, B, emit, n_rows_touched,
                                   min(50, max(5, args.steps)))

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu and w.name != "cfg4":     # a 56 GB host table is not a bounded sample
        wc = dir_b200.synth.cfg("cfg2") if w.name == "cfg3" else w
        r = cpu_restatement(wc, 3, 1, args.cpu_seconds, B)
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
               "sample": r["sample"] + "; PyTorch-CPU restatement of the reference's TF 1.x graph",
               "cpu_model": cpu_model_name()}
        try:
            cpu["cfg1"] = cpu_cfg1()
        except Exception as e:                                   # an extra, never worth the bench line
            print("bench.py: cfg1 CPU timing skipped (%s)" % e, file=sys.stderr)

    stages, nvlink, serial = None, None, None
    if sharded and micro == 1 and getattr(layer, "trace", None) is not None:
        # Stage times of the sharded step: a diagnostic pass AFTER the timed regions.  Eager launches, every stage
        # bracketed by CUDA events on its stream, one device sync per step.  Every rank takes part (the steps
        # contain the cross-rank barriers); rank 0 reports.
        try:                                  # the same code on every rank: a failure here is symmetric
            layer.trace.on = layer.trace_pre.on = True
            layer.trace.report()
            layer.trace_pre.report()
            for s_ in range(8):
                step(cursor[0] % R)
                cursor[0] += 1
            torch.cuda.synchronize()
            stages = (layer.trace.report(), layer.trace_pre.report())
            # the same stages with NOTHING overlapped: the id phase inline on the main stream (exclusive times)
            torch.cuda.current_stream().wait_stream(side)
            cur = cursor[0] % R                      # its id work is pending: run it, then go inline
            first, fm, emb, g, up, _ = model(cur)
            backward(first, fm, emb, g, up)
            for s_ in range(9):
                if s_ == 3:                          # the first inline steps allocate their handle: not timed
                    torch.cuda.synchronize()
                    layer.trace.report()
                    layer.trace_pre.report()
                idx_, val_, y_ = devs[s_ % R]
                first, fm, emb = layer(idx_, val_)
                with torch.no_grad():
                    g = torch.sigmoid(first + fm).sub_(y_.unsqueeze(1))
                backward(first, fm, emb, g, ups[s_ % R])
            torch.cuda.synchronize()
            serial = (layer.trace.report(), layer.trace_pre.report())
            cursor[0] = -1                           # the rotation is broken from here on: nothing may run() again
        except Exception as e:
            stages = None
            if rank == 0:
                print("bench.py: stage trace skipped (%s)" % e, file=sys.stderr)
        layer.trace.on = layer.trace_pre.on = False
        # The three exchange calls on their own, each replayed from a CUDA graph (no host gaps, nothing else on the
        # GPU), every rank at the same time so that the NVLink stores meet the traffic they meet in a step.  They run
        # on the state the last traced step left behind: ids and headers in the exchange buffers, the sorted list in
        # the handle, the slot map.  (The owner update re-applies the same sums: timing only, after every parity check.)
        calls_us = None
        try:
            calls_us = time_sharded_calls(dir_b200, layer, devs[8 % R], ups[8 % R], B, barrier)
        except Exception as e:
            if rank == 0:
                print("bench.py: sharded call timing skipped (%s)" % e, file=sys.stderr)
        if rank == 0 and stages is not None:
            try:
                main = serial[0] if serial else stages[0]     # exclusive stage times
                U = int(layer.last_exchange.get("unique_sent", 0))
                row_bytes = (K + 1) * 4                                   # (row, first-order weight) per distinct row
                key = "bwd.emit+push" if "bwd.emit+push" in main else "bwd.emit"
                # requester half of the backward: g, upstream u, per lookup id + value + one K-vector, per distinct
                # row the (G[K], g1) sums written to its owner
                nbytes = 4 * B + (B * d * 4 if emit else 0) + B * F * (8 + 4 + 4 * K) + U * row_bytes
                peak, src = RL.measured_peaks()
                t_emit, how = main[key], ("exclusive stage time (CUDA events, rank 0) from an eager, non-overlapped "
                                          "traced pass after the timed regions: host gaps included")
                if calls_us and key.endswith("push"):
                    t_emit, how = calls_us["dir_embed_bwd_reduce_emit_to"], (
                        "the call replayed from its own CUDA graph, CUDA events, every rank at the same time")
                gbs = nbytes / t_emit * 1e-3
                roof = {"bound": "hbm", "kernel": "dir_embed_bwd_reduce_emit_to" if key.endswith("push") else
                        "dir_embed_bwd_reduce_emit", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                        "peak_source": "%s (MEASURED_PEAKS.json hbm_gbs)" % src if src == "measured"
                        else "fallback (B200_PROFILING.md)", "traffic": None, "algorithmic_bytes_per_launch": int(nbytes),
                        "us_per_launch": t_emit, "how": how}
                link = U * row_bytes * (world - 1) / world                 # bytes that leave / reach this rank, each way
                t_fwd = calls_us["dir_shard_gather_send"] if calls_us else main.get("fwd.gather+send")
                nvlink = {"bytes_per_direction_per_rank": int(link), "peak": 770.0, "unit": "GB/s",
                          "peak_source": "measured peer copy per direction (B200_PROFILING.md); nominal 900",
                          "rows_gather_to_gbs": link / t_fwd * 1e-3 if t_fwd else None,
                          "frac": link / t_fwd * 1e-3 / 770.0 if t_fwd else None}
            except Exception as e:                                         # diagnostics must never cost the bench line
                print("bench.py: stage roofline skipped (%s)" % e, file=sys.stderr)
    if rank == 0:
        cfg = workload_config(w, args, world)
        if sharded:
            cfg["micro_batches"] = micro
        cfg.update({"l2_policy": "%d rotating input sets (%.0f MB of ids/values/upstream each) + a %.2f GB table: "
                                 "inputs larger than L2, no flush" % (
                                     R, (B * F * 12 + (B * d * 4 if emit else 0)) / 1e6,
                                     layer.rows.numel() * 4 / 1e9),
                    "cuda_graphs": use_graph, "rows_touched_per_step": int(np.mean(n_rows_touched))})
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "strong" if args.strong else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": cfg, "clocks": clocks.summary(), "e2e": e2e,
                "gpu_launches": launches_per_step * args.steps, "roofline": roof, "kernels": kernels,
                "cpu_baseline": cpu}
        if stages is not None:
            line["stages_us"] = {"main_stream": {k: round(v, 1) for k, v in stages[0].items()},
                                 "side_stream": {k: round(v, 1) for k, v in stages[1].items()},
                                 "serial_main": {k: round(v, 1) for k, v in serial[0].items()},
                                 "serial_id_phase": {k: round(v, 1) for k, v in serial[1].items()}}
            line["nvlink"] = nvlink
            if calls_us:
                line["sharded_calls_us"] = {k: round(v, 1) for k, v in calls_us.items()}
    if world > 1:
        dist.destroy_process_group()       # first: whatever NCCL still has to say must not follow the JSON line
    if rank == 0:
        sys.stdout.flush()
        print(json.dumps(line), flush=True)


DUMP_SEED = 1239
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path, outs, layer, cross):
    """Write one step's outputs (`outs`: the step's micro-batches in order, dicts of device tensors) and the layer's
    state after it as path/<name>.npy, float32; sampled positions as float64 `*_index` arrays.

    Per sample: logits, first_order, fm on up to 65 536 samples; embeddings and cross_out (the DCN cross output) on up
    to 4 MB worth of samples.  State: table, accumulator, linear, linear_accumulator on up to 262 144 rows of this
    rank's table, bias, and cross_w_grad_sum / cross_b_grad_sum: the cross parameters' .grad, which nothing zeroes,
    so the sum over every step run so far (warm-up and capture included).  Samples are drawn from a fixed seed, so two
    runs with the same arguments write the same positions.  .npy files already in `path` are removed first: the
    directory holds this run's arrays only."""
    import numpy as np
    import torch

    rng = np.random.default_rng(DUMP_SEED)

    def pick(n, k):
        return np.sort(rng.choice(n, size=min(n, k), replace=False))

    def rows_of(t, index):
        return t.index_select(0, torch.as_tensor(index, device=t.device)).cpu().numpy().astype(np.float32)

    step = {k: torch.cat([o[k] for o in outs]) for k in outs[0]}
    B = step["logits"].shape[0]
    arrays = {}
    s = pick(B, 1 << 16)
    arrays["sample_index"] = s.astype(np.float64)
    for k in ("logits", "first_order", "fm"):
        arrays[k] = rows_of(step[k].reshape(B), s)
    if step["embeddings"].numel():
        e = pick(B, max(1, (4 << 20) // (4 * step["embeddings"].shape[1])))
        arrays["embedding_sample_index"] = e.astype(np.float64)
        for k in ("embeddings", "cross_out"):
            if k in step:
                arrays[k] = rows_of(step[k].reshape(B, -1), e)
    n = layer.plan.n_local if hasattr(layer, "plan") else layer.n_rows
    r = pick(n, 1 << 18)
    arrays["table_row_index"] = r.astype(np.float64)
    for k, t in (("table", layer.table), ("accumulator", layer.accum), ("linear", layer.w1),
                 ("linear_accumulator", layer.w1_accum)):
        if t is not None:
            arrays[k] = rows_of(t, r)
    arrays["bias"] = layer.bias.detach().cpu().numpy().astype(np.float32)
    if cross is not None:
        for k in ("cross_w", "cross_b"):
            grad = getattr(cross, k).grad
            if grad is not None:
                arrays[k + "_grad_sum"] = grad.cpu().numpy().astype(np.float32)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit("bench.py: --dump-outputs would write %d bytes (limit %d)" % (total, DUMP_MAX_BYTES))
    os.makedirs(path, exist_ok=True)
    for f in os.listdir(path):
        if f.endswith(".npy"):
            os.remove(os.path.join(path, f))
    for k, a in arrays.items():
        np.save(os.path.join(path, k + ".npy"), a)
    print("bench.py: wrote %d arrays (%.1f MB) to %s" % (len(arrays), total / 1e6, path), file=sys.stderr)


def time_sharded_calls(pkg, layer, dev_set, up, B, barrier, iters=20):
    """CUDA-event time (us, this rank) of dir_shard_gather_send, dir_embed_bwd_reduce_emit_to and
    dir_shard_owner_update, each replayed from a CUDA graph of its own, on the state of the layer's last step."""
    import torch
    from dir_b200._lib import check, ptr
    from dir_b200.layers import _OPTIMIZERS, linear_opt_struct
    L = pkg._lib.lib()
    h = layer._last_handle
    px, p = layer.px, h.buf
    idx, val, _ = dev_set
    F, K = layer.field_size, layer.embedding_size
    dev = idx.device
    adagrad = layer.optimizer == "adagrad"
    S = torch.randn((B, K), device=dev) * 0.1
    g1 = torch.randn(B, device=dev) * 0.1
    n = B * layer.n_sel
    n_keys = layer.plan.cap * layer.plan.world_size
    ws = h.ws.get(L.dir_embed_bwd_workspace_bytes(max(n, 1), K), dev)
    nu = torch.zeros(1, dtype=torch.int64, device=dev)

    def gather_send(st):
        check(L.dir_shard_gather_send(px.ref(p), ptr(layer.table), layer.row_stride,
                                      ptr(layer.w1) if layer.first_order else None, layer.lin_stride,
                                      ptr(layer.dense_table) if layer.n_dense else None, layer.row_stride,
                                      ptr(layer.dense_lin) if (layer.n_dense and layer.first_order) else None,
                                      layer.gather_ctas_per_sm, st), "gather_send")

    def emit_to(st):
        check(L.dir_embed_bwd_reduce_emit_to(
            px.ref(p), ptr(val), ptr(g1) if layer.first_order else None, ptr(g1), ptr(S), ptr(up), ptr(h.uidx),
            ptr(h.owner_off), B, F, n_keys, ptr(layer.sparse_fields) if layer.n_sel < F else None, layer.n_sel,
            ptr(h.g1_local), ptr(ws), ws.numel(), st), "emit_to")

    def owner_update(st):
        check(L.dir_shard_owner_update(
            px.ref(p), ptr(layer.slot[p]), ptr(layer.table), ptr(layer.accum) if adagrad else None,
            layer.row_stride, ptr(layer.w1) if layer.first_order else None,
            ptr(layer.w1_accum) if layer.first_order else None, layer.lin_stride, layer.n_rows,
            ptr(layer.slot_epoch[p]), _OPTIMIZERS[layer.optimizer], layer.lr, None, linear_opt_struct(layer),
            None, None, None, nu.data_ptr(), st), "owner_update")

    calls = [("dir_shard_gather_send", gather_send), ("dir_embed_bwd_reduce_emit_to", emit_to),
             ("dir_shard_owner_update", owner_update)]
    torch.cuda.synchronize()
    graphs = {}
    cap = torch.cuda.Stream()
    cap.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(cap):
        for name, fn in calls:
            fn(cap.cuda_stream)                      # eager once
        cap.synchronize()
        for name, fn in calls:
            g_ = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_, stream=cap):
                fn(torch.cuda.current_stream().cuda_stream)
            graphs[name] = g_
    torch.cuda.current_stream().wait_stream(cap)
    torch.cuda.synchronize()
    out = {}
    for name, _ in calls:
        barrier()
        evs = []
        for it in range(3 + iters):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            graphs[name].replay()
            b.record()
            if it >= 3:
                evs.append((a, b))
        torch.cuda.synchronize()
        out[name] = 1e3 * sum(a.elapsed_time(b) for a, b in evs) / len(evs)
    return out


def time_calls(pkg, RL, layer, cross, devs, ups, w, B, emit, n_unique, iters):
    """CUDA-event time of each C-ABI call on torch's current stream (the one they are launched on),
    rotating inputs; returns (roofline of the dominant call, per-call table)."""
    import torch
    from dir_b200._lib import check, ptr
    lib = pkg._lib.lib()
    F, K = w.field_size, w.embedding_size
    L, d = w.cross_layer_num, F * K
    R = len(devs)
    dev = devs[0][0].device
    st = torch.cuda.current_stream().cuda_stream
    emb = torch.empty((B, d), device=dev) if emit else None
    S = torch.empty((B, K), device=dev)
    first, fm = torch.empty(B, device=dev), torch.empty(B, device=dev)
    keys = torch.empty(B * F, dtype=torch.int32, device=dev)
    g = (ups[0][:, 0] * 10.0).contiguous() if ups[0] is not None else torch.full((B,), 0.1, device=dev)
    ws = torch.empty(int(lib.dir_embed_bwd_workspace_bytes(B * F, K)), dtype=torch.uint8, device=dev)
    peak, src = RL.measured_peaks()
    U = sum(n_unique) / len(n_unique)
    n_sel = layer.n_sorted_fields

    def keys_sort(r):
        idx, val, _ = devs[r]
        check(lib.dir_shard_keys_sort(ptr(idx), ptr(val), ptr(layer.field_offset), ptr(layer.field_rows),
                                      layer.n_rows, B, F, 1, ptr(layer.sorted_fields), n_sel, ptr(keys), None,
                                      ptr(ws), ws.numel(), st), "keys_sort")

    def fwd(r):
        idx, val, _ = devs[r]
        check(lib.dir_embed_fm_fwd(ptr(layer.table), layer.row_stride, ptr(layer.w1), layer.lin_stride,
                                   ptr(layer.bias), ptr(idx), ptr(val), ptr(layer.field_offset),
                                   ptr(layer.field_rows), layer.n_rows, B, F, K, ptr(emb), ptr(S), ptr(first),
                                   ptr(fm), None, None, st), "fwd")

    ows = torch.empty(int(lib.dir_shard_dense_workspace_bytes(K)), dtype=torch.uint8, device=dev)
    nu = torch.zeros(2, dtype=torch.int64, device=dev)
    aux = layer.aux_stream(dev)

    def upd(r):
        # as the layer's backward runs it: the one-row fields' column sums on a second stream underneath the sorted
        # segmented reduce (disjoint rows); the events bracket both
        cur = torch.cuda.current_stream()
        if layer.n_onerow_fields:
            aux.wait_stream(cur)
            check(lib.dir_embed_bwd_onerow_update(
                ptr(layer.table), ptr(layer.accum), layer.row_stride, ptr(layer.w1), ptr(layer.w1_accum),
                layer.lin_stride, ptr(devs[r][0]), ptr(devs[r][1]), ptr(layer.field_offset), ptr(g), ptr(g), ptr(S),
                ptr(ups[r]) if emit else None, B, F, K, ptr(layer.onerow_fields), layer.n_onerow_fields, 1, LR, None, None, 0.0,
                ptr(ows), ows.numel(), nu[1:].data_ptr(), aux.cuda_stream), "onerow")
        check(lib.dir_embed_bwd_reduce_update(
            ptr(layer.table), ptr(layer.accum), layer.row_stride, ptr(layer.w1), ptr(layer.w1_accum),
            layer.lin_stride, ptr(devs[r][0]), ptr(devs[r][1]), ptr(layer.field_offset), ptr(g), ptr(g), ptr(S),
            ptr(ups[r]) if emit else None, B, F, K, layer.n_rows, ptr(layer.sorted_fields), n_sel,
            None, 0, 1, LR, None, None, ptr(ws), ws.numel(), nu.data_ptr(), st), "update")
        if layer.n_onerow_fields:
            cur.wait_stream(aux)

    calls = [("dir_embed_fm_fwd", fwd, RL.embed_fwd_bytes(B, F, K, True, emit)),
             ("dir_shard_keys_sort", keys_sort, 0),
             ("dir_embed_bwd_reduce_update", upd, RL.embed_bwd_bytes(B, F, K, U, True, emit, "adagrad"))]
    if cross is not None:
        xL, s = torch.empty((B, d), device=dev), torch.empty((B, L), device=dev)
        dx0, dw, db = torch.empty((B, d), device=dev), torch.empty((L, d), device=dev), torch.empty((L, d), device=dev)
        cws = torch.empty(int(lib.dir_cross_bwd_workspace_bytes(B, d, L)), dtype=torch.uint8, device=dev)

        def cf(r):
            check(lib.dir_cross_fwd(ptr(emb), ptr(cross.cross_w), ptr(cross.cross_b), B, d, L, ptr(xL), ptr(s), st), "cf")

        def cb(r):
            check(lib.dir_cross_bwd(ptr(emb), ptr(cross.cross_w), ptr(cross.cross_b), ptr(ups[r]), ptr(s), B, d, L,
                                    ptr(dx0), ptr(dw), ptr(db), ptr(cws), cws.numel(), st), "cb")
        calls += [("dir_cross_fwd", cf, RL.cross_fwd_bytes(B, d, L)), ("dir_cross_bwd", cb, RL.cross_bwd_bytes(B, d, L))]

    # One pass in order keeps each call's inputs valid; events bracket every call.  Each call is replayed from a
    # CUDA graph of its own (captured once per input set), so that the bracket holds the call's kernels and not the
    # host's launch gaps between them (a call is several launches, and the backward forks a second stream); if the
    # capture fails the calls are launched eagerly.
    evs = {name: [] for name, _, _ in calls}
    for r in range(R):                              # eager once: workspaces exist, errors surface here
        for name, fn, _ in calls:
            fn(r)
    torch.cuda.synchronize()
    replay, how = {}, "each call replayed from its own CUDA graph"
    try:
        cap = torch.cuda.Stream()
        cap.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(cap):
            for name, fn, _ in calls:
                for r in range(R):
                    g_ = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g_, stream=cap):
                        st = torch.cuda.current_stream().cuda_stream      # (the closures read `st`)
                        fn(r)
                    replay[(name, r)] = g_
        torch.cuda.current_stream().wait_stream(cap)
        torch.cuda.synchronize()
    except Exception as e:
        print("bench.py: per-call graph capture failed (%s); timing eager launches" % e, file=sys.stderr)
        replay, how = {}, "eager launches (host gaps between a call's kernels included)"
        torch.cuda.synchronize()
    st = torch.cuda.current_stream().cuda_stream
    for it in range(3 + iters):
        r = it % R
        for name, fn, _ in calls:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            if replay:
                replay[(name, r)].replay()
            else:
                fn(r)
            b.record()
            if it >= 3:
                evs[name].append((a, b))
    torch.cuda.synchronize()
    table = []
    for name, _, nbytes in calls:
        ms = sum(a.elapsed_time(b) for a, b in evs[name]) / len(evs[name])
        table.append({"call": name, "us": ms * 1e3, "algorithmic_bytes": int(nbytes),
                      "achieved_gbs": nbytes / (ms * 1e-3) / 1e9 if nbytes else None})
    top = max((t for t in table if t["algorithmic_bytes"]), key=lambda t: t["us"])
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath)).get(w.name, {}).get(top["call"])
        except Exception:
            traffic = None
    roof = {"bound": "hbm", "kernel": top["call"], "achieved": top["achieved_gbs"], "peak": peak, "unit": "GB/s",
            "frac": top["achieved_gbs"] / peak, "frac_of_nominal_8000": top["achieved_gbs"] / 8000.0,
            "traffic_source": "profiles/traffic.json: dram__bytes_read + write of one ncu --set full capture of this "
                              "kernel on this workload, committed with the profile; not re-measured in this run",
            "call_note": "dir_embed_bwd_reduce_update is timed as the layer runs it: dir_embed_bwd_onerow_update (the "
                         "one-row fields) on a second stream underneath the sorted segmented reduce", "peak_source": "%s (MEASURED_PEAKS.json hbm_gbs)" % src
            if src == "measured" else "fallback (B200_PROFILING.md)", "traffic": traffic,
            "algorithmic_bytes_per_launch": top["algorithmic_bytes"], "us_per_launch": top["us"], "timing": how}
    return roof, table


def watchdog(seconds):
    """A lost cross-rank barrier traps on the device after 20 s (sharded.BARRIER_TIMEOUT_MS); anything else that
    wedges the process is ended here rather than at the driver's limit."""
    def fire():
        print("bench.py: watchdog: no result after %d s, aborting" % seconds, file=sys.stderr, flush=True)
        os._exit(3)
    t = threading.Timer(seconds, fire)
    t.daemon = True
    t.start()
    return t


def main():
    args = parse_args()
    watchdog(float(os.environ.get("DIR_B200_WATCHDOG_S", "600")))
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
