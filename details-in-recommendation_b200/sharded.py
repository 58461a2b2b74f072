"""Row-sharded embedding + FM layer: one process per GPU, tables sharded by row over the ranks of a
process group, the FM / first-order / cross interaction data-parallel on the requesting rank
(SURVEY.md section 8e).

The reference's only hook for this is the partitioner around its embedding variables
(`input_layer_partitioner`, models/DeepFM/deepFM.py:163-175): with a TF parameter-server cluster
the variables are split by row and ids / IndexedSlices travel over gRPC.  Here only DISTINCT rows
travel: the requester sorts its lookups by (owner, local row), numbers the distinct ones, and after
the owner answered runs the ordinary forward kernel on the received rows; in the backward it sums
the gradients of each distinct row before shipping them, so a Zipf-hot row costs one row of traffic
per rank and step instead of one per lookup.  One-row (numeric) fields are replicated parameters.

The exchange runs over NVLink peer memory and is driven from the device: kernels store straight into the
peers' exchange buffers (symmetric memory), counts travel as headers read on the device, a device-side barrier
separates the phases.  No NCCL, no host read: the whole step replays from a CUDA graph (csrc/shard_peer.cu).
With one process the buffers are plain local memory.

`ShardPlan` (pure index arithmetic) carries no CUDA-only code: tests run it on CPU.
"""
import math
import os
import sys
from typing import Optional, Sequence

import torch
import torch.distributed as dist

from . import _lib
from ._lib import check, ptr
from .layers import (_CLIP_MAX_FIELDS, _K_OK, _LINEAR_OPTIMIZERS, _TABLE_OPTIMIZERS, _Workspace, _need_cuda,
                     _stream, linear_opt_struct, table_opt_struct, resolve_linear_optimizer)


class ShardPlan:
    """owner = global row mod G, local row = global row div G (modulo, so hot low rows spread)."""

    def __init__(self, rows_per_field: Sequence[int], world_size: int, rank: int):
        if world_size <= 0 or not 0 <= rank < world_size:
            raise ValueError("need 0 <= rank < world_size")
        self.rows_per_field = [int(r) for r in rows_per_field]
        self.world_size, self.rank = world_size, rank
        self.n_rows = sum(self.rows_per_field)
        off = [0]
        for r in self.rows_per_field[:-1]:
            off.append(off[-1] + r)
        self.field_offset = off
        self.cap = (self.n_rows + world_size - 1) // world_size          # rows every rank allocates
        self.n_local = (self.n_rows - rank + world_size - 1) // world_size if self.n_rows > rank else 0
        if self.cap * world_size >= 2 ** 32 - 1:
            raise ValueError("ceil(n_rows / world_size) * world_size must be < 2^32-1")

    def owner(self, global_rows):
        return global_rows % self.world_size

    def local_row(self, global_rows):
        return global_rows // self.world_size

    def global_row(self, local_rows, rank=None):
        return local_rows * self.world_size + (self.rank if rank is None else rank)

    def shard_of(self, full):
        """This rank's rows of a full [n_rows, ...] array (numpy or torch)."""
        return full[self.rank::self.world_size]

    def local_field_offset(self, rank=None):
        """[F + 1]: the first local row of each field on `rank`, then its local row count.  Local row l is global row
        l * G + rank, so a field's rows on one rank are contiguous; a field with fewer rows than G may have none."""
        r = self.rank if rank is None else rank
        G = self.world_size
        return [max(0, (x - r + G - 1) // G) for x in self.field_offset + [self.n_rows]]


class StageTrace:
    """Optional per-stage CUDA-event timing of the sharded step (DIR_B200_TRACE=1): mark(name) closes
    the stage that just ran; report() averages over the steps seen since the last report."""

    def __init__(self):
        self.on = os.environ.get("DIR_B200_TRACE", "0") == "1"
        self.marks, self.tot, self.steps = [], {}, 0

    def mark(self, name):
        if self.on:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.marks.append((name, ev))

    def close_step(self):
        if not self.on or len(self.marks) < 2:
            return
        torch.cuda.synchronize()
        for (_, a), (name, b) in zip(self.marks[:-1], self.marks[1:]):
            self.tot[name] = self.tot.get(name, 0.0) + a.elapsed_time(b) * 1e3
        self.marks, self.steps = [], self.steps + 1

    def report(self):
        out = {k: v / max(1, self.steps) for k, v in self.tot.items()}
        self.tot, self.steps = {}, 0
        return out


BARRIER_TIMEOUT_MS = int(os.environ.get("DIR_B200_BARRIER_TIMEOUT_MS", "20000"))


class PeerExchange:
    """The exchange buffers of the device-driven path: one per parity (consecutive steps alternate), laid out by
    `dir_peer_layout_init`, allocated as symmetric memory (torch.distributed._symmetric_memory: CUDA IPC mappings
    over NVLink + a device-side barrier) and mapped by every peer.  With one process they are plain local memory
    and the barrier is a no-op: the same kernels run.  `barrier(p, channel)` is a device-side cross-rank barrier on
    the current stream; a lost barrier traps after BARRIER_TIMEOUT_MS instead of spinning forever."""

    def __init__(self, group, world, rank, K, n_dense, seg_cap, u_cap, device, n_buf=2, norm_bytes=0):
        L = _lib.lib()
        self.world, self.rank, self.K, self.n_dense = world, rank, K, n_dense
        self.seg_cap, self.u_cap = int(seg_cap), int(u_cap)
        self.layouts, self.bufs, self.handles, self.peer_base = [], [], [], []
        for _ in range(n_buf):
            lay = _lib.PeerLayout()
            check(L.dir_peer_layout_init(world, rank, K, n_dense, self.seg_cap, self.u_cap, _lib.ctypes.byref(lay)),
                  "dir_peer_layout_init")
            buf, h, base = self._symmetric(group, world, int(lay.total_bytes), torch.uint8, device)
            lay.peer_base, lay.local = base.data_ptr(), buf.data_ptr()
            self.layouts.append(lay)
            self.bufs.append(buf)
            self.handles.append(h)
            self.peer_base.append(base)
        # clip_norm: one small norm buffer per exchange buffer ([G][F][kClipSlices][2] doubles), each with a barrier of
        # its own (its own symmetric allocation)
        self.norm_bufs, self.norm_handles, self.norm_peers = [], [], []
        for _ in range(n_buf if norm_bytes else 0):
            buf, h, base = self._symmetric(group, world, norm_bytes // 8, torch.float64, device)
            self.norm_bufs.append(buf)
            self.norm_handles.append(h)
            self.norm_peers.append(base)
        if world > 1:
            torch.cuda.synchronize(device)
            dist.barrier(group)                      # nobody stores into a buffer its owner is still zeroing

    @staticmethod
    def _symmetric(group, world, n, dtype, device):
        """(zeroed buffer, symmetric-memory handle or None, device array of the G ranks' addresses)"""
        if world > 1:
            import torch.distributed._symmetric_memory as symm_mem
            buf = symm_mem.empty(n, dtype=dtype, device=device)
            h = symm_mem.rendezvous(buf, group if group is not None else dist.group.WORLD)
            base = torch.tensor(list(h.buffer_ptrs), dtype=torch.int64, device=device)
        else:
            buf, h = torch.empty(n, dtype=dtype, device=device), None
            base = torch.tensor([buf.data_ptr()], dtype=torch.int64, device=device)
        buf.zero_()
        return buf, h, base

    def ref(self, p):
        return _lib.ctypes.byref(self.layouts[p])

    def rows(self, p):
        lay = self.layouts[p]
        n = self.u_cap + self.n_dense
        return self.bufs[p][lay.off_rows: lay.off_rows + n * self.K * 4].view(torch.float32).view(n, self.K)

    def w(self, p):
        lay = self.layouts[p]
        n = self.u_cap + self.n_dense
        return self.bufs[p][lay.off_w: lay.off_w + n * 4].view(torch.float32)

    def barrier(self, p, channel=0):
        if self.handles[p] is not None:
            self.handles[p].barrier(channel=channel, timeout_ms=BARRIER_TIMEOUT_MS)

    def norm_barrier(self, p):
        """Every rank has stored its column partials into norm buffer p."""
        if self.norm_handles[p] is not None:
            self.norm_handles[p].barrier(channel=0, timeout_ms=BARRIER_TIMEOUT_MS)


class ShardedLookups:
    """What `ShardedEmbeddingFM.presort` leaves behind for one batch -- everything that depends on the
    ids only: this rank's lookups sorted by (owner, local row), the distinct rows numbered, the ids
    already at their owners."""

    def __init__(self):
        self.ws, self.ws2 = _Workspace(), _Workspace()
        self.keys = self.uidx = self.ulocal = self.inv = self.owner_off = self.g1_local = None
        self.event = None
        self.src = None
        self.n_entries = 0          # lookups in the sorted list (B * sparse fields; bags: nnz)
        self.parity = None          # which exchange buffers this batch uses (set by presort)
        self.half = 0               # micro-batch of its batch (0, or 1 when the batch is exchanged as two halves)
        self.buf = None             # = parity * micro_batches + half: index of the exchange buffer / slot map
        self.gs_done = None         # event: this half's rows have been sent (the other half's exchange may start)
        self.shape = None

    @staticmethod
    def key_of(feature_index, feature_value):
        return (feature_index.data_ptr(), None if feature_value is None else feature_value.data_ptr(),
                tuple(feature_index.shape))


class _ShardedFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, anchor, bias, layer, idx, val, train, h, defer=False):
        B, F = idx.shape
        K = layer.embedding_size
        dev = idx.device
        L = _lib.lib()
        st = _stream()
        tr = layer.trace
        tr.mark("start")
        if h.event is not None and not layer.capturing:
            torch.cuda.current_stream().wait_event(h.event)
        emb = torch.empty((B, F * K), dtype=torch.float32, device=dev) if layer.emit_embeddings else None
        fm = torch.empty((B, 1), dtype=torch.float32, device=dev)
        first = torch.empty((B, 1), dtype=torch.float32, device=dev)
        S = torch.empty((B, K), dtype=torch.float32, device=dev) if train else None
        # the owner answers the ids it received: one kernel gathers the rows and stores them straight
        # into the requesters' buffers over NVLink
        px, p = layer.px, h.buf
        if train:
            # the owner marks who asked for which row (cells carry this use's epoch: nothing is cleared
            # afterwards).  Only the owner's update needs the marks: a second stream, underneath the row exchange
            # and the forward; the backward joins it.
            main, aux = torch.cuda.current_stream(), layer.aux_stream(dev, h.half)
            aux.wait_stream(main)
            check(L.dir_shard_slots(px.ref(p), ptr(layer.slot[p]), layer.n_rows, ptr(layer.slot_epoch[p]),
                                    ptr(layer.err_flag),
                                    layer._n_unique2.data_ptr() + 8 * h.parity if h.half == 0 else None,
                                    aux.cuda_stream), "dir_shard_slots")
        check(L.dir_shard_gather_send(px.ref(p), ptr(layer.table), layer.row_stride,
                                      ptr(layer.w1) if layer.first_order else None, layer.lin_stride,
                                      ptr(layer.dense_table) if layer.n_dense else None, layer.row_stride,
                                      ptr(layer.dense_lin) if (layer.n_dense and layer.first_order) else None,
                                      layer.gather_ctas_per_sm, st), "dir_shard_gather_send")
        h.gs_done = torch.cuda.Event()
        h.gs_done.record()
        tr.mark("fwd.gather+send")
        px.barrier(p, 0)
        layer._note_forward(h.half)
        tr.mark("fwd.barrier")
        rows, lin = px.rows(p), px.w(p) if layer.first_order else None
        check(L.dir_embed_fm_fwd(ptr(rows), K, ptr(lin), 1, ptr(bias) if layer.first_order else None,
                                 ptr(h.inv), ptr(val), ptr(layer.zero_offset), None, rows.shape[0], B, F, K,
                                 ptr(emb), ptr(S), ptr(first), ptr(fm), None, None, st), "dir_embed_fm_fwd")
        tr.mark("fwd.fm")
        if not layer.first_order:
            first.zero_()
        ctx.layer, ctx.train, ctx.shape, ctx.h = layer, train, (B, F, K), h
        ctx.idx, ctx.defer = idx, defer
        ctx.set_materialize_grads(False)
        if train:
            ctx.save_for_backward(val, S)
        if emb is None:
            emb = torch.empty((B, 0), dtype=torch.float32, device=dev)
            ctx.mark_non_differentiable(emb)
        return first, fm, emb

    @staticmethod
    def backward(ctx, g_first, g_fm, u):
        if not ctx.train:
            raise RuntimeError("ShardedEmbeddingFM.backward: forward ran without gradient tracking")
        layer, h = ctx.layer, ctx.h
        B, F, K = ctx.shape
        L = _lib.lib()
        st = _stream()
        val, S = ctx.saved_tensors
        dev = S.device
        g_first = (torch.zeros(B, dtype=torch.float32, device=dev) if g_first is None
                   else g_first.reshape(B).contiguous().float())
        g_fm = (torch.zeros(B, dtype=torch.float32, device=dev) if g_fm is None
                else g_fm.reshape(B).contiguous().float())
        if u is not None:
            u = u.contiguous().float()
        tr = layer.trace
        tr.mark("between")
        g_bias = None
        gfp = ptr(g_first) if layer.first_order else None
        n_keys = layer.plan.cap * layer.plan.world_size
        with torch.no_grad():
            px, p = layer.px, h.buf
            n = B * layer.n_sel
            # Next to the segmented reduce, on a second stream: the replicated one-row fields' column sums over
            # this rank's samples -> every rank's buffer, and the bias gradient.
            main, aux = torch.cuda.current_stream(), layer.aux_stream(dev, h.half)
            aux.wait_stream(main)
            with torch.cuda.stream(aux):
                if layer.first_order:
                    g_bias = g_first.sum().reshape(1)
                    g_bias.record_stream(main)
                if layer.n_dense:
                    ows = layer._dense_ws[h.half].get(L.dir_shard_dense_workspace_bytes(K), dev)
                    check(L.dir_shard_dense_emit(
                        px.ref(p), ptr(layer.dense_table), layer.row_stride, ptr(ctx.idx), ptr(val),
                        ptr(layer.dense_field_offset), gfp, ptr(g_fm), ptr(S), ptr(u), ptr(layer.onerow_fields), B, F,
                        ptr(ows), ows.numel(), aux.cuda_stream), "dir_shard_dense_emit")
            # per-distinct-row sums on the requester (the sorted list is in the handle's workspace), each
            # stored straight into its owner's buffer over NVLink as soon as its run is summed
            ws = h.ws.get(L.dir_embed_bwd_workspace_bytes(max(n, 1), K), dev)
            check(L.dir_embed_bwd_reduce_emit_to(
                px.ref(p), ptr(val), gfp, ptr(g_fm), ptr(S), ptr(u), ptr(h.uidx), ptr(h.owner_off), B, F, n_keys,
                ptr(layer.sparse_fields) if layer.n_sel < F else None, layer.n_sel, ptr(h.g1_local),
                ptr(ws), ws.numel(), st), "dir_embed_bwd_reduce_emit_to")
            check(L.dir_shard_g1_push(px.ref(p), ptr(h.g1_local), ptr(h.owner_off), n, st), "dir_shard_g1_push")
            main.wait_stream(aux)
            tr.mark("bwd.emit+push")
            if not ctx.defer:
                layer._owner_step([h])
            tr.close_step()
        if h is layer._inline:
            layer._inline_busy = False
        if not ctx.defer:
            layer._in_flight[h.buf] = False
        return None, g_bias, None, None, None, None, None, None


class ShardedEmbeddingFM(torch.nn.Module):
    """`EmbeddingFM` with its tables sharded by row over a process group (one process per GPU).

    Same call as EmbeddingFM: forward(feature_index[B_local, F] int64, feature_value | None) ->
    (first_order, fm_second_order, embeddings) for THIS rank's samples; `.backward()` updates the
    rows this rank owns with the gradients of every rank's samples.  `bias` is an ordinary
    replicated parameter: all-reduce its gradient like any dense parameter.

    `max_batch` sizes the exchange buffers.  `presort` may run at most one batch ahead of `forward`.

    clip_norm: tf.clip_by_norm of every column's gradient before the update, as `EmbeddingFM(clip_norm=...)` applies it
    (DeepCrossNetwork.py:282-289): one factor per column, over the column's per-row sums of the GLOBAL batch (every
    rank's requests of a row merged).  Each owner reduces its rows per column and the ranks exchange the partials
    (a few KB) over peer memory, so the step still replays from one CUDA graph.  SGD / Adagrad / Adam, one
    micro-batch.

    optimizer='adam': [TF] tf.train.AdamOptimizer(lr, optimizer_beta1, optimizer_beta2, optimizer_epsilon) on the
    tables, as `EmbeddingFM(optimizer='adam')` applies it (the reference's DCN optimizer,
    models/DeepCrossNetwork/train.py:104-124).  TF's sparse apply decays the moments of EVERY row, so after the grads
    barrier each owner sweeps its whole shard ([T | m | v] per row, `adam_m` / `adam_v`), adding the requesters'
    merged sums where a row has them; the beta powers live on the device (`beta_power`, the same on every rank).  The
    sweep runs every step, also when this rank's batch had no surviving lookup.  Every field goes through the
    exchange: `replicate_onerow` is ignored under Adam (a replicated one-row field would need an Adam step of its
    own, kept in step with the owner's sweep).  Adam does not train the first-order weights: with first_order=True a
    linear_optimizer must be named.  One micro-batch.
    """

    def __init__(self, field_size: int, embedding_size: int, rows_per_field: Sequence[int],
                 optimizer: str = "adagrad", lr: float = 0.01, initial_accumulator_value: float = 0.1,
                 first_order: bool = True, emit_embeddings: bool = True, check_bounds: bool = False,
                 process_group=None, max_batch: int = 65536, linear_optimizer: Optional[str] = None,
                 linear_lr: Optional[float] = None, l1_regularization_strength: float = 0.0,
                 l2_regularization_strength: float = 0.0, init: str = "trunc_normal", micro_batches: int = 1,
                 replicate_onerow: bool = True, max_entries: Optional[int] = None, optimizer_l1: float = 0.0,
                 optimizer_l2: float = 0.0, clip_norm: Optional[float] = None, device="cuda",
                 optimizer_beta1: float = 0.9, optimizer_beta2: float = 0.999, optimizer_epsilon: float = 1e-8):
        super().__init__()
        if micro_batches not in (1, 2):
            raise ValueError("micro_batches must be 1 or 2")
        self.micro_batches = int(micro_batches)
        adam = str(optimizer).lower() == "adam"     # kept out of _TABLE_OPTIMIZERS, as in layers.py
        if adam:
            if self.micro_batches != 1:
                # the owner's sweep reads one exchange buffer
                raise ValueError("optimizer='adam' needs micro_batches=1")
            if not lr > 0:
                raise ValueError("adam needs lr > 0")
            if not (0 <= optimizer_beta1 < 1 and 0 <= optimizer_beta2 < 1):
                raise ValueError("optimizer_beta1 / optimizer_beta2 must be in [0, 1)")
            if not optimizer_epsilon > 0:
                raise ValueError("optimizer_epsilon must be > 0")
            if first_order and linear_optimizer is None:
                raise ValueError("Adam does not train first-order weights: name a linear_optimizer "
                                 "(%s) or pass first_order=False" % ", ".join(sorted(_LINEAR_OPTIMIZERS)))
            if linear_optimizer is None:
                linear_lr = None
        self.optimizer_beta1, self.optimizer_beta2 = float(optimizer_beta1), float(optimizer_beta2)
        self.optimizer_epsilon = float(optimizer_epsilon)
        if clip_norm is not None and not clip_norm > 0:
            raise ValueError("clip_norm must be > 0 (or None)")
        self.clip_norm = None if clip_norm is None else float(clip_norm)
        if self.clip_norm is not None:
            if field_size > _CLIP_MAX_FIELDS:
                raise ValueError("clip_norm supports at most %d fields (one clip factor per column), got field_size=%d"
                                 % (_CLIP_MAX_FIELDS, field_size))
            if str(optimizer).lower() == "proximal_adagrad":
                raise ValueError("clip_norm is not available with proximal_adagrad")
            if self.micro_batches != 1:
                # the owner merges two buffers in one update: the norm pass would have to merge them as well
                raise ValueError("clip_norm needs micro_batches=1")
        if field_size <= 0:
            raise ValueError("empty columns.")                      # deepFM.py:104-105
        if embedding_size not in _K_OK:
            raise ValueError("embedding_size must be one of %r" % (_K_OK,))
        optimizer = optimizer.lower()
        if optimizer not in _TABLE_OPTIMIZERS and not adam:
            raise ValueError("optimizer must be 'adagrad', 'sgd', 'proximal_adagrad' or 'adam'")
        self.optimizer_l1, self.optimizer_l2 = float(optimizer_l1), float(optimizer_l2)
        if self.optimizer_l1 < 0 or self.optimizer_l2 < 0:
            raise ValueError("optimizer_l1 / optimizer_l2 must be >= 0")
        if init not in ("trunc_normal", "counter", "none"):
            raise ValueError("init must be 'trunc_normal', 'counter' or 'none'")
        self.l1, self.l2 = float(l1_regularization_strength), float(l2_regularization_strength)
        self.linear_optimizer, self.linear_lr, lin_needs_acc, lin_needs_z = resolve_linear_optimizer(
            optimizer, lr, linear_optimizer, linear_lr, self.l1, self.l2)
        rows = [int(r) for r in rows_per_field]
        if len(rows) != field_size:
            raise ValueError("rows_per_field must have field_size entries")
        self.group = process_group
        world = dist.get_world_size(process_group) if dist.is_initialized() else 1
        rank = dist.get_rank(process_group) if dist.is_initialized() else 0
        self.plan = ShardPlan(rows, world, rank)
        self.field_size, self.embedding_size = field_size, embedding_size
        self.optimizer, self.lr = optimizer, float(lr)
        self.first_order, self.emit_embeddings, self.check_bounds = first_order, emit_embeddings, check_bounds
        K = embedding_size
        adagrad = optimizer not in ("sgd", "adam")                  # the rule keeps an accumulator next to the row
        self.row_stride = 3 * K if adam else (2 * K if adagrad else K)
        self.lin_stride = 1
        self.n_rows = max(self.plan.cap, 1)                         # local rows allocated
        self.max_batch = int(max_batch)
        dev = torch.device(device)
        cap = self.n_rows
        self.register_buffer("field_offset", torch.tensor(self.plan.field_offset, dtype=torch.int64, device=dev))
        self.register_buffer("field_rows", torch.tensor(rows, dtype=torch.int64, device=dev))
        self.register_buffer("zero_offset", torch.zeros(field_size, dtype=torch.int64, device=dev))
        self.register_buffer("rows", torch.empty((cap, self.row_stride), dtype=torch.float32, device=dev))
        self.register_buffer("lin_rows", torch.zeros((cap, 1), dtype=torch.float32, device=dev))
        self.register_buffer("lin_acc", torch.zeros((cap, 1), dtype=torch.float32, device=dev) if lin_needs_acc else None)
        self.register_buffer("lin_z", torch.zeros((cap, 1), dtype=torch.float32, device=dev) if lin_needs_z else None)
        self.register_buffer("oob_flag", torch.zeros(1, dtype=torch.int32, device=dev))
        self.register_buffer("err_flag", torch.zeros(1, dtype=torch.int32, device=dev))
        # Adam's (beta1_power, beta2_power), advanced on the device by every owner sweep (every rank, every step)
        self.register_buffer("beta_power", torch.tensor([optimizer_beta1, optimizer_beta2], dtype=torch.float32,
                                                        device=dev) if adam else None)
        self.bias = torch.nn.Parameter(torch.zeros(1, dtype=torch.float32, device=dev))
        self._anchor = torch.nn.Parameter(torch.zeros(1, dtype=torch.float32, device=dev))
        self._n_unique2 = torch.zeros(2, dtype=torch.int64, device=dev)   # per exchange buffer: rows the owner updated
        self._last_parity = 0
        self._side = self._aux = self._micro = None
        self._inline, self._inline_busy = ShardedLookups(), False
        self._in_flight = [False] * (2 * self.micro_batches)
        # gather + send CTAs per SM: NVLink-bound, so with two micro-batches a small grid leaves the SMs to the forward
        # of the other half that runs next to it
        self.gather_ctas_per_sm = 8 if self.micro_batches == 1 else 3
        self.trace, self.trace_pre = StageTrace(), StageTrace()
        self.capturing = False
        if dev.type != "cuda":
            raise ValueError("ShardedEmbeddingFM needs a CUDA device: this layer has no CPU path")
        if world > 1 and dist.get_backend(process_group) != "nccl":
            raise ValueError("the peer-memory exchange needs the nccl backend (one process per GPU)")
        # One-row (numeric) fields are replicated parameters: every sample of every rank hits the same row, so they
        # stay out of the sort and the exchange; their gradients are column sums.
        onerow = [f for f, r in enumerate(rows) if r == 1][:64] if replicate_onerow and not adam else []
        sparse = [f for f in range(field_size) if f not in set(onerow)]
        self.n_dense, self.n_sel = len(onerow), len(sparse)
        self.register_buffer("onerow_fields", torch.tensor(onerow or [0], dtype=torch.int32, device=dev))
        self.register_buffer("sparse_fields", torch.tensor(sparse or [0], dtype=torch.int32, device=dev))
        self._ids_issued = self._fwd_issued = 0       # batches (their half 0) whose id exchange / forward was issued
        self._fwd_event = None
        # lookups of one batch that go through the exchange (bags: entries, `max_entries`)
        self.max_entries = int(max_entries) if max_entries else self.max_batch * max(self.n_sel, 1)
        seg_cap = max(1, min(self.max_entries, cap))   # rows one requester can ask of one owner
        u_cap = max(1, self.max_entries)               # distinct rows a requester can ask for
        if seg_cap >= 1 << 24:
            raise ValueError("max_batch * sparse fields must stay below 2^24 rows per requester and owner")
        if self.micro_batches == 2 and world > 32:
            raise ValueError("two micro-batches need world_size <= 32")
        n_buf = 2 * self.micro_batches          # two parities (consecutive steps alternate) x micro-batches
        L = _lib.lib()
        clip = self.clip_norm is not None
        self.px = PeerExchange(process_group, world, rank, K, self.n_dense, seg_cap, u_cap, dev, n_buf,
                               norm_bytes=world * L.dir_field_sqnorms_bytes(field_size) if clip else 0)
        # clip_norm: the columns' first local rows, the per-arrival squares (one scratch: steps run in stream order)
        # and the combined partials of the last step ([F][kClipSlices][2], the same on every rank)
        self.register_buffer("local_field_offset", torch.tensor(self.plan.local_field_offset(), dtype=torch.int64,
                                                                device=dev) if clip else None)
        self._clip_sq = torch.empty(2 * world * seg_cap, dtype=torch.float64, device=dev) if clip else None
        self.register_buffer("clip_partials", torch.zeros(L.dir_field_sqnorms_bytes(field_size) // 8,
                                                          dtype=torch.float64, device=dev) if clip else None)
        # who asked for which of my rows: one cell per (local row, requester), tagged with the buffer's epoch
        self.slot = [torch.zeros(cap * world, dtype=torch.int32, device=dev) for _ in range(n_buf)]
        self.slot_epoch = [torch.zeros(2, dtype=torch.int32, device=dev) for _ in range(n_buf)]
        with torch.no_grad():
            sd = 1.0 / math.sqrt(K)
            if init == "trunc_normal":
                torch.nn.init.trunc_normal_(self.table, 0.0, sd, -2.0 * sd, 2.0 * sd)
            elif init == "counter":
                self.init_counter(seed=1236, sd=sd)
            if adagrad:
                self.accum.fill_(initial_accumulator_value)
            if adam:
                self.rows[:, K:].zero_()
            if self.lin_acc is not None:
                self.lin_acc.fill_(initial_accumulator_value)
        if self.n_dense:
            self._init_dense_replicas(onerow, dev, initial_accumulator_value)

    @property
    def table(self):
        return self.rows[:, :self.embedding_size]

    @property
    def accum(self):
        return self.rows[:, self.embedding_size:] if self.optimizer not in ("sgd", "adam") else None

    @property
    def adam_m(self):
        K = self.embedding_size
        return self.rows[:, K:2 * K] if self.optimizer == "adam" else None

    @property
    def adam_v(self):
        K = self.embedding_size
        return self.rows[:, 2 * K:3 * K] if self.optimizer == "adam" else None

    @property
    def w1(self):
        return self.lin_rows[:, 0]

    @property
    def w1_accum(self):
        return self.lin_acc[:, 0] if self.lin_acc is not None else None

    @property
    def last_n_unique(self):
        """Local rows the last backward updated on this rank (+ the replicated one-row fields on rank 0)."""
        return self._n_unique2[self._last_parity:self._last_parity + 1]

    @torch.no_grad()
    def init_counter(self, seed=1236, sd=None):
        """Fill this rank's rows on the device from the counter hash of (seed, global row, component): tables too
        large to come from the host (cfg4), reproducible row by row (oracle.deepctr_oracle.counter_rows)."""
        sd = 1.0 / math.sqrt(self.embedding_size) if sd is None else float(sd)
        check(_lib.lib().dir_table_init_counter(ptr(self.table), self.row_stride, self.n_rows, self.embedding_size,
                                                self.plan.world_size, self.plan.rank, self.plan.n_rows, int(seed), sd,
                                                _stream()), "dir_table_init_counter")
        if self.n_dense and "dense_rows" in self._buffers:       # (the constructor builds the replicas afterwards)
            self._sync_dense_replicas()

    # -- replicated one-row fields ----------------------------------------------------------------------------
    @torch.no_grad()
    def _init_dense_replicas(self, onerow, dev, acc0):
        G, rank = self.plan.world_size, self.plan.rank
        n1 = len(onerow)
        dfo = [0] * self.field_size
        for j, f in enumerate(onerow):
            dfo[f] = j
        self.register_buffer("dense_field_offset", torch.tensor(dfo, dtype=torch.int64, device=dev))
        grow = [self.plan.field_offset[f] for f in onerow]                     # the fields' rows in the full table
        self.dense_global_rows = grow
        self.register_buffer("dense_shard_row", torch.tensor([g // G if g % G == rank else -1 for g in grow],
                                                             dtype=torch.int64, device=dev))
        self.register_buffer("dense_rows", torch.zeros((n1, self.row_stride), dtype=torch.float32, device=dev))
        self.register_buffer("dense_lin", torch.zeros(n1, dtype=torch.float32, device=dev))
        self.register_buffer("dense_lin_acc", torch.full((n1,), float(acc0), dtype=torch.float32, device=dev)
                             if self.lin_acc is not None else None)
        self.register_buffer("dense_lin_z", torch.zeros(n1, dtype=torch.float32, device=dev)
                             if self.lin_z is not None else None)
        self._dense_ws = [_Workspace(), _Workspace()]
        self._sync_dense_replicas()

    @torch.no_grad()
    def _sync_dense_replicas(self):
        """Replicas <- the owners' rows of the sharded table (all-reduce of rows that are zero off their owner)."""
        buf = torch.zeros((self.n_dense, self.row_stride + 3), dtype=torch.float32, device=self.rows.device)
        mine = self.dense_shard_row >= 0
        sr = self.dense_shard_row[mine]
        buf[mine, :self.row_stride] = self.rows[sr]
        buf[mine, self.row_stride] = self.lin_rows[sr, 0]
        if self.lin_acc is not None:
            buf[mine, self.row_stride + 1] = self.lin_acc[sr, 0]
        if self.lin_z is not None:
            buf[mine, self.row_stride + 2] = self.lin_z[sr, 0]
        if dist.is_initialized() and self.plan.world_size > 1:
            dist.all_reduce(buf, group=self.group)
        self.dense_rows.copy_(buf[:, :self.row_stride])
        self.dense_lin.copy_(buf[:, self.row_stride])
        if self.dense_lin_acc is not None:
            self.dense_lin_acc.copy_(buf[:, self.row_stride + 1])
        if self.dense_lin_z is not None:
            self.dense_lin_z.copy_(buf[:, self.row_stride + 2])

    @property
    def dense_table(self):
        return self.dense_rows[:, :self.embedding_size]

    @property
    def dense_accum(self):
        return self.dense_rows[:, self.embedding_size:] if self.optimizer != "sgd" else None

    def dense_linear_opt(self):
        """dir_linear_opt for the replicas (same rule as the sharded weights, the replicas' own Ftrl slot)."""
        if self.linear_optimizer is None:
            if self.optimizer == "proximal_adagrad":        # same rule, same strengths as the tables
                return _lib.ctypes.byref(_lib.LinearOpt(_lib.OPT_PROXIMAL_ADAGRAD, self.lr, self.optimizer_l1,
                                                        self.optimizer_l2, None))
            return None
        from .layers import _LINEAR_OPTIMIZERS
        z = self.dense_lin_z.data_ptr() if self.dense_lin_z is not None else None
        return _lib.ctypes.byref(_lib.LinearOpt(_LINEAR_OPTIMIZERS[self.linear_optimizer], self.linear_lr,
                                                self.l1, self.l2, z))

    @torch.no_grad()
    def load_tables(self, table=None, w1=None):
        """Takes the FULL [n_rows, K] table / [n_rows] first-order weights and keeps this rank's rows."""
        for dst, src in ((self.table, table), (self.w1, w1)):
            if src is not None:
                mine = torch.as_tensor(self.plan.shard_of(src), dtype=torch.float32)
                dst[:mine.shape[0]].copy_(mine.to(dst.device))
        if self.n_dense:
            self._sync_dense_replicas()

    def check_errors(self):
        """Raise if a kernel of the device-driven exchange flagged an overflow (one host read)."""
        code = int(self.err_flag.item())
        if code:
            self.err_flag.zero_()
            raise RuntimeError("sharded exchange: " + ("more distinct rows than the exchange buffers hold "
                               "(raise max_batch)" if code == 1 else "a received local row is out of range"))

    @property
    def last_exchange(self):
        """Sizes of the last inline step (host reads: diagnostics only)."""
        h = self._inline if self._last_handle is None else self._last_handle
        if h.owner_off is None:
            return {}
        off = h.owner_off.tolist()
        return {"unique_sent": int(off[-1]), "lookups": int(h.shape[0] * h.shape[1]) if h.shape else 0}

    _last_handle = None

    def _prepare(self, feature_index, feature_value):
        if feature_index.dim() != 2 or feature_index.shape[1] != self.field_size:
            raise ValueError("feature_index must be [B, field_size=%d]" % self.field_size)
        if feature_index.dtype != torch.int64:
            raise ValueError("feature_index must be int64")
        _need_cuda(feature_index, "feature_index")
        idx = feature_index.contiguous()
        val = None
        if feature_value is not None:
            if feature_value.shape != feature_index.shape:
                raise ValueError("feature_value must have feature_index's shape")
            _need_cuda(feature_value, "feature_value")
            val = feature_value.contiguous().float()
        return idx, val

    def side_stream(self, device):
        if self._side is None:
            self._side = torch.cuda.Stream(device=device, priority=-1)
        return self._side

    def aux_stream(self, device, half=0):
        if self._aux is None:
            # high priority: its small kernels must get SM slots while the big segmented reduce is running, not
            # queue behind that kernel's pending CTAs (profiles/r02_timeline_n2.txt); one per micro-batch
            self._aux = [torch.cuda.Stream(device=device, priority=-1) for _ in range(2)]
        return self._aux[half]

    def micro_stream(self, device):
        """The stream the second micro-batch of a step runs on (high priority: its row exchange must not queue
        behind the first half's forward)."""
        if self._micro is None:
            self._micro = torch.cuda.Stream(device=device, priority=-1)
        return self._micro

    @torch.no_grad()
    def _owner_step(self, handles):
        """Grads barrier, then the owner's half: the requesters' sums (of one exchange buffer, or of the two
        micro-batches' buffers) merged in a fixed order, fused row update; then the replicated one-row fields."""
        L = _lib.lib()
        st = _stream()
        tr = self.trace
        px = self.px
        h0 = handles[0]
        hb = handles[1] if len(handles) > 1 else None
        p = h0.buf
        adagrad = self.optimizer != "sgd"
        px.barrier(handles[-1].buf, 0)
        tr.mark("bwd.barrier")
        if self.optimizer == "adam":
            self._owner_step_adam(h0)
            return
        if self.clip_norm is not None:
            self._owner_step_clipped(h0)
            return
        check(L.dir_shard_owner_update(
            px.ref(p), ptr(self.slot[p]), ptr(self.table), ptr(self.accum) if adagrad else None,
            self.row_stride, ptr(self.w1) if self.first_order else None,
            ptr(self.w1_accum) if self.first_order else None, self.lin_stride, self.n_rows,
            ptr(self.slot_epoch[p]), _TABLE_OPTIMIZERS[self.optimizer], self.lr, table_opt_struct(self),
            linear_opt_struct(self),
            px.ref(hb.buf) if hb is not None else None, ptr(self.slot[hb.buf]) if hb is not None else None,
            ptr(self.slot_epoch[hb.buf]) if hb is not None else None,
            self._n_unique2.data_ptr() + 8 * h0.parity, st), "dir_shard_owner_update")
        self._last_parity = h0.parity
        tr.mark("bwd.owner_update")
        if self.n_dense:
            check(L.dir_shard_dense_apply(
                px.ref(p), ptr(self.dense_table), ptr(self.dense_accum) if adagrad else None,
                self.row_stride, ptr(self.dense_lin) if self.first_order else None,
                ptr(self.dense_lin_acc) if self.first_order else None, _TABLE_OPTIMIZERS[self.optimizer],
                self.lr, table_opt_struct(self), self.dense_linear_opt(), ptr(self.table), ptr(self.accum) if adagrad else None,
                self.row_stride, ptr(self.w1) if self.first_order else None,
                ptr(self.w1_accum) if self.first_order else None,
                ptr(self.lin_z) if (self.first_order and self.lin_z is not None) else None,
                self.lin_stride, ptr(self.dense_shard_row), px.ref(hb.buf) if hb is not None else None,
                self._n_unique2.data_ptr() + 8 * h0.parity if self.plan.rank == 0 else None, st),
                "dir_shard_dense_apply")
            tr.mark("bwd.dense_apply")

    def _owner_step_adam(self, h):
        """TF's Adam (one exchange buffer): with clip_norm the norm pass and its barrier first, as in
        `_owner_step_clipped`; then one sweep of this rank's shard that decays every row, adds the merged (clipped) sums
        and advances `beta_power`."""
        L = _lib.lib()
        st = _stream()
        px, p, F = self.px, h.buf, self.field_size
        clip = self.clip_norm is not None
        if clip:
            check(L.dir_shard_owner_sqnorms(px.ref(p), ptr(self.slot[p]), ptr(self.slot_epoch[p]), self.n_rows,
                                            ptr(self.local_field_offset), F, int(self.first_order), ptr(self._clip_sq),
                                            ptr(px.norm_peers[p]), st), "dir_shard_owner_sqnorms")
            self.trace.mark("bwd.sqnorms")
            px.norm_barrier(p)
            self.trace.mark("bwd.norm_barrier")
        opt = _lib.AdamOpt(self.lr, self.optimizer_beta1, self.optimizer_beta2, self.optimizer_epsilon,
                           self.beta_power.data_ptr())
        check(L.dir_shard_owner_apply_adam(
            px.ref(p), ptr(self.slot[p]), ptr(self.slot_epoch[p]), ptr(self.rows), self.row_stride, self.n_rows,
            ptr(self.w1) if self.first_order else None, ptr(self.w1_accum) if self.first_order else None,
            self.lin_stride, linear_opt_struct(self), ptr(self.local_field_offset) if clip else None, F,
            ptr(px.norm_bufs[p]) if clip else None, ptr(self.clip_partials) if clip else None,
            self.clip_norm if clip else 0.0, _lib.ctypes.byref(opt), self._n_unique2.data_ptr() + 8 * h.parity, st),
            "dir_shard_owner_apply_adam")
        self._last_parity = h.parity
        self.trace.mark("bwd.owner_adam")

    def _owner_step_clipped(self, h):
        """tf.clip_by_norm per column (one exchange buffer): the owner's per-column partials of the merged sums to every
        rank, a barrier, then the update scaled by the rank-order combined factors; the one-row replicas clip their
        own sums.  A step's norm buffer is written again only two steps later, by a norm pass that follows that step's
        grads barrier, which every rank reaches only after it has combined this step's partials (same stream)."""
        L = _lib.lib()
        st = _stream()
        px, p, F = self.px, h.buf, self.field_size
        adagrad = self.optimizer != "sgd"
        check(L.dir_shard_owner_sqnorms(px.ref(p), ptr(self.slot[p]), ptr(self.slot_epoch[p]), self.n_rows,
                                        ptr(self.local_field_offset), F, int(self.first_order), ptr(self._clip_sq),
                                        ptr(px.norm_peers[p]), st), "dir_shard_owner_sqnorms")
        self.trace.mark("bwd.sqnorms")
        px.norm_barrier(p)
        self.trace.mark("bwd.norm_barrier")
        check(L.dir_shard_owner_update_clipped(
            px.ref(p), ptr(self.slot[p]), ptr(self.table), ptr(self.accum) if adagrad else None, self.row_stride,
            ptr(self.w1) if self.first_order else None, ptr(self.w1_accum) if self.first_order else None,
            self.lin_stride, self.n_rows, ptr(self.slot_epoch[p]), _TABLE_OPTIMIZERS[self.optimizer], self.lr,
            linear_opt_struct(self), ptr(self.local_field_offset), F, ptr(px.norm_bufs[p]), ptr(self.clip_partials),
            self.clip_norm, self._n_unique2.data_ptr() + 8 * h.parity, st), "dir_shard_owner_update_clipped")
        self._last_parity = h.parity
        self.trace.mark("bwd.owner_update")
        if self.n_dense:
            check(L.dir_shard_dense_apply_clipped(
                px.ref(p), ptr(self.dense_table), ptr(self.dense_accum) if adagrad else None,
                self.row_stride, ptr(self.dense_lin) if self.first_order else None,
                ptr(self.dense_lin_acc) if self.first_order else None, _TABLE_OPTIMIZERS[self.optimizer],
                self.lr, self.dense_linear_opt(), ptr(self.table), ptr(self.accum) if adagrad else None,
                self.row_stride, ptr(self.w1) if self.first_order else None,
                ptr(self.w1_accum) if self.first_order else None,
                ptr(self.lin_z) if (self.first_order and self.lin_z is not None) else None,
                self.lin_stride, ptr(self.dense_shard_row), self.clip_norm,
                self._n_unique2.data_ptr() + 8 * h.parity if self.plan.rank == 0 else None, st),
                "dir_shard_dense_apply_clipped")
            self.trace.mark("bwd.dense_apply")

    def finish_step(self, handle_a, handle_b):
        """After the backward of both micro-batches of a batch (run with `defer_update=True`): the one owner update
        of the batch.  Call it on the stream both backwards have been joined into."""
        if self.micro_batches != 2:
            raise RuntimeError("finish_step needs micro_batches=2")
        if handle_a.parity != handle_b.parity or (handle_a.half, handle_b.half) != (0, 1):
            raise ValueError("finish_step takes the two halves (0, 1) of one batch")
        self._owner_step([handle_a, handle_b])
        self._in_flight[handle_a.buf] = self._in_flight[handle_b.buf] = False
        self.trace.close_step()

    def _note_forward(self, half=0):
        """Bookkeeping after the rows barrier of a step: every rank has finished the previous step, so the id
        exchange of the next batch may now overwrite the other parity's buffers."""
        if half == 0:
            self._fwd_issued += 1
        if not self.capturing:
            self._fwd_event = torch.cuda.Event()
            self._fwd_event.record()

    # ---- id phase ------------------------------------------------------------------------------------------
    @torch.no_grad()
    def id_local(self, h, idx, val):
        """Keys, sort, distinct-row numbering on the current stream: needs the ids only, touches no peer."""
        B, F = idx.shape
        K, G = self.embedding_size, self.plan.world_size
        dev = idx.device
        L = _lib.lib()
        st = _stream()
        n_sel = self.n_sel
        n = B * n_sel
        tr = self.trace_pre
        tr.mark("pre.start")
        if h.shape != (B, F) or h.keys is None or h.keys.device != dev:
            h.keys = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
            h.uidx = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
            h.ulocal = torch.empty(max(n, 1), dtype=torch.int32, device=dev)
            h.g1_local = torch.empty(max(n, 1), dtype=torch.float32, device=dev)
            h.inv = torch.empty((B, F), dtype=torch.int64, device=dev)
            h.owner_off = torch.zeros(G + 1, dtype=torch.int64, device=dev)
            h.shape = (B, F)
        h.n_entries = n
        sel = ptr(self.sparse_fields) if n_sel < F else None
        if self.n_dense:
            # the replicated one-row fields' part of `inv` needs the inputs only: first, off the chain that ends in
            # the id exchange (keys -> sort -> numbering -> push)
            check(L.dir_shard_dense_inv(ptr(idx), ptr(val), ptr(self.onerow_fields), self.n_dense, B, F,
                                        self.px.u_cap, ptr(h.inv),
                                        ptr(self.oob_flag) if self.check_bounds else None, st), "dir_shard_dense_inv")
        ws = h.ws.get(L.dir_embed_bwd_workspace_bytes(max(B * F, 1), K), dev)
        check(L.dir_shard_keys_sort(ptr(idx), ptr(val), ptr(self.field_offset), ptr(self.field_rows),
                                    self.plan.n_rows, B, F, G, sel, n_sel, ptr(h.keys),
                                    ptr(self.oob_flag) if self.check_bounds else None, ptr(ws), ws.numel(), st),
              "dir_shard_keys_sort")
        tr.mark("pre.keys+sort")
        if n > 0:
            skeys, spos = _lib.c_void_p(), _lib.c_void_p()
            check(L.dir_embed_bwd_sorted(ptr(ws), n, _lib.ctypes.byref(skeys), _lib.ctypes.byref(spos)),
                  "dir_embed_bwd_sorted")
        else:
            skeys = spos = None
        ws2 = h.ws2.get(max(L.dir_shard_unique_workspace_bytes(n), 1), dev)
        check(L.dir_shard_unique(skeys, spos, n, self.plan.n_rows, G, sel, n_sel, F, ptr(h.uidx), ptr(h.ulocal),
                                 ptr(h.inv), ptr(h.owner_off), ptr(ws2), ws2.numel(), st), "dir_shard_unique")
        tr.mark("pre.unique")

    @torch.no_grad()
    def id_exchange(self, h):
        """Ships the distinct ids to their owners (current stream): header + ids stored into the owners' buffers,
        a device-side barrier, then the owner marks who asked for which row."""
        L = _lib.lib()
        st = _stream()
        tr = self.trace_pre
        if h.half == 0:
            if self._ids_issued - self._fwd_issued >= 2 and not self.capturing:
                raise RuntimeError("ShardedEmbeddingFM.presort may run at most one batch ahead of forward")
            if h.parity is None or not self.capturing:
                h.parity = self._ids_issued % 2
            self._ids_issued += 1
        elif h.parity is None or not self.capturing:
            h.parity = (self._ids_issued - 1) % 2          # the second half follows its batch's first half
        h.buf = h.parity * self.micro_batches + h.half
        p, px = h.buf, self.px
        if self._fwd_event is not None and not self.capturing:
            torch.cuda.current_stream().wait_event(self._fwd_event)     # every rank is done with parity p
        check(L.dir_shard_ids_push(px.ref(p), ptr(h.ulocal), ptr(h.owner_off), h.n_entries,
                                   ptr(self.err_flag), ptr(self.slot_epoch[p]), st), "dir_shard_ids_push")
        tr.mark("pre.ids_push")
        px.barrier(p, 1)
        tr.mark("pre.barrier")

    @torch.no_grad()
    def presort(self, feature_index, feature_value=None, handle=None, after=None, fork=True, inline=False,
                phase="both", half=0):
        """Everything of a step that depends on the ids only: composite keys, sort, distinct-row numbering
        (phase "local": touches no peer), then the id exchange and the owner's bookkeeping (phase "exchange").
        By default on the side stream, so that issued for batch i+1 right after enqueueing step i it runs underneath
        step i.  `fork=False`: do not order the side stream after the work already queued on the current stream (the
        ids are already on the device, or `after` marks their arrival).  `inline=True`: on the current stream (a
        caller that captures CUDA graphs places the two phases itself).  At most one batch ahead of `forward`."""
        idx, val = self._prepare(feature_index, feature_value)
        if idx.shape[0] > self.max_batch:
            raise ValueError("batch %d exceeds max_batch=%d the exchange buffers were sized for" % (
                idx.shape[0], self.max_batch))
        if phase not in ("both", "local", "exchange"):
            raise ValueError("phase must be 'both', 'local' or 'exchange'")
        h = handle if handle is not None else ShardedLookups()
        if half not in (0, 1) or half >= self.micro_batches:
            raise ValueError("half must be 0 (or 1 with micro_batches=2)")
        h.half = half
        if inline:
            if phase != "exchange":
                self.id_local(h, idx, val)
            if phase != "local":
                self.id_exchange(h)
                self.trace_pre.close_step()
            h.event = None
        else:
            main, side = torch.cuda.current_stream(), self.side_stream(idx.device)
            if fork:        # order after whatever the current stream has queued (it may be producing the ids)
                ev = torch.cuda.Event()
                ev.record(main)
                side.wait_event(ev)
            if after is not None:
                side.wait_event(after)
            with torch.cuda.stream(side):
                self.id_local(h, idx, val)
                self.id_exchange(h)
                h.event = torch.cuda.Event()
                h.event.record(side)
                self.trace_pre.close_step()
        h.src = ShardedLookups.key_of(feature_index, feature_value)
        return h

    def forward(self, feature_index, feature_value=None, presorted=None, defer_update=False):
        """defer_update=True (micro_batches=2): the backward only ships this half's gradient sums; the caller runs
        `finish_step(half0, half1)` after both halves' backward."""
        idx, val = self._prepare(feature_index, feature_value)
        train = self.training and torch.is_grad_enabled()
        if defer_update and (self.micro_batches != 2 or presorted is None):
            raise ValueError("defer_update needs micro_batches=2 and a presorted handle")
        if presorted is None:
            # the layer's own handle serves one forward at a time (a second forward before the first one's backward
            # gets a handle of its own)
            mine = self._inline if not self._inline_busy else ShardedLookups()
            presorted = self.presort(feature_index, feature_value, handle=mine, inline=True)
            if mine is self._inline and train:
                self._inline_busy = True
        elif presorted.src != ShardedLookups.key_of(feature_index, feature_value):
            raise ValueError("presorted handle was made for other feature_index / feature_value tensors")
        if train:
            if self._in_flight[presorted.buf] and not self.capturing:
                raise RuntimeError("ShardedEmbeddingFM: two exchange buffers = at most two batches between forward and "
                                   "backward; run the backward of an earlier batch first")
            self._in_flight[presorted.buf] = True
        self._last_handle = presorted
        first, fm, emb = _ShardedFunction.apply(self._anchor, self.bias, self, idx, val, train, presorted,
                                                bool(defer_update))
        if self.check_bounds:
            if int(self.oob_flag.item()) != 0:
                self.oob_flag.zero_()
                raise IndexError("feature_index out of range for its field")
            self.check_errors()
        return first, fm, emb


# ------------------------------------------------------------------------------------------------------------------
# Multi-hot / weighted bags through the row-sharded tables (SURVEY.md section 8, rows f3 x e)
_COMBINER_CODE = {"sum": 0, "mean": 1, "sqrtn": 2}


class _ShardedBagFunction(torch.autograd.Function):
    """`_ShardedFunction` for bags: the exchange is the same (distinct rows travel once each way), the kernels
    either side of it are the bag ones -- dir_embed_bag_fm_fwd over the received rows, indexed by `inv` per ENTRY,
    and dir_embed_bag_bwd_reduce_emit_to for the per-distinct-row sums."""

    @staticmethod
    def forward(ctx, anchor, bias, layer, off, w, B, train, h):
        F, K = layer.field_size, layer.embedding_size
        dev = off.device
        L = _lib.lib()
        st = _stream()
        nnz = h.n_entries
        px, p = layer.px, h.buf
        emb = torch.empty((B, F * K), dtype=torch.float32, device=dev)
        fm = torch.empty((B, 1), dtype=torch.float32, device=dev)
        first = torch.empty((B, 1), dtype=torch.float32, device=dev)
        S = torch.empty((B, K), dtype=torch.float32, device=dev) if train else None
        if train:
            main, aux = torch.cuda.current_stream(), layer.aux_stream(dev, 0)
            aux.wait_stream(main)
            check(L.dir_shard_slots(px.ref(p), ptr(layer.slot[p]), layer.n_rows, ptr(layer.slot_epoch[p]),
                                    ptr(layer.err_flag), layer._n_unique2.data_ptr() + 8 * h.parity,
                                    aux.cuda_stream), "dir_shard_slots")
        check(L.dir_shard_gather_send(px.ref(p), ptr(layer.table), layer.row_stride,
                                      ptr(layer.w1) if layer.first_order else None, layer.lin_stride,
                                      None, layer.row_stride, None, layer.gather_ctas_per_sm, st),
              "dir_shard_gather_send")
        px.barrier(p, 0)
        layer._note_forward(0)
        rows, lin = px.rows(p), px.w(p) if layer.first_order else None
        slot = x = scratch = None
        if train and nnz > 0:
            scratch = torch.empty(nnz, dtype=torch.int32, device=dev)     # (the kernel's sort keys: not used here)
            slot = torch.empty(nnz, dtype=torch.int32, device=dev)
            x = torch.empty(nnz, dtype=torch.float32, device=dev)
        check(L.dir_embed_bag_fm_fwd(
            ptr(rows), K, ptr(lin), 1, ptr(bias) if layer.first_order else None, ptr(off), ptr(h.inv), ptr(w), nnz,
            ptr(layer.zero_offset), None, rows.shape[0], B, F, K, _COMBINER_CODE[layer.combiner], ptr(emb), ptr(S),
            ptr(first), ptr(fm), ptr(scratch), ptr(slot), ptr(x), None, st), "dir_embed_bag_fm_fwd")
        if not layer.first_order:
            first.zero_()
        ctx.layer, ctx.train, ctx.shape, ctx.h = layer, train, (B, F, K), h
        ctx.set_materialize_grads(False)
        if train:
            ctx.save_for_backward(w, slot, x, S, emb)
        return first, fm, emb

    @staticmethod
    def backward(ctx, g_first, g_fm, u):
        if not ctx.train:
            raise RuntimeError("ShardedEmbeddingBagFM.backward: forward ran without gradient tracking")
        layer, h = ctx.layer, ctx.h
        w, slot, x, S, emb = ctx.saved_tensors
        B, F, K = ctx.shape
        dev = S.device
        L = _lib.lib()
        st = _stream()
        nnz = h.n_entries
        g_first = (torch.zeros(B, dtype=torch.float32, device=dev) if g_first is None
                   else g_first.reshape(B).contiguous().float())
        g_fm = (torch.zeros(B, dtype=torch.float32, device=dev) if g_fm is None
                else g_fm.reshape(B).contiguous().float())
        if u is not None:
            u = u.contiguous().float()
        px, p = layer.px, h.buf
        n_keys = layer.plan.cap * layer.plan.world_size
        with torch.no_grad():
            main, aux = torch.cuda.current_stream(), layer.aux_stream(dev, 0)
            main.wait_stream(aux)                       # the slot marking of the forward
            if nnz > 0 and B > 0:
                ws = h.ws.get(L.dir_embed_bwd_workspace_bytes(nnz, K), dev)
                check(L.dir_embed_bag_bwd_reduce_emit_to(
                    px.ref(p), ptr(w), ptr(slot), ptr(x), nnz, ptr(emb), ptr(g_first) if layer.first_order else None,
                    ptr(g_fm), ptr(S), ptr(u), ptr(h.uidx), ptr(h.owner_off), B, F, n_keys, ptr(h.g1_local),
                    ptr(ws), ws.numel(), st), "dir_embed_bag_bwd_reduce_emit_to")
            check(L.dir_shard_g1_push(px.ref(p), ptr(h.g1_local), ptr(h.owner_off), nnz, st), "dir_shard_g1_push")
            layer._owner_step([h])
        layer._in_flight[h.buf] = False
        g_bias = g_first.sum().reshape(1) if layer.first_order else None
        return None, g_bias, None, None, None, None, None, None


class ShardedEmbeddingBagFM(ShardedEmbeddingFM):
    """`EmbeddingBagFM` with its tables sharded by row over a process group: `forward_bags(bag_offsets[B*F+1],
    bag_index[nnz], bag_weight[nnz] | None)` for THIS rank's samples; `.backward()` updates the rows this rank
    owns with every rank's gradients.  Every field goes through the exchange (a bag of a one-row field still has
    a length and weights).  `max_entries` bounds nnz of one call (it sizes the exchange buffers; default
    max_batch * field_size).  One batch at a time (no `presort`, no micro-batches)."""

    def __init__(self, field_size, embedding_size, rows_per_field, combiner="mean", max_entries=None, **kw):
        if combiner not in _COMBINER_CODE:
            raise ValueError("combiner must be 'sum', 'mean' or 'sqrtn'")
        if kw.get("micro_batches", 1) != 1:
            raise ValueError("ShardedEmbeddingBagFM exchanges a batch in one piece: micro_batches must be 1")
        if str(kw.get("optimizer", "adagrad")).lower() == "adam":
            raise ValueError("ShardedEmbeddingBagFM does not train with adam (nor does EmbeddingBagFM): adam is an "
                             "EmbeddingFM / ShardedEmbeddingFM option")
        super().__init__(field_size, embedding_size, rows_per_field, replicate_onerow=False,
                         max_entries=max_entries, **kw)
        self.combiner = combiner
        self._bag_handle = ShardedLookups()

    @torch.no_grad()
    def _id_local_bags(self, h, off, idx, w, B):
        """Keys per entry, sort, distinct-row numbering: `inv[j]` = entry j's row in the exchanged buffer."""
        F, K, G = self.field_size, self.embedding_size, self.plan.world_size
        dev = off.device
        L = _lib.lib()
        st = _stream()
        nnz = idx.numel()
        if h.keys is None or h.keys.numel() < max(nnz, 1) or h.keys.device != dev:
            for name, dt in (("keys", torch.int32), ("uidx", torch.int32), ("ulocal", torch.int32),
                             ("g1_local", torch.float32), ("inv", torch.int64)):
                setattr(h, name, torch.empty(max(nnz, 1), dtype=dt, device=dev))
            h.owner_off = torch.zeros(G + 1, dtype=torch.int64, device=dev)
        h.shape, h.n_entries = (B, F), nnz
        check(L.dir_shard_bag_keys(ptr(off), ptr(idx), ptr(w), nnz, ptr(self.field_offset), ptr(self.field_rows),
                                   self.plan.n_rows, B, F, G, ptr(h.keys),
                                   ptr(self.oob_flag) if self.check_bounds else None, st), "dir_shard_bag_keys")
        ws = h.ws.get(max(L.dir_embed_bwd_workspace_bytes(max(nnz, 1), K), 1), dev)
        check(L.dir_embed_bwd_sort(ptr(h.keys), nnz, self.plan.cap * G, ptr(ws), ws.numel(), st), "dir_embed_bwd_sort")
        skeys = spos = None
        if nnz > 0:
            skeys, spos = _lib.c_void_p(), _lib.c_void_p()
            check(L.dir_embed_bwd_sorted(ptr(ws), nnz, _lib.ctypes.byref(skeys), _lib.ctypes.byref(spos)),
                  "dir_embed_bwd_sorted")
        ws2 = h.ws2.get(max(L.dir_shard_unique_workspace_bytes(nnz), 1), dev)
        check(L.dir_shard_unique(skeys, spos, nnz, self.plan.n_rows, G, None, 0, F, ptr(h.uidx), ptr(h.ulocal),
                                 ptr(h.inv), ptr(h.owner_off), ptr(ws2), ws2.numel(), st), "dir_shard_unique")

    def forward(self, *a, **kw):
        raise RuntimeError("ShardedEmbeddingBagFM takes bags: call forward_bags(bag_offsets, bag_index, bag_weight)")

    def presort(self, *a, **kw):
        raise RuntimeError("ShardedEmbeddingBagFM runs its id phase inside forward_bags")

    def forward_bags(self, bag_offsets, bag_index, bag_weight=None):
        for t, name in ((bag_offsets, "bag_offsets"), (bag_index, "bag_index"), (bag_weight, "bag_weight")):
            _need_cuda(t, name)
        if bag_offsets.dtype != torch.int64 or bag_index.dtype != torch.int64:
            raise ValueError("bag_offsets and bag_index must be int64")
        if bag_offsets.dim() != 1 or (bag_offsets.numel() - 1) % self.field_size != 0 or bag_offsets.numel() < 1:
            raise ValueError("bag_offsets must be [B * field_size + 1]")
        if bag_weight is not None and bag_weight.shape != bag_index.shape:
            raise ValueError("bag_weight must have bag_index's shape")
        B = (bag_offsets.numel() - 1) // self.field_size
        if B > self.max_batch or bag_index.numel() > self.max_entries:
            raise ValueError("batch %d / %d entries exceed max_batch=%d / max_entries=%d the exchange buffers were "
                             "sized for" % (B, bag_index.numel(), self.max_batch, self.max_entries))
        off, idx = bag_offsets.contiguous(), bag_index.contiguous().reshape(-1)
        w = None if bag_weight is None else bag_weight.contiguous().float().reshape(-1)
        train = self.training and torch.is_grad_enabled()
        h = self._bag_handle
        h.half, h.event = 0, None
        self._id_local_bags(h, off, idx, w, B)
        self.id_exchange(h)
        if train:
            if self._in_flight[h.buf]:
                raise RuntimeError("ShardedEmbeddingBagFM: run the backward of the previous forward_bags first")
            self._in_flight[h.buf] = True
        self._last_handle = h
        first, fm, emb = _ShardedBagFunction.apply(self._anchor, self.bias, self, off, w, B, train, h)
        if self.check_bounds:
            if int(self.oob_flag.item()) != 0:
                self.oob_flag.zero_()
                raise IndexError("bag_index out of range for its field")
            self.check_errors()
        return first, fm, emb
