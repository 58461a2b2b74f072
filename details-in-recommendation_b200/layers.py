"""Host-side mirror of the reference's layer API for the Deep-CTR hot path.

The reference wires this path with four Python calls made while the TF graph is built
(SURVEY.md section 8b):
    myself_input_layer(features, columns)          models/DeepFM/deepFM.py:363-400
    linear_logit_fn(features)                      models/DeepFM/deepFM.py:255-275
    fm_logit_fn(inputs)                            models/DeepFM/deepFM.py:321-335
    _cross_architecture(input_layer, params)       models/DeepCrossNetwork/DeepCrossNetwork.py:350-367
`EmbeddingFM` stands in for the first three, `CrossNetwork` for the fourth, with the knobs the
reference exposes (field_size = len(column_names), embedding_size = fm_embedding_size,
cross_layer_num, cross_w / cross_b shaped [L, d]) and the dense, already-resolved inputs
feature_index / feature_value.  PyTorch here is plumbing (device memory, streams, autograd
hand-off); all arithmetic runs in libdir_b200.so.  There is no CPU path.
"""
import math
import os
from typing import Optional, Sequence, Union

import torch

from . import _lib
from ._lib import check, ptr

_COMBINERS = ("sum", "mean", "sqrtn")
_OPTIMIZERS = {"sgd": _lib.OPT_SGD, "adagrad": _lib.OPT_ADAGRAD}
_TABLE_OPTIMIZERS = dict(_OPTIMIZERS, proximal_adagrad=_lib.OPT_PROXIMAL_ADAGRAD)       # single-GPU layer
_LINEAR_OPTIMIZERS = dict(_TABLE_OPTIMIZERS, ftrl=_lib.OPT_FTRL)
_K_OK = (4, 8, 16, 32, 64)
_CLIP_MAX_FIELDS = 1024       # columns the clip's norm and apply kernels hold factors for (kClipMaxFields, update.cuh)


def table_opt_struct(layer):
    """dir_table_opt: l1 / l2 of a ProximalAdagrad table optimizer (None otherwise)."""
    if getattr(layer, "optimizer", None) != "proximal_adagrad":
        return None
    return _lib.ctypes.byref(_lib.TableOpt(layer.optimizer_l1, layer.optimizer_l2))


def linear_opt_struct(layer):
    """The dir_linear_opt the C ABI takes (None: the linear weights follow the tables' optimizer)."""
    if layer.linear_optimizer is None:
        if getattr(layer, "optimizer", None) == "proximal_adagrad":      # same rule, same strengths as the tables
            return _lib.ctypes.byref(_lib.LinearOpt(_lib.OPT_PROXIMAL_ADAGRAD, layer.lr, layer.optimizer_l1,
                                                    layer.optimizer_l2, None))
        return None
    z = layer.lin_z.data_ptr() if layer.lin_z is not None else None
    return _lib.ctypes.byref(_lib.LinearOpt(_LINEAR_OPTIMIZERS[layer.linear_optimizer], layer.linear_lr,
                                            layer.l1, layer.l2, z))


def resolve_linear_optimizer(optimizer, lr, linear_optimizer, linear_lr, l1, l2):
    """-> (linear_optimizer or None, linear_lr, needs_accumulator, needs_z).  None = same rule and rate as the
    tables (one optimizer over both scopes); the reference's DeepFM default is 'Ftrl' for the linear scope and
    'Adagrad' for the rest (models/DeepFM/deepFM.py:58-61)."""
    if linear_optimizer is not None:
        linear_optimizer = linear_optimizer.lower()
        if linear_optimizer not in _LINEAR_OPTIMIZERS:
            raise ValueError("linear_optimizer must be one of %r" % (sorted(_LINEAR_OPTIMIZERS),))
        if l1 < 0 or l2 < 0:
            raise ValueError("l1 / l2 regularization strengths must be >= 0")
    elif linear_lr is not None:
        linear_optimizer = optimizer
    eff = linear_optimizer or optimizer
    return (linear_optimizer, float(lr if linear_lr is None else linear_lr),
            eff in ("adagrad", "ftrl", "proximal_adagrad"), eff == "ftrl")


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _need_cuda(t, name):
    if t is not None and not t.is_cuda:
        raise ValueError("%s must be a CUDA tensor: this layer has no CPU path" % name)


class _Workspace:
    """Caller-owned scratch, grown on demand (the library never allocates)."""

    def __init__(self):
        self.buf = None

    def get(self, nbytes, device):
        if self.buf is None or self.buf.numel() < nbytes or self.buf.device != device:
            self.buf = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
        return self.buf


class SortedLookups:
    """What `EmbeddingFM.presort` leaves behind for one batch: the (row, position) list of its lookups
    sorted by row, inside a workspace of its own, and the event that marks the sort done.  The sort
    depends on the ids only -- not on the tables -- so it can run as soon as a batch is on the device,
    underneath the previous step (the reference's input pipeline likewise prefetches decoded batches,
    models/DeepCrossNetwork/train.py:148-156)."""

    def __init__(self):
        self.ws = _Workspace()
        self.keys = None
        self.event = None
        self.B = -1
        self.src = None

    @staticmethod
    def key_of(feature_index, feature_value):
        return (feature_index.data_ptr(), None if feature_value is None else feature_value.data_ptr(),
                tuple(feature_index.shape))


class _EmbeddingFMFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, anchor, bias, layer, idx, val, train, presorted):
        B, F = idx.shape
        K = layer.embedding_size
        dev = idx.device
        L = _lib.lib()
        emb = torch.empty((B, F * K), dtype=torch.float32, device=dev) if layer.emit_embeddings else None
        fm = torch.empty((B, 1), dtype=torch.float32, device=dev)
        first = torch.empty((B, 1), dtype=torch.float32, device=dev)
        S = torch.empty((B, K), dtype=torch.float32, device=dev) if train else None
        lin = layer.w1 if layer.first_order else None
        handle = None
        if train and B > 0:
            # The backward needs the lookups sorted by row.  That sort is latency-bound and leaves HBM
            # mostly idle, the gather below is HBM-bound: unless the caller already had the batch
            # sorted ahead of time (`presort`), fork it onto the side stream right here, underneath
            # the forward kernel and whatever the model does before this layer's backward.
            handle = presorted
            if handle is None:
                # the layer's own handle serves one forward at a time: a second forward before the first one's
                # backward (two towers sharing the layer) gets a handle of its own
                mine = layer._inline_sort if not layer._inline_busy else SortedLookups()
                handle = layer.presort(idx, val, handle=mine)
                if mine is layer._inline_sort:
                    layer._inline_busy = True
        check(L.dir_embed_fm_fwd(
            ptr(layer.table), layer.row_stride, ptr(lin), layer.lin_stride,
            ptr(bias) if layer.first_order else None, ptr(idx), ptr(val), ptr(layer.field_offset),
            ptr(layer.field_rows), layer.n_rows, B, F, K, ptr(emb), ptr(S), ptr(first), ptr(fm), None,
            ptr(layer.oob_flag) if layer.check_bounds else None, _stream()), "dir_embed_fm_fwd")
        if not layer.first_order:
            first.zero_()
        ctx.layer, ctx.train, ctx.handle = layer, train, handle
        ctx.shape = (B, F, K)
        ctx.set_materialize_grads(False)
        if train:
            ctx.save_for_backward(idx, val, S)
        if emb is None:
            emb = torch.empty((B, 0), dtype=torch.float32, device=dev)
            ctx.mark_non_differentiable(emb)
        return first, fm, emb

    @staticmethod
    def backward(ctx, g_first, g_fm, u):
        if not ctx.train:
            raise RuntimeError("EmbeddingFM.backward: forward ran without gradient tracking")
        layer = ctx.layer
        idx, val, S = ctx.saved_tensors
        B, F, K = ctx.shape
        dev = S.device
        g_first = (torch.zeros(B, dtype=torch.float32, device=dev) if g_first is None
                   else g_first.reshape(B).contiguous().float())
        g_fm = (torch.zeros(B, dtype=torch.float32, device=dev) if g_fm is None
                else g_fm.reshape(B).contiguous().float())
        if u is not None:
            u = u.contiguous().float()
        # Two independent pieces next to the sorted segmented reduce -- the one-row fields' column sums (rows no
        # sorted lookup touches) and the bias gradient -- run on a second stream underneath it.
        main, aux = torch.cuda.current_stream(), layer.aux_stream(dev)
        aux.wait_stream(main)
        g_bias = None
        with torch.cuda.stream(aux):
            if layer.first_order:
                g_bias = g_first.sum().reshape(1)
                g_bias.record_stream(main)
            if ctx.handle is not None:
                layer.apply_onerow_gradients(idx, val, g_first, g_fm, S, u, B)
        if layer.optimizer == "adam":          # TF's Adam steps every row, also after an empty batch
            if ctx.handle is not None and ctx.handle.event is not None:
                main.wait_event(ctx.handle.event)
            layer.apply_sorted_gradients_adam(ctx.handle, idx, val, g_first, g_fm, S, u, B)
        elif ctx.handle is not None:
            if ctx.handle.event is not None:
                main.wait_event(ctx.handle.event)
            if layer.clip_norm is None:
                layer.apply_sorted_gradients(ctx.handle, idx, val, g_first, g_fm, S, u, B)
            else:
                layer.apply_sorted_gradients_clipped(ctx.handle, idx, val, g_first, g_fm, S, u, B)
        main.wait_stream(aux)
        if ctx.handle is layer._inline_sort:
            layer._inline_busy = False
        return None, g_bias, None, None, None, None, None


class EmbeddingFM(torch.nn.Module):
    """Multi-field embedding lookup + first-order term + FM second-order interaction, with the
    backward's sparse row-wise Adagrad / SGD update fused in (tables are optimizer-owned state,
    not autograd Parameters; `.backward()` through the outputs updates them in place).

    forward(feature_index[B,F] int64, feature_value[B,F] fp32 | None)
        -> (first_order[B,1], fm_second_order[B,1], embeddings[B, F*K])
    which map 1:1 to `linear_logit_fn(features)`, `fm_logit_fn(inputs)` and the `net` fed to
    `dnn_logit_fn` (models/DeepFM/deepFM.py:214, 321-335, 288-291); `embeddings` is also DCN's
    x0 (models/DeepCrossNetwork/DeepCrossNetwork.py:126).

    rows_per_field: N_f per field (one reference embedding variable per column,
    deepFM.py:385-390), stored concatenated; or a single int `feature_size` with global ids.
    clip_norm: tf.clip_by_norm of every column's gradient before the update (DeepCrossNetwork.py:282-289; one
    factor per column variable, over its de-duplicated row sums): a two-pass backward, only when set.
    Storage is B200-first: with Adagrad each row and its accumulator share one 128-byte line
    ([N, 2K] fp32); the first-order weights and their accumulator are separate [N] arrays.
    optimizer='adam': [TF] tf.train.AdamOptimizer(lr, optimizer_beta1, optimizer_beta2, optimizer_epsilon) on the
    tables, the reference's DCN optimizer (models/DeepCrossNetwork/train.py:104-124).  TF's sparse apply decays the
    moments of EVERY row, so each backward sweeps the whole [N, 3K] storage ([T | m | v] per row); the beta powers
    live on the device (`beta_power`).  Every field goes through the sort (no one-row split).  Adam does not train
    the first-order weights: with first_order=True a linear_optimizer must be named.
    """

    def __init__(self, field_size: int, embedding_size: int,
                 rows_per_field: Union[int, Sequence[int]], optimizer: str = "adagrad",
                 lr: float = 0.01, initial_accumulator_value: float = 0.1,
                 combiner: str = "sum", first_order: bool = True, emit_embeddings: bool = True,
                 check_bounds: bool = False,
                 linear_optimizer: Optional[str] = None, linear_lr: Optional[float] = None,
                 l1_regularization_strength: float = 0.0, l2_regularization_strength: float = 0.0,
                 clip_norm: Optional[float] = None, optimizer_l1: float = 0.0, optimizer_l2: float = 0.0,
                 device="cuda", optimizer_beta1: float = 0.9, optimizer_beta2: float = 0.999,
                 optimizer_epsilon: float = 1e-8):
        super().__init__()
        if optimizer_l1 < 0 or optimizer_l2 < 0:
            raise ValueError("optimizer_l1 / optimizer_l2 must be >= 0")
        self.optimizer_l1, self.optimizer_l2 = float(optimizer_l1), float(optimizer_l2)
        if clip_norm is not None and not clip_norm > 0:
            raise ValueError("clip_norm must be > 0 (or None)")
        self.clip_norm = None if clip_norm is None else float(clip_norm)
        if field_size <= 0:
            raise ValueError("empty columns.")                      # deepFM.py:104-105
        if self.clip_norm is not None and field_size > _CLIP_MAX_FIELDS:
            raise ValueError("clip_norm supports at most %d fields (one clip factor per column), got field_size=%d"
                             % (_CLIP_MAX_FIELDS, field_size))
        if embedding_size not in _K_OK:
            raise ValueError("embedding_size must be one of %r" % (_K_OK,))
        optimizer = optimizer.lower()
        adam = optimizer == "adam"              # kept out of _TABLE_OPTIMIZERS: no other entry point learns Adam
        if optimizer not in _TABLE_OPTIMIZERS and not adam:
            raise ValueError("optimizer must be 'adagrad', 'sgd', 'proximal_adagrad' or 'adam'")
        if optimizer == "proximal_adagrad" and self.clip_norm is not None:
            raise ValueError("clip_norm is not available with proximal_adagrad")
        if adam:
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
        self.l1, self.l2 = float(l1_regularization_strength), float(l2_regularization_strength)
        self.linear_optimizer, self.linear_lr, lin_needs_acc, lin_needs_z = resolve_linear_optimizer(
            optimizer, lr, linear_optimizer, linear_lr, self.l1, self.l2)
        if combiner not in _COMBINERS:
            raise ValueError("combiner must be one of %r" % (_COMBINERS,))
        if isinstance(rows_per_field, int):                         # global ids: one shared table
            n_rows, offsets, rows = int(rows_per_field), [0] * field_size, None
        else:
            rows = [int(r) for r in rows_per_field]
            if len(rows) != field_size:
                raise ValueError("rows_per_field must have field_size entries")
            offsets = [0]
            for r in rows[:-1]:
                offsets.append(offsets[-1] + r)
            n_rows = sum(rows)
        if not 0 < n_rows < 2 ** 32 - 1:
            raise ValueError("total rows must be in (0, 2^32-1)")
        self.field_size, self.embedding_size, self.n_rows = field_size, embedding_size, n_rows
        self.shared_table = isinstance(rows_per_field, int)
        self.optimizer, self.lr = optimizer, float(lr)
        self.combiner, self.first_order = combiner, first_order
        self.emit_embeddings, self.check_bounds = emit_embeddings, check_bounds
        K = embedding_size
        adagrad = optimizer not in ("sgd", "adam")       # the rule keeps an accumulator next to the row
        self.row_stride = 3 * K if adam else (2 * K if adagrad else K)
        self.lin_stride = 1
        dev = torch.device(device)
        self.register_buffer("field_offset", torch.tensor(offsets, dtype=torch.int64, device=dev))
        self.register_buffer("field_rows", None if rows is None else
                             torch.tensor(rows, dtype=torch.int64, device=dev))
        self.register_buffer("rows", torch.empty((n_rows, self.row_stride), dtype=torch.float32, device=dev))
        self.register_buffer("lin_rows", torch.zeros((n_rows, 1), dtype=torch.float32, device=dev))
        self.register_buffer("lin_acc", torch.zeros((n_rows, 1), dtype=torch.float32, device=dev)
                             if lin_needs_acc else None)
        self.register_buffer("lin_z", torch.zeros((n_rows, 1), dtype=torch.float32, device=dev)    # Ftrl 'linear' slot
                             if lin_needs_z else None)
        self.register_buffer("oob_flag", torch.zeros(1, dtype=torch.int32, device=dev))
        # Adam's (beta1_power, beta2_power), advanced on the device by every apply
        self.register_buffer("beta_power", torch.tensor([optimizer_beta1, optimizer_beta2], dtype=torch.float32,
                                                        device=dev) if adam else None)
        # Field plan: a field whose table has ONE row (a numeric feature scaled by feature_value) needs no
        # sort -- every sample hits the same row -- so only the other fields' lookups are sorted.
        onerow = [f for f in range(field_size) if rows is not None and rows[f] == 1][:64]
        if os.environ.get("DIR_B200_SORT_ALL_FIELDS", "0") == "1" or adam:
            onerow = []             # Adam: the one apply kernel must see every gradient of the step
        srt = [f for f in range(field_size) if f not in set(onerow)]
        self.n_sorted_fields, self.n_onerow_fields = len(srt), len(onerow)
        self.register_buffer("sorted_fields", torch.tensor(srt or [0], dtype=torch.int32, device=dev))
        self.register_buffer("onerow_fields", torch.tensor(onerow or [0], dtype=torch.int32, device=dev))
        self.bias = torch.nn.Parameter(torch.zeros(1, dtype=torch.float32, device=dev))
        self._anchor = torch.nn.Parameter(torch.zeros(1, dtype=torch.float32, device=dev))
        self._nu_sorted = torch.zeros(1, dtype=torch.int64, device=dev)     # distinct rows the sorted reduce updated
        self._nu_onerow = torch.zeros(1, dtype=torch.int64, device=dev)     # one-row fields whose row was updated
        self._ws, self._onerow_ws = _Workspace(), _Workspace()
        self._side = self._aux = None
        self._clip_bufs = None
        self._inline_sort, self._inline_busy = SortedLookups(), False
        with torch.no_grad():
            # [TF] embedding_column initializer: truncated_normal(0, 1/sqrt(K)); linear weights zero
            torch.nn.init.trunc_normal_(self.table, 0.0, 1.0 / math.sqrt(K), -2.0 / math.sqrt(K), 2.0 / math.sqrt(K))
            if adagrad:
                self.accum.fill_(initial_accumulator_value)
            if adam:
                self.rows[:, K:].zero_()
            if self.w1_accum is not None:
                self.w1_accum.fill_(initial_accumulator_value)     # Adagrad and Ftrl both start at 0.1 in TF

    @property
    def last_n_unique(self):
        """Distinct rows the last backward updated (device int64[1])."""
        return self._nu_sorted + self._nu_onerow

    # views into the interleaved storage
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

    @torch.no_grad()
    def load_tables(self, table=None, w1=None, accum=None, w1_accum=None):
        for dst, src in ((self.table, table), (self.w1, w1), (self.accum, accum), (self.w1_accum, w1_accum)):
            if src is not None:
                dst.copy_(torch.as_tensor(src, dtype=torch.float32).to(dst.device))

    # -- checkpoint / warm start (the reference's `warm_start_from`, models/DeepFM/deepFM.py:71, and the
    #    per-column variables a TF checkpoint of it holds: one `embedding_weights` [N_f, K] and one linear
    #    `weights` [N_f, 1] per column, deepFM.py:385-390, :258-263).  The concatenated, accumulator-interleaved
    #    storage is this layer's business; what crosses the boundary is the reference's shape.
    @torch.no_grad()
    def export_columns(self, column_names=None, with_slots=False):
        """-> {name + '/embedding_weights': [N_f, K], name + '/weights': [N_f, 1]} on the CPU, one pair per field
        (plus '/embedding_weights/Adagrad', '/weights/Adagrad' / '/weights/Ftrl', '/weights/Ftrl_1' with
        `with_slots`; under Adam '/embedding_weights/Adam' (m), '/embedding_weights/Adam_1' (v) and the non-slot
        'beta1_power', 'beta2_power', TF's names).  column_names defaults to field_0 .. field_{F-1}."""
        if self.shared_table:
            raise ValueError("export_columns needs per-field tables (rows_per_field given as a list)")
        names = list(column_names) if column_names is not None else ["field_%d" % f for f in range(self.field_size)]
        if len(names) != self.field_size or len(set(names)) != len(names):
            raise ValueError("column_names must be field_size distinct names")
        off = self.field_offset.tolist()
        rows = self.field_rows.tolist()
        out = {}
        table, w1, acc, acc1 = self.table.cpu(), self.w1.cpu(), self.accum, self.w1_accum
        acc = None if acc is None else acc.cpu()
        acc1 = None if acc1 is None else acc1.cpu()
        z = None if self.lin_z is None else self.lin_z[:, 0].cpu()
        lin_slot = "Ftrl" if (self.linear_optimizer or self.optimizer) == "ftrl" else "Adagrad"
        adam_m = None if self.adam_m is None else self.adam_m.cpu()
        adam_v = None if self.adam_v is None else self.adam_v.cpu()
        if with_slots and adam_m is not None:
            bp = self.beta_power.cpu()
            out["beta1_power"], out["beta2_power"] = bp[0].clone(), bp[1].clone()
        for f, name in enumerate(names):
            sl = slice(off[f], off[f] + rows[f])
            out[name + "/embedding_weights"] = table[sl].clone()
            out[name + "/weights"] = w1[sl].clone().reshape(-1, 1)
            if with_slots:
                if acc is not None:
                    out[name + "/embedding_weights/Adagrad"] = acc[sl].clone()
                if adam_m is not None:
                    out[name + "/embedding_weights/Adam"] = adam_m[sl].clone()
                    out[name + "/embedding_weights/Adam_1"] = adam_v[sl].clone()
                if acc1 is not None:
                    out[name + "/weights/" + lin_slot] = acc1[sl].clone().reshape(-1, 1)
                if z is not None:
                    out[name + "/weights/Ftrl_1"] = z[sl].clone().reshape(-1, 1)
        return out

    @torch.no_grad()
    def import_columns(self, columns, column_names=None, strict=True):
        """Warm start from per-column arrays shaped as `export_columns` writes them (slots optional).
        strict=False skips columns that are absent (WarmStartSettings' vars_to_warm_start subset)."""
        if self.shared_table:
            raise ValueError("import_columns needs per-field tables (rows_per_field given as a list)")
        names = list(column_names) if column_names is not None else ["field_%d" % f for f in range(self.field_size)]
        if len(names) != self.field_size:
            raise ValueError("column_names must have field_size entries")
        off, rows, K = self.field_offset.tolist(), self.field_rows.tolist(), self.embedding_size
        lin_slot = "Ftrl" if (self.linear_optimizer or self.optimizer) == "ftrl" else "Adagrad"
        targets = [("/embedding_weights", self.table, K), ("/weights", self.w1, None),
                   ("/embedding_weights/Adagrad", self.accum, K), ("/weights/" + lin_slot, self.w1_accum, None),
                   ("/weights/Ftrl_1", None if self.lin_z is None else self.lin_z[:, 0], None),
                   ("/embedding_weights/Adam", self.adam_m, K), ("/embedding_weights/Adam_1", self.adam_v, K)]
        for f, name in enumerate(names):
            sl = slice(off[f], off[f] + rows[f])
            for suffix, dst, width in targets:
                src = columns.get(name + suffix)
                if src is None:
                    if strict and suffix in ("/embedding_weights", "/weights"):
                        raise KeyError("missing %s" % (name + suffix))
                    continue
                if dst is None:
                    raise ValueError("%s given but this layer keeps no such slot" % (name + suffix))
                src = torch.as_tensor(src, dtype=torch.float32)
                want = (rows[f], width) if width else (rows[f],)
                src = src.reshape(want) if src.numel() == rows[f] * (width or 1) else src
                if tuple(src.shape) != want:
                    raise ValueError("%s: expected shape %r, got %r" % (name + suffix, want, tuple(src.shape)))
                dst[sl].copy_(src.to(dst.device))
        for i, key in enumerate(("beta1_power", "beta2_power")):
            if key in columns:
                if self.beta_power is None:
                    raise ValueError("%s given but this layer keeps no such slot" % key)
                self.beta_power[i] = float(columns[key])

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
            if self.combiner != "sum":       # one id per field: mean / sqrtn reduce to a pruned gather
                val = (val > 0).float()
        return idx, val

    def forward(self, feature_index, feature_value=None, presorted=None):
        idx, val = self._prepare(feature_index, feature_value)
        train = self.training and torch.is_grad_enabled()
        if presorted is not None and presorted.src != SortedLookups.key_of(feature_index, feature_value):
            raise ValueError("presorted handle was made for other feature_index / feature_value tensors")
        first, fm, emb = _EmbeddingFMFunction.apply(self._anchor, self.bias, self, idx, val, train, presorted)
        if self.check_bounds and int(self.oob_flag.item()) != 0:
            self.oob_flag.zero_()
            raise IndexError("feature_index out of range for its field")   # TF CPU Gather raises
        return first, fm, emb

    @torch.no_grad()
    def presort(self, feature_index, feature_value=None, handle=None, after=None, record_event=True):
        """Sort the lookups of a batch by row on the side stream, ahead of `forward`.

        The sort needs only the ids, so a training loop can issue it for batch i+1 as soon as that batch
        is on the device and let it run underneath step i; pass the returned handle to
        `forward(..., presorted=handle)` with the SAME tensors.  `after`: an event the side stream must
        wait for first (e.g. the H2D copy of the batch).  `record_event=False` leaves the ordering to the
        caller (needed when the presort and its consumer are captured in different CUDA graphs).
        """
        idx, val = self._prepare(feature_index, feature_value)
        B, F, K = idx.shape[0], self.field_size, self.embedding_size
        dev = idx.device
        L = _lib.lib()
        h = handle if handle is not None else SortedLookups()
        ws = h.ws.get(L.dir_embed_bwd_workspace_bytes(max(B * F, 1), K), dev)
        n_sel = self.n_sorted_fields
        main, side = torch.cuda.current_stream(), self.side_stream(dev)
        if n_sel > 0 and B > 0:
            fork = torch.cuda.Event()
            fork.record(main)
            side.wait_event(fork)
            if after is not None:
                side.wait_event(after)
            if h.keys is None or h.keys.numel() != B * n_sel or h.keys.device != dev:
                h.keys = torch.empty((B * n_sel,), dtype=torch.int32, device=dev)
                h.keys.record_stream(side)
            check(L.dir_shard_keys_sort(ptr(idx), ptr(val), ptr(self.field_offset), ptr(self.field_rows),
                                        self.n_rows, B, F, 1, ptr(self.sorted_fields), n_sel, ptr(h.keys), None,
                                        ptr(ws), ws.numel(), side.cuda_stream), "dir_shard_keys_sort")
        h.event = None
        if record_event:
            h.event = torch.cuda.Event()
            h.event.record(side if (n_sel > 0 and B > 0) else main)
        h.B = B
        h.src = SortedLookups.key_of(feature_index, feature_value)
        return h

    def side_stream(self, device):
        if self._side is None:
            # high priority: the sort's few, latency-bound CTAs must not queue behind the thousands
            # of CTAs of the forward gather it is meant to run underneath
            self._side = torch.cuda.Stream(device=device, priority=-1)
        return self._side

    def aux_stream(self, device):
        if self._aux is None:
            # high priority: its small kernels must get SM slots while the big segmented reduce is running, not
            # queue behind that kernel's pending CTAs
            self._aux = torch.cuda.Stream(device=device, priority=-1)
        return self._aux

    @torch.no_grad()
    def apply_sorted_gradients(self, handle, feature_index, feature_value, g_first, g_fm, S, u, B):
        """segmented reduce -> fused row update (dir_embed_bwd_reduce_update) on the (row, position)
        list `presort` left sorted in the handle's workspace (the one-row fields: apply_onerow_gradients)."""
        F, K = self.field_size, self.embedding_size
        L = _lib.lib()
        ws = handle.ws.get(L.dir_embed_bwd_workspace_bytes(max(B * F, 1), K), S.device)
        adagrad = self.optimizer != "sgd"
        check(L.dir_embed_bwd_reduce_update(
            ptr(self.table), ptr(self.accum) if adagrad else None, self.row_stride,
            ptr(self.w1) if self.first_order else None,
            ptr(self.w1_accum) if self.first_order else None, self.lin_stride,
            ptr(feature_index), ptr(feature_value), ptr(self.field_offset), ptr(g_first), ptr(g_fm), ptr(S),
            ptr(u), B, F, K, self.n_rows, ptr(self.sorted_fields), self.n_sorted_fields,
            None, 0, _TABLE_OPTIMIZERS[self.optimizer], self.lr, table_opt_struct(self), linear_opt_struct(self),
            ptr(ws), ws.numel(),
            ptr(self._nu_sorted), _stream()), "dir_embed_bwd_reduce_update")

    @torch.no_grad()
    def apply_onerow_gradients(self, feature_index, feature_value, g_first, g_fm, S, u, B):
        """One-row (numeric) fields: every sample hits the same row, so the row's gradient is a column sum over the
        batch (fixed order, fp64-carried) -- no sort; independent of the sorted part (disjoint rows)."""
        F, K = self.field_size, self.embedding_size
        L = _lib.lib()
        if self.n_onerow_fields == 0:
            self._nu_onerow.zero_()
            return
        ows = self._onerow_ws.get(L.dir_shard_dense_workspace_bytes(K), S.device)
        adagrad = self.optimizer != "sgd"
        check(L.dir_embed_bwd_onerow_update(
            ptr(self.table), ptr(self.accum) if adagrad else None, self.row_stride,
            ptr(self.w1) if self.first_order else None,
            ptr(self.w1_accum) if self.first_order else None, self.lin_stride,
            ptr(feature_index), ptr(feature_value), ptr(self.field_offset), ptr(g_first), ptr(g_fm), ptr(S),
            ptr(u), B, F, K, ptr(self.onerow_fields), self.n_onerow_fields, _TABLE_OPTIMIZERS[self.optimizer], self.lr,
            table_opt_struct(self), linear_opt_struct(self), self.clip_norm or 0.0, ptr(ows), ows.numel(), ptr(self._nu_onerow), _stream()),
            "dir_embed_bwd_onerow_update")

    def _emit_unique_sums(self, handle, feature_value, g_first, g_fm, S, u, B):
        """First pass of the two-pass backward: number the distinct rows of the sorted list (dir_shard_unique), write
        their gradient sums gu[u] = (G[K], g1) (dir_embed_bwd_reduce_emit_local) and, with a clip norm, the
        per-column sums of squares (dir_field_sqnorms, fixed order).  -> (the buffers, device pointer of the
        distinct-row count, n lookups); n = 0: nothing was launched."""
        if self.clip_norm is not None and self.shared_table:
            raise ValueError("clip_norm needs per-field tables (one variable per column, as in the reference)")
        F, K = self.field_size, self.embedding_size
        n_sel = self.n_sorted_fields
        n = B * n_sel if handle is not None else 0
        if n == 0:
            return None, None, 0
        L = _lib.lib()
        dev = S.device
        ws = handle.ws.get(L.dir_embed_bwd_workspace_bytes(max(B * F, 1), K), dev)
        c = self._clip_bufs
        if c is None or c["n"] < n or c["uidx"].device != dev:
            c = self._clip_bufs = dict(
                n=n, uidx=torch.empty(n, dtype=torch.int32, device=dev), urows=torch.empty(n, dtype=torch.int32, device=dev),
                count=torch.zeros(2, dtype=torch.int64, device=dev), gu=torch.empty((n, K + 4), dtype=torch.float32, device=dev),
                ws2=torch.empty(max(int(L.dir_shard_unique_workspace_bytes(n)), 1), dtype=torch.uint8, device=dev),
                part=torch.empty(int(L.dir_field_sqnorms_bytes(F)), dtype=torch.uint8, device=dev))
        st = _stream()
        skeys, spos = _lib.c_void_p(), _lib.c_void_p()
        check(L.dir_embed_bwd_sorted(ptr(ws), n, _lib.ctypes.byref(skeys), _lib.ctypes.byref(spos)), "dir_embed_bwd_sorted")
        check(L.dir_shard_unique(skeys, spos, n, self.n_rows, 1, None, 0, F, ptr(c["uidx"]), ptr(c["urows"]), None,
                                 ptr(c["count"]), ptr(c["ws2"]), c["ws2"].numel(), st), "dir_shard_unique")
        check(L.dir_embed_bwd_reduce_emit_local(
            ptr(self.table), self.row_stride, ptr(feature_value), ptr(g_first) if self.first_order else None, ptr(g_fm),
            ptr(S), ptr(u), ptr(c["uidx"]), B, F, K, self.n_rows, ptr(self.sorted_fields), n_sel, ptr(c["gu"]), K + 4,
            ptr(ws), ws.numel(), st), "dir_embed_bwd_reduce_emit_local")
        n_dev = c["count"].data_ptr() + 8                      # count[1] = distinct rows (dir_shard_unique, G = 1)
        if self.clip_norm is not None:
            check(L.dir_field_sqnorms(ptr(c["gu"]), K + 4, ptr(c["urows"]), n_dev, ptr(self.field_offset), F, K,
                                      self.n_rows, ptr(c["part"]), st), "dir_field_sqnorms")
        return c, n_dev, n

    @torch.no_grad()
    def apply_sorted_gradients_clipped(self, handle, feature_index, feature_value, g_first, g_fm, S, u, B):
        """The backward with tf.clip_by_norm on every column's gradient (DeepCrossNetwork.py:282-289): a column's
        factor is known only once all of its row sums are, so the sums go to a buffer first (dir_embed_bwd_reduce_emit_local),
        the per-column norms are reduced in a fixed order (dir_field_sqnorms) and a second pass scales and applies
        (dir_rows_apply_clipped)."""
        c, n_dev, n = self._emit_unique_sums(handle, feature_value, g_first, g_fm, S, u, B)
        if n == 0:
            self._nu_sorted.zero_()
            return
        F, K = self.field_size, self.embedding_size
        adagrad = self.optimizer == "adagrad"
        check(_lib.lib().dir_rows_apply_clipped(
            ptr(self.table), ptr(self.accum) if adagrad else None, self.row_stride,
            ptr(self.w1) if self.first_order else None, ptr(self.w1_accum) if self.first_order else None,
            self.lin_stride, ptr(c["gu"]), K + 4, ptr(c["urows"]), n_dev, n, ptr(self.field_offset), F, K,
            ptr(c["part"]), self.clip_norm, _OPTIMIZERS[self.optimizer], self.lr, linear_opt_struct(self),
            ptr(self._nu_sorted), _stream()), "dir_rows_apply_clipped")

    @torch.no_grad()
    def apply_sorted_gradients_adam(self, handle, feature_index, feature_value, g_first, g_fm, S, u, B):
        """Adam (optimizer='adam'): the first pass of the clipped backward (`_emit_unique_sums`), then one sweep of
        the whole table (dir_rows_apply_adam) that decays every row's moments, adds the batch's de-duplicated
        (and, with clip_norm, clipped) gradients, moves every row and steps the first-order weights of the touched
        rows with the linear optimizer.  The beta powers advance on the device after the sweep."""
        c, n_dev, n = self._emit_unique_sums(handle, feature_value, g_first, g_fm, S, u, B)
        F, K = self.field_size, self.embedding_size
        opt = _lib.AdamOpt(self.lr, self.optimizer_beta1, self.optimizer_beta2, self.optimizer_epsilon,
                           self.beta_power.data_ptr())
        first = self.first_order and n > 0
        check(_lib.lib().dir_rows_apply_adam(
            ptr(self.rows), self.row_stride, self.n_rows, K, ptr(self.w1) if first else None,
            ptr(self.w1_accum) if first else None, self.lin_stride, linear_opt_struct(self) if first else None,
            ptr(c["gu"]) if n else None, K + 4, ptr(c["urows"]) if n else None, n_dev, n, ptr(self.field_offset), F,
            ptr(c["part"]) if (n and self.clip_norm is not None) else None, self.clip_norm or 0.0,
            _lib.ctypes.byref(opt), ptr(self._nu_sorted), _stream()), "dir_rows_apply_adam")


class _CrossFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x0, cross_w, cross_b, layer):
        B, d = x0.shape
        L = cross_w.shape[0]
        xL = torch.empty_like(x0)
        train = layer.training and (x0.requires_grad or cross_w.requires_grad or cross_b.requires_grad)
        s = torch.empty((B, L), dtype=torch.float32, device=x0.device) if train else None
        check(_lib.lib().dir_cross_fwd(ptr(x0), ptr(cross_w), ptr(cross_b), B, d, L, ptr(xL), ptr(s),
                                       _stream()), "dir_cross_fwd")
        ctx.layer = layer
        ctx.save_for_backward(x0, cross_w, cross_b, s)
        return xL

    @staticmethod
    def backward(ctx, dy):
        x0, cross_w, cross_b, s = ctx.saved_tensors
        B, d = x0.shape
        L = cross_w.shape[0]
        dy = dy.contiguous().float()
        dx0 = torch.empty_like(x0)
        dw = torch.empty_like(cross_w)
        db = torch.empty_like(cross_b)
        lib = _lib.lib()
        ws = ctx.layer._ws.get(lib.dir_cross_bwd_workspace_bytes(B, d, L), x0.device)
        check(lib.dir_cross_bwd(ptr(x0), ptr(cross_w), ptr(cross_b), ptr(dy), ptr(s), B, d, L,
                                ptr(dx0), ptr(dw), ptr(db), ptr(ws), ws.numel(), _stream()),
              "dir_cross_bwd")
        return dx0, dw, db, None


class CrossNetwork(torch.nn.Module):
    """DCN cross stack: x_{l+1} = x0 * (x_l . w_l) + b_l + x_l for l < cross_layer_num.

    Mirrors `_cross_architecture` / `_cross_variable_creat`
    (models/DeepCrossNetwork/DeepCrossNetwork.py:322-367): parameters `cross_w`, `cross_b`
    of shape [cross_layer_num, input_dim], both truncated_normal(0, 0.1) (the bias is not
    zero-initialised in the reference).  forward(x0[B,d]) -> x_L[B,d].
    """

    def __init__(self, input_dim: int, cross_layer_num: int = 2, device="cuda"):
        super().__init__()
        if not 0 < input_dim <= 1024:
            raise ValueError("input_dim must be in (0, 1024]")
        if not 0 < cross_layer_num <= 32:
            raise ValueError("cross_layer_num must be in (0, 32]")
        self.input_dim, self.cross_layer_num = input_dim, cross_layer_num
        w = torch.empty((cross_layer_num, input_dim), dtype=torch.float32, device=device)
        b = torch.empty((cross_layer_num, input_dim), dtype=torch.float32, device=device)
        torch.nn.init.trunc_normal_(w, 0.0, 0.1, -0.2, 0.2)
        torch.nn.init.trunc_normal_(b, 0.0, 0.1, -0.2, 0.2)
        self.cross_w = torch.nn.Parameter(w)
        self.cross_b = torch.nn.Parameter(b)
        self._ws = _Workspace()

    def forward(self, x0):
        _need_cuda(x0, "x0")
        if x0.dim() != 2 or x0.shape[1] != self.input_dim:
            raise ValueError("x0 must be [B, input_dim=%d]" % self.input_dim)
        return _CrossFunction.apply(x0.contiguous().float(), self.cross_w, self.cross_b, self)


class _InputLayerFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, emb, numeric, ind, layer):
        B = layer._batch(numeric, ind, emb)
        dev = layer.col_kind.device
        x0 = torch.empty((B, layer.output_dim), dtype=torch.float32, device=dev)
        check(_lib.lib().dir_input_layer_fwd(
            ptr(numeric), layer.n_numeric, ptr(ind), layer.n_indicator, ptr(emb), layer.emb_width,
            ptr(layer.col_kind), ptr(layer.col_src), ptr(layer.col_arg), B, layer.output_dim, ptr(x0), _stream()),
            "dir_input_layer_fwd")
        ctx.layer, ctx.B = layer, B
        return x0

    @staticmethod
    def backward(ctx, dx0):
        layer, B = ctx.layer, ctx.B
        if layer.emb_width == 0:
            return None, None, None, None
        dx0 = dx0.contiguous().float()
        u = torch.empty((B, layer.emb_width), dtype=torch.float32, device=dx0.device)
        check(_lib.lib().dir_input_layer_bwd(ptr(dx0), ptr(layer.emb_col), B, layer.output_dim, layer.emb_width,
                                             ptr(u), _stream()), "dir_input_layer_bwd")
        return u, None, None, None


class InputLayer(torch.nn.Module):
    """`tf.feature_column.input_layer(features, feature_columns)` in the reference's own DCN convention
    (models/DeepCrossNetwork/DeepCrossNetwork.py:126 over the columns of train.py:88-100): all dense columns
    side by side, **sorted by column name** -- numeric columns pass through 1-wide, indicator columns are one-hot
    vectors of their id, embedding columns are the K-wide rows of `EmbeddingFM` (census: d = 51).

    columns: [(name, kind, size)], kind 'numeric' (size 1), 'indicator' (size = vocabulary size) or
    'embedding' (size = K).  Inputs follow the LISTING order of each kind:
        forward(numeric[B, n_numeric] fp32 | None, indicator_ids[B, n_indicator] int64 | None,
                embeddings[B, sum K] | None)  ->  x0[B, output_dim]
    The backward returns the embedding columns' slice of dL/dx0 -- the upstream gradient the fused embedding
    backward takes; numeric and indicator columns carry no parameters.
    """

    def __init__(self, columns, device="cuda"):
        super().__init__()
        if not columns:
            raise ValueError("empty columns.")
        names = [c[0] for c in columns]
        if len(set(names)) != len(names):
            raise ValueError("column names must be unique")
        n_num = n_ind = emb_w = 0
        src = {}
        for name, kind, size in columns:
            size = int(size)
            if kind == "numeric":
                if size != 1:
                    raise ValueError("numeric column %r must have size 1" % name)
                src[name] = (0, n_num, size)
                n_num += 1
            elif kind == "indicator":
                if size <= 0:
                    raise ValueError("indicator column %r needs a positive vocabulary size" % name)
                src[name] = (1, n_ind, size)
                n_ind += 1
            elif kind == "embedding":
                if size <= 0:
                    raise ValueError("embedding column %r needs a positive dimension" % name)
                src[name] = (2, emb_w, size)
                emb_w += size
            else:
                raise ValueError("column kind must be 'numeric', 'indicator' or 'embedding', got %r" % (kind,))
        kind_l, src_l, arg_l, emb_col = [], [], [], [-1] * emb_w
        for name in sorted(names):                      # [TF] input_layer orders columns by name
            k, s, size = src[name]
            for t in range(size):
                if k == 2:
                    emb_col[s + t] = len(kind_l)
                kind_l.append(k)
                src_l.append(s + t if k == 2 else s)
                arg_l.append(t if k == 1 else 0)
        self.n_numeric, self.n_indicator, self.emb_width, self.output_dim = n_num, n_ind, emb_w, len(kind_l)
        dev = torch.device(device)
        self.register_buffer("col_kind", torch.tensor(kind_l, dtype=torch.int32, device=dev))
        self.register_buffer("col_src", torch.tensor(src_l, dtype=torch.int32, device=dev))
        self.register_buffer("col_arg", torch.tensor(arg_l, dtype=torch.int32, device=dev))
        self.register_buffer("emb_col", torch.tensor(emb_col or [-1], dtype=torch.int32, device=dev))

    def _batch(self, numeric, ind, emb):
        sizes = {t.shape[0] for t in (numeric, ind, emb) if t is not None}
        if len(sizes) != 1:
            raise ValueError("inputs must share one batch size")
        return sizes.pop()

    def forward(self, numeric=None, indicator_ids=None, embeddings=None):
        for t, n, w, dt in ((numeric, "numeric", self.n_numeric, torch.float32),
                            (indicator_ids, "indicator_ids", self.n_indicator, torch.int64),
                            (embeddings, "embeddings", self.emb_width, torch.float32)):
            if w == 0:
                continue
            if t is None or t.dim() != 2 or t.shape[1] != w or t.dtype != dt:
                raise ValueError("%s must be a [B, %d] %s tensor" % (n, w, dt))
            _need_cuda(t, n)
        numeric = numeric.contiguous() if self.n_numeric else None
        indicator_ids = indicator_ids.contiguous() if self.n_indicator else None
        embeddings = embeddings.contiguous() if self.emb_width else None
        return _InputLayerFunction.apply(embeddings, numeric, indicator_ids, self)
