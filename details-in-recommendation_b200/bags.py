"""Multi-hot / weighted bags through the same tables (SURVEY.md section 8f rank 3).

`myself_input_layer` exists so that DeepFM can take multi-hot columns -- a user's item history, a set
of tags -- each embedded with a combiner (models/DeepFM/deepFM.py:53, 77, 363-400; the weighted column of
dataset/SequenceTensorFlowDataset/test4.py:50-55, 113-116).  `EmbeddingBagFM` is `EmbeddingFM` with a
variable-length list of (id, weight) per (sample, field) in CSR form:

    forward(bag_offsets[B*F+1] int64, bag_index[nnz] int64, bag_weight[nnz] fp32 | None)
        -> (first_order[B,1], fm_second_order[B,1], embeddings[B, F*K])

Storage, optimizers (Adagrad / SGD for the tables, dir_linear_opt for the linear scope) and the in-place
fused update during `.backward()` are the parent's; the arithmetic runs in libdir_b200.so
(dir_embed_bag_fm_fwd, dir_embed_bwd_sort, dir_embed_bag_bwd_reduce_update).  No CPU path.
"""
import torch

from . import _lib
from ._lib import check, ptr
from .layers import _OPTIMIZERS, EmbeddingFM, _need_cuda, _stream, linear_opt_struct

_COMBINER_CODE = {"sum": 0, "mean": 1, "sqrtn": 2}


class _EmbeddingBagFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, anchor, bias, layer, off, idx, w, B, train):
        F, K = layer.field_size, layer.embedding_size
        dev = off.device
        nnz = idx.numel()
        L = _lib.lib()
        emb = torch.empty((B, F * K), dtype=torch.float32, device=dev)
        fm = torch.empty((B, 1), dtype=torch.float32, device=dev)
        first = torch.empty((B, 1), dtype=torch.float32, device=dev)
        S = torch.empty((B, K), dtype=torch.float32, device=dev) if train else None
        keys = slot = x = None
        if train and nnz > 0:
            keys = torch.empty(nnz, dtype=torch.int32, device=dev)
            slot = torch.empty(nnz, dtype=torch.int32, device=dev)
            x = torch.empty(nnz, dtype=torch.float32, device=dev)
        lin = layer.w1 if layer.first_order else None
        check(L.dir_embed_bag_fm_fwd(
            ptr(layer.table), layer.row_stride, ptr(lin), layer.lin_stride,
            ptr(bias) if layer.first_order else None, ptr(off), ptr(idx), ptr(w), nnz, ptr(layer.field_offset),
            ptr(layer.field_rows), layer.n_rows, B, F, K, _COMBINER_CODE[layer.combiner], ptr(emb), ptr(S),
            ptr(first), ptr(fm), ptr(keys), ptr(slot), ptr(x),
            ptr(layer.oob_flag) if layer.check_bounds else None, _stream()), "dir_embed_bag_fm_fwd")
        if not layer.first_order:
            first.zero_()
        ws = None
        if keys is not None:        # the backward needs the entries sorted by row; the list lives in this call's
            # own workspace, so two forwards may precede their backwards
            ws = torch.empty(int(L.dir_embed_bwd_workspace_bytes(nnz, K)), dtype=torch.uint8, device=dev)
            check(L.dir_embed_bwd_sort(ptr(keys), nnz, layer.n_rows, ptr(ws), ws.numel(), _stream()),
                  "dir_embed_bwd_sort")
        ctx.layer, ctx.train, ctx.shape, ctx.nnz, ctx.ws = layer, train, (B, F, K), nnz, ws
        ctx.set_materialize_grads(False)
        if train:
            ctx.save_for_backward(w, slot, x, S, emb)
        return first, fm, emb

    @staticmethod
    def backward(ctx, g_first, g_fm, u):
        if not ctx.train:
            raise RuntimeError("EmbeddingBagFM.backward: forward ran without gradient tracking")
        layer = ctx.layer
        w, slot, x, S, emb = ctx.saved_tensors
        B, F, K = ctx.shape
        dev = S.device
        L = _lib.lib()
        g_first = (torch.zeros(B, dtype=torch.float32, device=dev) if g_first is None
                   else g_first.reshape(B).contiguous().float())
        g_fm = (torch.zeros(B, dtype=torch.float32, device=dev) if g_fm is None
                else g_fm.reshape(B).contiguous().float())
        if u is not None:
            u = u.contiguous().float()
        if ctx.nnz > 0 and B > 0:
            adagrad = layer.optimizer == "adagrad"
            ws = ctx.ws
            with torch.no_grad():
                check(L.dir_embed_bag_bwd_reduce_update(
                    ptr(layer.table), ptr(layer.accum) if adagrad else None, layer.row_stride,
                    ptr(layer.w1) if layer.first_order else None,
                    ptr(layer.w1_accum) if layer.first_order else None, layer.lin_stride,
                    ptr(w), ptr(slot), ptr(x), ctx.nnz, ptr(emb), ptr(g_first), ptr(g_fm), ptr(S), ptr(u),
                    B, F, K, layer.n_rows, _OPTIMIZERS[layer.optimizer], layer.lr, linear_opt_struct(layer),
                    ptr(ws), ws.numel(), ptr(layer._nu_sorted), _stream()), "dir_embed_bag_bwd_reduce_update")
        else:
            layer._nu_sorted.zero_()
        layer._nu_onerow.zero_()
        g_bias = g_first.sum().reshape(1) if layer.first_order else None
        return None, g_bias, None, None, None, None, None, None


class EmbeddingBagFM(EmbeddingFM):
    """`EmbeddingFM` over multi-hot / weighted bags.  combiner: 'mean' (tf.feature_column.embedding_column's
    default), 'sum' or 'sqrtn' for the embedded part; the first-order term always sums
    (linear_sparse_combiner='sum', deepFM.py:59).  One-id-per-field inputs still go through the parent's
    `forward`; `forward_bags` takes the CSR form."""

    def __init__(self, field_size, embedding_size, rows_per_field, combiner="mean", **kw):
        if str(kw.get("optimizer", "adagrad")).lower() in ("proximal_adagrad", "adam"):
            raise ValueError("EmbeddingBagFM trains with 'adagrad' or 'sgd'; proximal_adagrad and adam are EmbeddingFM "
                             "options")
        if kw.get("clip_norm") is not None:
            raise ValueError("EmbeddingBagFM applies its gradients unclipped: clip_norm is an EmbeddingFM option")
        super().__init__(field_size, embedding_size, rows_per_field, combiner=combiner, **kw)

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
        off, idx = bag_offsets.contiguous(), bag_index.contiguous().reshape(-1)
        w = None if bag_weight is None else bag_weight.contiguous().float().reshape(-1)
        train = self.training and torch.is_grad_enabled()
        first, fm, emb = _EmbeddingBagFunction.apply(self._anchor, self.bias, self, off, idx, w, B, train)
        if self.check_bounds and int(self.oob_flag.item()) != 0:
            self.oob_flag.zero_()
            raise IndexError("bag_index out of range for its field")
        return first, fm, emb
