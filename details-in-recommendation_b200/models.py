"""The reference's two Deep-CTR graphs assembled around the B200 hot path (SURVEY.md section 8f, rank 1).

  DeepFM  models/DeepFM/deepFM.py:143-252   logits = linear_logits + fm_logit + dnn_logit
  DCN     models/DeepCrossNetwork/DeepCrossNetwork.py:124-141   dense(concat(cross(x0), deep(x0)))

The lookup, first-order, FM and cross arithmetic -- forward, backward and the sparse row update -- run in
libdir_b200.so (`EmbeddingFM` / `ShardedEmbeddingFM`, `CrossNetwork`).  The DNN tower is what consumes the
`embeddings[B, F*K]` output and produces the upstream gradient `u` the fused backward takes; it is a plain
stack of `torch.nn.Linear` (cuBLAS, fp32, TF32 off) because dense GEMMs are not this repository's subject.
Estimator orchestration, input_fn, metrics and checkpoints stay out of scope (DESIGN.md section 6).

Embedding tables and first-order weights are optimizer-owned state of the layer (updated in place during
`.backward()`); everything else is an ordinary Parameter stepped by `dense_optimizer()`, the dense
counterpart of the same rule ([TF] ApplyAdagrad: accumulator 0.1, no epsilon; `DCN(optimizer='adam')`: [TF] ApplyAdam,
`TFAdam`).
"""
from typing import Optional, Sequence

import torch

from .layers import CrossNetwork, EmbeddingFM
from .sharded import ShardedEmbeddingFM

_ADAGRAD_LR = 0.05        # [TF] canned estimators' default for 'Adagrad' (deepFM.py:61)


class _Tower(torch.nn.Module):
    """dnn_logit_fn (deepFM.py:284-319) / _deep_architecture (DeepCrossNetwork.py:370-410): dense + activation per
    hidden layer, optional dropout and batch normalisation, optional activation-free final layer."""

    def __init__(self, d_in, hidden_units, final_units, activation, dropout, batch_norm, bn_momentum,
                 bn_on_last, init, device, bn_before_dropout=False):
        super().__init__()
        self.bn_before_dropout = bn_before_dropout
        sizes = [d_in] + [int(h) for h in hidden_units]
        self.hidden = torch.nn.ModuleList(torch.nn.Linear(a, b, device=device) for a, b in zip(sizes[:-1], sizes[1:]))
        n = len(self.hidden)
        self.bn = torch.nn.ModuleList(
            (torch.nn.BatchNorm1d(b, momentum=1.0 - bn_momentum, eps=1e-3, device=device)       # TF momentum / epsilon
             if batch_norm and (bn_on_last or i < n - 1) else torch.nn.Identity())
            for i, b in enumerate(sizes[1:]))
        self.final = torch.nn.Linear(sizes[-1], final_units, device=device) if final_units else None
        self.activation, self.dropout = activation, dropout
        self.out_features = final_units or sizes[-1]
        for lin in list(self.hidden) + ([self.final] if self.final is not None else []):
            init(lin.weight)
            torch.nn.init.zeros_(lin.bias)

    def forward(self, x):
        for lin, bn in zip(self.hidden, self.bn):
            x = self.activation(lin(x))
            if self.bn_before_dropout:            # DCN: dense(act) -> batch norm -> dropout (DeepCrossNetwork.py:397-408)
                x = bn(x)
            if self.dropout is not None and self.training:
                x = torch.nn.functional.dropout(x, self.dropout, True)
            if not self.bn_before_dropout:        # DeepFM: dense(act) -> dropout -> batch norm (deepFM.py:297-306)
                x = bn(x)
        return self.final(x) if self.final is not None else x


def _embedding_layer(sharded, *args, **kw):
    return (ShardedEmbeddingFM if sharded else EmbeddingFM)(*args, **kw)


class TFAdam(torch.optim.Optimizer):
    """[TF] ApplyAdam, tf.train.AdamOptimizer's rule for dense variables (the reference's DCN optimizer,
    models/DeepCrossNetwork/train.py:104-124), in fp32:
        lr_t = lr * sqrt(1 - beta2_power) / (1 - beta1_power)
        m += (g - m) * (1 - beta1);  v += (g * g - v) * (1 - beta2);  var -= (m * lr_t) / (sqrt(v) + epsilon)
        then beta1_power *= beta1, beta2_power *= beta2 (once per step, shared by every parameter)
    Not torch.optim.Adam, which adds epsilon after the bias correction of v.  The beta powers are one device tensor
    (`beta_power`, kept in the optimizer's state so state_dict() / load_state_dict() carry it), so a captured step
    replays with the right bias correction."""

    def __init__(self, params, lr, beta1=0.9, beta2=0.999, epsilon=1e-8):
        if not lr > 0 or not (0 <= beta1 < 1 and 0 <= beta2 < 1) or not epsilon > 0:
            raise ValueError("TFAdam needs lr > 0, 0 <= beta1, beta2 < 1 and epsilon > 0")
        super().__init__(params, dict(lr=float(lr)))
        self.beta1, self.beta2, self.epsilon = float(beta1), float(beta2), float(epsilon)
        # 1 - beta as TF evaluates it, in fp32 (1 - 0.9 in fp64 rounds to a different fp32 value)
        self._omb1 = float(torch.tensor(1.0) - torch.tensor(self.beta1))
        self._omb2 = float(torch.tensor(1.0) - torch.tensor(self.beta2))
        self._betas = None

    @property
    def beta_power(self):
        """(beta1_power, beta2_power), float32[2] on the parameters' device (None before the first step)."""
        return self.state.get("beta_power")

    @torch.no_grad()
    def step(self, closure=None):
        loss = closure() if closure is not None else None
        params = [p for g in self.param_groups for p in g["params"]]
        if not params:
            return loss
        dev = params[0].device
        bp = self.state.get("beta_power")
        if bp is None:
            bp = torch.tensor([self.beta1, self.beta2], dtype=torch.float32, device=dev)
        elif bp.device != dev:                   # loaded from a checkpoint on another device
            bp = bp.to(dev)
        self.state["beta_power"] = bp            # not a parameter's state: load_state_dict copies it as it is
        if self._betas is None or self._betas.device != dev:
            self._betas = torch.tensor([self.beta1, self.beta2], dtype=torch.float32, device=dev)
        for group in self.param_groups:
            lr_t = (group["lr"] * torch.sqrt(1 - bp[1])) / (1 - bp[0])
            for p in group["params"]:
                if p.grad is None:
                    continue
                st = self.state[p]
                if not st:
                    st["m"], st["v"] = torch.zeros_like(p), torch.zeros_like(p)
                g, m, v = p.grad, st["m"], st["v"]
                m.add_((g - m) * self._omb1)
                v.add_((g * g - v) * self._omb2)
                p.sub_((m * lr_t) / (v.sqrt() + self.epsilon))
        bp.mul_(self._betas)
        return loss


def clip_by_norm_(parameters, clip_norm):
    """tf.clip_by_norm applied to EACH gradient tensor (DeepCrossNetwork.py:284), not a global norm."""
    for p in parameters:
        if p.grad is not None:
            p.grad.mul_(clip_norm / torch.clamp(p.grad.norm(), min=clip_norm))


class DeepFM(torch.nn.Module):
    """DeepFM as `_DeepFM_model_fn` builds it (deepFM.py:143-252).

    Constructor knobs follow the reference's (deepFM.py:55-73): fm_embedding_size, dnn_hidden_units,
    dnn_activation_fn, dnn_dropout, batch_norm, dnn_optimizer ('Adagrad'), loss_reduction (SUM);
    field_size = len(column_names), rows_per_field = the columns' bucket sizes.  linear_optimizer
    ('ftrl' | 'adagrad' | 'sgd', the reference's default is 'Ftrl'; None = dnn_optimizer) trains the first-order
    weights inside the fused backward; l1_/l2_regularization_strength pass through to the layer.  The scalar
    linear bias is stepped by `dense_optimizer()` with the tower.
    forward(feature_index[B,F], feature_value[B,F] | None) -> logits[B,1].
    """

    def __init__(self, field_size: int, fm_embedding_size: int, rows_per_field: Sequence[int],
                 dnn_hidden_units: Sequence[int] = (256, 128), dnn_activation_fn=torch.relu,
                 dnn_dropout: Optional[float] = None, batch_norm: bool = False, dnn_optimizer: str = "adagrad",
                 dnn_learning_rate: float = _ADAGRAD_LR, linear_optimizer: Optional[str] = None,
                 linear_learning_rate: Optional[float] = None, loss_reduction: str = "sum", sharded: bool = False,
                 device="cuda", **layer_kw):
        super().__init__()
        if str(dnn_optimizer).lower() == "adam":
            raise ValueError("DeepFM trains with Adagrad (the reference's dnn_optimizer) or SGD; adam is a DCN option")
        if not dnn_hidden_units:
            raise ValueError("dnn_hidden_units must name at least one layer")
        if loss_reduction not in ("sum", "mean"):
            raise ValueError("loss_reduction must be 'sum' or 'mean'")
        self.loss_reduction, self.dnn_learning_rate = loss_reduction, float(dnn_learning_rate)
        self.embedding = _embedding_layer(sharded, field_size, fm_embedding_size, list(rows_per_field),
                                          optimizer=dnn_optimizer, lr=dnn_learning_rate,
                                          linear_optimizer=linear_optimizer, linear_lr=linear_learning_rate,
                                          device=device, **layer_kw)
        self.dnn = _Tower(field_size * fm_embedding_size, dnn_hidden_units, 1, dnn_activation_fn, dnn_dropout,
                          batch_norm, 0.999, True, torch.nn.init.xavier_uniform_, device)     # glorot_uniform (:300)

    def forward(self, feature_index, feature_value=None, presorted=None):
        first, fm, emb = self.embedding(feature_index, feature_value, presorted=presorted)
        return first + fm + self.dnn(emb)                                   # :337-338 then add_n (:223)

    def loss(self, logits, labels):
        """_binary_logistic_head_with_sigmoid_cross_entropy_loss, loss_reduction SUM by default (:72, :107-111)."""
        return torch.nn.functional.binary_cross_entropy_with_logits(
            logits.reshape(-1), labels.reshape(-1).float(), reduction=self.loss_reduction)

    def dense_parameters(self):
        return [p for n, p in self.named_parameters() if not n.endswith("_anchor")]

    def dense_optimizer(self):
        return torch.optim.Adagrad(self.dense_parameters(), lr=self.dnn_learning_rate,
                                   initial_accumulator_value=0.1, eps=0.0)

    def train_step(self, optimizer, feature_index, feature_value, labels):
        """forward, loss, backward (tables updated in place by the fused kernel), dense step."""
        optimizer.zero_grad(set_to_none=True)
        loss = self.loss(self(feature_index, feature_value), labels)
        loss.backward()
        optimizer.step()
        return loss.detach()


class DCN(torch.nn.Module):
    """Deep & Cross network as `dcn_logits_fn` builds it (DeepCrossNetwork.py:124-141): x0 = the embedded
    input, `cross_layer_num` cross layers beside a deep tower, concat, dense(1).  hidden_units,
    cross_layer_num, dnn_dropout, batch_norm, learning rate and clip norm as in DeepCrossNetwork.py:35-49,
    :282-289; MEAN-reduced loss (:209-225).  x0 is the [B, F*K] embedding output (every field embedded
    to K: BASELINE.json's d = 624 convention).
    The per-tensor clip_by_norm(100) is applied to every gradient, as the reference does: the dense ones here, each
    column's table gradient inside the layer (`EmbeddingFM(clip_norm=...)`, a two-pass backward).  The sharded
    layer clips its table gradients only with clip_sharded_tables=True (`ShardedEmbeddingFM(clip_norm=...)`: each
    column's norm over the merged sums of the global batch, reduced across ranks on the device); by default it
    applies them unclipped, as it always has.
    optimizer='adam' is the reference's own (train.py:104-124, epsilon = adam_epsilon = 1e-4): TF's Adam on the
    tables (`EmbeddingFM(optimizer='adam')`, or `ShardedEmbeddingFM(optimizer='adam')` with sharded=True, where each
    owner sweeps its own shard; every row's moments decay at every step) and `TFAdam` on the dense parameters.  With
    sharded=True and clip_sharded_tables=True that is the reference's full rule across GPUs: every column's table
    gradient clipped, then Adam.
    """

    def __init__(self, field_size: int, embedding_size: int, rows_per_field: Sequence[int],
                 cross_layer_num: int = 2, hidden_units: Sequence[int] = (256, 128), dnn_activation_fn=torch.relu,
                 dnn_dropout: Optional[float] = None, batch_norm: bool = False, optimizer: str = "adagrad",
                 learning_rate: float = _ADAGRAD_LR, clip_norm: Optional[float] = 100.0, sharded: bool = False,
                 device="cuda", adam_epsilon: float = 1e-4, clip_sharded_tables: bool = False, **layer_kw):
        super().__init__()
        d = field_size * embedding_size
        self.learning_rate, self.clip_norm = float(learning_rate), clip_norm
        self.optimizer, self.adam_epsilon = optimizer.lower(), float(adam_epsilon)
        if clip_norm and (clip_sharded_tables or not sharded):
            layer_kw = dict(layer_kw, clip_norm=clip_norm)      # every column's gradient is clipped too (:284)
        if self.optimizer == "adam":
            layer_kw = dict(layer_kw, optimizer_epsilon=self.adam_epsilon)
        self.embedding = _embedding_layer(sharded, field_size, embedding_size, list(rows_per_field), optimizer=optimizer,
                                          lr=learning_rate, first_order=False, device=device, **layer_kw)
        self.cross = CrossNetwork(d, cross_layer_num, device=device)
        self.deep = _Tower(d, hidden_units, 0, dnn_activation_fn, dnn_dropout, batch_norm, 0.999, False,
                           torch.nn.init.xavier_normal_, device, bn_before_dropout=True)        # glorot_normal (:393)
        self.logits = torch.nn.Linear(d + self.deep.out_features, 1, device=device)             # :137
        torch.nn.init.xavier_uniform_(self.logits.weight)      # tf.layers.dense default kernel init
        torch.nn.init.zeros_(self.logits.bias)

    def forward(self, feature_index, feature_value=None, presorted=None):
        _, _, x0 = self.embedding(feature_index, feature_value, presorted=presorted)
        return self.logits(torch.cat([self.cross(x0), self.deep(x0)], dim=-1))

    def loss(self, logits, labels):
        return torch.nn.functional.binary_cross_entropy_with_logits(
            logits.reshape(-1), labels.reshape(-1).float(), reduction="mean")

    def dense_parameters(self):
        skip = ("_anchor", "embedding.bias")
        return [p for n, p in self.named_parameters() if not n.endswith(skip)]

    def dense_optimizer(self):
        if self.optimizer == "adam":
            return TFAdam(self.dense_parameters(), self.learning_rate, epsilon=self.adam_epsilon)
        return torch.optim.Adagrad(self.dense_parameters(), lr=self.learning_rate,
                                   initial_accumulator_value=0.1, eps=0.0)

    def train_step(self, optimizer, feature_index, feature_value, labels):
        optimizer.zero_grad(set_to_none=True)
        loss = self.loss(self(feature_index, feature_value), labels)
        loss.backward()
        if self.clip_norm:
            clip_by_norm_(self.dense_parameters(), float(self.clip_norm))
        optimizer.step()
        return loss.detach()
