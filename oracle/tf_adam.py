"""TEST INFRASTRUCTURE -- [TF] tf.train.AdamOptimizer as the reference's DCN trains with it
(models/DeepCrossNetwork/train.py:104-124: AdamOptimizer(learning_rate, epsilon=1e-4) after clip_by_norm(., 100) on
every gradient, DeepCrossNetwork.py:264-290).

PARITY UNPINNED like oracle/tf_semantics.py: TensorFlow 1.x cannot run here, so the rules below are TF's
adam.py / training_ops as recalled from its sources, in TF's evaluation order.  tests/test_oracle_adam.py pins
them against closed forms.  Only tests/ may import this.

  sparse_adam   Adam._apply_sparse_shared on an IndexedSlices gradient (an embedding table): the moments of EVERY
                row decay, the batch's de-duplicated rows scatter-add, every row moves.  Not LazyAdam.
  dense_adam    ApplyAdam on a dense variable: the same rule, rounded differently.
  finish        Adam._finish: both powers advance once per apply_gradients, shared by all variables.
"""
import numpy as np

from . import deepctr_oracle as O
from . import full_models as FM
from . import tf_semantics as tfs

# tf.train.AdamOptimizer defaults; the reference's DCN passes epsilon = 1e-4 (train.py:104-124)
BETA1, BETA2, EPSILON = 0.9, 0.999, 1e-8
DCN_EPSILON = 1e-4


def _scalars(beta1, beta2, epsilon, dt):
    """beta1, beta2, 1 - beta1, 1 - beta2, epsilon as TF evaluates them for an fp32 variable -- in fp32 (fp32(1) -
    fp32(0.999) is 1.3e-5 away from 0.001) -- then carried in dt."""
    f = np.float32
    return (dt(f(beta1)), dt(f(beta2)), dt(f(1) - f(beta1)), dt(f(1) - f(beta2)), dt(f(epsilon)))


def initial_powers(beta1=BETA1, beta2=BETA2, dtype=np.float32):
    """beta1_power, beta2_power as Adam._create_slots makes them: they start at beta1 and beta2 (fp32 values)."""
    return np.asarray(np.float32([beta1, beta2]), dtype=dtype)


def adam_lr(lr, beta_power):
    """lr * sqrt(1 - beta2_power) / (1 - beta1_power), from the powers as they stand before this step's _finish."""
    dt = beta_power.dtype.type
    return dt(lr) * np.sqrt(dt(1) - beta_power[1]) / (dt(1) - beta_power[0])


def sparse_adam(var, m, v, rows, grad, lr, beta_power, beta1=BETA1, beta2=BETA2, epsilon=EPSILON):
    """Adam._apply_sparse_shared after _apply_sparse_duplicate_indices summed duplicate rows; in place, `rows` unique:
        m = m * beta1;  m[r] += g_r * (1 - beta1)          (assign, then scatter_add)
        v = v * beta2;  v[r] += (g_r * g_r) * (1 - beta2)
        var -= (lr_t * m) / (sqrt(v) + epsilon)            every row; epsilon outside the sqrt, no bias-corrected v
    Rows the batch does not touch still decay, and still move while their m is not zero."""
    dt = var.dtype.type
    b1, b2, omb1, omb2, eps = _scalars(beta1, beta2, epsilon, dt)
    lr_t = adam_lr(lr, beta_power)
    m[...] = m * b1
    m[rows] = m[rows] + grad * omb1
    v[...] = v * b2
    v[rows] = v[rows] + (grad * grad) * omb2
    var[...] = var - (lr_t * m) / (np.sqrt(v) + eps)


def dense_adam(var, m, v, grad, lr, beta_power, beta1=BETA1, beta2=BETA2, epsilon=EPSILON):
    """ApplyAdam (training_ops, use_nesterov = False); in place:
        m += (g - m) * (1 - beta1);  v += (g * g - v) * (1 - beta2);  var -= (m * lr_t) / (sqrt(v) + epsilon)"""
    dt = var.dtype.type
    b1, b2, omb1, omb2, eps = _scalars(beta1, beta2, epsilon, dt)
    lr_t = adam_lr(lr, beta_power)
    m += (grad - m) * omb1
    v += (grad * grad - v) * omb2
    var -= (m * lr_t) / (np.sqrt(v) + eps)


def finish(beta_power, beta1=BETA1, beta2=BETA2):
    """Adam._finish: beta1_power *= beta1, beta2_power *= beta2 (once per apply_gradients)."""
    dt = beta_power.dtype.type
    beta_power[0] = beta_power[0] * dt(np.float32(beta1))
    beta_power[1] = beta_power[1] * dt(np.float32(beta2))


def adam_state(p, beta1=BETA1, beta2=BETA2):
    """Zero m / v slots shaped like every entry of a parameter dict (lists kept), and the shared powers."""
    dt = p["table"].dtype
    st = {"m": {}, "v": {}, "beta_power": initial_powers(beta1, beta2, dt)}
    for k, val in p.items():
        for s in ("m", "v"):
            st[s][k] = [np.zeros_like(a) for a in val] if isinstance(val, list) else np.zeros_like(np.asarray(val))
    return st


def dcn_gradients(p, field_offset, idx, val, labels, clip_norm=100.0):
    """The gradients full_models.dcn_train_step applies (DeepCrossNetwork.py:124-141 backward, MEAN loss), clipped as
    the reference clips them (:282-289): each table column's IndexedSlices on its own, every dense tensor on its own.
    -> dict(loss, logits, rows, G, G_unclipped, dense={name: grad or [grads]}).  tests/test_oracle_adam.py pins it to
    full_models.dcn_train_step, so the two restatements of the DCN backward cannot drift apart."""
    dt = p["table"].dtype.type
    logits, c = FM.dcn_forward(p, field_offset, idx, val)
    loss, g = FM.sigmoid_ce_grad(logits, labels.astype(dt), "mean")
    d = p["cross_w"].shape[1]
    dWl = c["m"].T @ g[:, None]
    dbl = np.asarray([g.sum()], dtype=dt)
    dm = g[:, None] @ p["Wl"].T
    dx0_c, dcw, dcb = O.cross_backward(c["x0"], p["cross_w"], p["cross_b"], dm[:, :d])
    dx0_d, dWs, dbs = FM.mlp_backward(c["acts"], p["W"], dm[:, d:], final_linear=False)
    u = (dx0_c + dx0_d).reshape(c["e"].shape)
    zero = np.zeros(idx.shape[0], dtype=dt)
    rows, G, _, _ = O.embedding_backward(p["table"], field_offset, idx, val, zero, zero, u, "sum", dt)
    clip = (lambda t: tfs.clip_by_norm(t, clip_norm)) if clip_norm else (lambda t: t)
    G_unclipped = G
    if clip_norm:
        G = tfs.clip_indexed_slices_per_column(rows, G, field_offset, p["table"].shape[0], clip_norm)
    dense = dict(cross_w=clip(dcw), cross_b=clip(dcb), Wl=clip(dWl), bl=clip(dbl),
                 W=[clip(x) for x in dWs], b=[clip(x) for x in dbs])
    return dict(loss=loss, logits=logits, rows=rows, G=G, G_unclipped=G_unclipped, dense=dense)


def dcn_train_step(p, st, field_offset, idx, val, labels, lr, clip_norm=100.0, epsilon=DCN_EPSILON,
                   beta1=BETA1, beta2=BETA2, sparse=None, dense=None):
    """full_models.dcn_train_step with the reference's optimizer (train.py:104-124): the clipped gradients of
    dcn_gradients, Adam on the table (sparse_adam) and on every dense variable (dense_adam), then one _finish.
    In place; st from adam_state.  sparse / dense replace the two rules (tests use it for rules that must be told
    apart from TF's).  Returns dcn_gradients' dict."""
    sparse, dense = sparse or sparse_adam, dense or dense_adam
    out = dcn_gradients(p, field_offset, idx, val, labels, clip_norm)
    bp, M, V = st["beta_power"], st["m"], st["v"]
    hp = dict(beta1=beta1, beta2=beta2, epsilon=epsilon)
    sparse(p["table"], M["table"], V["table"], out["rows"], out["G"], lr, bp, **hp)
    for k, grad in out["dense"].items():
        if isinstance(grad, list):
            for i, gi in enumerate(grad):
                dense(p[k][i], M[k][i], V[k][i], gi, lr, bp, **hp)
        else:
            dense(p[k], M[k], V[k], grad, lr, bp, **hp)
    finish(bp, beta1, beta2)
    return out
