"""TF 1.x Adam on the embedding tables (dir_rows_apply_adam, `EmbeddingFM(optimizer='adam')`, `DCN(optimizer='adam')`)
against oracle/tf_adam.py.

Two levels, because Adam divides by sqrt(v) + eps: a gradient component that cancels to |G| ~ eps moves by up to
lr_t whatever its sign, so an error in G that is harmless elsewhere can move such a component by lr_t.
  * the apply kernel on a gradient the test supplies: the oracle sees the same fp32 inputs, so T, m, v are held to REL;
  * the layer: the kernel's gradient sums may differ from the oracle's by the band the full-size tests allow them
    (REL * Gfloor, the cancellation-aware magnitude being summed, SURVEY 7.2).  `_adam_step_band` pushes that band
    through one update by interval arithmetic and adds a few ulp of fp32 rounding; that is the bound, checked step
    by step from the state the kernel started from.  Negative controls check that it still rejects LazyAdam, torch's epsilon placement and a step
    without bias correction."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import deepctr_oracle as O
from oracle import full_models as FM
from oracle import tf_adam as A
from oracle import tf_semantics as tfs
from tests._util import REL, make_case, rel_err, to_dev, torch_embedding_reference

pytestmark = pytest.mark.gpu

B1, B2 = 0.9, 0.999
ULP = 2.0 ** -23


def _adam_step_band(T, m, v, p1, p2, G, d, has, lr, eps, b1=B1, b2=B2, lazy=False, torch_eps=False, no_bias=False):
    """One TF Adam step in fp64 from the state the kernel started from: T, m, v [R,K], powers p1, p2 (the fp32 values
    on the device), the oracle's gradient G [R,K] (0 where has[R] is False) and its band d = REL * Gabs.
    -> T', m', v' and bounds on |kernel - T'| etc. that hold for any gradient within G +- d (interval arithmetic
    through m, v and the division), plus a few ulp of fp32 rounding.  lazy / torch_eps / no_bias change T' to the
    rules the bound must reject (LazyAdam, torch.optim.Adam's epsilon, no bias correction); the bounds stay TF's."""
    f = np.float32                       # the scalars as TF evaluates them: fp32, 1 - beta included
    b1, b2, o1, o2, eps = float(f(b1)), float(f(b2)), float(f(1) - f(b1)), float(f(1) - f(b2)), float(f(eps))
    lr_t = lr * np.sqrt(1 - p2) / (1 - p1)
    m1 = b1 * m + o1 * G
    v1 = b2 * v + o2 * G * G
    slack = 4 * ULP * (b1 * m.abs() + o1 * (G.abs() + d))
    m_lo, m_hi = b1 * m + o1 * (G - d) - slack, b1 * m + o1 * (G + d) + slack
    sq_lo = torch.where(G.abs() <= d, torch.zeros_like(G), (G.abs() - d) ** 2)
    v_lo = (b2 * v + o2 * sq_lo) * (1 - 4 * ULP)
    v_hi = (b2 * v + o2 * (G.abs() + d) ** 2) * (1 + 4 * ULP)
    step = lr_t * m1 / (v1.sqrt() + eps)
    dlo, dhi = v_lo.sqrt() + eps, v_hi.sqrt() + eps
    s_lo = lr_t * torch.where(m_lo >= 0, m_lo / dhi, m_lo / dlo)
    s_hi = lr_t * torch.where(m_hi >= 0, m_hi / dlo, m_hi / dhi)
    bT = torch.maximum(s_hi - step, step - s_lo) + 8 * ULP * torch.maximum(s_lo.abs(), s_hi.abs()) + ULP * T.abs()
    bm = torch.maximum(m_hi - m1, m1 - m_lo)
    bv = torch.maximum(v_hi - v1, v1 - v_lo)
    if no_bias:
        step = lr * m1 / (v1.sqrt() + eps)
    if torch_eps:
        step = lr * (m1 / (1 - p1)) / ((v1 / (1 - p2)).sqrt() + eps)
    if lazy:
        step = torch.where(has[:, None], step, torch.zeros_like(step))
    return T - step, m1, v1, bT, bm, bv


def _lib_call(L, table, row_stride, n_rows, K, gu, urows, count, n_cap, off, F, part, clip, opt, lin=None,
              lin_acc=None, lin_opt=None):
    from dir_b200 import _lib
    _lib.check(L.dir_rows_apply_adam(table.data_ptr(), row_stride, n_rows, K,
                                     None if lin is None else lin.data_ptr(), None if lin_acc is None else lin_acc.data_ptr(),
                                     1, lin_opt, None if gu is None else gu.data_ptr(), K + 4,
                                     None if urows is None else urows.data_ptr(),
                                     None if count is None else count.data_ptr(), n_cap, off.data_ptr(), F,
                                     None if part is None else part.data_ptr(), clip, ctypes.byref(opt), None,
                                     torch.cuda.current_stream().cuda_stream), "dir_rows_apply_adam")


@pytest.mark.parametrize("K", [4, 8, 16, 32, 64])
@pytest.mark.parametrize("clip", [None, 0.5])
def test_apply_kernel_three_steps(pkg, cuda, K, clip):
    from dir_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(K + (7 if clip else 0))
    rows_per_field = [1, 700, 1, 2500, 3, 1300]              # tiles of 1024 rows cross field boundaries
    F, N = len(rows_per_field), sum(rows_per_field)
    off = np.concatenate([[0], np.cumsum(rows_per_field)[:-1]]).astype(np.int64)
    lr, eps = 0.01, 1e-4
    T0 = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
    rows = torch.zeros((N, 3 * K + 4), dtype=torch.float32, device="cuda")     # row_stride > 3K
    rows[:, :K] = to_dev(T0)
    bp = torch.tensor([B1, B2], dtype=torch.float32, device="cuda")
    opt = _lib.AdamOpt(lr, B1, B2, eps, bp.data_ptr())
    part = torch.empty(int(L.dir_field_sqnorms_bytes(F)), dtype=torch.uint8, device="cuda")
    offd = to_dev(off)
    t, m, v = T0.astype(np.float64), np.zeros((N, K)), np.zeros((N, K))
    bp64 = A.initial_powers(B1, B2, np.float32)
    edges = np.concatenate([off, off + np.asarray(rows_per_field) - 1, [1023, 1024, 2047, 2048, N - 1]])
    choices = [np.unique(np.concatenate([edges, rng.choice(N, 900, replace=False)])),       # boundaries + random
               np.arange(N), np.zeros(0, np.int64)]                                         # U = n_rows, U = 0
    touched = np.zeros(N, bool)
    for ur in choices:
        U = ur.size
        G = (rng.standard_normal((U, K)) * rng.choice([1e-6, 1e-2, 1.0], size=(U, 1))).astype(np.float32)
        gu = torch.zeros((max(U, 1), K + 4), dtype=torch.float32, device="cuda")
        gu[:U, :K] = to_dev(G)
        urows = to_dev(ur.astype(np.int32)) if U else torch.zeros(1, dtype=torch.int32, device="cuda")
        count = torch.tensor([0, U], dtype=torch.int64, device="cuda")
        n_dev = count[1:]
        if clip is not None and U:
            _lib.check(L.dir_field_sqnorms(gu.data_ptr(), K + 4, urows.data_ptr(), n_dev.data_ptr(), offd.data_ptr(), F,
                                           K, N, part.data_ptr(), torch.cuda.current_stream().cuda_stream), "sqnorms")
            Gc = tfs.clip_indexed_slices_per_column(ur, G.astype(np.float64), off, N, clip)
        else:
            Gc = G.astype(np.float64)
        _lib_call(L, rows, 3 * K + 4, N, K, gu if U else None, urows if U else None, n_dev if U else None, U, offd, F,
                  part if (clip is not None and U) else None, clip or 0.0, opt)
        A.sparse_adam(t, m, v, ur, Gc, lr, bp64.astype(np.float64), B1, B2, eps)
        A.finish(bp64, B1, B2)
        touched[ur] = True
    torch.cuda.synchronize()
    got = rows.cpu().numpy()
    assert rel_err(got[:, :K], t, np.abs(T0).max() + lr) <= REL
    assert rel_err(got[:, K:2 * K], m, np.abs(m).max()) <= REL
    assert rel_err(got[:, 2 * K:3 * K], v, np.abs(v).max()) <= REL
    assert np.array_equal(bp.cpu().numpy(), bp64), "beta powers: the repeated fp32 product, bit for bit"
    assert not got[:, 3 * K:].any(), "the row padding beyond 3K is never written"


def test_apply_kernel_untouched_rows_bit_exact_and_graph_replay(pkg, cuda):
    from dir_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(3)
    N, K, F = 5000, 16, 1
    offd = torch.zeros(1, dtype=torch.int64, device="cuda")
    rows0 = torch.zeros((N, 3 * K), dtype=torch.float32, device="cuda")
    rows0[:, :K] = torch.randn((N, K), device="cuda")
    ur = np.sort(rng.choice(N, 300, replace=False)).astype(np.int32)
    gu = torch.zeros((300, K + 4), device="cuda")
    gu[:, :K] = torch.randn((300, K), device="cuda")
    urows, count = to_dev(ur), torch.tensor([300], dtype=torch.int64, device="cuda")

    def run(rows, bp, n):
        opt = _lib.AdamOpt(0.01, B1, B2, 1e-8, bp.data_ptr())
        for _ in range(n):
            _lib_call(L, rows, 3 * K, N, K, gu, urows, count, 300, offd, F, None, 0.0, opt)

    eager, bp_e = rows0.clone(), torch.tensor([B1, B2], device="cuda")
    run(eager, bp_e, 3)
    never = np.setdiff1d(np.arange(N), ur)
    assert torch.equal(eager[never], rows0[never]), "never-touched rows: T unchanged, m = v = 0, bit for bit"
    graphed, bp_g = rows0.clone(), torch.tensor([B1, B2], device="cuda")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):          # warm the launch path outside the capture, then restore the state
        run(graphed, bp_g, 1)
    torch.cuda.current_stream().wait_stream(side)
    graphed.copy_(rows0)
    bp_g.copy_(torch.tensor([B1, B2]))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        run(graphed, bp_g, 1)
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    assert torch.equal(graphed, eager) and torch.equal(bp_g, bp_e), "3 replays must equal 3 eager calls, bitwise"


SHAPES = [(64, [50, 1, 9, 1000, 3, 17, 1], 16), (257, [100] * 26 + [1] * 13, 16), (700, [5, 1, 3], 8),
          (3000, [40, 2000, 1], 32)]


@pytest.mark.parametrize("B,rows,K", SHAPES)
@pytest.mark.parametrize("lin_opt", [None, "ftrl"])
@pytest.mark.parametrize("eps", [1e-4, 1e-8])
def test_layer_three_steps_against_the_band(pkg, cuda, B, rows, K, lin_opt, eps):
    """Three steps of EmbeddingFM(optimizer='adam') on the test_gpu_ftrl shapes (weighted, pruned, skewed, one-row
    fields).  Each step is checked from the state the kernel started from: the oracle takes its gradient at the
    layer's own table, so the band of one step does not have to carry the previous steps' rounding."""
    case = make_case(31, B, rows, K, weighted=True, prune=True, skew=2.0)
    rng, F, N = case["rng"], case["F"], case["N"]
    lr, lin_lr = 0.01, 0.2
    steps = []
    for s in range(3):               # the batches differ: rows touched earlier go untouched later
        c = make_case(100 + s, B, rows, K, weighted=True, prune=True, skew=2.0)
        steps.append((c["idx"], c["val"], rng.standard_normal(B).astype(np.float32),
                      (rng.standard_normal(B) * 0.1).astype(np.float32),
                      (rng.standard_normal((B, F, K)) * 0.1).astype(np.float32)))
    kw = dict(linear_optimizer=lin_opt, linear_lr=lin_lr) if lin_opt else dict(first_order=False)
    layer = pkg.EmbeddingFM(F, K, [int(r) for r in rows], optimizer="adam", lr=lr, optimizer_epsilon=eps, **kw).train()
    layer.load_tables(case["table"], case["w1"])
    w, n1, z1 = case["w1"].astype(np.float64), np.full(N, 0.1), np.zeros(N)
    touched = np.zeros(N, bool)
    rejected = dict(lazy=False, no_bias=False, torch_eps=False)
    stale = False
    for s, (idx, val, g_first, g_fm, u) in enumerate(steps):
        st = torch.tensor(layer.rows.cpu().numpy().astype(np.float64))
        T, m, v = st[:, :K], st[:, K:2 * K], st[:, 2 * K:]
        p1, p2 = (float(x) for x in layer.beta_power.cpu())
        r, G, g1, _ = O.embedding_backward(T.numpy(), case["off"], idx, val, g_first, g_fm, u, "sum", np.float64)
        # the band of the kernel's row sums: REL of the cancellation-aware magnitude |x| (|g_fm| sum_f |e_f| + |u|)
        # (SURVEY 7.2); the oracle's sum of |per-lookup term| misses the rounding of S where S - e cancels
        Gfloor = torch_embedding_reference(st[:, :K].float(), torch.zeros(N), 0.0, torch.tensor(case["off"]),
                                           torch.tensor(idx), torch.tensor(val), torch.tensor(g_first),
                                           torch.tensor(g_fm), torch.tensor(u))["Gfloor"]
        first, fm, emb = layer(to_dev(idx), to_dev(val))
        torch.autograd.backward((first, fm, emb), (to_dev(g_first)[:, None], to_dev(g_fm)[:, None],
                                                   to_dev(u.reshape(B, -1))))
        torch.cuda.synchronize()
        Gd, dd, has = torch.zeros((N, K), dtype=torch.float64), torch.zeros((N, K), dtype=torch.float64), torch.zeros(N, dtype=torch.bool)
        Gd[r], has[r] = torch.tensor(G), True
        dd = REL * Gfloor
        T1, m1, v1, bT, bm, bv = _adam_step_band(T, m, v, p1, p2, Gd, dd, has, lr, eps)
        got = torch.tensor(layer.rows.cpu().numpy().astype(np.float64))
        errT = (got[:, :K] - T1).abs()
        assert bool((errT <= bT).all()), (s, float((errT - bT).max()), int((errT > bT).sum()))
        assert bool(((got[:, K:2 * K] - m1).abs() <= bm).all()), s
        assert bool(((got[:, 2 * K:] - v1).abs() <= bv).all()), s
        assert int(layer.last_n_unique.item()) == r.size
        for name in rejected:
            T_x = _adam_step_band(T, m, v, p1, p2, Gd, dd, has, lr, eps, **{name: True})[0]
            rejected[name] |= bool(((T_x - T1).abs() > bT).any())
        if lin_opt:
            O.sparse_ftrl(w, n1, z1, r, g1, lin_lr)
        stale |= bool((touched & ~has.numpy()).any())     # rows with a nonzero m and no gradient in this step
        touched[r] = True
    final = layer.rows.cpu().numpy()
    assert np.array_equal(final[~touched, :K], case["table"][~touched]) and not final[~touched, K:].any()
    bp = A.initial_powers(B1, B2, np.float32)
    for _ in range(3):
        A.finish(bp, B1, B2)
    assert np.array_equal(layer.beta_power.cpu().numpy(), bp)
    # negative controls: the same bound rejects the wrong rules (torch's epsilon placement only shows at a large eps)
    assert stale or N < B, "some rows touched earlier must go untouched later (every batch covers the [5, 1, 3] table)"
    assert (rejected["lazy"] or not stale) and rejected["no_bias"], rejected
    assert rejected["torch_eps"] or eps < 1e-4, rejected
    if lin_opt:
        got_w = layer.w1.cpu().numpy()
        assert rel_err(got_w, w, np.abs(case["w1"]).max() + lin_lr) <= 2 * REL
        assert np.array_equal(got_w[~touched], case["w1"][~touched])
    # run to run: bit-identical
    again = pkg.EmbeddingFM(F, K, [int(r) for r in rows], optimizer="adam", lr=lr, optimizer_epsilon=eps, **kw).train()
    again.load_tables(case["table"], case["w1"])
    for idx, val, g_first, g_fm, u in steps:
        first, fm, emb = again(to_dev(idx), to_dev(val))
        torch.autograd.backward((first, fm, emb), (to_dev(g_first)[:, None], to_dev(g_fm)[:, None],
                                                   to_dev(u.reshape(B, -1))))
    torch.cuda.synchronize()
    assert torch.equal(again.rows, layer.rows) and torch.equal(again.lin_rows, layer.lin_rows)


def _wrong_rule(kind):
    """(sparse, dense) rules with tf_adam's signature that differ from TF's Adam in one respect: 'lazy' (LazyAdam:
    only the batch's rows decay and move), 'torch_eps' (torch.optim.Adam: eps after the bias correction of v),
    'no_bias' (no bias correction)."""
    def move(var, m, v, lr, bp, eps):
        if kind == "torch_eps":
            return lr * (m / (1 - bp[0])) / (np.sqrt(v / (1 - bp[1])) + eps)
        if kind == "no_bias":
            return lr * m / (np.sqrt(v) + eps)
        return A.adam_lr(lr, bp) * m / (np.sqrt(v) + eps)

    def dense(var, m, v, grad, lr, bp, beta1, beta2, epsilon):
        m += (grad - m) * (1 - beta1)
        v += (grad * grad - v) * (1 - beta2)
        var -= move(var, m, v, lr, bp, epsilon)

    def sparse(var, m, v, rows, grad, lr, bp, beta1, beta2, epsilon):
        if kind == "lazy":
            sv, sm, sw = var[rows], m[rows], v[rows]
            dense(sv, sm, sw, grad, lr, bp, beta1, beta2, epsilon)
            var[rows], m[rows], v[rows] = sv, sm, sw
            return
        m[...] = m * beta1
        m[rows] += grad * (1 - beta1)
        v[...] = v * beta2
        v[rows] += grad * grad * (1 - beta2)
        var[...] = var - move(var, m, v, lr, bp, epsilon)

    return sparse, (A.dense_adam if kind == "lazy" else dense)


_VARIANTS = {k: _wrong_rule(k) for k in ("lazy", "torch_eps", "no_bias")}


def _copy(p):
    return {k: ([a.copy() for a in v] if isinstance(v, list) else np.copy(v)) for k, v in p.items()}


@pytest.mark.parametrize("clip", [100.0, 0.05])
def test_dcn_adam_two_steps(pkg, cuda, clip):
    """DCN with the reference's optimizer (Adam, eps = 1e-4, clip_by_norm on every gradient) against
    tf_adam.dcn_train_step in fp64, for the logits, the loss and every parameter over two steps on two different
    batches.  Bound per tensor: REL of its scale plus 8x the distance between the fp32 and the fp64 restatements of
    the same steps (how far fp32 arithmetic alone moves Adam's result on this case; the GPU plays no part in it).
    Negative controls: the same bounds reject LazyAdam, torch's epsilon placement and a step without bias
    correction, run through the same oracle."""
    B, K, hidden, L, lr = 192, 16, (64, 32), 3, 0.01
    ROWS = [50, 1, 9, 1000, 3, 17, 1]
    case = make_case(12, B, ROWS, K, weighted=True, prune=True)
    rng, F = case["rng"], case["F"]
    d = F * K
    labels = (rng.random(B) < 0.3).astype(np.float32)
    W, b = FM.make_tower(rng, d, hidden, 0, np.float32)
    p32 = dict(table=case["table"], cross_w=tfs.truncated_normal(rng, (L, d), 0.1),
               cross_b=tfs.truncated_normal(rng, (L, d), 0.1), W=W, b=b,
               Wl=FM.glorot_uniform(rng, d + hidden[-1], 1, np.float32), bl=np.asarray([0.02], np.float32))
    p = {k: ([a.astype(np.float64) for a in v] if isinstance(v, list) else np.asarray(v, np.float64)) for k, v in p32.items()}
    model = pkg.DCN(F, K, ROWS, cross_layer_num=L, hidden_units=hidden, learning_rate=lr, clip_norm=clip,
                    optimizer="adam").train()
    model.embedding.load_tables(case["table"], None)
    lins = list(model.deep.hidden)
    with torch.no_grad():
        for lin, ww, bb in zip(lins, W, b):
            lin.weight.copy_(to_dev(ww.T))
            lin.bias.copy_(to_dev(bb))
        model.cross.cross_w.copy_(to_dev(p32["cross_w"]))
        model.cross.cross_b.copy_(to_dev(p32["cross_b"]))
        model.logits.weight.copy_(to_dev(p32["Wl"].T))
        model.logits.bias.copy_(to_dev(p32["bl"]))
    second = make_case(13, B, ROWS, K, weighted=True, prune=True)      # rows of batch 0 go untouched in batch 1
    batches = [(case["idx"], case["val"], labels), (second["idx"], second["val"], (rng.random(B) < 0.3).astype(np.float32))]
    p0, p32 = _copy(p), _copy(p32)
    variants = {name: (_copy(p), A.adam_state(p)) for name in _VARIANTS}
    st, st32 = A.adam_state(p), A.adam_state(p32)
    opt = model.dense_optimizer()
    assert isinstance(opt, pkg.TFAdam)
    for step, (bi, bv, bl) in enumerate(batches):
        idx, val, y = to_dev(bi), to_dev(bv), to_dev(bl)
        with torch.no_grad():
            got_logits = model(idx, val)[:, 0].cpu().numpy()
        c = FM.dcn_forward(p, case["off"], bi, bv)[1]
        floor = np.abs(c["m"] * p["Wl"][:, 0][None, :]).sum(1) + 1e-3
        out = A.dcn_train_step(p, st, case["off"], bi, bv, bl.astype(np.float64), lr, clip_norm=clip)
        out32 = A.dcn_train_step(p32, st32, case["off"], bi, bv, bl, lr, clip_norm=clip)
        for name, (pv, sv) in variants.items():
            sparse, dense = _VARIANTS[name]
            A.dcn_train_step(pv, sv, case["off"], bi, bv, bl.astype(np.float64), lr, clip_norm=clip, sparse=sparse,
                             dense=dense)
        if clip < 1.0 and step == 0:      # the clip must bind on at least one column's table gradient
            off = list(case["off"]) + [case["N"]]
            r_, G_ = out["rows"], out["G_unclipped"]
            assert max(np.linalg.norm(G_[(r_ >= off[f]) & (r_ < off[f + 1])]) for f in range(F)) > clip
        err = np.abs(got_logits - out["logits"])
        assert np.all(err <= REL * floor + 8 * np.abs(out32["logits"] - out["logits"]).max()), (step, err.max())
        loss = model.train_step(opt, idx, val, y)
        torch.cuda.synchronize()
        assert abs(float(loss) - out["loss"]) <= 1e-5 * abs(out["loss"]) + 8 * abs(float(out32["loss"]) - out["loss"]) + 1e-7

    rejected = dict.fromkeys(_VARIANTS, False)

    def check(got, want64, want32, scale, key, i=None):
        got, want64, want32 = (np.asarray(a, np.float64) for a in (got, want64, want32))
        bound = REL * scale + 8 * np.abs(want32 - want64).max()
        assert np.abs(got - want64).max() <= bound, (key, np.abs(got - want64).max(), bound)
        for name, (pv, _) in variants.items():
            other = pv[key] if i is None else pv[key][i]
            rejected[name] |= bool(np.abs(np.asarray(other) - want64).max() > bound)

    check(model.embedding.table.cpu().numpy(), p["table"], p32["table"], np.abs(p0["table"]).max(), "table")
    check(model.cross.cross_w.detach().cpu().numpy(), p["cross_w"], p32["cross_w"], np.abs(p0["cross_w"]).max(), "cross_w")
    check(model.cross.cross_b.detach().cpu().numpy(), p["cross_b"], p32["cross_b"], np.abs(p0["cross_b"]).max(), "cross_b")
    for i, (lin, w64, w32, b64, b32, ww0) in enumerate(zip(lins, p["W"], p32["W"], p["b"], p32["b"], p0["W"])):
        check(lin.weight.detach().cpu().numpy().T, w64, w32, np.abs(ww0).max(), "W", i)
        check(lin.bias.detach().cpu().numpy(), b64, b32, np.abs(ww0).max(), "b", i)
    check(model.logits.weight.detach().cpu().numpy().T, p["Wl"], p32["Wl"], np.abs(p0["Wl"]).max(), "Wl")
    check(model.logits.bias.detach().cpu().numpy(), p["bl"], p32["bl"], 1.0, "bl")
    assert all(rejected.values()), rejected
    touched = np.zeros(case["N"], bool)
    for bi, bv, _ in batches:
        keep = tfs.keep_mask(bi, bv)
        touched[O.global_rows(np.where(keep, bi, 0), case["off"])[keep]] = True
    assert np.array_equal(model.embedding.table.cpu().numpy()[~touched], case["table"][~touched])
    assert np.array_equal(model.embedding.beta_power.cpu().numpy(), st32["beta_power"])
    assert np.array_equal(opt.beta_power.cpu().numpy(), st32["beta_power"])


def test_storage_beyond_2_31_floats(pkg, cuda):
    """[T | m | v] of 12 M rows at K = 64 is 2.3e9 floats, so every row offset must be 64-bit.  Two steps, each
    checked from the state the kernel started from against a torch fp64 sweep on the device, with the gradient band
    of tests/_util.torch_embedding_reference (REL * Gfloor) pushed through the update as in the layer test."""
    K, B, lr, eps = 64, 4096, 0.01, 1e-4
    rows = [4_000_000, 3_000_000, 5_000_000]
    F, N = len(rows), sum(rows)
    layer = pkg.EmbeddingFM(F, K, rows, optimizer="adam", lr=lr, optimizer_epsilon=eps, first_order=False).train()
    assert layer.rows.numel() > 2 ** 31
    T0 = layer.table.clone()
    gen = torch.Generator(device="cuda").manual_seed(5)
    rows_t = torch.tensor(rows, device="cuda")
    touched = torch.zeros(N, dtype=torch.bool, device="cuda")
    for s in range(2):
        idx = (torch.rand((B, F), device="cuda", generator=gen) * rows_t).long()
        if s == 0:                                           # the last rows of the table: offsets beyond 2^31 floats
            idx[:64, 2] = rows[2] - 1 - torch.arange(64, device="cuda")
        val = torch.rand((B, F), device="cuda", generator=gen) + 0.25
        g_fm = torch.randn(B, device="cuda", generator=gen) * 0.1
        u = torch.randn((B, F * K), device="cuda", generator=gen) * 0.1
        ref = torch_embedding_reference(layer.table.clone(), torch.zeros(N, device="cuda"), 0.0, layer.field_offset,
                                        idx, val, torch.zeros(B, device="cuda"), g_fm, u)
        has = ref["touched"]
        sel = (touched | has).nonzero()[:, 0]                # rows with a nonzero m, v after this step
        before = layer.rows[sel].double()
        p1, p2 = (float(x) for x in layer.beta_power.cpu())
        G, d = ref["G"][sel], REL * ref["Gfloor"][sel]
        del ref
        first, fm, emb = layer(idx, val)
        torch.autograd.backward((fm, emb), (g_fm[:, None], u))
        torch.cuda.synchronize()
        assert int(layer.last_n_unique.item()) == int(has.sum())
        T1, m1, v1, bT, bm, bv = _adam_step_band(before[:, :K], before[:, K:2 * K], before[:, 2 * K:], p1, p2, G, d,
                                                 has[sel], lr, eps)
        got = layer.rows[sel].double()
        assert bool(((got[:, :K] - T1).abs() <= bT).all()), s
        assert bool(((got[:, K:2 * K] - m1).abs() <= bm).all()), s
        assert bool(((got[:, 2 * K:] - v1).abs() <= bv).all()), s
        touched |= has
        del G, d, before, got
    assert bool(touched[N - 64:].all())
    never = (~touched).nonzero()[:, 0]
    assert torch.equal(layer.rows[never, :K], T0[never]) and not bool(layer.rows[never, K:].any())
