"""TF's Adam on the row-sharded tables (`ShardedEmbeddingFM(optimizer='adam')`, dir_shard_owner_apply_adam,
`DCN(sharded=True, optimizer='adam')`) against oracle/tf_adam.py.  Every step is checked from the state the kernel
started from with test_gpu_adam's band (the oracle's fp64 step, widened by the band of the gradient sums, pushed
through Adam by interval arithmetic); with a clip the gradient and its band are clipped per column first
(test_gpu_backward_widths._clip_center).  At world 1 `EmbeddingFM(optimizer='adam')` is held to the same bands on the
same inputs; with 2 / 4 / 8 GPUs (skipped otherwise) the union of the shards is held to the band of the concatenated
batch, and the ranks must agree bit for bit on the beta powers and the combined clip partials."""
import os
import types

import numpy as np
import pytest
import torch

from oracle import full_models as FM
from oracle import tf_adam as A
from oracle import tf_semantics as tfs
from tests._util import REL, make_case, to_dev, torch_embedding_reference
from tests.test_gpu_adam import B1, B2, _adam_step_band
from tests.test_gpu_backward_widths import (CLIP_LIN, _band, _clip_batch, _clip_center, _field_ids, _lin_rule, _same,
                                            _state, _step, _upstream)
from tests.test_gpu_sharded import SHAPES, _free_port
from tests.test_gpu_sharded_clip import _all_binding_clip

pytestmark = pytest.mark.gpu

LR, EPS = 0.01, 1e-4


def _powers_after(steps):
    bp = A.initial_powers(B1, B2, np.float32)
    for _ in range(steps):
        A.finish(bp, B1, B2)
    return bp


def _targets(ref, layer, clip):
    """(G, d, g1, d1): the oracle's per-row sums and their bands, clipped per column when clip is set."""
    G, d, g1, d1 = ref["G"], REL * ref["Gfloor"], ref["g1"], REL * ref["g1abs"]
    if clip is not None:
        fid, F = _field_ids(layer), layer.field_size
        _, G, d, _, _ = _clip_center(G, d, ref["touched"], fid, F, clip)
        _, g1, d1, _, _ = _clip_center(g1, d1, ref["touched"], fid, F, clip)
    return G, d, g1, d1


def _check_adam_step(layer, before, p1, p2, G, d, g1, d1, touched, lr=LR, eps=EPS):
    """The table (T, m, v of every row) and the first-order weights against the band of one step."""
    K = layer.embedding_size
    st = before["rows"].double()
    T1, m1, v1, bT, bm, bv = _adam_step_band(st[:, :K], st[:, K:2 * K], st[:, 2 * K:3 * K], p1, p2, G, d, touched,
                                             lr, eps)
    got = layer.rows.double()
    out = {"T": int(((got[:, :K] - T1).abs() > bT).sum()), "m": int(((got[:, K:2 * K] - m1).abs() > bm).sum()),
           "v": int(((got[:, 2 * K:3 * K] - v1).abs() > bv).sum())}
    assert int(layer.last_n_unique.item()) == int(touched.sum())
    if layer.first_order:
        kind, llr, l1, l2 = _lin_rule(layer)
        n0 = None if before["n"] is None else before["n"][:, 0].double()
        z0 = None if before["z"] is None else before["z"][:, 0].double()
        (ww, _, _), (bw, _, _) = _band(kind, before["lin"][:, 0].double(), n0, g1, d1, llr, l1, l2, z0)
        out["w1"] = int((((layer.w1.double() - ww).abs() > bw) & touched).sum())
        assert torch.equal(layer.lin_rows[~touched], before["lin"][~touched]), "first-order weights without a gradient"
    return out


def _checked_adam_step(layer, idx, val, g_first, g_fm, u, clip):
    K = layer.embedding_size
    before = _state(layer)
    ref = torch_embedding_reference(before["rows"][:, :K], before["lin"][:, 0], 0.0, layer.field_offset, idx, val,
                                    g_first, g_fm, u)
    G, d, g1, d1 = _targets(ref, layer, clip)
    p1, p2 = (float(x) for x in layer.beta_power.cpu())
    _step(layer, idx, val, g_first, g_fm, u)
    bad = _check_adam_step(layer, before, p1, p2, G, d, g1, d1, ref["touched"])
    assert not any(bad.values()), bad
    return ref["touched"]


@pytest.mark.parametrize("B,rows,K", SHAPES)
@pytest.mark.parametrize("lin", ["none", "adagrad", "ftrl"])
@pytest.mark.parametrize("clipped", [False, True])
def test_world1_three_steps_against_the_band(pkg, cuda, B, rows, K, lin, clipped):
    """Three steps of the sharded layer and of EmbeddingFM(optimizer='adam') on the same inputs, each held to the band
    of the fp64 oracle; rows never touched stay bit-identical with zero moments; beta_power is the fp32 product."""
    F, N = len(rows), sum(rows)
    rng = np.random.default_rng(B + K)
    table = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
    w1 = (rng.standard_normal(N) * 0.1).astype(np.float32)
    kw = dict(optimizer="adam", lr=LR, optimizer_epsilon=EPS, clip_norm=1.0 if clipped else None, **CLIP_LIN[lin])
    sh = pkg.ShardedEmbeddingFM(F, K, rows, max_batch=B, **kw).train()   # (the clip is chosen from the first batch)
    loc = pkg.EmbeddingFM(F, K, rows, **kw).train()
    assert sh.accum is None and sh.adam_m is not None and sh.n_dense == 0
    for layer in (sh, loc):
        layer.load_tables(table, w1)
    touched = torch.zeros(N, dtype=torch.bool, device="cuda")
    clip = None
    for s in range(3):
        idx, val = _clip_batch(rows, B, 7 + B + s)
        g_first, g_fm, u = _upstream(11 + B + s, B, F, K)
        if clipped and clip is None:                    # binds on every live column of the first step
            st = _state(sh)
            ref = torch_embedding_reference(st["rows"][:, :K], st["lin"][:, 0], 0.0, sh.field_offset, idx, val,
                                            g_first, g_fm, u)
            clip = _all_binding_clip(ref, sh, sh.first_order)
            sh.clip_norm = loc.clip_norm = clip
        for layer in (sh, loc):
            t = _checked_adam_step(layer, idx, val, g_first, g_fm, u, clip)
        sh.check_errors()
        touched |= t
    never = ~touched
    assert torch.equal(sh.table[never], torch.as_tensor(table).cuda()[never]) and not bool(sh.rows[never, K:].any())
    bp = _powers_after(3)
    assert np.array_equal(sh.beta_power.cpu().numpy(), bp) and np.array_equal(loc.beta_power.cpu().numpy(), bp)


@pytest.mark.parametrize("B,rows,K", [(64, [50, 1, 9, 1000, 3, 17, 1], 16), (257, [100] * 26 + [1] * 13, 16)])
def test_clip_that_never_binds_is_bit_exact(pkg, cuda, B, rows, K):
    """clip_norm = 2^100 scales every merged sum by 2^100 / 2^100: two steps equal unclipped Adam bit for bit."""
    F = len(rows)
    case = make_case(5, B, rows, K, weighted=True, prune=True)
    kw = dict(optimizer="adam", lr=LR, linear_optimizer="adagrad", linear_lr=0.1, max_batch=B)
    a = pkg.ShardedEmbeddingFM(F, K, rows, clip_norm=2.0 ** 100, **kw).train()
    b = pkg.ShardedEmbeddingFM(F, K, rows, **kw).train()
    for layer in (a, b):
        layer.load_tables(case["table"], case["w1"])
    for s in range(2):
        idx, val = _clip_batch(rows, B, 30 + s)
        g_first, g_fm, u = _upstream(40 + s, B, F, K)
        _step(a, idx, val, g_first, g_fm, u)
        _step(b, idx, val, g_first, g_fm, u)
        assert _same(_state(a), _state(b)), s
        assert torch.equal(a.beta_power, b.beta_power)
        assert int(a.last_n_unique.item()) == int(b.last_n_unique.item())


@pytest.mark.parametrize("clip", [None, 0.05])
def test_graph_replay_equals_eager(pkg, cuda, clip):
    """One step captured into a CUDA graph (norm pass and barrier included when clipping) and replayed twice equals
    two eager steps, bit for bit, beta_power included: the sweep reads the powers on the device."""
    B, rows, K = 257, [100] * 26 + [1] * 13, 16
    F = len(rows)
    case = make_case(9, B, rows, K, weighted=True, prune=True)
    idx, val = _clip_batch(rows, B, 50)
    g_first, g_fm, u = _upstream(51, B, F, K)
    layers = []
    for _ in range(2):
        layer = pkg.ShardedEmbeddingFM(F, K, rows, optimizer="adam", lr=LR, linear_optimizer="ftrl", linear_lr=0.1,
                                       clip_norm=clip, max_batch=B).train()
        layer.load_tables(case["table"], case["w1"])
        for _ in range(2):                              # both parities warmed eagerly
            _step(layer, idx, val, g_first, g_fm, u)
        layers.append(layer)
    eager, graphed = layers
    for _ in range(2):
        _step(eager, idx, val, g_first, g_fm, u)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    graphed.capturing = True
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s, capture_error_mode="thread_local"):
            first, fm, emb = graphed(idx, val)
            torch.autograd.backward((first, fm, emb), (g_first[:, None], g_fm[:, None], u.reshape(B, -1)))
    graphed.capturing = False
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    for _ in range(2):
        graph.replay()
    torch.cuda.synchronize()
    graphed.check_errors()
    assert _same(_state(eager), _state(graphed))
    assert torch.equal(eager.beta_power, graphed.beta_power)
    assert np.array_equal(eager.beta_power.cpu().numpy(), _powers_after(4))
    if clip is not None:
        assert torch.equal(eager.clip_partials, graphed.clip_partials)


def test_fully_pruned_step_still_decays(pkg, cuda):
    """A step in which every lookup is pruned: every row with a nonzero m still moves and decays, the powers still
    advance, no row counts as updated."""
    B, rows, K = 300, [400, 1, 50, 7], 8
    F = len(rows)
    layer = pkg.ShardedEmbeddingFM(F, K, rows, optimizer="adam", lr=LR, optimizer_epsilon=EPS, first_order=False,
                                   max_batch=B).train()
    idx, val = _clip_batch(rows, B, 3)
    g_first, g_fm, u = _upstream(4, B, F, K)
    touched = _checked_adam_step(layer, idx, val, g_first, g_fm, u, None)
    before = _state(layer)
    p1, p2 = (float(x) for x in layer.beta_power.cpu())
    _step(layer, idx, torch.zeros_like(val), g_first, g_fm, u)        # value 0 prunes every lookup
    layer.check_errors()
    N = sum(rows)
    zero = torch.zeros((N, K), dtype=torch.float64, device="cuda")
    none = torch.zeros(N, dtype=torch.bool, device="cuda")
    bad = _check_adam_step(layer, before, p1, p2, zero, zero, None, None, none)
    assert not any(bad.values()), bad
    assert int(layer.last_n_unique.item()) == 0
    assert not torch.equal(layer.table[touched], before["rows"][touched, :K]), "live rows move without a gradient"
    assert torch.equal(layer.rows[~touched], before["rows"][~touched])
    assert np.array_equal(layer.beta_power.cpu().numpy(), _powers_after(2))


def test_storage_beyond_2_31_floats(pkg, cuda):
    """[T | m | v] of 12 M local rows at K = 64 is 2.3e9 floats, so every row offset of the sweep must be 64-bit.
    Two steps, each checked from the state the kernel started from, as test_gpu_adam checks the local layer."""
    K, B, lr, eps = 64, 4096, 0.01, 1e-4
    rows = [4_000_000, 3_000_000, 5_000_000]
    F, N = len(rows), sum(rows)
    layer = pkg.ShardedEmbeddingFM(F, K, rows, optimizer="adam", lr=lr, optimizer_epsilon=eps, first_order=False,
                                   max_batch=B).train()
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
        layer.check_errors()
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


def test_dcn_sharded_adam_clipped_two_steps(pkg, cuda):
    """DCN(sharded=True, optimizer='adam', clip_sharded_tables=True): the reference's full rule (clip per column, Adam
    on the tables, TFAdam on the dense parameters) over two steps against tf_adam.dcn_train_step with a clip that
    binds on the table gradients.  Bound per tensor as in test_gpu_adam.test_dcn_adam_two_steps."""
    from tests.test_gpu_models import ROWS
    B, K, hidden, L, lr, clip = 192, 16, (64, 32), 3, 0.01, 0.05
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
                    optimizer="adam", sharded=True, clip_sharded_tables=True, max_batch=B).train()
    emb = model.embedding
    assert isinstance(emb, pkg.ShardedEmbeddingFM) and emb.optimizer == "adam" and emb.clip_norm == clip
    assert emb.optimizer_epsilon == model.adam_epsilon == A.DCN_EPSILON
    emb.load_tables(case["table"], None)
    lins = list(model.deep.hidden)
    with torch.no_grad():
        for lin, ww, bb in zip(lins, W, b):
            lin.weight.copy_(to_dev(ww.T))
            lin.bias.copy_(to_dev(bb))
        model.cross.cross_w.copy_(to_dev(p32["cross_w"]))
        model.cross.cross_b.copy_(to_dev(p32["cross_b"]))
        model.logits.weight.copy_(to_dev(p32["Wl"].T))
        model.logits.bias.copy_(to_dev(p32["bl"]))
    second = make_case(13, B, ROWS, K, weighted=True, prune=True)
    batches = [(case["idx"], case["val"], labels), (second["idx"], second["val"], (rng.random(B) < 0.3).astype(np.float32))]
    p0 = {k: ([a.copy() for a in v] if isinstance(v, list) else np.copy(v)) for k, v in p.items()}
    st, st32 = A.adam_state(p), A.adam_state(p32)
    opt = model.dense_optimizer()
    assert isinstance(opt, pkg.TFAdam)
    for step, (bi, bv, bl) in enumerate(batches):
        out = A.dcn_train_step(p, st, case["off"], bi, bv, bl.astype(np.float64), lr, clip_norm=clip)
        out32 = A.dcn_train_step(p32, st32, case["off"], bi, bv, bl, lr, clip_norm=clip)
        if step == 0:
            off = list(case["off"]) + [case["N"]]
            r_, G_ = out["rows"], out["G_unclipped"]
            assert max(np.linalg.norm(G_[(r_ >= off[f]) & (r_ < off[f + 1])]) for f in range(F)) > clip
        loss = model.train_step(opt, to_dev(bi), to_dev(bv), to_dev(bl))
        torch.cuda.synchronize()
        emb.check_errors()
        assert abs(float(loss) - out["loss"]) <= 1e-5 * abs(out["loss"]) + 8 * abs(float(out32["loss"]) - out["loss"]) + 1e-7

    def check(got, want64, want32, scale, key):
        got, want64, want32 = (np.asarray(a, np.float64) for a in (got, want64, want32))
        bound = REL * scale + 8 * np.abs(want32 - want64).max()
        assert np.abs(got - want64).max() <= bound, (key, np.abs(got - want64).max(), bound)

    check(emb.table.cpu().numpy()[:case["N"]], p["table"], p32["table"], np.abs(p0["table"]).max(), "table")
    check(model.cross.cross_w.detach().cpu().numpy(), p["cross_w"], p32["cross_w"], np.abs(p0["cross_w"]).max(), "cross_w")
    check(model.cross.cross_b.detach().cpu().numpy(), p["cross_b"], p32["cross_b"], np.abs(p0["cross_b"]).max(), "cross_b")
    for i, (lin, w64, w32, b64, b32, ww0) in enumerate(zip(lins, p["W"], p32["W"], p["b"], p32["b"], p0["W"])):
        check(lin.weight.detach().cpu().numpy().T, w64, w32, np.abs(ww0).max(), "W%d" % i)
        check(lin.bias.detach().cpu().numpy(), b64, b32, np.abs(ww0).max(), "b%d" % i)
    check(model.logits.weight.detach().cpu().numpy().T, p["Wl"], p32["Wl"], np.abs(p0["Wl"]).max(), "Wl")
    assert np.array_equal(emb.beta_power.cpu().numpy(), st32["beta_power"])
    assert np.array_equal(opt.beta_power.cpu().numpy(), st32["beta_power"])


# ---------------------------------------------------------------------------------------------------------------
# several ranks
ROWS_MR, K_MR, BL_MR = [50, 1, 9, 1000, 3, 17, 1, 5], 16, 96


def _union(layer, world, t):
    """[cap * world, ...] of a per-rank tensor: local row l of rank r is global row l * world + r."""
    import torch.distributed as dist
    parts = [torch.empty_like(t) for _ in range(world)]
    dist.all_gather(parts, t.contiguous())
    full = torch.zeros((t.shape[0] * world,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
    for r in range(world):
        full[r::world] = parts[r]
    return full[:sum(ROWS_MR)]


def _adam_run(pkg_mod, rank, world, batches, table, w1, clip, check):
    """Three steps of this rank's slices; with check, each step's union held to the band of the global batch."""
    import torch.distributed as dist
    F, K = len(ROWS_MR), K_MR
    sl = slice(rank * BL_MR, (rank + 1) * BL_MR)
    layer = pkg_mod.ShardedEmbeddingFM(F, K, ROWS_MR, optimizer="adam", lr=LR, optimizer_epsilon=EPS,
                                       linear_optimizer="adagrad", linear_lr=0.1, clip_norm=clip,
                                       max_batch=BL_MR).train()
    layer.load_tables(table, w1)
    off = torch.tensor([0] + list(np.cumsum(ROWS_MR)[:-1]), dtype=torch.int64, device="cuda")
    probe = types.SimpleNamespace(field_rows=torch.tensor(ROWS_MR, device="cuda"), field_size=F)
    for idx, val, (g_first, g_fm, u) in batches:
        if check:
            before = dict(rows=_union(layer, world, layer.rows), lin=_union(layer, world, layer.lin_rows),
                          n=_union(layer, world, layer.lin_acc), z=None)
            ref = torch_embedding_reference(before["rows"][:, :K], before["lin"][:, 0], 0.0, off, idx, val, g_first,
                                            g_fm, u)
            G, d, g1, d1 = _targets(ref, probe, clip)
            p1, p2 = (float(x) for x in layer.beta_power.cpu())
        _step(layer, idx[sl], val[sl], g_first[sl], g_fm[sl], u[sl])
        layer.check_errors()
        if check:
            nu = layer.last_n_unique.clone()
            dist.all_reduce(nu)
            union = types.SimpleNamespace(
                embedding_size=K, rows=_union(layer, world, layer.rows), lin_rows=_union(layer, world, layer.lin_rows),
                first_order=True, linear_optimizer="adagrad", linear_lr=0.1, l1=0.0, l2=0.0, optimizer="adam",
                last_n_unique=nu)
            union.w1 = union.lin_rows[:, 0]
            bad = _check_adam_step(union, before, p1, p2, G, d, g1, d1, ref["touched"])
            assert not any(bad.values()), bad
    return layer


def _adam_rank_main(rank, world, port, out):
    import torch.distributed as dist
    import dir_b200
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        F, K, Bg = len(ROWS_MR), K_MR, BL_MR * world
        rng = np.random.default_rng(61)
        table = (rng.standard_normal((sum(ROWS_MR), K)) / np.sqrt(K)).astype(np.float32)
        w1 = (rng.standard_normal(sum(ROWS_MR)) * 0.1).astype(np.float32)
        batches = []                                     # the global batches, the same on every rank
        for s in range(3):
            idx, val = _clip_batch(ROWS_MR, Bg, 62 + s)
            batches.append((idx, val, _upstream(70 + s, Bg, F, K)))
        T0, W0 = torch.as_tensor(table).cuda(), torch.as_tensor(w1).cuda()
        off = torch.tensor([0] + list(np.cumsum(ROWS_MR)[:-1]), dtype=torch.int64, device="cuda")
        ref = torch_embedding_reference(T0, W0, 0.0, off, batches[0][0], batches[0][1], *batches[0][2])
        probe = types.SimpleNamespace(field_rows=torch.tensor(ROWS_MR, device="cuda"), field_size=F)
        c = torch.tensor([_all_binding_clip(ref, probe, True) if rank == 0 else 0.0], dtype=torch.float32,
                         device="cuda")
        dist.broadcast(c, 0)
        clip = float(c.item())
        layers = [_adam_run(dir_b200, rank, world, batches, table, w1, clip, check) for check in (True, False)]
        layer = layers[0]
        # two runs: bit-identical on the rows this rank owns (a rank with fewer than ceil(N / G) rows pads its shard
        # with a row that is never asked for and keeps each layer's own random initialisation)
        n = layer.plan.n_local
        assert torch.equal(layers[0].rows[:n], layers[1].rows[:n])
        assert torch.equal(layers[0].lin_rows[:n], layers[1].lin_rows[:n])
        assert torch.equal(layers[0].clip_partials, layers[1].clip_partials)
        # every rank holds the same powers and divides by the same combined partials
        for t, what in ((layer.beta_power, "beta_power"), (layer.clip_partials, "clip partials")):
            parts = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(parts, t)
            assert all(torch.equal(parts[0], p) for p in parts), what + " differ between ranks"
        assert np.array_equal(layer.beta_power.cpu().numpy(), _powers_after(3))
        out.put((rank, "ok"))
    except Exception:
        import traceback
        out.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_multi_rank_adam_matches_oracle(pkg, cuda, world):
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_adam_rank_main, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    res = [out.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(r, "ok") for r in range(world)], res
