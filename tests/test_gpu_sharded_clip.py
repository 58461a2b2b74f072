"""tf.clip_by_norm per column on the row-sharded tables (`ShardedEmbeddingFM(clip_norm=...)`,
DeepCrossNetwork.py:282-289): the owner's norm pass over the merged per-row sums, the exchange of the column
partials, the clipped owner update and the clipped one-row replicas.  At world 1 the layer is held to the fp64 oracle
(embedding backward -> per-column clip -> update) with the bands of the local clipped update, and to
`EmbeddingFM(clip_norm=...)`; with 2 / 4 / 8 GPUs (skipped otherwise) the union of the shards is held to the oracle on
the concatenated batch, and the ranks must agree bit for bit on the combined partials and the replicas."""
import os
import types

import numpy as np
import pytest
import torch

from oracle import full_models as FM
from oracle import tf_semantics as tfs
from tests._util import REL, make_case, to_dev, torch_embedding_reference
from tests.test_gpu_backward_widths import (CLIP_LIN, _bag_reference, _choose_clip, _clip_batch, _clip_center,
                                            _clip_check, _field_ids, _reference, _same, _state, _step, _upstream)
from tests.test_gpu_sharded import SHAPES, _free_port

pytestmark = pytest.mark.gpu


def _all_binding_clip(ref, layer, with_g1):
    """A clip (fp32-exact) below every live column's norm band: every column binds (G, and g1 when trained)."""
    fid, F = _field_ids(layer), layer.field_size
    lows = []
    for key, floor in (("G", "Gfloor"), ("g1", "g1abs")) if with_g1 else (("G", "Gfloor"),):
        _, _, _, nrm, dn = _clip_center(ref[key], REL * ref[floor], ref["touched"], fid, F, 1.0)
        live = nrm > 0
        lows.append(float((nrm - dn)[live].min()))
    clip = float(np.float32(0.5 * min(lows)))
    assert clip > 0
    return clip


W1_CASES = [(B, rows, K, mode) for B, rows, K in SHAPES for mode in ("all", "some") if not (mode == "some" and len(rows) < 2)]


@pytest.mark.parametrize("B,rows,K,mode", W1_CASES)
@pytest.mark.parametrize("optimizer", ["adagrad", "sgd"])
@pytest.mark.parametrize("lin", ["same", "adagrad"])
def test_world1_clipped_matches_oracle_and_local(pkg, cuda, B, rows, K, mode, optimizer, lin):
    F = len(rows)
    rng = np.random.default_rng(B + K)
    table = (rng.standard_normal((sum(rows), K)) / np.sqrt(K)).astype(np.float32)
    w1 = (rng.standard_normal(sum(rows)) * 0.1).astype(np.float32)
    kw = dict(optimizer=optimizer, lr=1.0 if optimizer == "sgd" else 0.05, **CLIP_LIN[lin])
    sh = pkg.ShardedEmbeddingFM(F, K, rows, clip_norm=1.0, max_batch=B, **kw).train()
    loc = pkg.EmbeddingFM(F, K, rows, clip_norm=1.0, **kw).train()
    for layer in (sh, loc):
        layer.load_tables(table, w1)
    idx, val = _clip_batch(rows, B, 7 + B)
    scale = torch.tensor([2.0 ** (f % 4) for f in range(F)], device="cuda")
    g_first, g_fm, u = _upstream(11 + B, B, F, K, scale)
    before = _state(sh)
    ref = _reference(sh, before, idx, val, g_first, g_fm, u)
    if mode == "all":
        clip = _all_binding_clip(ref, sh, True)
    else:
        clip = _choose_clip(ref, sh)
        fid = _field_ids(sh)
        _, _, _, n1, _ = _clip_center(ref["g1"], REL * ref["g1abs"], ref["touched"], fid, F, 1.0)
        g_first = g_first * float(np.float32(4 * clip / float(n1[n1 > 0].median())))     # some g1 columns bind too
        ref = _reference(sh, before, idx, val, g_first, g_fm, u)
    sh.clip_norm = loc.clip_norm = clip
    _step(sh, idx, val, g_first, g_fm, u)
    sh.check_errors()
    bad = _clip_check(sh, before, ref, clip)
    assert not any(bad.values()), bad
    _step(loc, idx, val, g_first, g_fm, u)
    bad = _clip_check(loc, before, ref, clip)
    assert not any(bad.values()), bad
    # the two layers agree to the fp32 rounding of the same clipped step
    touched = ref["touched"]
    assert torch.allclose(sh.rows[touched], loc.rows[touched], rtol=1e-5, atol=1e-6)
    assert torch.allclose(sh.lin_rows[touched], loc.lin_rows[touched], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("B,rows,K", [(64, [50, 1, 9, 1000, 3, 17, 1], 16), (257, [100] * 26 + [1] * 13, 16)])
@pytest.mark.parametrize("optimizer", ["adagrad", "sgd"])
def test_clip_that_never_binds_is_bit_exact(pkg, cuda, B, rows, K, optimizer):
    """clip_norm = 2^100 scales every sum by 2^100 / 2^100: two steps equal the unclipped sharded layer bit for bit."""
    F = len(rows)
    case = make_case(5, B, rows, K, weighted=True, prune=True)
    a = pkg.ShardedEmbeddingFM(F, K, rows, optimizer=optimizer, lr=0.05, clip_norm=2.0 ** 100, max_batch=B).train()
    b = pkg.ShardedEmbeddingFM(F, K, rows, optimizer=optimizer, lr=0.05, max_batch=B).train()
    for layer in (a, b):
        layer.load_tables(case["table"], case["w1"])
    for s in range(2):
        idx, val = _clip_batch(rows, B, 30 + s)
        g_first, g_fm, u = _upstream(40 + s, B, F, K)
        _step(a, idx, val, g_first, g_fm, u)
        _step(b, idx, val, g_first, g_fm, u)
        assert _same(_state(a), _state(b)), s
        assert torch.equal(a.dense_rows, b.dense_rows)
        assert int(a.last_n_unique.item()) == int(b.last_n_unique.item())


def test_graph_replay_equals_eager(pkg, cuda):
    """One clipped step captured into a CUDA graph (norm pass, norm barrier, clipped update and replicas included)
    and replayed equals the same step run eagerly, bit for bit."""
    B, rows, K = 257, [100] * 26 + [1] * 13, 16
    F = len(rows)
    case = make_case(9, B, rows, K, weighted=True, prune=True)
    idx, val = _clip_batch(rows, B, 50)
    g_first, g_fm, u = _upstream(51, B, F, K)
    layers = []
    for _ in range(2):
        layer = pkg.ShardedEmbeddingFM(F, K, rows, lr=0.05, clip_norm=0.05, max_batch=B).train()
        layer.load_tables(case["table"], case["w1"])
        for _ in range(2):                              # both parities warmed eagerly
            _step(layer, idx, val, g_first, g_fm, u)
        layers.append(layer)
    eager, graphed = layers
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
    graph.replay()
    torch.cuda.synchronize()
    graphed.check_errors()
    assert _same(_state(eager), _state(graphed))
    assert torch.equal(eager.dense_rows, graphed.dense_rows)
    assert torch.equal(eager.clip_partials, graphed.clip_partials)


def test_bags_world1_clipped(pkg, cuda):
    """ShardedEmbeddingBagFM(clip_norm=...) (combiner 'sum') against the fp64 bag reference, clipped per column."""
    B, rows, K = 300, [400, 1, 50, 7], 8
    F = len(rows)
    gen = torch.Generator(device="cuda").manual_seed(3)
    cnt = torch.randint(0, 4, (B * F,), device="cuda", generator=gen)
    off = torch.cat([torch.zeros(1, dtype=torch.int64, device="cuda"), cnt.cumsum(0)])
    slot = torch.repeat_interleave(torch.arange(B * F, device="cuda"), cnt)
    hi = torch.tensor(rows, device="cuda")[slot % F]
    bag_idx = (torch.rand(slot.numel(), device="cuda", generator=gen) * hi).long()
    bag_w = torch.rand(slot.numel(), device="cuda", generator=gen) + 0.25
    rng = np.random.default_rng(3)
    table = (rng.standard_normal((sum(rows), K)) / np.sqrt(K)).astype(np.float32)
    w1 = (rng.standard_normal(sum(rows)) * 0.1).astype(np.float32)
    layer = pkg.ShardedEmbeddingBagFM(F, K, rows, combiner="sum", lr=0.05, clip_norm=1.0, max_batch=B,
                                      max_entries=int(slot.numel())).train()
    layer.load_tables(table, w1)
    g_first, g_fm, u = _upstream(4, B, F, K)
    before = _state(layer)
    ref = _bag_reference(before["rows"][:, :K], before["lin"][:, 0], layer.field_offset, off, bag_idx, bag_w, B, F,
                         g_first, g_fm, u)
    clip = _choose_clip(ref, layer)
    layer.clip_norm = clip
    first, fm, emb = layer.forward_bags(off, bag_idx, bag_w)
    torch.autograd.backward((first, fm, emb), (g_first[:, None], g_fm[:, None], u.reshape(B, -1)))
    torch.cuda.synchronize()
    layer.check_errors()
    bad = _clip_check(layer, before, ref, clip)
    assert not any(bad.values()), bad


def test_dcn_sharded_clipped_one_step(pkg, cuda):
    """DCN(sharded=True, clip_sharded_tables=True): one step against full_models.dcn_train_step(clip_tables=True) with
    a clip that binds on the table gradients."""
    from tests.test_gpu_models import ROWS, _copy, _load_tower, _tower_err
    from tests._util import rel_err
    B, K, hidden, L, lr, clip = 192, 16, (64, 32), 3, 0.05, 0.05
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
                    sharded=True, clip_sharded_tables=True, max_batch=B).train()
    assert model.embedding.clip_norm == clip
    model.embedding.load_tables(case["table"], None)
    _load_tower(model.deep, W, b, False)
    with torch.no_grad():
        model.cross.cross_w.copy_(to_dev(p32["cross_w"]))
        model.cross.cross_b.copy_(to_dev(p32["cross_b"]))
        model.logits.weight.copy_(to_dev(p32["Wl"].T))
        model.logits.bias.copy_(to_dev(p32["bl"]))
    p0, st = _copy(p), FM.adagrad_state(p)
    out = FM.dcn_train_step(p, st, case["off"], case["idx"], case["val"], labels.astype(np.float64), lr,
                            clip_norm=clip, clip_tables=True)
    off = list(case["off"]) + [case["N"]]
    norms = [np.linalg.norm(out["G_unclipped"][(out["rows"] >= off[f]) & (out["rows"] < off[f + 1])]) for f in range(F)]
    assert max(norms) > clip, "clip too loose for this test to mean anything"
    loss = model.train_step(model.dense_optimizer(), to_dev(case["idx"]), to_dev(case["val"]), to_dev(labels))
    torch.cuda.synchronize()
    assert abs(float(loss) - out["loss"]) <= 1e-5 * abs(out["loss"]) + 1e-7
    assert rel_err(model.embedding.table.cpu().numpy(), p["table"], np.abs(p0["table"]).max()) <= REL
    assert rel_err(model.cross.cross_w.detach().cpu().numpy(), p["cross_w"], np.abs(p0["cross_w"]).max()) <= REL
    assert _tower_err(model.deep, p["W"], p["b"], p0["W"], False) <= REL


# ---------------------------------------------------------------------------------------------------------------
# several ranks
ROWS_MR, K_MR, BL_MR = [50, 1, 9, 1000, 3, 17, 1, 5], 16, 96


def _run_rank(pkg_mod, rank, world, idx_all, val_all, up, table, w1, clip):
    """One clipped step of this rank's slice; returns the layer."""
    g_first, g_fm, u = up
    sl = slice(rank * BL_MR, (rank + 1) * BL_MR)
    F = len(ROWS_MR)
    layer = pkg_mod.ShardedEmbeddingFM(F, K_MR, ROWS_MR, lr=0.05, clip_norm=clip, max_batch=BL_MR).train()
    layer.load_tables(table, w1)
    _step(layer, idx_all[sl], val_all[sl], g_first[sl], g_fm[sl], u[sl])
    layer.check_errors()
    return layer


def _clip_rank_main(rank, world, port, out):
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
        idx, val = _clip_batch(ROWS_MR, Bg, 62)                          # the global batch, the same on every rank
        up = _upstream(63, Bg, F, K)
        T0 = torch.as_tensor(table).cuda()
        W0 = torch.as_tensor(w1).cuda()
        off = torch.tensor([0] + list(np.cumsum(ROWS_MR)[:-1]), dtype=torch.int64, device="cuda")
        ref = torch_embedding_reference(T0, W0, 0.0, off, idx, val, *up)
        probe = types.SimpleNamespace(field_rows=torch.tensor(ROWS_MR, device="cuda"), field_size=F)
        c = torch.tensor([_choose_clip(ref, probe) if rank == 0 else 0.0], dtype=torch.float32, device="cuda")
        dist.broadcast(c, 0)
        clip = float(c.item())
        layers = [_run_rank(dir_b200, rank, world, idx, val, up, table, w1, clip) for _ in range(2)]
        layer = layers[0]
        # two runs: bit-identical on the rows this rank owns (a rank with fewer than ceil(N / G) rows pads its shard
        # with a row that is never asked for and keeps each layer's own random initialisation)
        n = layer.plan.n_local
        assert torch.equal(layers[0].rows[:n], layers[1].rows[:n])
        assert torch.equal(layers[0].lin_rows[:n], layers[1].lin_rows[:n])
        assert torch.equal(layers[0].clip_partials, layers[1].clip_partials)
        # every rank divides by the same combined partials
        parts = [torch.empty_like(layer.clip_partials) for _ in range(world)]
        dist.all_gather(parts, layer.clip_partials)
        assert all(torch.equal(parts[0], p) for p in parts), "combined partials differ between ranks"
        # replicas equal on every rank and mirror the owner's row
        for j, g in enumerate(layer.dense_global_rows):
            own = [torch.zeros_like(layer.dense_rows[j]) for _ in range(world)]
            dist.all_gather(own, layer.dense_rows[j].contiguous())
            assert all(torch.equal(own[0], o) for o in own), "replicas diverged"
            if rank == g % world:
                assert torch.equal(layer.rows[g // world], layer.dense_rows[j])
        # the union of the shards against the oracle on the concatenated batch
        shards = [torch.empty_like(layer.rows) for _ in range(world)]
        lins = [torch.empty_like(layer.lin_rows) for _ in range(world)]
        accs = [torch.empty_like(layer.lin_acc) for _ in range(world)]
        dist.all_gather(shards, layer.rows)
        dist.all_gather(lins, layer.lin_rows)
        dist.all_gather(accs, layer.lin_acc)
        nu = layer.last_n_unique.clone()
        dist.all_reduce(nu)
        N = sum(ROWS_MR)
        cap = layer.plan.cap
        full = torch.zeros((cap * world, 2 * K), device="cuda")
        fw = torch.zeros((cap * world, 1), device="cuda")
        fa = torch.zeros((cap * world, 1), device="cuda")
        for r in range(world):
            full[r::world], fw[r::world], fa[r::world] = shards[r], lins[r], accs[r]
        before = dict(rows=torch.cat([T0, torch.full_like(T0, 0.1)], 1), lin=W0[:, None].clone(),
                      n=torch.full_like(W0[:, None], 0.1), z=None)
        union = types.SimpleNamespace(
            embedding_size=K, optimizer="adagrad", lr=0.05, optimizer_l1=0.0, optimizer_l2=0.0, linear_optimizer=None,
            field_rows=probe.field_rows, field_size=F, rows=full[:N], accum=full[:N, K:], lin_rows=fw[:N],
            lin_acc=fa[:N], lin_z=None, w1=fw[:N, 0], w1_accum=fa[:N, 0], first_order=True, last_n_unique=nu)
        bad = _clip_check(union, before, ref, clip)
        assert not any(bad.values()), bad
        out.put((rank, "ok"))
    except Exception:
        import traceback
        out.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4, 8])
def test_multi_rank_clipped_matches_oracle(pkg, cuda, world):
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_clip_rank_main, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    res = [out.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(r, "ok") for r in range(world)], res


def test_requester_segments_ascend_on_device(pkg, cuda):
    """The norm pass finds a column's arrivals with lower_bound: after the id phase each owner's segment of the
    distinct local rows is strictly ascending (fields, G = 3 keys, pruned lookups)."""
    from dir_b200 import _lib
    from dir_b200.sharded import ShardedLookups
    rows, K, B = [50, 1, 9, 1000, 3, 17, 1], 16, 500
    layer = pkg.ShardedEmbeddingFM(len(rows), K, rows, max_batch=B)
    idx, val = _clip_batch(rows, B, 70)
    for G in (1, 3, 8):
        layer.plan.world_size = G                       # keys for G owners; nothing is exchanged
        h = ShardedLookups()
        layer.plan.cap = -(-sum(rows) // G)
        layer.id_local(h, idx, val)
        torch.cuda.synchronize()
        o = h.owner_off.cpu().numpy()
        ul = h.ulocal.cpu().numpy()
        for q in range(G):
            seg = ul[o[q]:o[q + 1]]
            assert np.all(np.diff(seg) > 0), (G, q)
            assert np.all(seg * G + q < sum(rows))
