"""GPU parity of the row-sharded path.  With one process (world_size 1) every kernel of the device-driven
exchange runs against local buffers -- composite keys, sort, distinct-row numbering, id push, the owner's slot
map, gather + send, forward on the exchanged rows, per-row gradient sums, owner-side merge + update, the
replicated one-row fields -- and must match the oracle like the single-GPU layer does.  With 2 / 4 / 8 GPUs
(skipped otherwise) the ranks each feed their own samples over NVLink peer memory and the union of their
shards must match the oracle run on the concatenated batch."""
import os
import socket

import numpy as np
import pytest
import torch

from oracle import deepctr_oracle as O
from tests._util import REL, make_case, oracle_forward, rel_err, to_dev

pytestmark = pytest.mark.gpu

SHAPES = [(1, [5], 4), (64, [50, 1, 9, 1000, 3, 17, 1], 16), (257, [100] * 26 + [1] * 13, 16),
          (1024, [10_000] * 26 + [1] * 13, 8), (130, [33] * 70, 32), (5000, [3, 1], 16)]


def _layer(pkg, case, optimizer="adagrad", lr=0.05):
    layer = pkg.ShardedEmbeddingFM(case["F"], case["K"], [int(r) for r in case["rows"]], optimizer=optimizer,
                                   lr=lr).train()
    layer.load_tables(case["table"], case["w1"])
    return layer


@pytest.mark.parametrize("B,rows,K", SHAPES)
@pytest.mark.parametrize("optimizer", ["adagrad", "sgd"])
def test_world1_matches_oracle(pkg, cuda, B, rows, K, optimizer):
    case = make_case(31, B, rows, K, weighted=True, prune=True)
    rng, F = case["rng"], case["F"]
    g_first = rng.standard_normal(B).astype(np.float32)
    g_fm = (rng.standard_normal(B) * 0.1).astype(np.float32)
    u = (rng.standard_normal((B, F, K)) * 0.1).astype(np.float32)
    layer = _layer(pkg, case, optimizer)
    first, fm, emb = layer(to_dev(case["idx"]), to_dev(case["val"]))
    e, first_o, fm_o, _ = oracle_forward(case)
    assert np.array_equal(emb.detach().cpu().numpy().reshape(B, F, K), e), "gathered rows must be bit-exact"
    e64, first64, fm64, _ = oracle_forward(case, dtype=np.float64)
    assert rel_err(fm.detach().cpu().numpy(), fm64, 0.5 * (e64 ** 2).sum((1, 2))[:, None] + 1e-30) <= REL
    assert rel_err(first.detach().cpu().numpy(), first64, np.abs(case["w1"]).max() * F + 1e-3) <= REL
    loss = (first[:, 0] * to_dev(g_first)).sum() + (fm[:, 0] * to_dev(g_fm)).sum() + (emb * to_dev(u.reshape(B, -1))).sum()
    loss.backward()
    torch.cuda.synchronize()
    t, w = case["table"].astype(np.float64), case["w1"].astype(np.float64)
    acc, acc1 = np.full_like(t, 0.1), np.full_like(w, 0.1)
    urows, G, g1, _, Gabs, g1abs = O.embedding_backward(t, case["off"], case["idx"], case["val"], g_first, g_fm, u,
                                                        "sum", np.float64, return_abs=True)
    if optimizer == "adagrad":
        O.sparse_adagrad(t, acc, urows, G, 0.05)
        O.sparse_adagrad(w, acc1, urows, g1, 0.05)
    else:
        O.sparse_sgd(t, urows, G, 0.05)
        O.sparse_sgd(w, urows, g1, 0.05)
    got_t, got_w = layer.table.cpu().numpy(), layer.w1.cpu().numpy()
    assert int(layer.last_n_unique.item()) == len(urows)
    untouched = np.ones(case["N"], bool)
    untouched[urows] = False
    assert np.array_equal(got_t[untouched], case["table"][untouched])
    assert rel_err(got_t[urows], t[urows], np.abs(case["table"]).max()) <= REL
    assert rel_err(got_w[urows], w[urows], np.abs(case["w1"]).max() + 1e-3) <= REL
    if optimizer == "adagrad":
        floor = 0.1 + 2 * np.abs(G) * Gabs
        assert rel_err(layer.accum.cpu().numpy()[urows], acc[urows], floor) <= REL
    ex = layer.last_exchange
    keep = (case["idx"] >= 0) & (case["val"] > 0)
    # one-row fields are replicated parameters: they do not travel
    dense_touched = sum(1 for f in range(F) if int(case["rows"][f]) == 1 and keep[:, f].any()) if layer.n_dense else 0
    assert ex["unique_sent"] == len(urows) - dense_touched and ex["lookups"] == B * F
    layer.check_errors()
    # a second step from the updated state (the other exchange buffer; the owner's marks of step 1 were taken back)
    first2, fm2, emb2 = layer(to_dev(case["idx"]), to_dev(case["val"]))
    e2, _ = O.embedding_lookup(got_t, case["off"], case["idx"], case["val"], "sum", np.float32)
    assert np.array_equal(emb2.detach().cpu().numpy().reshape(B, F, K), e2), "step 2 must see step 1's rows"
    (first2.sum() + fm2.sum() + emb2.sum()).backward()
    torch.cuda.synchronize()
    layer.check_errors()
    # the owner's marks are never cleared: they expire with their epoch, and both buffers have been used once
    assert [int(e[0]) for e in layer.slot_epoch] == [1, 1]


@pytest.mark.parametrize("B,rows,K", [(64, [50, 1, 9, 1000, 3, 17, 1], 16), (1024, [10_000] * 26 + [1] * 13, 8)])
@pytest.mark.parametrize("l1,l2", [(0.0, 0.0), (0.002, 0.01)])
def test_world1_proximal_adagrad(pkg, cuda, B, rows, K, l1, l2):
    """ProximalAdagrad (models/ESMM/train.py:137-139) through the sharded layer: the owner's update and the
    replicated one-row fields apply [TF] SparseApplyProximalAdagrad to the de-duplicated sums."""
    case = make_case(37, B, rows, K, weighted=True, prune=True)
    rng, F = case["rng"], case["F"]
    g_first = rng.standard_normal(B).astype(np.float32)
    g_fm = (rng.standard_normal(B) * 0.1).astype(np.float32)
    u = (rng.standard_normal((B, F, K)) * 0.1).astype(np.float32)
    layer = pkg.ShardedEmbeddingFM(F, K, [int(r) for r in rows], optimizer="proximal_adagrad", lr=0.05,
                                   optimizer_l1=l1, optimizer_l2=l2).train()
    layer.load_tables(case["table"], case["w1"])
    first, fm, emb = layer(to_dev(case["idx"]), to_dev(case["val"]))
    loss = (first[:, 0] * to_dev(g_first)).sum() + (fm[:, 0] * to_dev(g_fm)).sum() + (emb * to_dev(u.reshape(B, -1))).sum()
    loss.backward()
    torch.cuda.synchronize()
    layer.check_errors()
    t, w = case["table"].astype(np.float64), case["w1"].astype(np.float64)
    acc, acc1 = np.full_like(t, 0.1), np.full_like(w, 0.1)
    urows, G, g1, _ = O.embedding_backward(t, case["off"], case["idx"], case["val"], g_first, g_fm, u, "sum", np.float64)
    O.sparse_proximal_adagrad(t, acc, urows, G, 0.05, l1, l2)
    O.sparse_proximal_adagrad(w, acc1, urows, g1, 0.05, l1, l2)
    got_t, got_w = layer.table.cpu().numpy(), layer.w1.cpu().numpy()
    untouched = np.ones(case["N"], bool)
    untouched[urows] = False
    assert np.array_equal(got_t[untouched], case["table"][untouched])
    assert rel_err(got_t[urows], t[urows], np.abs(case["table"]).max()) <= REL
    assert rel_err(got_w[urows], w[urows], np.abs(case["w1"]).max() + 1e-3) <= REL
    if l1 > 0:      # the shrinkage really acted on some component
        plain = case["table"].astype(np.float64).copy()
        O.sparse_proximal_adagrad(plain, np.full_like(plain, 0.1), urows, G, 0.05, 0.0, 0.0)
        assert np.abs(plain[urows] - t[urows]).max() > 1e-5


@pytest.mark.parametrize("n,n_rows,G,sel", [(3_000_017, 1_000_003, 4, False), (70_001, 500, 8, False),
                                             (26 * 40_000, 10_000_003, 2, True)])
def test_unique_numbering_against_numpy(pkg, cuda, n, n_rows, G, sel):
    """dir_shard_unique on its own, at sizes where the scan of the tile counts takes several rounds: uidx, the
    distinct local rows, inv and owner_off against numpy on the same sorted list (pruned entries included)."""
    from dir_b200 import _lib
    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    rng = np.random.default_rng(51)
    cap = (n_rows + G - 1) // G
    pruned = cap * G
    rows = rng.integers(0, n_rows, size=n)
    rows[rng.integers(0, n, size=n // 50)] = -1                            # pruned lookups
    keys = np.where(rows >= 0, (rows % G) * cap + rows // G, pruned).astype(np.int64)
    order = np.argsort(keys, kind="stable")
    skeys, spos = keys[order], order.astype(np.int64)
    F, n_sel = (39, 26) if sel else (1, 1)
    fsel = np.r_[0:13, 20:33].astype(np.int32) if sel else None                       # 26 of the 39 fields
    d_k, d_p = to_dev(skeys.astype(np.uint32).view(np.int32)), to_dev(spos.astype(np.uint32).view(np.int32))
    uidx = torch.empty(n, dtype=torch.int32, device="cuda")
    ulocal = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    n_pos = (n // n_sel) * F if sel else n
    inv = torch.full((n_pos,), -5, dtype=torch.int64, device="cuda")
    owner_off = torch.full((G + 1,), -3, dtype=torch.int64, device="cuda")
    ws = torch.empty(max(int(L.dir_shard_unique_workspace_bytes(n)), 1), dtype=torch.uint8, device="cuda")
    d_sel = to_dev(fsel) if sel else None
    _lib.check(L.dir_shard_unique(d_k.data_ptr(), d_p.data_ptr(), n, n_rows, G, d_sel.data_ptr() if sel else None,
                                  n_sel, F, uidx.data_ptr(), ulocal.data_ptr(), inv.data_ptr(), owner_off.data_ptr(),
                                  ws.data_ptr(), ws.numel(), st), "unique")
    torch.cuda.synchronize()
    live = skeys != pruned
    head = live & np.concatenate([[True], skeys[1:] != skeys[:-1]])
    incl = np.cumsum(head)
    want_u = np.where(live, incl - 1, 0)
    assert np.array_equal(uidx.cpu().numpy(), want_u.astype(np.int32))
    U = int(head.sum())
    assert np.array_equal(ulocal.cpu().numpy()[:U], (skeys[head] % cap).astype(np.int32))
    want_off = np.array([int((skeys[head] < g * cap).sum()) for g in range(G + 1)], np.int64)
    assert np.array_equal(owner_off.cpu().numpy(), want_off)
    pos = spos
    if sel:
        b, j = spos // n_sel, spos % n_sel
        pos = b * F + fsel[j]
    want_inv = np.full(n_pos, -5, np.int64)
    want_inv[pos] = np.where(live, incl - 1, -1)
    assert np.array_equal(inv.cpu().numpy(), want_inv)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


CASES = {"small": ([50, 1, 9, 1000, 3, 17, 1], 16, 96),          # at world 8: ceil(n_rows / G) = 136 < distinct rows of a rank
         "wide": ([300, 1, 400, 350, 1, 500], 8, 600)}           # at world 2: ceil(n_rows / G) = 776 < ~1 200 distinct rows


def _rank_main(rank, world, port, out, case_name="small"):
    import torch.distributed as dist
    import dir_b200
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        rows, K, Bl = CASES[case_name]
        case = make_case(41, Bl * world, rows, K, weighted=True, prune=True,
                         skew=2.0 if case_name == "small" else None)                     # global batch
        rng, F = case["rng"], case["F"]
        g_first = rng.standard_normal(Bl * world).astype(np.float32)
        g_fm = (rng.standard_normal(Bl * world) * 0.1).astype(np.float32)
        u = (rng.standard_normal((Bl * world, F, K)) * 0.1).astype(np.float32)
        sl = slice(rank * Bl, (rank + 1) * Bl)
        layer = dir_b200.ShardedEmbeddingFM(F, K, rows, optimizer="adagrad", lr=0.05, max_batch=Bl,
                                            device="cuda").train()
        layer.load_tables(case["table"], case["w1"])
        d = "cuda"
        first, fm, emb = layer(to_dev(case["idx"][sl], d), to_dev(case["val"][sl], d))
        e, first_o, fm_o, _ = oracle_forward(case)
        assert np.array_equal(emb.detach().cpu().numpy().reshape(Bl, F, K), e[sl])
        e64, first64, fm64, _ = oracle_forward(case, dtype=np.float64)
        assert rel_err(fm.detach().cpu().numpy(), fm64[sl], 0.5 * (e64[sl] ** 2).sum((1, 2))[:, None] + 1e-30) <= REL
        loss = ((first[:, 0] * to_dev(g_first[sl], d)).sum() + (fm[:, 0] * to_dev(g_fm[sl], d)).sum()
                + (emb * to_dev(u[sl].reshape(Bl, -1), d)).sum())
        loss.backward()
        torch.cuda.synchronize()
        layer.check_errors()
        shards = [torch.empty_like(layer.rows) for _ in range(world)]
        lins = [torch.empty_like(layer.lin_rows) for _ in range(world)]
        dist.all_gather(shards, layer.rows)
        dist.all_gather(lins, layer.lin_rows)
        if rank == 0:
            N = case["N"]
            full = np.zeros((layer.plan.cap * world, 2 * K), np.float32)
            fw = np.zeros(layer.plan.cap * world, np.float32)
            for r in range(world):
                full[r::world] = shards[r].cpu().numpy()
                fw[r::world] = lins[r].cpu().numpy()[:, 0]
            t, w = case["table"].astype(np.float64), case["w1"].astype(np.float64)
            acc, acc1 = np.full_like(t, 0.1), np.full_like(w, 0.1)
            urows, G, g1, _ = O.embedding_backward(t, case["off"], case["idx"], case["val"], g_first, g_fm, u,
                                                   "sum", np.float64)
            O.sparse_adagrad(t, acc, urows, G, 0.05)
            O.sparse_adagrad(w, acc1, urows, g1, 0.05)
            assert rel_err(full[:N, :K], t, np.abs(case["table"]).max()) <= REL
            assert rel_err(fw[:N], w, np.abs(case["w1"]).max() + 1e-3) <= REL
            untouched = np.ones(N, bool)
            untouched[urows] = False
            assert np.array_equal(full[:N, :K][untouched], case["table"][untouched])
            floor = 0.1 + 2 * np.abs(G) * np.abs(G)
            assert rel_err(full[:N, K:][urows], acc[urows], floor + 1e-3) <= 10 * REL
        if layer.n_dense:
            # every rank's replica of a one-row field equals the owner's row of the sharded table
            for j, g in enumerate(layer.dense_global_rows):
                own = [torch.zeros_like(layer.dense_rows[j]) for _ in range(world)]
                dist.all_gather(own, layer.dense_rows[j].contiguous())
                assert all(torch.equal(own[0], o) for o in own), "replicas diverged"
                if rank == g % world:
                    assert torch.equal(layer.rows[g // world], layer.dense_rows[j])
        # a presorted second step (id phase on the side stream, one batch ahead) from the updated state
        idx2, val2 = to_dev(case["idx"][sl], d), to_dev(case["val"][sl], d)
        h = layer.presort(idx2, val2)
        f2, m2, e2 = layer(idx2, val2, presorted=h)
        (f2.sum() + m2.sum() + e2.sum()).backward()
        torch.cuda.synchronize()
        layer.check_errors()
        if rank == 0:
            e_want, _ = O.embedding_lookup(full[:N, :K], case["off"], case["idx"][sl], case["val"][sl], "sum", np.float32)
            assert np.array_equal(e2.detach().cpu().numpy().reshape(Bl, F, K), e_want), "step 2 must see step 1's rows"
        out.put((rank, "ok"))
    except Exception as ex:
        import traceback
        out.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("case_name", [pytest.param("small", id="peer-small"), pytest.param("wide", id="peer-wide")])
def test_multi_rank_matches_oracle(pkg, cuda, case_name, world):
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs (gpurun --gpus %d)" % (world, world))
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_rank_main, args=(r, world, port, out, case_name)) for r in range(world)]
    for p in procs:
        p.start()
    res = [out.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(r, "ok") for r in range(world)], res


def test_slot_epoch_wraps(pkg, cuda):
    """The owner's marks carry an 8-bit epoch per exchange buffer and are never cleared; after 255 uses of a buffer
    the epoch wraps and the map is zeroed on the device.  530 steps cross the wrap of both buffers: the sharded layer
    must keep following the plain layer step for step (a stale mark read as live would merge a gradient twice)."""
    case = make_case(77, 48, [40, 1, 7, 300, 1], 8, weighted=True, prune=True, skew=2.0)
    a = _layer(pkg, case, "sgd", 0.01)
    b = pkg.EmbeddingFM(case["F"], case["K"], [int(r) for r in case["rows"]], optimizer="sgd", lr=0.01).train()
    b.load_tables(case["table"], case["w1"])
    rng = np.random.default_rng(5)
    idxs = [to_dev(np.stack([rng.integers(0, r, size=48) for r in case["rows"]], 1).astype(np.int64)) for _ in range(7)]
    val = to_dev(case["val"])
    for s in range(530):
        for layer in (a, b):
            first, fm, emb = layer(idxs[s % 7], val)
            (first.sum() + 0.1 * fm.sum() + 0.05 * emb.sum()).backward()
    torch.cuda.synchronize()
    a.check_errors()
    assert all(0 < int(e[0]) < 20 for e in a.slot_epoch), "530 steps = 265 uses per buffer: both epochs have wrapped"
    ta, tb = a.table.cpu().numpy(), b.table.cpu().numpy()
    assert np.abs(ta - tb).max() <= 1e-4 * max(1.0, np.abs(tb).max())
    assert np.abs(a.w1.cpu().numpy() - b.w1.cpu().numpy()).max() <= 1e-4


def _micro_step(layer, idx, val, g_first, g_fm, u, d="cuda"):
    """One batch as two micro-batches: both halves presorted, forward on two streams, backward, ONE owner update."""
    B = idx.shape[0]
    Bh = B // 2
    hs, outs = [], []
    ti, tv = to_dev(idx, d), to_dev(val, d)
    for x in range(2):
        sl = slice(x * Bh, (x + 1) * Bh)
        hs.append(layer.presort(ti[sl], tv[sl], half=x))
    main, sb = torch.cuda.current_stream(), layer.micro_stream(ti.device)
    fa = layer(ti[:Bh], tv[:Bh], presorted=hs[0], defer_update=True)
    sb.wait_event(hs[0].gs_done)
    with torch.cuda.stream(sb):
        fb = layer(ti[Bh:], tv[Bh:], presorted=hs[1], defer_update=True)
    tg1, tg2, tu = to_dev(g_first, d), to_dev(g_fm, d), to_dev(u.reshape(B, -1), d)
    torch.autograd.backward(fa, (tg1[:Bh, None], tg2[:Bh, None], tu[:Bh]))
    with torch.cuda.stream(sb):
        torch.autograd.backward(fb, (tg1[Bh:, None], tg2[Bh:, None], tu[Bh:]))
    main.wait_stream(sb)
    layer.finish_step(hs[0], hs[1])
    torch.cuda.synchronize()
    return torch.cat([fa[2], fb[2]]).detach()


@pytest.mark.parametrize("B,rows,K", [(64, [50, 1, 9, 1000, 3, 17, 1], 16), (1024, [10_000] * 26 + [1] * 13, 8),
                                      (600, [3, 1, 40], 4)])
def test_world1_two_micro_batches(pkg, cuda, B, rows, K):
    """The batch exchanged as two micro-batches (each through an exchange buffer and slot map of its own) and merged by
    ONE owner update: rows that both halves touch must get the summed gradient once (Adagrad: one step per batch)."""
    case = make_case(53, B, rows, K, weighted=True, prune=True, skew=2.0)
    rng, F = case["rng"], case["F"]
    g_first = rng.standard_normal(B).astype(np.float32)
    g_fm = (rng.standard_normal(B) * 0.1).astype(np.float32)
    u = (rng.standard_normal((B, F, K)) * 0.1).astype(np.float32)
    layer = pkg.ShardedEmbeddingFM(F, K, [int(r) for r in rows], optimizer="adagrad", lr=0.05, micro_batches=2).train()
    layer.load_tables(case["table"], case["w1"])
    t, w = case["table"].astype(np.float64), case["w1"].astype(np.float64)
    acc, acc1 = np.full_like(t, 0.1), np.full_like(w, 0.1)
    for step in range(3):                            # three steps: both parities and a re-used buffer
        emb = _micro_step(layer, case["idx"], case["val"], g_first, g_fm, u)
        e, _ = O.embedding_lookup(t.astype(np.float32), case["off"], case["idx"], case["val"], "sum", np.float32)
        if step == 0:
            assert np.array_equal(emb.cpu().numpy().reshape(B, F, K), e), "gathered rows must be bit-exact"
        urows, G, g1, _, Gabs, _ = O.embedding_backward(t, case["off"], case["idx"], case["val"], g_first, g_fm, u,
                                                        "sum", np.float64, return_abs=True)
        O.sparse_adagrad(t, acc, urows, G, 0.05)
        O.sparse_adagrad(w, acc1, urows, g1, 0.05)
        layer.check_errors()
        assert int(layer.last_n_unique.item()) == len(urows)
    got_t, got_w = layer.table.cpu().numpy(), layer.w1.cpu().numpy()
    assert rel_err(got_t, t, np.abs(case["table"]).max()) <= 3 * REL
    assert rel_err(got_w, w, np.abs(case["w1"]).max() + 1e-3) <= 3 * REL
    assert rel_err(layer.accum.cpu().numpy(), acc, 0.1 + np.abs(acc).max()) <= 3 * REL


def _rank_main_micro(rank, world, port, out):
    import torch.distributed as dist
    import dir_b200
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        rows, K, Bl = CASES["wide"]
        case = make_case(43, Bl * world, rows, K, weighted=True, prune=True)
        rng, F = case["rng"], case["F"]
        g_first = rng.standard_normal(Bl * world).astype(np.float32)
        g_fm = (rng.standard_normal(Bl * world) * 0.1).astype(np.float32)
        u = (rng.standard_normal((Bl * world, F, K)) * 0.1).astype(np.float32)
        sl = slice(rank * Bl, (rank + 1) * Bl)
        layer = dir_b200.ShardedEmbeddingFM(F, K, rows, optimizer="adagrad", lr=0.05, max_batch=Bl, micro_batches=2,
                                            device="cuda").train()
        layer.load_tables(case["table"], case["w1"])
        t, w = case["table"].astype(np.float64), case["w1"].astype(np.float64)
        acc, acc1 = np.full_like(t, 0.1), np.full_like(w, 0.1)
        for step in range(2):
            emb = _micro_step(layer, case["idx"][sl], case["val"][sl], g_first[sl], g_fm[sl], u[sl])
            e, _ = O.embedding_lookup(t.astype(np.float32), case["off"], case["idx"], case["val"], "sum", np.float32)
            if step == 0:
                assert np.array_equal(emb.cpu().numpy().reshape(Bl, F, K), e[sl])
            urows, G, g1, _ = O.embedding_backward(t, case["off"], case["idx"], case["val"], g_first, g_fm, u, "sum", np.float64)
            O.sparse_adagrad(t, acc, urows, G, 0.05)
            O.sparse_adagrad(w, acc1, urows, g1, 0.05)
            layer.check_errors()
        shards = [torch.empty_like(layer.rows) for _ in range(world)]
        dist.all_gather(shards, layer.rows)
        if rank == 0:
            N = case["N"]
            full = np.zeros((layer.plan.cap * world, 2 * K), np.float32)
            for r in range(world):
                full[r::world] = shards[r].cpu().numpy()
            assert rel_err(full[:N, :K], t, np.abs(case["table"]).max()) <= 3 * REL
        out.put((rank, "ok"))
    except Exception:
        import traceback
        out.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])
def test_multi_rank_two_micro_batches(pkg, cuda, world):
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs (gpurun --gpus %d)" % (world, world))
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_rank_main_micro, args=(r, world, port, out)) for r in range(world)]
    for p in procs:
        p.start()
    res = [out.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(r, "ok") for r in range(world)], res
