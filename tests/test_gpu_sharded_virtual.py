"""The row-sharded layer with G ranks on ONE GPU: G threads of one process, each rank on a stream of its own, their
exchange buffers on the same device (tests/_virtual_world.py).  The exchange kernels reach their peers only through
the rank-ordered address array, so every code path that needs G > 1 runs here -- the leader rule and the rank-order
merge over requesters, the slot cells of requesters >= 8, bits 32-63 of the `more` mask, the norm partials stored
into every rank, Adam's per-tile leader map -- at any G up to the ABI's 64.  NVLink and the device-side barrier of
symmetric memory are not exercised: the multi-process tests (test_multi_rank_*) remain the only check of those.

a. The multi-rank bodies of test_gpu_sharded / _bags / _clip / _adam, imported and run unchanged.
b. Checks that need every rank's state at hand, which one process has without a collective:
   - the exchange buffers after an Adagrad step, against numpy on the same ids: headers, id segments (strictly
     ascending), slot cells (exactly the segment's rows carry the current epoch), the rows and first-order weights
     each requester received (bit for bit), the gradient sums it stored at each owner (within the fp64 band);
   - forward invariance: every rank's outputs bit-identical to a world-1 layer's on the same slice;
   - determinism: two fresh worlds end bit-identical;
   - a table with fewer rows than ranks: ranks that own nothing still request (Adagrad, a binding clip, Adam)."""
import traceback
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist

import dir_b200
from tests import test_gpu_sharded as TS
from tests import test_gpu_sharded_adam as TA
from tests import test_gpu_sharded_bags as TB
from tests import test_gpu_sharded_clip as TC
from tests._util import REL, make_case, to_dev, torch_embedding_reference
from tests._virtual_world import run_world
from tests.test_gpu_backward_widths import _clip_batch, _clip_check, _state, _step, _upstream, _violations

pytestmark = pytest.mark.gpu


def _all_ok(res, G):
    bad = [(r, v) for r, v in res if v != "ok"]
    assert not bad, "\n".join("rank %d:\n%s" % b for b in bad)
    assert [r for r, _ in res] == list(range(G))


def _payloads(res, G):
    bad = [(r, v) for r, v in res if isinstance(v, str)]
    assert not bad, "\n".join("rank %d:\n%s" % b for b in bad)
    assert [r for r, _ in res] == list(range(G))
    return [v for _, v in res]


# ---------------------------------------------------------------------------------------------------------------
# a. the multi-rank bodies, unchanged

@pytest.mark.parametrize("G", [2, 3, 4, 8, 12, 64])
def test_rank_main_small(pkg, cuda, G):
    _all_ok(run_world(G, TS._rank_main, "small"), G)


@pytest.mark.parametrize("G", [2, 3, 8, 12])
def test_rank_main_wide(pkg, cuda, G):
    _all_ok(run_world(G, TS._rank_main, "wide"), G)


@pytest.mark.parametrize("G", [2, 3, 17, 32])
def test_rank_main_two_micro_batches(pkg, cuda, G):
    """Half s of rank q is virtual requester s * G + q: from G = 17 the second halves use bits >= 32 of `more`;
    32 is the layer's limit for two micro-batches."""
    _all_ok(run_world(G, TS._rank_main_micro), G)


@pytest.mark.parametrize("G", [2, 3, 8])
@pytest.mark.parametrize("combiner", ["sum", "mean"])
def test_bags_rank_main(pkg, cuda, combiner, G):
    _all_ok(run_world(G, TB._rank_main, combiner), G)


@pytest.mark.parametrize("G", [2, 3, 8, 12])
def test_clip_rank_main(pkg, cuda, G):
    _all_ok(run_world(G, TC._clip_rank_main), G)


@pytest.mark.parametrize("G", [2, 3, 8, 12])
def test_adam_rank_main(pkg, cuda, G):
    _all_ok(run_world(G, TA._adam_rank_main), G)


# ---------------------------------------------------------------------------------------------------------------
# b. checks across every rank's state
ROWS, K, BL = TS.CASES["small"]                  # two one-row fields (replicated), skewed ids: hot rows of every rank
F, N = len(ROWS), sum(ROWS)
OFF = np.concatenate([[0], np.cumsum(ROWS)[:-1]]).astype(np.int64)
STEPS = 3                                        # the last step reuses buffer 0: its slot map holds step 1's cells


def _batch(seed, Bg):
    case = make_case(seed, Bg, ROWS, K, weighted=True, prune=True, skew=2.0)
    rng = case["rng"]
    g_first = rng.standard_normal(Bg).astype(np.float32)
    g_fm = (rng.standard_normal(Bg) * 0.1).astype(np.float32)
    u = (rng.standard_normal((Bg, F, K)) * 0.1).astype(np.float32)
    return case, g_first, g_fm, u


def _adagrad_body(rank, world, port, out):
    """STEPS Adagrad steps of this rank's slices (a new batch each step) -> the layer, its state before the last step
    and its outputs of the first forward."""
    dist.init_process_group("nccl", rank=rank, world_size=world)
    try:
        sl = slice(rank * BL, (rank + 1) * BL)
        batches = [_batch(41 + s, BL * world) for s in range(STEPS)]
        layer = dir_b200.ShardedEmbeddingFM(F, K, ROWS, optimizer="adagrad", lr=0.05, max_batch=BL).train()
        layer.load_tables(batches[0][0]["table"], batches[0][0]["w1"])
        fwd = before = None
        for s, (case, g_first, g_fm, u) in enumerate(batches):
            before = _state(layer)
            first, fm, emb = layer(to_dev(case["idx"][sl]), to_dev(case["val"][sl]))
            if s == 0:
                fwd = [t.detach().clone() for t in (first, fm, emb)]
            torch.autograd.backward((first, fm, emb), (to_dev(g_first[sl])[:, None], to_dev(g_fm[sl])[:, None],
                                                       to_dev(u[sl].reshape(BL, -1))))
            torch.cuda.synchronize()
            layer.check_errors()
        out.put((rank, dict(layer=layer, before=before, fwd=fwd)))
    except Exception:
        out.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


def _unite(parts, G):
    """[cap * G, ...] from the G ranks' [cap, ...]: local row l of rank r is global row l * G + r."""
    full = torch.zeros((parts[0].shape[0] * G,) + tuple(parts[0].shape[1:]), dtype=parts[0].dtype,
                       device=parts[0].device)
    for r, t in enumerate(parts):
        full[r::G] = t
    return full


def _buffer(layer, p):
    """Exchange buffer p of a rank as numpy views, by the offsets of its dir_peer_layout."""
    lay = layer.px.layouts[p]
    b = layer.px.bufs[p].cpu().numpy()
    G, sc, n = lay.G, lay.seg_cap, lay.u_cap + lay.n_dense

    def v(off, dt, cnt):
        return b[off: off + cnt * np.dtype(dt).itemsize].view(dt)
    return dict(hdr=v(lay.off_hdr, np.int64, 4 * G).reshape(G, 4), ids=v(lay.off_ids, np.int32, G * sc).reshape(G, sc),
                rows=v(lay.off_rows, np.float32, n * lay.K).reshape(n, lay.K), w=v(lay.off_w, np.float32, n),
                g=v(lay.off_g, np.float32, G * sc * lay.K).reshape(G, sc, lay.K),
                g1=v(lay.off_g1, np.float32, G * sc).reshape(G, sc))


def _check_exchange(pls, G, mutate=None):
    """The last step's exchange buffers against numpy on the same ids (the rules tests/test_sharded_cpu.py restates).
    mutate(bufs, slots, epochs) edits the host copies first (negative controls)."""
    layers = [p["layer"] for p in pls]
    p = layers[0]._last_handle.buf
    assert all(l._last_handle.buf == p for l in layers) and p == 0
    case, g_first, g_fm, u = _batch(41 + STEPS - 1, BL * G)
    T = _unite([pl["before"]["rows"][:, :K] for pl in pls], G)[:N]          # the table the step started from
    W = _unite([pl["before"]["lin"][:, 0] for pl in pls], G)[:N]
    Tn, Wn = T.cpu().numpy(), W.cpu().numpy()
    bufs = [_buffer(l, p) for l in layers]
    slots = [l.slot[p].cpu().numpy().view(np.uint32).reshape(-1, G) for l in layers]
    epochs = [int(l.slot_epoch[p][0]) for l in layers]
    assert epochs == [2] * G, "buffer 0 is in its second use"
    if mutate is not None:
        mutate(bufs, slots, epochs)
    sparse = np.array([r != 1 for r in ROWS])                               # one-row fields do not travel
    fo = torch.tensor(OFF, device="cuda")
    stale = 0
    for q in range(G):
        sl = slice(q * BL, (q + 1) * BL)
        idx, val = case["idx"][sl], case["val"][sl]
        keep = (idx >= 0) & (val > 0) & sparse[None, :]
        grows = np.unique((idx + OFF[None, :])[keep])                       # q's distinct rows, ascending
        ref = torch_embedding_reference(T, W, 0.0, fo, to_dev(idx), to_dev(val), to_dev(g_first[sl]),
                                        to_dev(g_fm[sl]), to_dev(u[sl]))
        Gr, Gf = ref["G"].cpu().numpy(), ref["Gfloor"].cpu().numpy()
        g1r, g1f = ref["g1"].cpu().numpy(), ref["g1abs"].cpu().numpy()
        for o in range(G):
            mine = grows[grows % G == o]
            seg, cnt, base = mine // G, len(mine), int((grows % G < o).sum())
            b = bufs[o]
            where = "owner %d, requester %d" % (o, q)
            assert b["hdr"][q, 0] == cnt and b["hdr"][q, 1] == base, where
            got = b["ids"][q, :cnt]
            assert np.all(np.diff(got.astype(np.int64)) > 0), "segment not strictly ascending: " + where
            assert np.array_equal(got, seg), where
            col = slots[o][:, q]
            live = np.nonzero((col >> 24) == epochs[o])[0]
            assert np.array_equal(live, seg), "cells with the current epoch != the segment: " + where
            assert np.array_equal(col[seg], (epochs[o] << 24) | (np.arange(cnt) + 1)), where
            stale += int(((col >> 24) != 0).sum()) - cnt
            # what q received from o: bit-exact copies of the table's rows
            assert np.array_equal(bufs[q]["rows"][base: base + cnt], Tn[mine]), "rows: " + where
            assert np.array_equal(bufs[q]["w"][base: base + cnt], Wn[mine]), "first-order weights: " + where
            # what q stored at o: its per-distinct-row sums on its own slice
            assert np.all(np.abs(b["g"][q, :cnt] - Gr[mine]) <= REL * Gf[mine]), "g: " + where
            assert np.all(np.abs(b["g1"][q, :cnt] - g1r[mine]) <= REL * g1f[mine]), "g1: " + where
    assert stale > 0, "some cells of step 1 are left with the old epoch: the epoch check is exercised"


def _swap_ids(bufs, slots, epochs):
    """two ids of a segment out of order"""
    o, q = next((o, q) for o, b in enumerate(bufs) for q in range(len(b["hdr"])) if b["hdr"][q, 0] >= 2)
    bufs[o]["ids"][q, [0, 1]] = bufs[o]["ids"][q, [1, 0]]


def _stale_cell(bufs, slots, epochs):
    """a cell of a row requester 0 did not ask for this time that carries the current epoch anyway (what an owner that
    ignored the epoch would read from a stale cell)"""
    col = slots[0][:, 0]
    r = int(np.nonzero((col >> 24) != epochs[0])[0][0])
    col[r] = (epochs[0] << 24) | 1


def _nudge_g(bufs, slots, epochs):
    """one component of one stored gradient sum off by 1e-3 of the sum's largest component"""
    o, q = next((o, q) for o, b in enumerate(bufs) for q in range(len(b["hdr"])) if b["hdr"][q, 0] >= 1)
    g = bufs[o]["g"][q, 0]
    g[0] += np.float32(1e-3 * max(float(np.abs(g).max()), 1e-2))


@pytest.mark.parametrize("G", [2, 3, 8, 12, 64])
def test_exchange_buffers_and_forward(pkg, cuda, G):
    """After STEPS Adagrad steps: every owner's headers, id segments and slot map, every requester's received rows and
    stored gradient sums against numpy (catches unsorted segments, a cell written without the epoch or for the wrong
    arrival, a row sent to the wrong place, a sum stored in another requester's segment).  And every rank's first
    forward bit-identical to a world-1 layer's on the same slice and table: the same kernel over the same row values in
    the same field order, whatever the exchange did in between."""
    pls = _payloads(run_world(G, _adagrad_body), G)
    assert all(int(pl["layer"].err_flag.item()) == 0 for pl in pls)
    _check_exchange(pls, G)
    if G == 3:      # the check rejects each of these edits
        for mutate, what in ((_swap_ids, "ascending"), (_stale_cell, "current epoch"), (_nudge_g, "g: ")):
            with pytest.raises(AssertionError, match=what):
                _check_exchange(pls, G, mutate)
    case = _batch(41, BL * G)[0]
    for r, pl in enumerate(pls):
        one = pkg.ShardedEmbeddingFM(F, K, ROWS, optimizer="adagrad", lr=0.05, max_batch=BL).train()
        one.load_tables(case["table"], case["w1"])
        sl = slice(r * BL, (r + 1) * BL)
        want = one(to_dev(case["idx"][sl]), to_dev(case["val"][sl]))
        for name, a, b in zip(("first", "fm", "emb"), pl["fwd"], want):
            assert torch.equal(a, b.detach()), "rank %d: %s differs from world 1" % (r, name)


def test_two_worlds_are_bit_identical(pkg, cuda):
    """The same STEPS steps in two fresh worlds of 8 ranks, each rank on its own stream: the union of the shards
    (rows and accumulators), the first-order weights and the summed last_n_unique agree bit for bit.  Hot rows are
    asked for by every rank, so a merge whose order followed arrival timing (a float atomic) would show here."""
    runs = []
    for _ in range(2):
        pls = _payloads(run_world(8, _adagrad_body), 8)
        runs.append((_unite([pl["layer"].rows for pl in pls], 8), _unite([pl["layer"].lin_rows for pl in pls], 8),
                     sum(int(pl["layer"].last_n_unique.item()) for pl in pls)))
    (ra, la, na), (rb, lb, nb) = runs
    # (rows past N pad the shards of ranks with fewer than ceil(N / G) rows: each layer's own random initialisation)
    assert torch.equal(ra[:N], rb[:N]) and torch.equal(la[:N], lb[:N]) and na == nb
    assert not torch.equal(ra[:N, :K], torch.as_tensor(_batch(41, BL * 8)[0]["table"]).cuda()), "the steps moved rows"


# fewer rows than ranks: at G = 8, ranks 6 and 7 own no row (each allocates one padding row) and still request
ROWS0, K0, BL0, G0 = [3, 1, 2], 8, 24, 8
LR, EPS = TA.LR, TA.EPS
MODES = {"adagrad": dict(optimizer="adagrad", lr=0.05), "clip": dict(optimizer="adagrad", lr=0.05),
         "adam": dict(optimizer="adam", lr=LR, optimizer_epsilon=EPS, linear_optimizer="adagrad", linear_lr=0.1)}


def _sparse_body(rank, world, port, out, mode, table, w1, idx, val, up, clip):
    dist.init_process_group("nccl", rank=rank, world_size=world)
    try:
        sl = slice(rank * BL0, (rank + 1) * BL0)
        layer = dir_b200.ShardedEmbeddingFM(len(ROWS0), K0, ROWS0, max_batch=BL0, clip_norm=clip,
                                            **MODES[mode]).train()
        layer.load_tables(table, w1)
        before = _state(layer)
        bp = None if layer.beta_power is None else [float(x) for x in layer.beta_power.cpu()]
        g_first, g_fm, u = up
        _step(layer, idx[sl], val[sl], g_first[sl], g_fm[sl], u[sl])
        layer.check_errors()
        out.put((rank, dict(layer=layer, before=before, bp=bp)))
    except Exception:
        out.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("mode", ["adagrad", "clip", "adam"])
def test_ranks_that_own_nothing(pkg, cuda, mode):
    """rows = [3, 1, 2] at G = 8: one Adagrad step, one with a clip that binds on every column, one Adam step (the
    owners sweep their shards, the two empty ranks their padding row).  The union of the shards is held to the helpers
    the multi-rank bodies use; err_flag is clean, the padding rows do not move, and the ranks agree bit for bit on the
    combined clip partials and the beta powers."""
    G, F0, N0 = G0, len(ROWS0), sum(ROWS0)
    rng = np.random.default_rng(71)
    table = (rng.standard_normal((N0, K0)) / np.sqrt(K0)).astype(np.float32)
    w1 = (rng.standard_normal(N0) * 0.1).astype(np.float32)
    idx, val = _clip_batch(ROWS0, BL0 * G, 72)
    up = _upstream(73, BL0 * G, F0, K0)
    fo = torch.tensor([0] + list(np.cumsum(ROWS0)[:-1]), dtype=torch.int64, device="cuda")
    ref = torch_embedding_reference(torch.as_tensor(table).cuda(), torch.as_tensor(w1).cuda(), 0.0, fo, idx, val, *up)
    probe = types.SimpleNamespace(field_rows=torch.tensor(ROWS0, device="cuda"), field_size=F0)
    clip = TC._all_binding_clip(ref, probe, True) if mode == "clip" else None
    torch.cuda.synchronize()
    pls = _payloads(run_world(G, _sparse_body, mode, table, w1, idx, val, up, clip), G)
    layers = [pl["layer"] for pl in pls]
    assert [l.plan.n_local for l in layers] == [1] * N0 + [0] * (G - N0)
    assert all(int(l.err_flag.item()) == 0 for l in layers)
    rows = _unite([l.rows for l in layers], G)
    lin = _unite([l.lin_rows for l in layers], G)
    acc = _unite([l.lin_acc for l in layers], G)
    b_rows = _unite([pl["before"]["rows"] for pl in pls], G)
    assert torch.equal(b_rows[:N0, :K0], torch.as_tensor(table).cuda())
    assert torch.equal(rows[N0:], b_rows[N0:]), "padding rows moved"
    before = dict(rows=b_rows[:N0], lin=_unite([pl["before"]["lin"] for pl in pls], G)[:N0],
                  n=_unite([pl["before"]["n"] for pl in pls], G)[:N0], z=None)
    nu = sum(l.last_n_unique for l in layers)
    if mode == "adam":
        union = types.SimpleNamespace(embedding_size=K0, rows=rows[:N0], lin_rows=lin[:N0], first_order=True,
                                      linear_optimizer="adagrad", linear_lr=0.1, l1=0.0, l2=0.0, optimizer="adam",
                                      last_n_unique=nu)
        union.w1 = union.lin_rows[:, 0]
        p1, p2 = pls[0]["bp"]
        bad = TA._check_adam_step(union, before, p1, p2, *TA._targets(ref, probe, None), ref["touched"])
        for l in layers:
            assert np.array_equal(l.beta_power.cpu().numpy(), TA._powers_after(1)), "beta powers differ between ranks"
    else:
        union = types.SimpleNamespace(
            embedding_size=K0, optimizer="adagrad", lr=0.05, optimizer_l1=0.0, optimizer_l2=0.0, linear_optimizer=None,
            field_rows=probe.field_rows, field_size=F0, rows=rows[:N0], accum=rows[:N0, K0:], lin_rows=lin[:N0],
            lin_acc=acc[:N0], lin_z=None, w1=lin[:N0, 0], w1_accum=acc[:N0, 0], first_order=True, last_n_unique=nu)
        if mode == "clip":
            bad = _clip_check(union, before, ref, clip)
            assert all(torch.equal(l.clip_partials, layers[0].clip_partials) for l in layers), \
                "combined partials differ between ranks"
            assert bool(layers[0].clip_partials.any())
        else:
            bad = _violations(union, before, ref["G"], REL * ref["Gfloor"], ref["g1"], REL * ref["g1abs"],
                              ref["touched"])
    assert not any(bad.values()), bad
