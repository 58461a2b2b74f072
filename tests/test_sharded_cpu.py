"""Host-side logic of the row-sharded path on CPU: the shard plan's index arithmetic, and the device-driven
exchange restated with numpy for several simulated ranks.  Rows seen through the exchange must equal a direct
lookup in the full table, and the owners' merged gradient sums must equal a global scatter-add."""
import numpy as np
import pytest
import torch

from oracle import deepctr_oracle as O


def test_shard_plan_arithmetic():
    from dir_b200.sharded import ShardPlan
    rows = [5, 1, 9]
    g = torch.arange(15)
    full = np.arange(30).reshape(15, 2)
    for world in (1, 2, 3, 8):
        seen = []
        for rank in range(world):
            p = ShardPlan(rows, world, rank)
            assert p.n_rows == 15 and p.cap == -(-15 // world)
            mine = [r for r in range(15) if r % world == rank]
            assert p.n_local == len(mine)
            assert [int(p.global_row(torch.tensor(l))) for l in range(p.n_local)] == mine
            assert torch.equal(p.global_row(p.local_row(g), p.owner(g)), g)
            assert p.shard_of(full).shape[0] == p.n_local and np.array_equal(p.shard_of(full), full[mine])
            seen += mine
        assert sorted(seen) == list(range(15))
    with pytest.raises(ValueError):
        ShardPlan(rows, 2, 2)
    assert np.array_equal(ShardPlan(rows, 4, 1).shard_of(full), full[1::4])


def _peer_protocol(world, rows, K, B, seed, seg_cap=None):
    """The device-driven exchange of csrc/shard_peer.cu restated with numpy, every rank simulated in one process:
    headers (count, base_u) + id segments, the owner's slot map (slot[row, q] = i + 1, no sort), rows stored at
    base_u + i of the requester, per-distinct-row sums stored at segment q of the owner, the lowest asking rank
    merging in rank order.  Returns (rows each rank's lookups see, per-global-row gradient sums, slot maps)."""
    from dir_b200.sharded import ShardPlan
    rng = np.random.default_rng(seed)
    N = sum(rows)
    F = len(rows)
    table = rng.standard_normal((N, K)).astype(np.float32)
    plans = [ShardPlan(rows, world, r) for r in range(world)]
    cap = plans[0].cap
    seg_cap = seg_cap or min(B * F, cap)
    idx = [np.stack([rng.integers(0, r, size=B) for r in rows], 1).astype(np.int64) for _ in range(world)]
    grads = [rng.standard_normal((B * F, K)).astype(np.float32) for _ in range(world)]
    off = np.asarray(plans[0].field_offset)
    # requester side: distinct (owner, local) keys, owner-major; header + ids into the owners' buffers
    hdr = np.zeros((world, world, 2), np.int64)                     # hdr[o][q] = (count, base_u)
    ids = np.full((world, world, seg_cap), -1, np.int64)            # ids[o][q][i]
    inv, uk = [], []
    for q in range(world):
        grow = (idx[q] + off[None, :]).reshape(-1)
        key = (grow % world) * cap + grow // world
        ukeys, iv = np.unique(key, return_inverse=True)
        inv.append(iv)
        uk.append(ukeys)
        owner_off = np.searchsorted(ukeys, np.arange(world + 1) * cap)
        for o in range(world):
            c = owner_off[o + 1] - owner_off[o]
            assert c <= seg_cap
            hdr[o, q] = (c, owner_off[o])
            ids[o, q, :c] = ukeys[owner_off[o]:owner_off[o + 1]] % cap
    # owner side: slot map, gather + send
    slot = np.zeros((world, cap, world), np.int64)
    rowsbuf = [np.zeros((len(uk[q]), K), np.float32) for q in range(world)]
    for o in range(world):
        local = table[o::world]
        for q in range(world):
            c, base = hdr[o, q]
            r = ids[o, q, :c]
            assert (slot[o, r, q] == 0).all()                         # a requester sends a row at most once
            slot[o, r, q] = np.arange(c) + 1
            rowsbuf[q][base:base + c] = local[r]
    seen = [rowsbuf[q][inv[q]].reshape(B, F, K) for q in range(world)]
    # backward: per-distinct-row sums into the owner's segment q; the lowest asking rank merges in rank order
    gbuf = np.zeros((world, world, seg_cap, K), np.float32)
    for q in range(world):
        gu = np.zeros((len(uk[q]), K), np.float32)
        np.add.at(gu, inv[q], grads[q])
        for o in range(world):
            c, base = hdr[o, q]
            gbuf[o, q, :c] = gu[base:base + c]
    total = np.zeros((cap * world, K), np.float64)
    merges = 0
    for o in range(world):
        for q in range(world):
            for i in range(hdr[o, q, 0]):
                r = ids[o, q, i]
                if (slot[o, r, :q] != 0).any():
                    continue                                           # an earlier rank merges this row
                g = gbuf[o, q, i].astype(np.float64)
                for p in range(q + 1, world):
                    if slot[o, r, p]:
                        g = g + gbuf[o, p, slot[o, r, p] - 1]
                total[r * world + o] = g
                merges += 1
    return table, idx, grads, off, seen, total, merges


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_peer_protocol_restated(world):
    """Host-checkable statement of the N > 1 device-driven exchange (the kernels themselves need GPUs:
    tests/test_gpu_sharded.py).  Rows seen through the exchange equal a direct lookup; merged sums equal a global
    scatter-add; every touched row is merged exactly once.  Includes the case ceil(n_rows / G) < distinct rows of
    one requester (world 8), which round 1's buffer sizing got wrong."""
    rows, K, B = [40, 1, 90, 300, 3, 1], 4, 64
    table, idx, grads, off, seen, total, merges = _peer_protocol(world, rows, K, B, seed=11)
    F = len(rows)
    ref = np.zeros_like(total)
    touched = set()
    for q in range(world):
        want, _ = O.embedding_lookup(table, off, idx[q], None)
        assert np.array_equal(seen[q], want)
        grow = (idx[q] + off[None, :]).reshape(-1)
        np.add.at(ref, grow, grads[q].astype(np.float64))
        touched |= set(grow.tolist())
    assert merges == len(touched)
    assert np.allclose(total[:sum(rows)], ref[:sum(rows)], atol=1e-5)
    if world == 8:
        from dir_b200.sharded import ShardPlan
        cap = ShardPlan(rows, world, 0).cap
        assert max(len(set((idx[q] + off[None, :]).reshape(-1).tolist())) for q in range(world)) > cap
