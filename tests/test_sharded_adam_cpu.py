"""TF's Adam on the row-sharded tables, host side: the owner sweep of csrc/shard_peer.cu (dir_shard_owner_apply_adam)
restated with numpy for several simulated ranks -- per tile and requester the arrivals found with lower_bound, a
map in which the lowest requester wins, the rank-order fp32 merge, the clip factors from the rank-order combined
partials, the fp32 Adam step on every local row -- and the union of the shards held to oracle.tf_adam.sparse_adam
(after tf_semantics' per-column clip) on the concatenated batch over three steps; the constructor's refusals."""
import numpy as np
import pytest

from oracle import tf_adam as A
from oracle import tf_semantics as tfs

TILE = 1024                     # kAdamTile
EMPTY = 0xFFFFFFFF
K = 4
ROWS = [2600, 1, 9, 1500, 3, 17, 1, 4100]        # N = 8231: several tiles per owner at G <= 3, two at G = 8
LR, B1, B2, EPS = 0.01, 0.9, 0.999, 1e-8


def _requests(world, step, B=60):
    """Per requester: {global row: fp32 per-row sum [K + 1]} (g and g1) of its own samples.  Requester 0 asks only
    for rows of the first column after step 0, so later tiles see no arrival of it; every requester asks for the
    rows on both sides of each owner's first tile boundary."""
    rng = np.random.default_rng(100 * world + step)
    off = np.r_[0, np.cumsum(ROWS)[:-1]]
    out = []
    for q in range(world):
        r = {}
        fields = [0] if (q == 0 and step > 0 and world > 1) else range(len(ROWS))
        for f in fields:
            n = ROWS[f]
            lo = 0 if step == 0 else n // 2          # steps 1, 2 leave the lower half of each column alone
            for i in rng.integers(lo, n, size=B):
                g = (rng.standard_normal(K + 1) * (1 + f % 3)).astype(np.float32)
                row = int(off[f] + i)
                r[row] = (r[row] + g).astype(np.float32) if row in r else g
        if q > 0 or step == 0 or world == 1:
            for o in range(world):
                for l in (TILE - 1, TILE):
                    row = l * world + o
                    if row < sum(ROWS):
                        g = rng.standard_normal(K + 1).astype(np.float32)
                        r[row] = (r[row] + g).astype(np.float32) if row in r else g
        out.append(r)
    return out


def _segment(req, owner, G):
    """What requester q sends owner o: its distinct local rows for o, ascending (the key order)."""
    return np.asarray(sorted(row // G for row in req if row % G == owner), dtype=np.int64)


def _owner_sweep(world, o, reqs, state, bp, clip, den, den1, stats):
    """One dir_shard_owner_apply_adam on owner o (fp32), in place on state = (T, m, v) of its local rows.
    -> {global row: merged, clipped [K + 1]} of the rows that had a gradient."""
    from dir_b200.sharded import ShardPlan
    plan = ShardPlan(ROWS, world, o)
    n_local = plan.cap
    lfo = plan.local_field_offset()
    segs = [_segment(reqs[q], o, world) for q in range(world)]
    slot = [{int(l): i for i, l in enumerate(segs[q])} for q in range(world)]     # slot[row][q] = i + 1
    T, m, v = state
    f32 = np.float32
    b1, b2, omb1, omb2, eps = f32(B1), f32(B2), f32(1) - f32(B1), f32(1) - f32(B2), f32(EPS)
    lr_t = f32(f32(LR) * np.sqrt(f32(1) - bp[1])) / (f32(1) - bp[0])
    merged = {}
    for r0 in range(0, n_local, TILE):
        r1 = min(r0 + TILE, n_local)
        smap = np.full(r1 - r0, EMPTY, dtype=np.uint32)
        seen = []
        for q in range(world):
            lo, hi = np.searchsorted(segs[q], r0), np.searchsorted(segs[q], r1)     # the two warp lower_bounds
            seen.append(hi > lo)
            np.minimum.at(smap, segs[q][lo:hi] - r0, (np.uint32(q) << 24) | np.arange(lo, hi, dtype=np.uint32))
        if any(seen) and not all(seen):
            stats["tile_without_some_requester"] = True
        if r1 - r0 < TILE:
            stats["partial_tile"] = True
        G = np.zeros((r1 - r0, K + 1), dtype=np.float32)
        has = smap != EMPTY
        for t in np.nonzero(has)[0]:
            l = r0 + int(t)
            q0, i0 = int(smap[t] >> 24), int(smap[t] & 0xFFFFFF)
            row = l * world + o
            assert segs[q0][i0] == l and all(l not in slot[p] for p in range(q0))    # the lowest requester leads
            g = reqs[q0][row].copy()
            for p in range(q0 + 1, world):                                          # rank order, fp32 adds
                if l in slot[p]:
                    g = (g + reqs[p][row]).astype(np.float32)
            if clip is not None:
                f = int(np.searchsorted(lfo, l, side="right") - 1)
                g[:K] = (g[:K] * f32(clip)) / den[f]
                g[K] = (g[K] * f32(clip)) / den1[f]
            G[t] = g
            merged[row] = g
            if sum(l in slot[p] for p in range(world)) == world and world > 1:
                stats["asked_by_all"] = True
            if l % TILE in (0, TILE - 1) and l > 0:
                stats["tile_edges"] = stats.get("tile_edges", 0) + 1
        sl = slice(r0, r1)
        mm, vv = m[sl] * b1, v[sl] * b2
        mm[has] = mm[has] + G[has, :K] * omb1
        vv[has] = vv[has] + (G[has, :K] * G[has, :K]) * omb2
        T[sl] = T[sl] - (lr_t * mm) / (np.sqrt(vv) + eps)
        m[sl], v[sl] = mm, vv
    return merged


def _combined_factors(world, reqs, clip):
    """Per column: max(||G_f||, clip) and max(||g1_f||, clip) from the partials of every owner (fp64 squares of the
    merged rows), combined in rank order -- the same denominators on every rank."""
    from dir_b200.sharded import ShardPlan
    F = len(ROWS)
    part = np.zeros((F, 2))
    for o in range(world):
        lfo = ShardPlan(ROWS, world, o).local_field_offset()
        own = np.zeros((F, 2))
        rows = sorted({r for q in range(world) for r in reqs[q] if r % world == o})
        for row in rows:
            g = None
            for q in range(world):                                                  # rank order, fp32 adds
                if row in reqs[q]:
                    g = reqs[q][row].copy() if g is None else (g + reqs[q][row]).astype(np.float32)
            f = int(np.searchsorted(lfo, row // world, side="right") - 1)
            own[f] += ((g[:K].astype(np.float64) ** 2).sum(), np.float64(g[K]) ** 2)
        part = part + own
    den = np.maximum(np.sqrt(part[:, 0]).astype(np.float32), np.float32(clip))
    den1 = np.maximum(np.sqrt(part[:, 1]).astype(np.float32), np.float32(clip))
    return den, den1


def _concatenated(reqs):
    full = {}
    for r in reqs:
        for row, g in r.items():
            full[row] = full.get(row, 0) + g.astype(np.float64)
    rws = np.array(sorted(full))
    return rws, np.stack([full[r] for r in rws])


@pytest.mark.parametrize("clipped", [False, True])
@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_owner_sweep_matches_adam_of_concatenated_batch(world, clipped):
    from dir_b200.sharded import ShardPlan
    N = sum(ROWS)
    off = list(np.r_[0, np.cumsum(ROWS)[:-1]])
    rng = np.random.default_rng(world)
    T0 = (rng.standard_normal((N, K)) / np.sqrt(K)).astype(np.float32)
    plans = [ShardPlan(ROWS, world, o) for o in range(world)]
    shards = []
    for o, p in enumerate(plans):
        t = np.zeros((p.cap, K), np.float32)
        t[:p.n_local] = p.shard_of(T0)
        shards.append((t, np.zeros((p.cap, K), np.float32), np.zeros((p.cap, K), np.float32)))
    bp = A.initial_powers(B1, B2, np.float32)                # every rank holds the same powers
    t64, m64, v64 = T0.astype(np.float64), np.zeros((N, K)), np.zeros((N, K))
    bp64 = A.initial_powers(B1, B2, np.float32)
    stats, touched_by_step = {}, []
    clip = None
    for step in range(3):
        reqs = _requests(world, step)
        rws, vals = _concatenated(reqs)
        if clipped and clip is None:                         # between two column norms: some bind, some do not
            norms = sorted(np.linalg.norm(vals[(rws >= a) & (rws < b), :K]) for a, b in zip(off, off[1:] + [N]))
            clip = float(np.float32(np.sqrt(norms[3] * norms[4])))
            all_norms = [np.linalg.norm(vals[(rws >= a) & (rws < b), :K]) for a, b in zip(off, off[1:] + [N])]
            assert max(all_norms) > clip and min(n for n in all_norms if n > 0) < clip
        den = den1 = None
        if clip is not None:
            den, den1 = _combined_factors(world, reqs, clip)
        merged = {}
        for o in range(world):
            merged.update(_owner_sweep(world, o, reqs, shards[o], bp, clip, den, den1, stats))
        A.finish(bp, B1, B2)
        assert sorted(merged) == list(rws), "every requested row is merged exactly once, by its leading requester"
        # the oracle: tf_semantics' clip of the concatenated batch, then TF's sparse Adam (fp64)
        G = vals[:, :K]
        if clip is not None:
            G = tfs.clip_indexed_slices_per_column(rws, G, off, N, clip)
            g1 = tfs.clip_indexed_slices_per_column(rws, vals[:, K:], off, N, clip)
            have1 = np.stack([merged[r][K:] for r in rws]).astype(np.float64)
            assert np.abs(have1 - g1).max() <= 1e-5 * np.abs(vals).max()
        have = np.stack([merged[r][:K] for r in rws]).astype(np.float64)
        assert np.abs(have - G).max() <= 1e-5 * np.abs(vals).max()
        A.sparse_adam(t64, m64, v64, rws, G, LR, bp64.astype(np.float64), B1, B2, EPS)
        A.finish(bp64, B1, B2)
        touched_by_step.append(set(rws.tolist()))
        # the union of the shards
        T = np.zeros((plans[0].cap * world, K))
        Mu, Vu = np.zeros_like(T), np.zeros_like(T)
        for o in range(world):
            T[o::world], Mu[o::world], Vu[o::world] = shards[o]
        assert np.abs(T[:N] - t64).max() <= 1e-5 * (np.abs(T0).max() + LR), step
        assert np.abs(Mu[:N] - m64).max() <= 1e-5 * np.abs(m64).max(), step
        assert np.abs(Vu[:N] - v64).max() <= 1e-5 * np.abs(v64).max(), step
        assert not T[N:].any() and not Mu[N:].any(), "padding rows of the last shard stay zero"
    assert np.array_equal(bp, bp64), "beta powers: the repeated fp32 product, on every rank"
    never = sorted(set(range(N)) - set().union(*touched_by_step))
    assert np.array_equal(T[never], T0[never].astype(np.float64)) and not Mu[never].any()
    stale = touched_by_step[0] - touched_by_step[1] - touched_by_step[2]
    assert len(stale) > 100, "rows touched in step 1 only decay and move in steps 2 and 3"
    assert stats.get("partial_tile"), "n_local is not a multiple of the tile"
    assert stats.get("tile_edges", 0) >= 2 * world
    if world > 1:
        assert stats.get("tile_without_some_requester") and stats.get("asked_by_all"), stats


def test_adam_is_not_a_table_optimizer_of_the_other_entry_points():
    from dir_b200.layers import _TABLE_OPTIMIZERS
    assert "adam" not in _TABLE_OPTIMIZERS


ADAM = dict(optimizer="adam", first_order=False)


@pytest.mark.parametrize("kw,msg", [(dict(ADAM, micro_batches=2), "micro_batches=1"),
                                    (dict(optimizer="adam"), "Adam does not train first-order weights"),
                                    (dict(ADAM, lr=0.0), "adam needs lr > 0"),
                                    (dict(ADAM, lr=-1.0), "adam needs lr > 0"),
                                    (dict(ADAM, optimizer_beta1=1.0), r"\[0, 1\)"),
                                    (dict(ADAM, optimizer_beta2=-0.1), r"\[0, 1\)"),
                                    (dict(ADAM, optimizer_epsilon=0.0), "optimizer_epsilon must be > 0")])
def test_sharded_adam_refusals(kw, msg):
    import dir_b200
    with pytest.raises(ValueError, match=msg):
        dir_b200.ShardedEmbeddingFM(3, 8, [4, 5, 6], device="cpu", **kw)


def test_valid_adam_gets_as_far_as_the_device():
    import dir_b200
    for kw in (ADAM, dict(optimizer="ADAM", linear_optimizer="ftrl"), dict(ADAM, clip_norm=1.0),
               dict(ADAM, replicate_onerow=True)):
        with pytest.raises(ValueError, match="CUDA device"):
            dir_b200.ShardedEmbeddingFM(3, 8, [4, 1, 6], device="cpu", **kw)
    with pytest.raises(ValueError, match="does not train with adam"):
        dir_b200.ShardedEmbeddingBagFM(3, 8, [4, 5, 6], device="cpu", **ADAM)
    with pytest.raises(ValueError, match="CUDA device"):          # DCN no longer refuses Adam with the sharded layer
        dir_b200.DCN(3, 8, [4, 5, 6], sharded=True, optimizer="adam", clip_sharded_tables=True, device="cpu")
