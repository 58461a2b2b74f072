"""tf.clip_by_norm per column on the row-sharded tables, host side: the owner-side protocol of csrc/shard_peer.cu
restated with numpy for several simulated ranks (leader rule, rank-order merge, per-column partials over each
requester's ascending segment, rank-order combine) against tf_semantics' clip of the concatenated batch; the key
order the norm pass relies on; the columns' local row offsets; and the constructor's refusals."""
import numpy as np
import pytest

from oracle import tf_semantics as tfs

SLICES, CTA = 16, 256          # kClipSlices, threads of the reduce kernel


def _requests(rows, world, seed, B=40):
    """Per requester: {global row: fp32 per-row sum [K + 1]} of its own samples (g and g1)."""
    rng = np.random.default_rng(seed)
    N, K = sum(rows), 4
    out = []
    for _ in range(world):
        r = {}
        off = np.r_[0, np.cumsum(rows)[:-1]]
        for f, n in enumerate(rows):
            for i in rng.integers(0, n, size=B):
                g = (rng.standard_normal(K + 1) * (1 + f)).astype(np.float32)
                row = int(off[f] + i)
                r[row] = (r[row] + g).astype(np.float32) if row in r else g
        out.append(r)
    return out, N, K


def _keys_segment(req, owner, G):
    """What requester q sends owner o: its distinct local rows for o in key order, (owner, local row) ascending."""
    keys = sorted(((row % G), row // G) for row in req)
    return [l for (o, l) in keys if o == owner]


def _protocol(rows, world, seed, clip):
    """-> ({global row: clipped fp32 [K + 1]}, combined partials [F][S][2]) as the ranks would compute them."""
    from dir_b200.sharded import ShardPlan
    reqs, N, K = _requests(rows, world, seed)
    F = len(rows)
    norm = np.zeros((world, F, SLICES, 2))                      # norm buffer contents: [rank that stored][f][s][2]
    merged = {}
    for o in range(world):
        plan = ShardPlan(rows, world, o)
        lfo = plan.local_field_offset()
        segs = [_keys_segment(reqs[q], o, world) for q in range(world)]
        sq = []                                                 # per arrival, in arrival order (q, then i)
        for q in range(world):
            for l in segs[q]:
                row = l * world + o
                asked = [p for p in range(world) if l in set(segs[p])]
                if asked[0] != q:                               # an earlier requester merges this row
                    sq.append((0.0, 0.0))
                    continue
                g = reqs[q][row].copy()
                for p in asked[1:]:                             # rank order, fp32 adds
                    g = (g + reqs[p][row]).astype(np.float32)
                merged[row] = g
                sq.append((float((g[:K].astype(np.float64) ** 2).sum()), float(np.float64(g[K]) ** 2)))
        pre = np.r_[0, np.cumsum([len(s) for s in segs])]
        for f in range(F):
            for s in range(SLICES):
                acc = np.zeros(2)
                for q in range(world):
                    seg = np.asarray(segs[q], dtype=np.int64)
                    lo, hi = np.searchsorted(seg, lfo[f]), np.searchsorted(seg, lfo[f + 1])
                    for i in range(lo + s * CTA, hi, SLICES * CTA):
                        for t in range(i, min(i + CTA, hi)):
                            acc += sq[pre[q] + t]
                norm[o, f, s] = acc
    part = norm[0].copy()
    for q in range(1, world):                                   # rank-order combine: the same on every rank
        part = part + norm[q]
    tot = part.sum(1)
    den = np.maximum(np.sqrt(tot[:, 0]).astype(np.float32), np.float32(clip))
    den1 = np.maximum(np.sqrt(tot[:, 1]).astype(np.float32), np.float32(clip))
    off = np.r_[0, np.cumsum(rows)[:-1]]
    out = {}
    for row, g in merged.items():
        f = int(np.searchsorted(off, row, side="right") - 1)
        c = g.copy()
        c[:K] = (g[:K] * np.float32(clip)) / den[f]
        c[K] = (g[K] * np.float32(clip)) / den1[f]
        out[row] = c
    return out, reqs, N, K, part


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_protocol_matches_clip_of_concatenated_batch(world):
    rows = [50, 1, 9, 300, 3, 17, 1, 2]
    reqs, N, K = _requests(rows, world, 5 + world)
    full = {}
    for r in reqs:                                              # the concatenated batch's de-duplicated sums, fp64
        for row, g in r.items():
            full[row] = full.get(row, 0) + g.astype(np.float64)
    rws = np.array(sorted(full))
    vals = np.stack([full[r] for r in rws])
    off = list(np.r_[0, np.cumsum(rows)[:-1]])
    norms = sorted(np.linalg.norm(vals[(rws >= a) & (rws < b), :K]) for a, b in zip(off, off[1:] + [N]))
    clip = float(np.float32(np.sqrt(norms[3] * norms[4])))     # between two column norms: some bind, some do not
    got, _, _, _, part = _protocol(rows, world, 5 + world, clip)
    want_G = tfs.clip_indexed_slices_per_column(rws, vals[:, :K], off, N, clip)
    want_g1 = tfs.clip_indexed_slices_per_column(rws, vals[:, K:], off, N, clip)
    assert sorted(got) == list(rws), "every requested row is merged exactly once, by its leading requester"
    have = np.stack([got[r] for r in rws]).astype(np.float64)
    scale = np.abs(vals).max()
    assert np.abs(have[:, :K] - want_G).max() <= 1e-5 * scale
    assert np.abs(have[:, K:] - want_g1).max() <= 1e-5 * scale
    # the clip binds on some columns and not on others (the test means something)
    norms = [np.linalg.norm(vals[(rws >= a) & (rws < b), :K]) for a, b in zip(off, off[1:] + [N])]
    assert max(norms) > clip and min(n for n in norms if n > 0) < clip


def _sorted_keys(rows, world, B, seed):
    """The id phase's key order (keys.cuh / dir_shard_bag_keys): key = (row mod G) * cap + row div G, pruned lookups
    last; distinct keys numbered in sorted order, ulocal[u] = key mod cap."""
    rng = np.random.default_rng(seed)
    N = sum(rows)
    cap = -(-N // world)
    off = np.r_[0, np.cumsum(rows)[:-1]]
    ids = np.stack([rng.integers(-1, n, B) for n in rows], 1)
    row = off[None, :] + ids
    key = np.where(ids >= 0, (row % world) * cap + row // world, world * cap).reshape(-1)
    u = np.unique(key)
    u = u[u < world * cap]
    return u // cap, u % cap


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_requester_segments_ascend_in_local_row(world):
    owner, local = _sorted_keys([50, 1, 9, 1000, 3, 17, 1], world, 300, world)
    assert np.all(np.diff(owner) >= 0)
    for o in range(world):
        seg = local[owner == o]
        assert np.all(np.diff(seg) > 0)


def test_local_field_offsets():
    from dir_b200.sharded import ShardPlan
    rows = [5, 1, 9, 2, 1, 30]                                  # fields with fewer rows than G
    N = sum(rows)
    off = np.r_[0, np.cumsum(rows)]
    for world in (1, 2, 3, 8):
        for rank in range(world):
            p = ShardPlan(rows, world, rank)
            lfo = p.local_field_offset()
            assert len(lfo) == len(rows) + 1 and lfo[-1] == p.n_local
            assert all(a <= b for a, b in zip(lfo, lfo[1:]))
            for f in range(len(rows)):
                mine = [l for l in range(p.n_local) if off[f] <= l * world + rank < off[f + 1]]
                assert mine == list(range(lfo[f], lfo[f + 1])), (world, rank, f)
            assert p.local_field_offset(rank) == lfo


@pytest.mark.parametrize("kw,msg", [(dict(clip_norm=0.0), "clip_norm must be > 0"),
                                    (dict(clip_norm=-1.0), "clip_norm must be > 0"),
                                    (dict(clip_norm=1.0, optimizer="proximal_adagrad"), "proximal_adagrad"),
                                    (dict(clip_norm=1.0, micro_batches=2), "micro_batches=1")])
def test_sharded_clip_refusals(kw, msg):
    import dir_b200
    with pytest.raises(ValueError, match=msg):
        dir_b200.ShardedEmbeddingFM(3, 8, [4, 5, 6], device="cpu", **kw)
    with pytest.raises(ValueError, match="at most 1024 fields"):
        dir_b200.ShardedEmbeddingFM(1025, 8, [2] * 1025, clip_norm=1.0, device="cpu")
    with pytest.raises(ValueError, match="CUDA device"):                       # a valid clip gets as far as the device
        dir_b200.ShardedEmbeddingFM(3, 8, [4, 5, 6], clip_norm=1.0, device="cpu")


def test_bag_layer_and_dcn_forward_the_clip():
    import dir_b200
    with pytest.raises(ValueError, match="clip_norm must be > 0"):
        dir_b200.ShardedEmbeddingBagFM(3, 8, [4, 5, 6], clip_norm=-2.0, device="cpu")
    with pytest.raises(ValueError, match="micro_batches=1"):
        dir_b200.DCN(3, 8, [4, 5, 6], sharded=True, clip_sharded_tables=True, micro_batches=2, device="cpu")
