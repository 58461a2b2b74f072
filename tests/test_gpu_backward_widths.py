"""The table backward at every embedding width K in {4, 8, 16, 32, 64}, at the branches that depend on K, on the
number of one-row fields and on the length of a run of equal rows:

  A  one-row column sums (embed_bwd_onerow_kernel<LPR, P> + finish): every (LPR, P) pair a width can reach, 1 to 8
     launches, the 64-field cap, B = 1 and a grid-stride wrap, every table rule and linear optimizer;
  B  long-run finishing (embed_bwd_finish_kernel<LPR>): runs laid out on exact chunk boundaries -- the 32 / 33-chunk
     boundary between phase 2 and phase 3, the 256 / 257 boundary of phase 3's probe loop, two long runs in one
     finish CTA, a run that ends the list -- in the fused, emit (clipped), Adam and bag modes;
  C  the clipped two-pass update (dir_embed_bwd_reduce_emit_local -> dir_field_sqnorms -> dir_rows_apply_clipped, and
     the clip in the one-row finish) at the layer: SGD / Adagrad, every linear optimizer, up to 1024 columns;
  D  a negative control per section: the same bound rejects a reference that is wrong by one sample, one chunk or
     one clip factor.

Bounds.  The kernels' gradient sums may differ from the fp64 reference (tests/_util.torch_embedding_reference) by
REL * Gfloor, the cancellation-aware magnitude being summed (SURVEY 7.2), as in test_gpu_zz_fullsize.py.  That band
is pushed through the update rule (`_band`) and a few ulp of fp32 rounding are added; every touched element is held
to it, and everything the batch did not touch must be bit-identical.  Each step is checked from the state the kernel
started from.
"""
import math
import os

import numpy as np
import pytest
import torch

from oracle import tf_adam as A
from oracle import tf_semantics as tfs
from tests._util import REL, torch_embedding_reference
from tests.test_gpu_adam import _adam_step_band
from tests.test_gpu_embedding import _sorted_lists

pytestmark = pytest.mark.gpu

ULP = 2.0 ** -23
CHUNK = 128               # kChunk of embed_bwd.cu
LONG_RUN = 32             # kLongRun: a run whose head is followed by more than this many chunks goes to phase 3
ONEROW_PASSES, ONEROW_MAX = 4, 64      # kOneRowPasses, kOneRowMax


def _lib():
    from dir_b200 import _lib as L
    return L


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ---------------------------------------------------------------------------------------------------------------
# the update rules in fp64 and the gradient band pushed through them

def _rule(kind, t, a, g, lr, l1=0.0, l2=0.0, z=None):
    """One step of a table / linear rule in fp64 -> (t', a', z')."""
    if kind == "sgd":
        return t - lr * g, a, z
    a2 = a + g * g
    if kind == "adagrad":
        return t - lr * g / a2.sqrt(), a2, z
    if kind == "proximal_adagrad":
        eta = lr / a2.sqrt()
        p = t - g * eta
        return torch.sign(p) * (p.abs() - eta * l1).clamp_min(0.0) / (1.0 + l2 * eta), a2, z
    assert kind == "ftrl"
    sq = a2.sqrt()
    z2 = z + g - (sq - a.sqrt()) / lr * t
    w = torch.where(z2.abs() > l1, (torch.sign(z2) * l1 - z2) / (sq / lr + 2.0 * l2), torch.zeros_like(z2))
    return w, a2, z2


def _band(kind, t, a, g, d, lr, l1=0.0, l2=0.0, z=None):
    """The rule at the reference gradient g, and bounds on |kernel - that| valid for any gradient in [g - d, g + d]
    plus the fp32 rounding of the update itself.  Over an interval this narrow (d ~ 1e-5 |g|) every rule here is
    monotone or smooth, so the deviations at the ends and the midpoints, with a quarter of margin, bound it."""
    want = _rule(kind, t, a, g, lr, l1, l2, z)
    dev = [torch.zeros_like(t) for _ in range(3)]
    for s in (-1.0, -0.5, 0.5, 1.0):
        o = _rule(kind, t, a, g + s * d, lr, l1, l2, z)
        for i in range(3):
            if o[i] is not None:
                dev[i] = torch.maximum(dev[i], (o[i] - want[i]).abs())
    t2, a2, z2 = want
    bt = 1.25 * dev[0] + 8 * ULP * (t.abs() + (t2 - t).abs() + t2.abs())
    ba = None if kind == "sgd" else 1.25 * dev[1] + 2 * ULP * a2
    bz = None
    if kind == "ftrl":     # sigma * w: the difference of two square roots, divided by lr, times w
        sq = a2.sqrt()
        bz = 1.25 * dev[2] + 4 * ULP * (z2.abs() + g.abs() + (sq + a.sqrt()) / lr * t.abs())
        bt = 1.25 * dev[0] + 8 * ULP * t2.abs() + bz / (sq / lr + 2.0 * l2)
    return want, (bt, ba, bz)


def _lin_rule(layer):
    """(kind, lr, l1, l2) of the first-order weights, as layers.linear_opt_struct resolves it."""
    if layer.linear_optimizer is None:
        if layer.optimizer == "proximal_adagrad":
            return "proximal_adagrad", layer.lr, layer.optimizer_l1, layer.optimizer_l2
        return layer.optimizer, layer.lr, 0.0, 0.0
    return layer.linear_optimizer, layer.linear_lr, layer.l1, layer.l2


def _state(layer):
    return {k: None if t is None else t.detach().clone()
            for k, t in (("rows", layer.rows), ("lin", layer.lin_rows), ("n", layer.lin_acc), ("z", layer.lin_z))}


def _load(layer, st):
    with torch.no_grad():
        for k, t in (("rows", layer.rows), ("lin", layer.lin_rows), ("n", layer.lin_acc), ("z", layer.lin_z)):
            if t is not None:
                t.copy_(st[k])


def _same(a, b):
    return all((x is None and y is None) or torch.equal(x, y) for x, y in zip(a.values(), b.values()))


def _violations(layer, before, G, d, g1, d1, touched):
    """Elements of the step outside the band -> {what: count}.  Asserts that what the batch did not touch is
    bit-identical and that last_n_unique counts the touched rows."""
    K = layer.embedding_size
    tm = touched[:, None]
    r0 = before["rows"].double()
    T0 = r0[:, :K]
    A0 = r0[:, K:2 * K] if layer.accum is not None else None
    (Tw, Aw, _), (bt, ba, _) = _band(layer.optimizer, T0, A0, G, d, layer.lr, layer.optimizer_l1, layer.optimizer_l2)
    got = layer.rows.double()
    out = {"T": int((((got[:, :K] - Tw).abs() > bt) & tm).sum())}
    if A0 is not None:
        out["acc"] = int((((got[:, K:2 * K] - Aw).abs() > ba) & tm).sum())
    unt = ~touched
    assert torch.equal(layer.rows[unt], before["rows"][unt]), "rows the batch did not touch must stay bit-identical"
    assert int(layer.last_n_unique.item()) == int(touched.sum())
    if layer.first_order:
        kind, lr, l1, l2 = _lin_rule(layer)
        w0 = before["lin"][:, 0].double()
        n0 = None if before["n"] is None else before["n"][:, 0].double()
        z0 = None if before["z"] is None else before["z"][:, 0].double()
        (ww, nw, zw), (bw, bn, bz) = _band(kind, w0, n0, g1, d1, lr, l1, l2, z0)
        out["w1"] = int((((layer.w1.double() - ww).abs() > bw) & touched).sum())
        if bn is not None:
            out["w1_acc"] = int((((layer.w1_accum.double() - nw).abs() > bn) & touched).sum())
        if bz is not None:
            out["w1_z"] = int((((layer.lin_z[:, 0].double() - zw).abs() > bz) & touched).sum())
        for k in ("lin", "n", "z"):
            if before[k] is not None:
                now = {"lin": layer.lin_rows, "n": layer.lin_acc, "z": layer.lin_z}[k]
                assert torch.equal(now[unt], before[k][unt]), k
    return out


def _reference(layer, before, idx, val, g_first, g_fm, u):
    K = layer.embedding_size
    return torch_embedding_reference(before["rows"][:, :K], before["lin"][:, 0], 0.0, layer.field_offset, idx, val,
                                     g_first, g_fm, u)


def _step(layer, idx, val, g_first, g_fm, u):
    first, fm, emb = layer(idx, val)
    torch.autograd.backward((first, fm, emb), (g_first[:, None], g_fm[:, None], u.reshape(idx.shape[0], -1)))
    torch.cuda.synchronize()


def _upstream(seed, B, F, K, u_scale=None):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    g_first = torch.randn(B, device="cuda", generator=gen)
    g_fm = torch.randn(B, device="cuda", generator=gen) * 0.1
    u = torch.randn((B, F, K), device="cuda", generator=gen) * 0.1
    if u_scale is not None:
        u *= u_scale[None, :, None]
    return g_first, g_fm, u


def _checked_step(layer, idx, val, g_first, g_fm, u):
    """One step, checked against the band -> (state before, reference)."""
    before = _state(layer)
    ref = _reference(layer, before, idx, val, g_first, g_fm, u)
    _step(layer, idx, val, g_first, g_fm, u)
    bad = _violations(layer, before, ref["G"], REL * ref["Gfloor"], ref["g1"], REL * ref["g1abs"], ref["touched"])
    assert not any(bad.values()), bad
    return before, ref


# ---------------------------------------------------------------------------------------------------------------
# A. one-row fields

def _onerow_plan(K, n):
    """(LPR, [P of each launch of embed_bwd_onerow_kernel]) for n one-row fields (launch_onerow_partials)."""
    lpr = K // 4
    slots = 32 // lpr
    per = ONEROW_PASSES * slots
    n = min(n, ONEROW_MAX)
    return lpr, [-(-min(per, n - f0) // slots) for f0 in range(0, n, per)]


# n one-row fields per K; in the comments (P of each launch).  Every (LPR, P) a width reaches and 1 to 8 launches.
ONEROW_N = {
    4: (1, 32, 33, 64),                              # (1) (1) (2) (2)               LPR 1: P <= 2 below the cap
    8: (1, 17, 33, 49, 64),                          # (1) (2) (3) (4) (4)
    16: (8, 9, 24, 32, 33, 64),                      # (1) (2) (3) (4) (4 1) (4 4)
    32: (3, 6, 13, 16, 17, 27, 64),                  # (1) (2) (4) (4) (4 1) (4 3) (4 4 4 4)
    64: (1, 5, 8, 9, 20, 37, 42, 55, 64),            # (1) (3) (4) (4 1) (4 4 2) 5, 6, 7 and 8 launches
}
ONEROW_VARIANT_N = {4: 33, 8: 49, 16: 33, 32: 17, 64: 9}
ONEROW_VARIANTS = ("B1", "B9000", "sgd", "proximal_adagrad", "ftrl")
ONEROW_CASES = ([(K, n, "base") for K, ns in ONEROW_N.items() for n in ns] + [(K, 70, "base") for K in ONEROW_N]
                + [(K, ONEROW_VARIANT_N[K], v) for K in ONEROW_N for v in ONEROW_VARIANTS])


def test_onerow_grid_covers_every_pass_and_launch_count():
    pairs, launches = set(), set()
    for K, n, _ in ONEROW_CASES:
        lpr, ps = _onerow_plan(K, n)
        pairs.update((lpr, p) for p in ps)
        launches.add(len(ps))
    reachable = {(K // 4, p) for K in ONEROW_N for n in range(1, ONEROW_MAX + 1) for p in _onerow_plan(K, n)[1]}
    assert pairs == reachable and launches == set(range(1, 9)), (sorted(reachable - pairs), sorted(launches))


def _onerow_case(K, n, B, seed):
    """Sorted fields of 37 and 300 rows around n one-row fields; scattered pruning; with n >= 2 the last one-row
    field has every lookup pruned."""
    rng = np.random.default_rng(seed)
    rows = [37] + [1] * n
    rows.insert(n // 2 + 1, 300)
    F = len(rows)
    idx = np.stack([rng.integers(0, r, B) for r in rows], 1).astype(np.int64)
    val = (rng.random((B, F)) + 0.25).astype(np.float32)
    m = rng.random((B, F))
    val[m < 0.04] = 0.0
    val[(m >= 0.04) & (m < 0.06)] = -0.5
    idx[(m >= 0.06) & (m < 0.08)] = -1
    onerow = [f for f in range(F) if rows[f] == 1]
    dead = onerow[-1] if n >= 2 else None
    if dead is not None:
        val[:, dead] = 0.0
    table = (rng.standard_normal((sum(rows), K)) / np.sqrt(K)).astype(np.float32)
    w1 = (rng.standard_normal(sum(rows)) * 0.1).astype(np.float32)
    return rows, torch.as_tensor(idx).cuda(), torch.as_tensor(val).cuda(), table, w1, dead


def _onerow_layer(pkg, K, rows, variant, table, w1):
    kw = dict(optimizer="adagrad", lr=0.05)
    if variant == "sgd":
        kw = dict(optimizer="sgd", lr=1.0)
    elif variant == "proximal_adagrad":
        kw = dict(optimizer="proximal_adagrad", lr=0.05, optimizer_l1=0.01, optimizer_l2=0.001)
    elif variant == "ftrl":
        kw = dict(optimizer="adagrad", lr=0.05, linear_optimizer="ftrl", linear_lr=0.1,
                  l1_regularization_strength=0.001, l2_regularization_strength=0.001)
    layer = pkg.EmbeddingFM(len(rows), K, rows, first_order=True, **kw).train()
    layer.load_tables(table, w1)
    return layer


def _direct_onerow(pkg, twin, idx, val, g_first, g_fm, u):
    """dir_embed_fm_fwd for S, then one dir_embed_bwd_onerow_update call on the twin's tables -> launches it made."""
    from dir_b200 import layers as LY
    _l = _lib()
    L = _l.lib()
    B, F = idx.shape
    K = twin.embedding_size
    S = torch.empty((B, K), device="cuda")
    first, fm = torch.empty(B, device="cuda"), torch.empty(B, device="cuda")
    _l.check(L.dir_embed_fm_fwd(twin.table.data_ptr(), twin.row_stride, twin.w1.data_ptr(), twin.lin_stride, None,
                                idx.data_ptr(), val.data_ptr(), twin.field_offset.data_ptr(), twin.field_rows.data_ptr(),
                                twin.n_rows, B, F, K, None, S.data_ptr(), first.data_ptr(), fm.data_ptr(), None, None,
                                _stream()), "dir_embed_fm_fwd")
    ws = torch.empty(int(L.dir_shard_dense_workspace_bytes(K)), dtype=torch.uint8, device="cuda")
    nu = torch.zeros(1, dtype=torch.int64, device="cuda")
    ptr = _l.ptr
    n0 = L.dir_launch_count()
    _l.check(L.dir_embed_bwd_onerow_update(
        ptr(twin.table), ptr(twin.accum), twin.row_stride, ptr(twin.w1), ptr(twin.w1_accum), twin.lin_stride, ptr(idx),
        ptr(val), ptr(twin.field_offset), ptr(g_first), ptr(g_fm), ptr(S), ptr(u), B, F, K, ptr(twin.onerow_fields),
        twin.n_onerow_fields, LY._TABLE_OPTIMIZERS[twin.optimizer], twin.lr, LY.table_opt_struct(twin),
        LY.linear_opt_struct(twin), 0.0, ptr(ws), ws.numel(), ptr(nu), _stream()), "dir_embed_bwd_onerow_update")
    launches = int(L.dir_launch_count() - n0)
    torch.cuda.synchronize()
    return launches, int(nu.item())


@pytest.mark.parametrize("K,n,variant", ONEROW_CASES)
def test_onerow_fields(pkg, cuda, monkeypatch, K, n, variant):
    B = {"B1": 1, "B9000": 9000}.get(variant, 1001)
    rows, idx, val, table, w1, dead = _onerow_case(K, n, B, 1000 * K + n)
    F = len(rows)
    g_first, g_fm, u = _upstream(K + n, B, F, K)
    layer = _onerow_layer(pkg, K, rows, variant, table, w1)
    assert layer.n_onerow_fields == min(n, ONEROW_MAX) and layer.n_sorted_fields == F - min(n, ONEROW_MAX)
    before, ref = _checked_step(layer, idx, val, g_first, g_fm, u)
    onerow_rows = layer.field_offset[layer.onerow_fields.long()][:layer.n_onerow_fields]
    if dead is not None:
        r = int(layer.field_offset[dead])
        assert not bool(ref["touched"][r])
        assert torch.equal(layer.rows[r], before["rows"][r]) and torch.equal(layer.lin_rows[r], before["lin"][r])

    # D: the same band rejects a reference that lacks one sample's term of a one-row field (the largest one)
    f = int(layer.onerow_fields[0])
    r = int(layer.field_offset[f])
    if bool(ref["touched"][r]) and B > 1:
        x = torch.where(ref["keep"][:, f], val[:, f].double(), torch.zeros_like(val[:, f].double()))
        term = x[:, None] * (g_fm.double()[:, None] * (ref["S"] - ref["e"][:, f]) + u[:, f].double())
        b = int(term.abs().sum(1).argmax())
        val_x = val.clone()
        val_x[b, f] = 0.0
        wrong = _reference(layer, before, idx, val_x, g_first, g_fm, u)
        bad = _violations(layer, before, wrong["G"], REL * wrong["Gfloor"], wrong["g1"], REL * wrong["g1abs"],
                          ref["touched"])
        assert bad["T"] > 0, "the band must reject a column sum that misses one sample"

    # the same kernels called directly: launches = ceil(n / fields per launch) + the finish, bit-identical rows
    twin = _onerow_layer(pkg, K, rows, variant, table, w1)
    _load(twin, before)
    launches, nu = _direct_onerow(pkg, twin, idx, val, g_first, g_fm, u)
    lpr, ps = _onerow_plan(K, n)
    assert launches == len(ps) + 1, (launches, ps)
    assert nu == int(ref["touched"][onerow_rows].sum())
    assert torch.equal(twin.rows[onerow_rows], layer.rows[onerow_rows])
    assert torch.equal(twin.lin_rows[onerow_rows], layer.lin_rows[onerow_rows])

    # every field through the sort: the same step, held to the same band
    monkeypatch.setenv("DIR_B200_SORT_ALL_FIELDS", "1")
    srt = _onerow_layer(pkg, K, rows, variant, table, w1)
    assert srt.n_onerow_fields == 0
    _checked_step(srt, idx, val, g_first, g_fm, u)


# ---------------------------------------------------------------------------------------------------------------
# B. long runs with exact chunk geometry

C = CHUNK
# exclusive end of the run of row r in the sorted list (rows 0..10 in order; rows 11..15 are never looked up)
RUN_ENDS = [33 * C + 50,      # r0: starts at 0 (a chunk boundary), M = 33: phase 3
            66 * C + 1,       # r1: starts mid-chunk, M = 33: phase 3, its head in the same finish CTA as r0's (K <= 16)
            99 * C,           # r2: M = 32 (phase 2's last), ends exactly at a chunk end
            130 * C + 60,     # r3: starts at a chunk boundary, M = 31
            131 * C + 10,     # r4: M = 1
            131 * C + 30,     # r5: inside one chunk (phase 1)
            386 * C + 5,      # r6: M = 255: one probe round
            642 * C + 7,      # r7: M = 256: a full round, then an empty one
            899 * C + 9,      # r8: M = 257
            1499 * C + 11,    # r9: M = 600: three rounds
            1539 * C + 77]    # r10: M = 40, the last valid run
RUN_M = [33, 33, 32, 31, 1, 0, 255, 256, 257, 600, 40]
N_LONG_ROWS = 16
PRUNED_TAIL = 40 * C + 3       # value-0 lookups (they sort last): longer than 33 chunks, must update nothing


def _runs_of(keys):
    """(key, start, end) of each run of a sorted key list."""
    k = np.asarray(keys)
    cut = np.flatnonzero(np.diff(k)) + 1
    starts = np.concatenate([[0], cut])
    ends = np.concatenate([cut, [k.size]])
    return [(int(k[s]), int(s), int(e)) for s, e in zip(starts, ends)]


def _assert_layout(keys, last, K):
    """The sorted keys (device, int32) hold rows 0..10 at RUN_ENDS, then the run `last` = (key, length) ends the list."""
    runs = _runs_of(keys.cpu().numpy().view(np.uint32))
    assert [r for r, _, _ in runs[:11]] == list(range(11)), "rows 0..10 first, in order"
    assert [(s, e) for _, s, e in runs[:11]] == list(zip([0] + RUN_ENDS[:-1], RUN_ENDS)), "intended layout"
    M = [(e - 1) // C - s // C for _, s, e in runs[:11]]             # chunks after the head that start with the row
    assert M == RUN_M and M[0] > LONG_RUN and M[1] > LONG_RUN and M[2] == LONG_RUN
    assert runs[0][1] % C == 0 and runs[1][1] % C != 0 and runs[2][2] % C == 0 and runs[3][1] % C == 0
    ng = 256 // (K // 4)                                              # chunks per finish CTA
    assert (runs[0][1] // C) // ng == (runs[1][1] // C) // ng or K > 16, "two phase-3 runs in one finish CTA"
    assert (runs[-1][0], runs[-1][2] - runs[-1][1]) == last and runs[-1][2] == keys.numel()


def _long_case(K, tail, seed):
    rng = np.random.default_rng(seed)
    lengths = np.diff([0] + RUN_ENDS)
    idx = np.repeat(np.arange(11), lengths)
    val = (rng.random(idx.size) + 0.25).astype(np.float32)
    if tail == "pruned":
        idx = np.concatenate([idx, rng.integers(0, N_LONG_ROWS, PRUNED_TAIL)])
        val = np.concatenate([val, np.zeros(PRUNED_TAIL, np.float32)])
    perm = rng.permutation(idx.size)                     # samples in random order: the sort makes the runs
    table = (rng.standard_normal((N_LONG_ROWS, K)) / np.sqrt(K)).astype(np.float32)
    w1 = (rng.standard_normal(N_LONG_ROWS) * 0.1).astype(np.float32)
    return (torch.as_tensor(idx[perm][:, None]).cuda(), torch.as_tensor(val[perm][:, None]).cuda(), table, w1)


def _bag_reference(T0, w1_0, off, bag_off, bag_idx, bag_w, B, F, g_first, g_fm, u):
    """EmbeddingBagFM (combiner 'sum') forward / backward in fp64: what torch_embedding_reference gives for one id
    per field, per bag entry.  The floor sums |x T| over every entry of a sample (the rounding of S and of e_s)."""
    N, K = T0.shape
    cnt = bag_off[1:] - bag_off[:-1]
    slot = torch.repeat_interleave(torch.arange(B * F, device=T0.device), cnt)
    b, f = slot // F, slot % F
    row = bag_idx + off[f]
    x = bag_w.double()
    te = T0[row].double() * x[:, None]
    e = torch.zeros((B * F, K), dtype=torch.float64, device=T0.device).index_add_(0, slot, te)
    ea = torch.zeros((B * F, K), dtype=torch.float64, device=T0.device).index_add_(0, slot, te.abs())
    S, Sa = e.view(B, F, K).sum(1), ea.view(B, F, K).sum(1)
    uu = u.reshape(B * F, K).double()
    gfm = g_fm.double()
    per = x[:, None] * (gfm[b, None] * (S[b] - e[slot]) + uu[slot])
    floor = x.abs()[:, None] * (gfm[b, None].abs() * Sa[b] + uu[slot].abs())
    z = torch.zeros((N, K), dtype=torch.float64, device=T0.device)
    t1 = g_first.double()[b] * x
    z1 = torch.zeros(N, dtype=torch.float64, device=T0.device)
    touched = torch.zeros(N, dtype=torch.bool, device=T0.device)
    touched[row] = True
    return dict(G=z.clone().index_add_(0, row, per), Gfloor=z.clone().index_add_(0, row, floor),
                g1=z1.clone().index_add_(0, row, t1), g1abs=z1.clone().index_add_(0, row, t1.abs()), touched=touched)


LONG_CASES = [(K, mode, tail) for K in (4, 8, 16, 32, 64) for mode in ("adagrad", "sgd", "clip", "adam", "bag")
              for tail in ("end", "pruned") if not (mode == "bag" and tail == "pruned")]


@pytest.mark.parametrize("K,mode,tail", LONG_CASES)
def test_long_runs(pkg, cuda, K, mode, tail):
    idx, val, table, w1 = _long_case(K, tail, 7 + K)
    if mode == "bag":
        return _long_runs_bags(pkg, K, idx, val, table, w1)
    B = idx.shape[0]
    g_first, g_fm, u = _upstream(3 * K, B, 1, K)
    kw = {"adagrad": dict(optimizer="adagrad", lr=0.05), "sgd": dict(optimizer="sgd", lr=1.0),
          "clip": dict(optimizer="adagrad", lr=0.05, clip_norm=2.0 ** 100),
          "adam": dict(optimizer="adam", lr=0.01, first_order=False)}[mode]

    def run():
        layer = pkg.EmbeddingFM(1, K, [N_LONG_ROWS], **kw).train()
        layer.load_tables(table, w1)
        before = _state(layer)
        _step(layer, idx, val, g_first, g_fm, u)
        return layer, before

    layer, before = run()
    keys, _ = _sorted_lists(layer._inline_sort.ws.buf, B)
    _assert_layout(keys, (N_LONG_ROWS, PRUNED_TAIL) if tail == "pruned" else (10, RUN_ENDS[-1] - RUN_ENDS[-2]), K)
    assert (PRUNED_TAIL - 1) // C > LONG_RUN
    again, _ = run()
    assert _same(_state(layer), _state(again)), "two runs must be bit-identical"
    ref = _reference(layer, before, idx, val, g_first, g_fm, u)
    G, d, touched = ref["G"], REL * ref["Gfloor"], ref["touched"]
    assert int(touched.sum()) == 11
    if mode == "adam":
        st = before["rows"].double().cpu()
        p1, p2 = (float(x) for x in A.initial_powers())
        T1, m1, v1, bT, bm, bv = _adam_step_band(st[:, :K], st[:, K:2 * K], st[:, 2 * K:], p1, p2, G.cpu(), d.cpu(),
                                                 touched.cpu(), layer.lr, layer.optimizer_epsilon)
        t, m, v = (st[:, i * K:(i + 1) * K].numpy().copy() for i in range(3))
        r = np.flatnonzero(touched.cpu().numpy())
        A.sparse_adam(t, m, v, r, G.cpu().numpy()[r], layer.lr, A.initial_powers(dtype=np.float64),
                      epsilon=layer.optimizer_epsilon)
        assert np.allclose(T1.numpy(), t, rtol=1e-12, atol=0) and np.allclose(m1.numpy(), m, rtol=1e-12, atol=0)
        got = layer.rows.double().cpu()
        assert bool(((got[:, :K] - T1).abs() <= bT).all()) and bool(((got[:, K:2 * K] - m1).abs() <= bm).all())
        assert bool(((got[:, 2 * K:] - v1).abs() <= bv).all())
        assert torch.equal(layer.rows[~touched], before["rows"][~touched])
        assert int(layer.last_n_unique.item()) == 11
        return
    bad = _violations(layer, before, G, d, ref["g1"], REL * ref["g1abs"], touched)
    assert not any(bad.values()), bad
    if mode == "clip":     # a power-of-two clip that never binds: the emit mode equals the fused mode bit for bit
        kw.pop("clip_norm")
        layer_x, _ = run()
        assert _same(_state(layer), _state(layer_x))
        return
    # D: the band rejects a reference that misses one chunk of 128 lookups of r9's phase-3 run
    _, pos = _sorted_lists(layer._inline_sort.ws.buf, B)
    drop = pos[1000 * C:1001 * C].long()
    assert bool((keys[1000 * C:1001 * C] == 9).all())
    val_x = val.clone()
    val_x[drop] = 0.0
    wrong = _reference(layer, before, idx, val_x, g_first, g_fm, u)
    bad = _violations(layer, before, wrong["G"], REL * wrong["Gfloor"], wrong["g1"], REL * wrong["g1abs"], touched)
    assert bad["T"] > 0, "the band must reject a run sum that misses one chunk"


def _long_runs_bags(pkg, K, idx, val, table, w1):
    """EmbeddingBagFM (sum): field 0 holds one entry per bag, laid out as above; field 1's bags (1 to 3 entries) all
    hit its row 0, one run of ~2 B entries that ends the list."""
    from dir_b200 import _lib as _l
    B = idx.shape[0]
    F = 2
    n1 = 1 + torch.arange(B, device="cuda") % 3
    cnt = torch.stack([torch.ones(B, dtype=torch.int64, device="cuda"), n1], 1).reshape(-1)
    bag_off = torch.cat([torch.zeros(1, dtype=torch.int64, device="cuda"), cnt.cumsum(0)])
    slot = torch.repeat_interleave(torch.arange(B * F, device="cuda"), cnt)
    bag_idx = torch.where(slot % F == 0, idx[:, 0][slot // F], torch.zeros_like(slot))
    gen = torch.Generator(device="cuda").manual_seed(K)
    bag_w = torch.rand(bag_idx.numel(), device="cuda", generator=gen) + 0.25
    rows = [N_LONG_ROWS, 3]
    tbl = np.concatenate([table, np.full((3, K), 0.125, np.float32)])
    lin = np.concatenate([w1, np.zeros(3, np.float32)])
    g_first, g_fm, u = _upstream(5 * K, B, F, K)

    def run():
        layer = pkg.EmbeddingBagFM(F, K, rows, combiner="sum", optimizer="adagrad", lr=0.05).train()
        layer.load_tables(tbl, lin)
        before = _state(layer)
        first, fm, emb = layer.forward_bags(bag_off, bag_idx, bag_w)
        torch.autograd.backward((first, fm, emb), (g_first[:, None], g_fm[:, None], u.reshape(B, -1)))
        torch.cuda.synchronize()
        return layer, before

    layer, before = run()
    # the layout of the entries' sorted list (the bag layer sorts the same keys with the same call)
    keys = (bag_idx + layer.field_offset[slot % F]).to(torch.int32)
    ws = torch.zeros(int(_l.lib().dir_embed_bwd_workspace_bytes(keys.numel(), K)), dtype=torch.uint8, device="cuda")
    _l.check(_l.lib().dir_embed_bwd_sort(keys.data_ptr(), keys.numel(), layer.n_rows, ws.data_ptr(), ws.numel(),
                                         _stream()), "dir_embed_bwd_sort")
    torch.cuda.synchronize()
    sk, _ = _sorted_lists(ws, keys.numel())
    _assert_layout(sk, (N_LONG_ROWS, int(n1.sum())), K)
    again, _ = run()
    assert _same(_state(layer), _state(again)), "two runs must be bit-identical"
    ref = _bag_reference(before["rows"][:, :K], before["lin"][:, 0], layer.field_offset, bag_off, bag_idx, bag_w, B, F,
                         g_first, g_fm, u)
    bad = _violations(layer, before, ref["G"], REL * ref["Gfloor"], ref["g1"], REL * ref["g1abs"], ref["touched"])
    assert not any(bad.values()), bad


# ---------------------------------------------------------------------------------------------------------------
# C. the clipped update at the layer

def _field_ids(layer):
    rows = layer.field_rows
    return torch.repeat_interleave(torch.arange(layer.field_size, device=rows.device), rows)


def _clip_center(V, dV, touched, fid, F, clip):
    """tf.clip_by_norm per column of the per-row sums V ([N, K] or [N]) with their band dV -> (factor c_f, the
    clipped sums c_f V, their band, column norms, norm bands).  |d||V_f||| <= ||dV_f|| (triangle inequality) and
    max(., clip) is 1-Lipschitz, so |dc_f| <= c_f ||dV_f|| / max(||V_f||, clip), plus the fp32 rounding of the norm."""
    t = touched.double()
    sq = (V * V).reshape(V.shape[0], -1).sum(1) * t
    dsq = (dV * dV).reshape(V.shape[0], -1).sum(1) * t
    z = torch.zeros(F, dtype=torch.float64, device=V.device)
    nrm, dn = z.clone().index_add_(0, fid, sq).sqrt(), z.clone().index_add_(0, fid, dsq).sqrt()
    den = torch.clamp(nrm, min=clip)
    c = clip / den
    dc = c * dn / den + 4 * ULP * c
    cr, dcr = c[fid], dc[fid]
    if V.dim() == 2:
        cr, dcr = cr[:, None], dcr[:, None]
    return c, cr * V, cr * dV + dcr * V.abs() + 4 * ULP * cr * V.abs(), nrm, dn


def _clip_check(layer, before, ref, clip, wrong=None):
    """Violations of the clipped step.  wrong: 'neighbour' (column f gets column f+1's factor) or 'g1' (g1 unclipped)."""
    fid = _field_ids(layer)
    F = layer.field_size
    touched = ref["touched"]
    c, Gc, dG, _, _ = _clip_center(ref["G"], REL * ref["Gfloor"], touched, fid, F, clip)
    c1, g1c, dg1, _, _ = _clip_center(ref["g1"], REL * ref["g1abs"], touched, fid, F, clip)
    if wrong == "neighbour":
        touched_f = torch.zeros(F, dtype=torch.bool, device=fid.device).index_fill_(0, fid[touched], True)
        pick = [f for f in range(F - 1) if touched_f[f] and touched_f[f + 1] and abs(float(c[f] - c[f + 1])) > 0.01 * float(c[f])]
        assert pick, "some neighbouring columns must have different factors"
        f = pick[0]
        m = (fid == f)[:, None]
        Gc = torch.where(m, ref["G"] * c[f + 1], Gc)
    if wrong == "g1":
        g1c = ref["g1"]
    return _violations(layer, before, Gc, dG, g1c, dg1, touched)


def _choose_clip(ref, layer):
    """A clip (fp32-exact, as the kernels see it) between two column norms in the middle: some columns bind, some
    do not, none within its norm band of the clip."""
    fid = _field_ids(layer)
    _, _, _, nrm, dn = _clip_center(ref["G"], REL * ref["Gfloor"], ref["touched"], fid, layer.field_size, 1.0)
    live = nrm > 0
    s = torch.sort(nrm[live]).values
    i = s.numel() // 2 - 1
    clip = float(np.float32(math.sqrt(float(s[i]) * float(s[i + 1]))))
    binds = live & (nrm - dn > clip * (1 + 1e-6))
    free = live & (nrm + dn < clip * (1 - 1e-6))
    assert bool(binds.any()) and bool(free.any())
    return clip


CLIP_ROWS = [30000, 1, 50, 3, 1, 700, 5, 9]     # column 0: > 16 * 256 distinct rows at B = 6000; column 6: all pruned
CLIP_DEAD = 6
CLIP_LIN = {"none": dict(first_order=False), "same": dict(), "ftrl": dict(linear_optimizer="ftrl", linear_lr=0.1),
            "adagrad": dict(linear_optimizer="adagrad", linear_lr=0.2)}


def _clip_batch(rows, B, seed, dead=None):
    rng = np.random.default_rng(seed)
    F = len(rows)
    idx = np.stack([rng.integers(0, r, B) for r in rows], 1).astype(np.int64)
    val = (rng.random((B, F)) + 0.25).astype(np.float32)
    m = rng.random((B, F))
    val[m < 0.03] = 0.0
    idx[(m >= 0.03) & (m < 0.05)] = -1
    if dead is not None:
        val[:, dead] = 0.0
    return torch.as_tensor(idx).cuda(), torch.as_tensor(val).cuda()


def _clip_steps(pkg, rows, K, opt, lin, B, steps, dead=None, neg=True, seed=0):
    F = len(rows)
    rng = np.random.default_rng(seed)
    table = (rng.standard_normal((sum(rows), K)) / np.sqrt(K)).astype(np.float32)
    w1 = (rng.standard_normal(sum(rows)) * 0.1).astype(np.float32)
    lr = 1.0 if opt == "sgd" else 0.05
    kw = dict(optimizer=opt, lr=lr, **CLIP_LIN[lin])

    def make(**extra):
        layer = pkg.EmbeddingFM(F, K, rows, **kw, **extra).train()
        layer.load_tables(table, w1)
        return layer

    scale = torch.tensor([2.0 ** (f % 4) for f in range(F)], device="cuda")
    main = make(clip_norm=1.0)
    assert main.n_onerow_fields == min(sum(r == 1 for r in rows), ONEROW_MAX)
    exact, plain = make(clip_norm=2.0 ** 100), make()
    os.environ["DIR_B200_SORT_ALL_FIELDS"] = "1"
    try:
        srt = make(clip_norm=1.0)
    finally:
        del os.environ["DIR_B200_SORT_ALL_FIELDS"]
    assert srt.n_onerow_fields == 0
    for s in range(steps):
        idx, val = _clip_batch(rows, B, seed + 10 + s, dead)
        g_first, g_fm, u = _upstream(seed + 20 + s, B, F, K, scale)
        before = _state(main)
        ref = _reference(main, before, idx, val, g_first, g_fm, u)
        clip = _choose_clip(ref, main)
        if main.first_order:            # scale g_first so that some first-order columns bind as well
            fid = _field_ids(main)
            _, _, _, n1, _ = _clip_center(ref["g1"], REL * ref["g1abs"], ref["touched"], fid, F, 1.0)
            g_first = g_first * float(np.float32(4 * clip / float(n1[n1 > 0].median())))
            ref = _reference(main, before, idx, val, g_first, g_fm, u)
            _, _, _, n1, d1 = _clip_center(ref["g1"], REL * ref["g1abs"], ref["touched"], fid, F, 1.0)
            assert bool((n1 - d1 > clip).any())
        # the center is tf_semantics' clip_indexed_slices_per_column of the de-duplicated sums
        r = ref["touched"].nonzero()[:, 0]
        want = tfs.clip_indexed_slices_per_column(r.cpu().numpy(), ref["G"][r].cpu().numpy(),
                                                  main.field_offset.cpu().numpy(), main.n_rows, clip)
        got = _clip_center(ref["G"], REL * ref["Gfloor"], ref["touched"], _field_ids(main), F, clip)[1][r].cpu().numpy()
        assert np.allclose(got, want, rtol=1e-12, atol=1e-300)
        main.clip_norm = srt.clip_norm = clip
        _step(main, idx, val, g_first, g_fm, u)
        bad = _clip_check(main, before, ref, clip)
        assert not any(bad.values()), (s, bad)
        if neg and s == 0:              # D: the band rejects a neighbour's factor and an unclipped g1
            assert _clip_check(main, before, ref, clip, "neighbour")["T"] > 0
            if main.first_order:
                assert _clip_check(main, before, ref, clip, "g1")["w1"] > 0
        if dead is not None:
            r0 = int(main.field_offset[dead])
            assert torch.equal(main.rows[r0:r0 + rows[dead]], before["rows"][r0:r0 + rows[dead]])
        _sqnorm_check(main)
        # one-row fields through the sort, the same clip, held to the same band
        before_s = _state(srt)
        ref_s = _reference(srt, before_s, idx, val, g_first, g_fm, u)
        _step(srt, idx, val, g_first, g_fm, u)
        bad = _clip_check(srt, before_s, ref_s, clip)
        assert not any(bad.values()), (s, bad)
        # clip_norm = 2^100: the clipped backward equals the fused one bit for bit
        _step(exact, idx, val, g_first, g_fm, u)
        _step(plain, idx, val, g_first, g_fm, u)
        assert _same(_state(exact), _state(plain)), s
        assert int(exact.last_n_unique.item()) == int(plain.last_n_unique.item())


def _sqnorm_check(layer):
    """dir_field_sqnorms' partials of the last step: each column's sum over its 16 slices equals the fp64 sum of squares
    of the fp32 per-row sums it read (G and g1), to 1e-12."""
    c = layer._clip_bufs
    F, K = layer.field_size, layer.embedding_size
    U = int(c["count"][1].item())
    part = c["part"][:F * 16 * 2 * 8].view(torch.float64).reshape(F, 16, 2).sum(1).cpu().numpy()
    gu = c["gu"][:U].double().cpu().numpy()
    urows = c["urows"][:U].long().cpu().numpy()
    assert np.all(np.diff(urows) > 0)
    fid = np.searchsorted(layer.field_offset.cpu().numpy(), urows, side="right") - 1
    want = np.zeros((F, 2))
    np.add.at(want[:, 0], fid, (gu[:, :K] ** 2).sum(1))
    np.add.at(want[:, 1], fid, gu[:, K] ** 2)
    assert np.all(np.abs(part - want) <= 1e-12 * np.abs(want)), np.abs(part - want).max()


@pytest.mark.parametrize("K", [4, 8, 16, 32, 64])
@pytest.mark.parametrize("opt", ["sgd", "adagrad"])
@pytest.mark.parametrize("lin", list(CLIP_LIN))
def test_clipped_update(pkg, cuda, K, opt, lin):
    """Two steps of EmbeddingFM(clip_norm=...): accumulators carry over, each step checked from its own start."""
    _clip_steps(pkg, CLIP_ROWS, K, opt, lin, 6000, 2, dead=CLIP_DEAD, seed=K)


@pytest.mark.parametrize("F", [300, 1024])
def test_clipped_update_many_columns(pkg, cuda, F):
    """More columns than the 256 threads that form their clip denominators in one pass."""
    rows = [[1, 3, 7, 40][f % 4] for f in range(F)]
    _clip_steps(pkg, rows, 8, "adagrad", "ftrl", 64, 1, neg=False, seed=F)


# ---------------------------------------------------------------------------------------------------------------
# E. clip_norm is refused beyond the clip's column limit, at construction

@pytest.mark.parametrize("opt", ["sgd", "adagrad", "adam"])
def test_clip_norm_refuses_more_than_1024_columns(pkg, cuda, opt):
    kw = dict(first_order=False) if opt == "adam" else {}
    with pytest.raises(ValueError, match="1024"):
        pkg.EmbeddingFM(1025, 8, [2] * 1025, optimizer=opt, clip_norm=1.0, **kw)
    pkg.EmbeddingFM(1024, 8, [2] * 1024, optimizer=opt, clip_norm=1.0, **kw)


def test_dcn_refuses_more_than_1024_columns(pkg, cuda):
    with pytest.raises(ValueError, match="1024"):
        pkg.DCN(1025, 4, [2] * 1025)                        # DCN clips every column's gradient by default
    with pytest.raises(ValueError, match="1024"):
        pkg.DCN(1025, 4, [2] * 1025, optimizer="adam")


def test_adam_without_clip_takes_more_than_1024_columns(pkg, cuda):
    F, K, B = 1100, 4, 8
    layer = pkg.EmbeddingFM(F, K, [2] * F, optimizer="adam", lr=0.01, first_order=False).train()
    idx = torch.randint(0, 2, (B, F), device="cuda")
    val = torch.ones((B, F), device="cuda")
    g_first, g_fm, u = _upstream(1, B, F, K)
    before = _state(layer)
    _step(layer, idx, val, g_first, g_fm, u)
    ref = _reference(layer, before, idx, val, g_first, g_fm, u)
    assert int(layer.last_n_unique.item()) == int(ref["touched"].sum())
    moved = (layer.rows[:, :K] != before["rows"][:, :K]).any(1)
    assert torch.equal(moved, ref["touched"] & (ref["G"] != 0).any(1))
