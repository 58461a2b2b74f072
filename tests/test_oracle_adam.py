"""TF 1.x Adam (oracle/tf_adam.py) pinned to closed forms, the dense optimizer of models.DCN pinned to the oracle, and
everything about optimizer='adam' that is decided before a kernel runs: argument validation of dir_rows_apply_adam,
the layers and models that refuse Adam, the layer's storage and its checkpoint names.  No GPU needed."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import tf_adam as A

LR, B1, B2 = 0.01, 0.875, 1 - 2.0 ** -9       # exact in fp32, as are 1 - B1 and 1 - B2: the closed forms hold in fp64


def test_step_one_closed_form():
    """Step 1: m = (1-b1) g, v = (1-b2) g^2, lr_t = lr sqrt(1-b2) / (1-b1), so the move is
    lr sqrt(1-b2) g / (sqrt(1-b2) |g| + eps)."""
    rng = np.random.default_rng(1)
    for eps in (1e-8, 1e-4, 0.5):
        var = rng.standard_normal((20, 4))
        m, v = np.zeros_like(var), np.zeros_like(var)
        rows = np.array([1, 4, 7, 19])
        g = rng.standard_normal((4, 4)) * np.array([1e-6, 1e-3, 1.0, 100.0])
        bp = A.initial_powers(B1, B2, np.float64)
        want = var.copy()
        e32 = float(np.float32(eps))             # TF's epsilon is an fp32 scalar too
        want[rows] -= LR * np.sqrt(1 - B2) * g / (np.sqrt(1 - B2) * np.abs(g) + e32)
        A.sparse_adam(var, m, v, rows, g, LR, bp, B1, B2, eps)
        np.testing.assert_allclose(var, want, rtol=1e-13, atol=1e-15)
        np.testing.assert_allclose(m[rows], (1 - B1) * g, rtol=1e-15)
        np.testing.assert_allclose(v[rows], (1 - B2) * g * g, rtol=1e-15)


def test_untouched_rows_and_the_decay_of_touched_ones():
    rng = np.random.default_rng(2)
    eps = 1e-4
    var = rng.standard_normal((50, 8)).astype(np.float32)
    var0 = var.copy()
    m, v = np.zeros_like(var), np.zeros_like(var)
    bp = A.initial_powers(B1, B2, np.float32)
    r1 = np.array([3, 10, 11, 40])
    g1 = rng.standard_normal((4, 8)).astype(np.float32)
    A.sparse_adam(var, m, v, r1, g1, LR, bp, B1, B2, eps)
    A.finish(bp, B1, B2)
    never = np.setdiff1d(np.arange(50), r1)
    assert np.array_equal(var[never], var0[never]) and not m[never].any() and not v[never].any()
    m1, v1, after1 = m.copy(), v.copy(), var.copy()
    r2 = np.array([10, 41])                      # rows 3, 11, 40 are touched at step 1 only
    g2 = rng.standard_normal((2, 8)).astype(np.float32)
    A.sparse_adam(var, m, v, r2, g2, LR, bp, B1, B2, eps)
    A.finish(bp, B1, B2)
    never = np.setdiff1d(np.arange(50), np.concatenate([r1, r2]))
    assert np.array_equal(var[never], var0[never]) and not m[never].any() and not v[never].any()
    lr_t2 = LR * np.sqrt(1 - B2 ** 2) / (1 - B1 ** 2)
    for r in (3, 11, 40):                        # the step-1-only rows still move (this is not LazyAdam)
        want = lr_t2 * B1 * m1[r].astype(np.float64) / (np.sqrt(B2 * v1[r].astype(np.float64)) + eps)
        np.testing.assert_allclose(after1[r] - var[r], want, rtol=2e-5, atol=1e-9)
        assert np.all(after1[r] != var[r])
    assert bp.dtype == np.float32 and bp[0] == np.float32(B1 ** 3)


def test_scalars_are_evaluated_in_fp32():
    """TF evaluates 1 - beta2 in the variable's dtype: for fp32 and beta2 = 0.999 that is 1.3e-5 away from 0.001,
    which the oracle carries into fp64 rather than the exact value."""
    var, m, v = np.zeros((1, 1)), np.zeros((1, 1)), np.zeros((1, 1))
    A.sparse_adam(var, m, v, np.array([0]), np.ones((1, 1)), LR, A.initial_powers(dtype=np.float64))
    assert v[0, 0] == np.float64(np.float32(1) - np.float32(0.999)) and v[0, 0] != 1 - 0.999
    assert m[0, 0] == np.float64(np.float32(1) - np.float32(0.9))


def test_sparse_equals_dense_on_the_scattered_gradient():
    rng = np.random.default_rng(3)
    var = rng.standard_normal((30, 4))
    ds = [var.copy(), np.zeros_like(var), np.zeros_like(var)]
    ss = [var.copy(), np.zeros_like(var), np.zeros_like(var)]
    bp_d, bp_s = A.initial_powers(dtype=np.float64), A.initial_powers(dtype=np.float64)
    for _ in range(4):
        rows = np.unique(rng.integers(0, 30, 9))
        g = rng.standard_normal((rows.size, 4))
        dense = np.zeros_like(var)
        dense[rows] = g
        A.dense_adam(*ds, dense, LR, bp_d, epsilon=1e-4)
        A.sparse_adam(*ss, rows, g, LR, bp_s, epsilon=1e-4)
        A.finish(bp_d)
        A.finish(bp_s)
    for a, b in zip(ds, ss):
        np.testing.assert_allclose(a, b, rtol=1e-12, atol=1e-15)


def test_tf_adam_torch_optimizer_matches_dense_adam(pkg):
    rng = np.random.default_rng(4)
    shapes = [(7, 5), (5,), (1,)]
    p0 = [rng.standard_normal(s).astype(np.float32) for s in shapes]
    params = [torch.nn.Parameter(torch.tensor(a)) for a in p0]
    opt = pkg.TFAdam(params, LR, epsilon=1e-4)          # TF's defaults 0.9 / 0.999, whose 1 - beta round in fp32
    ref = [[a.copy(), np.zeros_like(a), np.zeros_like(a)] for a in p0]
    bp = A.initial_powers(dtype=np.float32)
    for _ in range(3):
        grads = [rng.standard_normal(s).astype(np.float32) * 0.1 for s in shapes]
        for p, g in zip(params, grads):
            p.grad = torch.tensor(g)
        opt.step()
        for r, g in zip(ref, grads):
            A.dense_adam(*r, g, LR, bp, epsilon=1e-4)
        A.finish(bp)
    for p, r in zip(params, ref):
        np.testing.assert_allclose(p.detach().numpy(), r[0], rtol=2e-6, atol=1e-7)
        st = opt.state[p]
        np.testing.assert_allclose(st["m"].numpy(), r[1], rtol=2e-6, atol=1e-9)
        np.testing.assert_allclose(st["v"].numpy(), r[2], rtol=2e-6, atol=1e-12)
    assert np.array_equal(opt.beta_power.numpy(), bp)
    with pytest.raises(ValueError):
        pkg.TFAdam(params, LR, epsilon=0.0)
    with pytest.raises(ValueError):
        pkg.TFAdam(params, LR, beta1=1.0)


def _call(lib, _lib, opt, K=16, row_stride=48, n_rows=100, table=16, partials=None, F=2, clip=100.0, lin=None,
          linear_opt=None, n_capacity=0):
    return lib.dir_rows_apply_adam(table, row_stride, n_rows, K, lin, None, 1, linear_opt, None, K + 4, None, None,
                                   n_capacity, 16, F, partials, clip, ctypes.byref(opt) if opt else None, None, None)


def test_apply_adam_validates_before_any_launch(pkg):
    from dir_b200 import _lib
    lib = _lib.lib()
    P = 16                                    # any non-NULL, 16-byte aligned "pointer": nothing dereferences it

    def opt(lr=0.01, b1=0.9, b2=0.999, eps=1e-8, bp=P):
        return _lib.AdamOpt(lr, b1, b2, eps, bp)

    cases = [(dict(opt=opt(b1=1.0)), b"beta"), (dict(opt=opt(b2=-0.1)), b"beta"), (dict(opt=opt(b1=float("nan"))), b"beta"),
             (dict(opt=opt(eps=0.0)), b"epsilon"), (dict(opt=opt(lr=0.0)), b"lr"), (dict(opt=opt(bp=None)), b"null"),
             (dict(opt=None), b"null"), (dict(opt=opt(), K=12), b"K must be"), (dict(opt=opt(), row_stride=32), b"row_stride"),
             (dict(opt=opt(), table=P + 4), b"aligned"), (dict(opt=opt(), n_rows=0), b"n_rows"),
             (dict(opt=opt(), n_capacity=8), b"null"), (dict(opt=opt(), partials=P, clip=0.0), b"clip_norm"),
             (dict(opt=opt(), partials=P, F=0), b"F"), (dict(opt=opt(), lin=P), b"linear_opt")]
    for kw, msg in cases:
        rc = _call(lib, _lib, **kw)
        assert rc == -22 and msg in lib.dir_last_error(), (kw, lib.dir_last_error())
    bad_lin = _lib.LinearOpt(_lib.OPT_FTRL, 0.2, 0.0, 0.0, None)
    rc = _call(lib, _lib, opt(), lin=P, linear_opt=ctypes.byref(bad_lin))
    assert rc == -22 and b"lin_accum" in lib.dir_last_error()


def test_layer_and_models_arguments(pkg):
    kw = dict(device="cpu")
    lay = pkg.EmbeddingFM(2, 8, [4, 5], optimizer="adam", first_order=False, **kw)
    assert lay.row_stride == 24 and lay.accum is None and lay.n_onerow_fields == 0
    assert lay.adam_m.shape == (9, 8) and not lay.adam_m.any() and not lay.adam_v.any()
    assert lay.beta_power.dtype == torch.float32 and lay.beta_power.tolist() == [np.float32(0.9), np.float32(0.999)]
    one = pkg.EmbeddingFM(3, 8, [4, 1, 1], optimizer="adam", linear_optimizer="ftrl", **kw)
    assert one.n_onerow_fields == 0 and one.n_sorted_fields == 3 and one.lin_z is not None
    assert pkg.EmbeddingFM(3, 8, [4, 1, 1], **kw).n_onerow_fields == 2        # the default layer keeps its split
    for bad in (dict(optimizer_beta1=1.0), dict(optimizer_beta2=-0.5), dict(optimizer_epsilon=0.0), dict(lr=0.0)):
        with pytest.raises(ValueError):
            pkg.EmbeddingFM(2, 8, [4, 5], optimizer="adam", first_order=False, **bad, **kw)
    with pytest.raises(ValueError, match="first-order"):
        pkg.EmbeddingFM(2, 8, [4, 5], optimizer="adam", **kw)
    with pytest.raises(ValueError):
        pkg.EmbeddingFM(2, 8, [4, 5], optimizer="adam", linear_optimizer="adam", **kw)
    with pytest.raises(ValueError):
        pkg.ShardedEmbeddingFM(2, 8, [4, 5], optimizer="adam", first_order=False, **kw)
    with pytest.raises(ValueError):
        pkg.EmbeddingBagFM(2, 8, [4, 5], optimizer="adam", first_order=False, **kw)
    with pytest.raises(ValueError):
        pkg.DeepFM(2, 8, [4, 5], dnn_optimizer="adam", linear_optimizer="ftrl", **kw)
    with pytest.raises(ValueError):
        pkg.DCN(2, 8, [4, 5], optimizer="adam", sharded=True, **kw)
    dcn = pkg.DCN(2, 8, [4, 5], optimizer="adam", hidden_units=(8,), **kw)
    assert dcn.embedding.optimizer == "adam" and dcn.embedding.optimizer_epsilon == 1e-4
    assert dcn.embedding.clip_norm == 100.0 and isinstance(dcn.dense_optimizer(), pkg.TFAdam)
    assert pkg.DCN(2, 8, [4, 5], hidden_units=(8,), **kw).embedding.optimizer == "adagrad"
    from dir_b200 import layers
    assert "adam" not in layers._TABLE_OPTIMIZERS and "adam" not in layers._LINEAR_OPTIMIZERS


def test_checkpoint_names_round_trip(pkg):
    lay = pkg.EmbeddingFM(2, 4, [3, 5], optimizer="adam", linear_optimizer="ftrl", device="cpu")
    rng = np.random.default_rng(5)
    with torch.no_grad():
        lay.rows.copy_(torch.tensor(rng.standard_normal((8, 12)).astype(np.float32)))
        lay.beta_power.copy_(torch.tensor([0.729, 0.997003]))
    out = lay.export_columns(["a", "b"], with_slots=True)
    assert out["b/embedding_weights/Adam"].shape == (5, 4) and out["a/embedding_weights/Adam_1"].shape == (3, 4)
    assert np.array_equal(out["b/embedding_weights/Adam"].numpy(), lay.rows[3:, 4:8].numpy())
    assert np.array_equal(out["a/embedding_weights/Adam_1"].numpy(), lay.rows[:3, 8:].numpy())
    assert float(out["beta1_power"]) == np.float32(0.729) and "a/embedding_weights/Adagrad" not in out
    fresh = pkg.EmbeddingFM(2, 4, [3, 5], optimizer="adam", linear_optimizer="ftrl", device="cpu")
    fresh.import_columns(out, ["a", "b"])
    assert torch.equal(fresh.rows, lay.rows) and torch.equal(fresh.beta_power, lay.beta_power)
    adagrad = pkg.EmbeddingFM(2, 4, [3, 5], device="cpu")
    with pytest.raises(ValueError):
        adagrad.import_columns(out, ["a", "b"])


@pytest.mark.parametrize("clip", [100.0, 0.05])
def test_dcn_gradients_are_full_models_gradients(clip):
    """tf_adam.dcn_gradients restates the DCN backward of full_models.dcn_train_step; pin the two together.  Adagrad
    with accumulator A and lr = sqrt(A) moves a variable by g / sqrt(1 + g^2 / A): with A = 1e30 that is g to fp64
    precision, so full_models' step exposes the gradients it applies as p_before - p_after."""
    from oracle import full_models as FM
    from oracle import tf_semantics as tfs
    from tests._util import make_case
    rows = [50, 1, 9, 1000, 3, 17, 1]
    case = make_case(12, 96, rows, 8, weighted=True, prune=True)
    rng, F, d = case["rng"], case["F"], case["F"] * 8
    labels = (rng.random(96) < 0.3).astype(np.float64)
    W, b = FM.make_tower(rng, d, (16, 8), 0, np.float64)
    p = dict(table=case["table"].astype(np.float64), cross_w=tfs.truncated_normal(rng, (2, d), 0.1, np.float64),
             cross_b=tfs.truncated_normal(rng, (2, d), 0.1, np.float64), W=W, b=b,
             Wl=FM.glorot_uniform(rng, d + 8, 1, np.float64), bl=np.asarray([0.02]))
    p0 = {k: ([a.copy() for a in v] if isinstance(v, list) else np.copy(v)) for k, v in p.items()}
    want = A.dcn_gradients(p0, case["off"], case["idx"], case["val"], labels, clip_norm=clip)
    ref = FM.dcn_train_step(p, FM.adagrad_state(p, init=1e30), case["off"], case["idx"], case["val"], labels, 1e15,
                            clip_norm=clip)
    assert ref["loss"] == want["loss"] and np.array_equal(ref["logits"], want["logits"])
    assert np.array_equal(ref["rows"], want["rows"]) and np.array_equal(ref["G"], want["G"])
    if clip < 1:
        assert not np.array_equal(want["G"], want["G_unclipped"]), "the clip must bind on a column"

    def close(before, after, grad):
        np.testing.assert_allclose(before - after, grad, rtol=1e-8, atol=1e-14 * (1 + np.abs(before).max()))

    close(p0["table"][want["rows"]], p["table"][want["rows"]], want["G"])
    for k, g in want["dense"].items():
        for before, after, gi in (zip(p0[k], p[k], g) if isinstance(g, list) else [(p0[k], p[k], g)]):
            close(before, after, gi)


def test_tf_adam_state_dict_carries_the_powers(pkg):
    params = [torch.nn.Parameter(torch.ones(3))]
    opt = pkg.TFAdam(params, LR, epsilon=1e-4)
    for _ in range(2):
        params[0].grad = torch.full((3,), 0.5)
        opt.step()
    import io
    buf = io.BytesIO()
    torch.save(opt.state_dict(), buf)             # a checkpoint: nothing shared with the running optimizer
    buf.seek(0)
    sd = torch.load(buf)
    again = pkg.TFAdam([torch.nn.Parameter(params[0].detach().clone())], LR, epsilon=1e-4)
    again.load_state_dict(sd)
    assert torch.equal(again.beta_power, opt.beta_power)
    bp = A.initial_powers(dtype=np.float32)
    A.finish(bp)
    A.finish(bp)
    assert np.array_equal(again.beta_power.numpy(), bp)
    for o in (opt, again):
        o.param_groups[0]["params"][0].grad = torch.full((3,), 0.5)
        o.step()
    assert torch.equal(again.param_groups[0]["params"][0], params[0]) and torch.equal(again.beta_power, opt.beta_power)
