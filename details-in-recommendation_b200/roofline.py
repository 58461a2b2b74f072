"""ALGORITHMIC bytes of each kernel of the path (SURVEY.md section 8d, BASELINE.md section 2).

These are the only byte counts `bench.py`'s `roofline.achieved` may use: sort passes, `S[B,K]`,
workspaces and cache re-reads are excluded by definition.  I = 8 (int64 id), V = 4 (fp32 value, 0
when feature_value is None), R = 4K (one row), E = B*F*R when [B,F,K] embeddings / upstream
gradients cross the layer boundary (a DNN or cross consumer is attached) else 0, U = distinct
rows a batch touches, c = 4 for Adagrad (read+write row, read+write accumulator), 2 for SGD.
"""
import json
import os

I_BYTES = 8
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def embed_fwd_bytes(B, F, K, weighted=True, emit=True):
    """lookup + first order + FM forward: ids, values, K-row, first-order weight per lookup;
    write first + fm per sample; + emitted embeddings."""
    V, R = (4 if weighted else 0), 4 * K
    return B * F * (I_BYTES + V + R + 4) + 8 * B + (B * F * R if emit else 0)


def embed_bwd_bytes(B, F, K, U, weighted=True, upstream=True, optimizer="adagrad"):
    """backward + fused row update: g per sample, upstream u, per lookup id + value + one K-vector,
    per distinct row (row + first-order weight) x c."""
    V, R = (4 if weighted else 0), 4 * K
    c = 4 if optimizer == "adagrad" else 2
    return 4 * B + (B * F * R if upstream else 0) + B * F * (I_BYTES + V + R) + U * (R + 4) * c


def adam_apply_bytes(n_rows, K, U, first_order=False, linear_optimizer=None):
    """dir_rows_apply_adam: TF's Adam decays every row's moments, so the sweep reads and writes all n_rows rows
    [T | m | v] (3R each way) plus, per distinct row, its index (4 B) and its gradient G and, with first-order
    weights, g1 and the weight's state (as embed_bwd_bytes counts it: c = 4 for Adagrad / Ftrl-like, 2 for SGD)."""
    R = 4 * K
    lin = 0
    if first_order:
        c = 2 if linear_optimizer == "sgd" else 4
        lin = U * (4 + 4 * c + (8 if linear_optimizer == "ftrl" else 0))
    return n_rows * 3 * R * 2 + U * (4 + R) + lin


def shard_adam_apply_bytes(n_local, K, arrivals, G, U=None, first_order=False, linear_optimizer=None):
    """dir_shard_owner_apply_adam on one owner: the sweep reads and writes all n_local rows [T | m | v] (3R each way);
    each of the `arrivals` (every requester's distinct rows that reached this owner) costs its id (4 B, the tile map),
    its gradient sum (R) and its row's slot cells (4G, the rank-order merge).  With first-order weights, per distinct
    row U (default: arrivals) its g1 (4 B) and the weight's state as adam_apply_bytes counts it."""
    R = 4 * K
    U = arrivals if U is None else U
    lin = 0
    if first_order:
        c = 2 if linear_optimizer == "sgd" else 4
        lin = arrivals * 4 + U * (4 * c + (8 if linear_optimizer == "ftrl" else 0))
    return n_local * 3 * R * 2 + arrivals * (4 + R + 4 * G) + lin


def cross_fwd_bytes(B, d, L):
    return 2 * B * d * 4 + 2 * L * d * 4


def cross_bwd_bytes(B, d, L):
    return 3 * B * d * 4 + 4 * L * d * 4


def measured_peaks():
    """(hbm GB/s, source): MEASURED_PEAKS.json (driver-written) else the profiling recipe's fallback."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except (OSError, KeyError, ValueError):
        return 6650.0, "fallback"
