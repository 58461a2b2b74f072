"""ctypes binding of libdir_b200.so (the C ABI declared in include/dir_b200.h).

No CPU fallback: if the shared library is missing or a call fails, this raises.
"""
import ctypes
import os
import subprocess
from ctypes import c_char_p, c_float, c_int, c_int64, c_size_t, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdir_b200.so")
CSRC = os.path.join(_HERE, "csrc")

OPT_SGD, OPT_ADAGRAD, OPT_FTRL, OPT_PROXIMAL_ADAGRAD = 0, 1, 2, 3


class LinearOpt(ctypes.Structure):
    """struct dir_linear_opt (include/dir_b200.h): the linear scope's own optimizer."""
    _fields_ = [("optimizer", c_int), ("lr", c_float), ("l1", c_float), ("l2", c_float), ("z", c_void_p)]


class TableOpt(ctypes.Structure):
    """struct dir_table_opt (include/dir_b200.h): l1 / l2 of a ProximalAdagrad table optimizer."""
    _fields_ = [("l1", c_float), ("l2", c_float)]


class AdamOpt(ctypes.Structure):
    """struct dir_adam_opt (include/dir_b200.h): Adam's hyper-parameters and its device-resident beta powers."""
    _fields_ = [("lr", c_float), ("beta1", c_float), ("beta2", c_float), ("epsilon", c_float), ("beta_power", c_void_p)]


class PeerLayout(ctypes.Structure):
    """struct dir_peer_layout (include/dir_b200.h): the exchange buffer every rank owns, per parity."""
    _fields_ = [("G", c_int), ("rank", c_int), ("K", c_int), ("n_dense", c_int),
                ("seg_cap", c_int64), ("u_cap", c_int64),
                ("off_hdr", c_int64), ("off_ids", c_int64), ("off_rows", c_int64), ("off_w", c_int64),
                ("off_g", c_int64), ("off_g1", c_int64), ("off_dense", c_int64), ("total_bytes", c_int64),
                ("peer_base", c_void_p), ("local", c_void_p)]


_EINVAL, _ENOMEM, _EIO = -22, -12, -5

# name -> (restype, argtypes); must list every symbol include/dir_b200.h declares
SIGNATURES = {
    "dir_version": (c_int, []),
    "dir_last_error": (c_char_p, []),
    "dir_launch_count": (c_uint64, []),
    "dir_embed_fm_fwd": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_void_p, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dir_embed_bwd_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "dir_embed_bwd_sort": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_size_t, c_void_p]),
    "dir_embed_bwd_reduce_update": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64,
                                            c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                            c_int64, c_int, c_int, c_int64, c_void_p, c_int, c_void_p, c_int,
                                            c_int, c_float, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p]),
    "dir_embed_bwd_onerow_update": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p,
                                            c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64,
                                            c_int, c_int, c_void_p, c_int, c_int, c_float, c_void_p, c_void_p, c_float,
                                            c_void_p, c_size_t, c_void_p, c_void_p]),
    "dir_embed_bwd_reduce_emit_local": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                c_void_p, c_int64, c_int, c_int, c_int64, c_void_p, c_int, c_void_p,
                                                c_int64, c_void_p, c_size_t, c_void_p]),
    "dir_field_sqnorms_bytes": (c_size_t, [c_int]),
    "dir_field_sqnorms": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int64, c_void_p,
                                  c_void_p]),
    "dir_rows_apply_clipped": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_int64,
                                       c_void_p, c_void_p, c_int64, c_void_p, c_int, c_int, c_void_p, c_float, c_int,
                                       c_float, c_void_p, c_void_p, c_void_p]),
    "dir_rows_apply_adam": (c_int, [c_void_p, c_int64, c_int64, c_int, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                    c_int64, c_void_p, c_void_p, c_int64, c_void_p, c_int, c_void_p, c_float, c_void_p,
                                    c_void_p, c_void_p]),
    "dir_embed_bwd_sorted": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "dir_shard_keys": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int,
                               c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "dir_shard_bag_keys": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64,
                                   c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "dir_embed_bag_bwd_reduce_emit_to": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                                 c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int,
                                                 c_int64, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dir_shard_keys_sort": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int,
                                    c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dir_shard_unique_workspace_bytes": (c_size_t, [c_int64]),
    "dir_shard_unique": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int, c_void_p, c_int, c_int, c_void_p,
                                 c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "dir_shard_dense_inv": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int, c_int64, c_void_p, c_void_p,
                                    c_void_p]),
    "dir_peer_layout_init": (c_int, [c_int, c_int, c_int, c_int, c_int64, c_int64, c_void_p]),
    "dir_shard_ids_push": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "dir_shard_slots": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dir_shard_gather_send": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_void_p,
                                      c_int, c_void_p]),
    "dir_embed_bwd_reduce_emit_to": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                             c_void_p, c_int64, c_int, c_int64, c_void_p, c_int, c_void_p, c_void_p,
                                             c_size_t, c_void_p]),
    "dir_shard_g1_push": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "dir_shard_dense_workspace_bytes": (c_size_t, [c_int]),
    "dir_shard_dense_emit": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_size_t, c_void_p]),
    "dir_shard_owner_update": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64,
                                       c_int64, c_void_p, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_void_p]),
    "dir_shard_dense_apply": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_float,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p,
                                      c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dir_shard_owner_sqnorms": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int, c_int, c_void_p,
                                        c_void_p, c_void_p]),
    "dir_shard_owner_update_clipped": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                               c_int64, c_int64, c_void_p, c_int, c_float, c_void_p, c_void_p, c_int,
                                               c_void_p, c_void_p, c_float, c_void_p, c_void_p]),
    "dir_shard_dense_apply_clipped": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int,
                                              c_float, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p,
                                              c_void_p, c_int64, c_void_p, c_float, c_void_p, c_void_p]),
    "dir_shard_owner_apply_adam": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p,
                                           c_void_p, c_int64, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_float,
                                           c_void_p, c_void_p, c_void_p]),
    "dir_table_init_counter": (c_int, [c_void_p, c_int64, c_int64, c_int, c_int, c_int, c_int64, c_uint64, c_float,
                                       c_void_p]),
    "dir_embed_bag_fm_fwd": (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_int64, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_int, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "dir_embed_bag_bwd_reduce_update": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_void_p,
                                                c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                                c_void_p, c_int64, c_int, c_int, c_int64, c_int, c_float, c_void_p,
                                                c_void_p, c_size_t, c_void_p, c_void_p]),
    "dir_fingerprint64_host": (c_uint64, [c_void_p, c_int64]),
    "dir_fingerprint64": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "dir_hash_bucket": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_void_p]),
    "dir_vocabulary_lookup": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_void_p,
                                      c_int64, c_void_p]),
    "dir_bucketize": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_int, c_void_p, c_int64, c_void_p]),
    "dir_expand_features": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int64, c_int, c_int, c_int,
                                    c_void_p, c_void_p, c_void_p]),
    "dir_input_layer_fwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                                    c_int64, c_int, c_void_p, c_void_p]),
    "dir_input_layer_bwd": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p]),
    "dir_cross_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p,
                              c_void_p, c_void_p]),
    "dir_cross_bwd_workspace_bytes": (c_size_t, [c_int64, c_int, c_int]),
    "dir_cross_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int,
                              c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
}

_lib = None


def build(verbose=False):
    """Compile csrc/*.cu for sm_100a into libdir_b200.so (nvcc cross-compiles without a GPU)."""
    out = subprocess.run(["make", "-C", CSRC, "-j8"], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout[-4000:])
        print(out.stderr[-4000:])
    if out.returncode != 0:
        raise RuntimeError("building libdir_b200.so failed")
    return LIB_PATH


def lib():
    """The loaded library; raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libdir_b200.so is missing (%s): build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` or `make -C %s`.  There is no CPU fallback." % (LIB_PATH, CSRC))
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)      # AttributeError if the symbol is not exported
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(rc, what):
    if rc == 0:
        return
    msg = lib().dir_last_error().decode("utf-8", "replace")
    if rc == _EINVAL:
        raise ValueError("%s: %s" % (what, msg))
    if rc == _ENOMEM:
        raise MemoryError("%s: %s" % (what, msg))
    raise RuntimeError("%s failed (%d): %s" % (what, rc, msg))


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def launch_count():
    return int(lib().dir_launch_count())
