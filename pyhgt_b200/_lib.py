"""ctypes binding of libhgt_b200.so (C ABI declared in include/hgt_b200.h).

The library is built in-tree by ``pyhgt_b200/build.py`` (nvcc, sm_100a).  There is NO fallback: if the
shared object is missing or a symbol is absent, loading raises.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libhgt_b200.so")

_c = ctypes
_p = _c.c_void_p
_i32 = _c.c_int32
_i64 = _c.c_int64
_sz = _c.c_size_t

# name -> argtypes; every function returns int except where noted.  Mirrors include/hgt_b200.h.
SIGNATURES = {
    "hgt_abi_version": [],
    "hgt_plan_workspace_bytes": [_i64, _i64, _c.POINTER(_sz)],
    "hgt_plan_nodes": [_p, _i64, _i32, _p, _p, _p, _p, _p, _sz, _p],
    "hgt_plan_edges_sort": [_p, _p, _p, _p, _i64, _i64, _i32, _i32, _p, _p, _p, _p, _p, _sz, _p],
    "hgt_plan_edges_fill": [_p, _p, _p, _p, _p, _p, _i64, _i64, _i32, _i32, _p, _p, _p, _i32, _i32, _p, _p, _p, _p],
    "hgt_plan_tiles": [_p, _i64, _i64, _i32, _i32, _p, _i64, _p, _i64, _p, _c.POINTER(_i32), _p, _sz, _p],
    "hgt_gather_rows": [_p, _p, _i64, _i32, _p, _p],
    "hgt_halo_pull": [_c.c_uint64, _p, _p, _i64, _i32, _i64, _p, _p],
    "hgt_halo_pull_split": [_c.c_uint64, _p, _p, _p, _i64, _i32, _i32, _i64, _p, _p, _p, _p],
    "hgt_halo_push_split": [_p, _p, _p, _p, _i64, _i32, _i32, _i64, _c.c_uint64, _c.c_uint64, _p, _p],
    "hgt_fold_weights": [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p, _p, _p,
                         _p, _p, _p],
    "hgt_concat_linears": [_p, _p, _i32, _i32, _i32, _p, _p, _p],
    "hgt_typed_linear_workspace_bytes": [_p, _i32, _i32, _i32, _i32, _c.POINTER(_sz)],
    "hgt_typed_linear": [_p, _i64, _p, _p, _i32, _i32, _p, _p, _i32, _p, _p, _i32, _p, _sz, _p],
    "hgt_edge_workspace_bytes": [_i32, _i32, _i32, _c.POINTER(_sz)],
    "hgt_edge_forward": [_p, _p, _p, _p, _p, _p, _p, _p, _i32, _i32, _p, _i32, _i64, _i64, _i32, _i32, _i32, _p, _p,
                         _p, _p, _p, _p, _sz, _i32, _p, _p, _i32, _p, _p],
    "hgt_typed_linear_presplit_workspace_bytes": [_p, _i32, _i32, _i32, _c.POINTER(_sz)],
    "hgt_typed_linear_presplit": [_p, _p, _p, _p, _i32, _i32, _p, _p, _i32, _p, _p, _p, _sz, _p],
    "hgt_edge_backward": [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i32, _i64, _i32, _i32, _i64, _i64, _p, _p, _p, _p, _sz,
                          _p, _p],
    "hgt_typed_linear_bwd_workspace_bytes": [_p, _i32, _p, _i32, _i32, _i64, _i64, _i32, _i32, _i32, _c.POINTER(_sz)],
    "hgt_typed_linear_bwd": [_p, _p, _p, _i64, _p, _i64, _p, _p, _p, _i32, _i32, _p, _p, _i32, _p, _p, _i32, _p, _p, _p,
                             _i32, _p, _sz, _p],
    "hgt_act_split": [_p, _i64, _i64, _i32, _i32, _p, _p, _p, _p],
    "hgt_update_backward": [_p, _p, _p, _p, _i32, _p, _p, _p, _p, _i64, _i32, _p, _p, _p, _p, _p, _p],
    "hgt_fold_backward": [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p, _p, _p, _p, _p,
                          _p, _p, _p, _p, _p],
    "hgt_conv_workspace_bytes": [_p, _c.POINTER(_sz)],
    "hgt_conv_forward": [_p, _p, _sz, _p],
    "hgt_update_epilogue": [_p, _p, _p, _i32, _p, _p, _p, _p, _p, _i64, _i32, _p, _p, _p, _p],
    # deterministic backward (torch.use_deterministic_algorithms)
    "hgt_plan_group_by_workspace_bytes": [_i64, _i32, _c.POINTER(_sz)],
    "hgt_plan_group_by": [_p, _i64, _i32, _p, _p, _p, _sz, _p],
    "hgt_plan_csr_dst": [_p, _i64, _i64, _p, _p],
    "hgt_edge_backward_det_workspace_bytes": [_i64, _i32, _i32, _p, _p, _p, _c.POINTER(_sz)],
    "hgt_edge_backward_det": [_p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _i64, _i32, _i32, _p, _p, _p, _p, _sz, _p],
    "hgt_typed_linear_bwd_det_workspace_bytes": [_p, _i32, _p, _i32, _i32, _i64, _i64, _i32, _i32, _i32,
                                                 _c.POINTER(_sz)],
    "hgt_typed_linear_bwd_det": [_p, _p, _p, _i64, _p, _i64, _p, _p, _p, _i32, _i32, _p, _p, _i32, _p, _p, _i32, _p, _p,
                                 _p, _i32, _p, _sz, _p],
    "hgt_update_backward_det_workspace_bytes": [_i64, _i32, _i32, _c.POINTER(_sz)],
    "hgt_update_backward_det": [_p, _p, _p, _p, _i32, _p, _p, _p, _p, _i64, _i32, _p, _p, _p, _p, _p, _p, _sz, _p],
    "hgt_fold_backward_det_workspace_bytes": [_i32, _i32, _i32, _c.POINTER(_sz)],
    "hgt_fold_backward_det": [_p, _p, _p, _p, _p, _p, _p, _p, _p, _i32, _i32, _i32, _i32, _i32, _i32, _p, _p, _p, _p, _p,
                              _p, _p, _p, _p, _p, _p, _sz, _p],
}


class TileSet(ctypes.Structure):
    """Mirror of `hgt_tile_set` (include/hgt_b200.h): one edge index of the deterministic edge backward."""
    _fields_ = [("ptr", ctypes.c_void_p), ("pos", ctypes.c_void_p), ("tiles", ctypes.c_void_p),
                ("hubs", ctypes.c_void_p), ("d_counts", ctypes.c_void_p), ("n_tiles", ctypes.c_int32),
                ("n_split", ctypes.c_int32), ("n_hubs", ctypes.c_int32), ("reserved", ctypes.c_int32)]

class ConvArgs(ctypes.Structure):
    """Mirror of `hgt_conv_args` (include/hgt_b200.h); field order and types must match the C struct exactly
    (checked against hgt_conv_args_size() in tests/test_capi.py)."""
    _I64 = ["n_nodes", "n_edges", "kv_rows", "cat_rows", "q_off", "kv_off", "proj_elems"]
    _I32 = ["num_types", "num_relations", "n_heads", "d_in", "d_out", "n_pairs", "use_rte", "use_norm", "edge_variant",
            "linear_impl", "n_tiles", "n_split", "n_hubs", "n_proj_groups", "n_rte_groups", "n_upd_groups"]
    _PTR = ["perm", "type_row0", "type_active", "out_map", "row_ptr", "kv_row", "rte_row", "csr_eid", "tiles", "hubs",
            "d_tile_counts", "pair_type", "pair_rel", "cat_row0", "q_row0",
            "proj_groups", "h_proj_groups", "proj_cblocks", "rte_groups", "h_rte_groups", "rte_cblocks",
            "rt_groups", "h_rt_groups", "rt_cblocks", "upd_groups", "h_upd_groups", "upd_cblocks",
            "wq", "bq", "wk", "bk", "wv", "bv", "wa", "ba", "norm_w", "norm_b",
            "relation_att", "relation_msg", "relation_pri", "skip", "emb_weight", "emb_lin_w", "emb_lin_b",
            "x", "x_hi", "x_lo", "out", "att", "out_hi", "out_lo"]
    _fields_ = ([(n, ctypes.c_int64) for n in _I64] + [(n, ctypes.c_int32) for n in _I32] +
                [(n, ctypes.c_void_p) for n in _PTR])


LIN_GROUP_DTYPE = np.dtype([("a_row0", "<i8"), ("m", "<i8"), ("w_row0", "<i4"), ("n_cblocks", "<i4"),
                            ("cb_first", "<i4"), ("has_bias", "<i4")])
LIN_CBLOCK_DTYPE = np.dtype([("out_off", "<i8"), ("ld", "<i8")])
assert LIN_GROUP_DTYPE.itemsize == 32 and LIN_CBLOCK_DTYPE.itemsize == 16

_lib = None


class HgtError(RuntimeError):
    pass


def load():
    """Load the shared library once and attach argtypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise HgtError("libhgt_b200.so not found at %s — run `python -m pyhgt_b200.build` "
                       "(or __graft_entry__.build()); there is no CPU fallback" % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    lib.hgt_last_error.restype = _c.c_char_p
    lib.hgt_last_error.argtypes = []
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing: loud by design
        fn.restype = _c.c_int
        fn.argtypes = args
    lib.hgt_kernel_launches.restype = _c.c_uint64
    lib.hgt_kernel_launches.argtypes = []
    lib.hgt_conv_args_size.restype = _c.c_uint64
    lib.hgt_conv_args_size.argtypes = []
    lib.hgt_sampler_budget_update.restype = _c.c_int64       # host helper of sampler.py: returns a count, not a status
    lib.hgt_sampler_budget_update.argtypes = [_p, _p, _i64, _i64, _i64, _i64, _i64, _p, _p, _p, _p, _p, _p, _p]
    lib.hgt_sampler_add_budget.restype = _c.c_int64
    lib.hgt_sampler_add_budget.argtypes = [_p, _p, _i64, _p, _c.c_int32, _p, _c.c_int32, _i64, _p, _p, _i64, _i64, _p]
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().hgt_last_error()
        raise HgtError("%s failed (code %d): %s" % (what, rc, msg.decode() if msg else "?"))


def call(name, *args):
    lib = load()
    check(getattr(lib, name)(*args), name)


def kernel_launches():
    return int(load().hgt_kernel_launches())


def ptr(t):
    """Device (or host) address of a torch tensor, or None."""
    return None if t is None else t.data_ptr()
