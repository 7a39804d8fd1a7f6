"""ctypes binding of ``libbotgat.so`` (C ABI declared in ``include/botgat.h``).

There is no CPU fallback: if the shared library is missing or a call fails, a
``RuntimeError`` is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BOTGAT_LIB") or os.path.join(_HERE, "libbotgat.so")  # BOTGAT_LIB: developer A/B builds
ABI_VERSION = 5

c_i64p = C.POINTER(C.c_int64)
c_vp = C.c_void_p

# order of BOTGAT_* array ids in include/botgat.h
ARRAYS = ("in_indptr", "in_indices", "in_eid", "out_indptr", "out_indices", "out_eid", "in_deg", "out_deg")
ORDER_IN, ORDER_OUT = 0, 1


class GraphInfo(C.Structure):
    _fields_ = [
        ("n_src", C.c_int64), ("n_dst", C.c_int64), ("n_edges", C.c_int64),
        ("max_in_deg", C.c_int64), ("max_out_deg", C.c_int64),
        ("has_zero_in_degree", C.c_int32), ("device", C.c_int32),
        ("n_slots_in", C.c_int64), ("n_slots_out", C.c_int64),
        ("in_eid_identity", C.c_int32), ("tiles_src", C.c_int32), ("tiles_dst", C.c_int32),
        ("n_seg_in", C.c_int32), ("n_seg_out", C.c_int32), ("reserved_", C.c_int32),
    ]


class EdgeSubset(C.Structure):
    """``botgat_edge_subset``: the kept-edge adjacency of one CSR order (device pointers)."""
    _fields_ = [("indptr", c_vp), ("indices", c_vp), ("eid", c_vp), ("kept", c_vp), ("base", c_vp), ("seg_beg", c_vp), ("seg_end", c_vp)]


class FwdArgs(C.Structure):
    _fields_ = [
        ("H", C.c_int32), ("D", C.c_int32),
        ("ld_ft", C.c_int64), ("ld_out", C.c_int64),
        ("ft", c_vp), ("el", c_vp), ("er", c_vp), ("eb", c_vp),
        ("Hb", C.c_int32), ("col_parts", C.c_int32),
        ("am", c_vp), ("ee", c_vp), ("keep", c_vp), ("attn_mul", c_vp), ("src_scale", c_vp), ("dst_scale", c_vp),
        ("slope", C.c_float), ("attn_p", C.c_float), ("seed", C.c_uint64),
        ("out", c_vp), ("row_max", c_vp), ("row_sum", c_vp), ("scratch", c_vp),
        ("h_begin", C.c_int32), ("h_count", C.c_int32),
        ("res", c_vp), ("ld_res", C.c_int64), ("res2", c_vp), ("ld_res2", C.c_int64),
        ("ep_scale", c_vp), ("ep_shift", c_vp), ("y", c_vp), ("ld_y", C.c_int64),
        ("ep_relu", C.c_int32), ("reserved_", C.c_int32),
        ("subset", C.POINTER(EdgeSubset)),
    ]


class BwdArgs(C.Structure):
    _fields_ = [
        ("H", C.c_int32), ("D", C.c_int32),
        ("ld_ft", C.c_int64), ("ld_out", C.c_int64), ("ld_gft", C.c_int64),
        ("ft", c_vp), ("el", c_vp), ("er", c_vp), ("eb_out", c_vp),
        ("Hb", C.c_int32), ("phases", C.c_int32),
        ("am_out", c_vp), ("ee", c_vp), ("keep", c_vp), ("attn_mul", c_vp), ("src_scale", c_vp), ("dst_scale", c_vp),
        ("slope", C.c_float), ("attn_p", C.c_float), ("seed", C.c_uint64),
        ("out", c_vp), ("row_max", c_vp), ("row_sum", c_vp), ("gout", c_vp),
        ("drec", c_vp), ("gprime", c_vp), ("scratch", c_vp), ("gz", c_vp),
        ("grad_ft", c_vp), ("grad_el", c_vp), ("grad_ee", c_vp), ("ld_gee", C.c_int64), ("grad_er", c_vp),
        ("h_begin", C.c_int32), ("h_count", C.c_int32),
        ("subset_out", C.POINTER(EdgeSubset)),
    ]


# symbol -> (restype, argtypes); every symbol include/botgat.h declares
SIGNATURES = {
    "botgat_abi_version": (C.c_int, []),
    "botgat_last_error": (C.c_char_p, []),
    "botgat_launch_count": (C.c_int64, []),
    "botgat_graph_create": (C.c_int, [C.c_int64, C.c_int64, C.c_int64, c_vp, c_vp, C.c_int, c_vp, C.POINTER(c_vp)]),
    "botgat_graph_destroy": (None, [c_vp]),
    "botgat_graph_destroy_async": (None, [c_vp, c_vp]),
    "botgat_graph_get": (C.c_int, [c_vp, C.c_int, C.POINTER(c_vp), c_i64p]),
    "botgat_graph_get_info": (C.c_int, [c_vp, C.POINTER(GraphInfo)]),
    "botgat_coo_to_bidirected": (C.c_int, [C.c_int64, C.c_int64, c_vp, c_vp, c_vp, c_vp, c_i64p, C.c_int, c_vp]),
    "botgat_coo_remove_self_loop": (C.c_int, [C.c_int64, c_vp, c_vp, c_vp, c_vp, c_i64p, C.c_int, c_vp]),
    "botgat_coo_add_self_loop": (C.c_int, [C.c_int64, C.c_int64, c_vp, c_vp, c_vp, c_vp, C.c_int, c_vp]),
    "botgat_edge_stage": (C.c_int, [c_vp, C.c_int, C.c_int32, c_vp, C.c_int64, c_vp, c_vp, C.c_int64, c_vp, c_vp,
                                    C.POINTER(EdgeSubset), c_vp]),
    "botgat_edge_unstage": (C.c_int, [c_vp, C.c_int, C.c_int32, c_vp, c_vp, C.c_int64, C.POINTER(EdgeSubset), c_vp]),
    "botgat_edge_reduce_dst": (C.c_int, [c_vp, C.c_int32, c_vp, C.c_int64, c_vp, c_vp, c_vp]),
    "botgat_sample_workspace_bytes": (C.c_int64, [C.c_int64]),
    "botgat_sample_count": (C.c_int, [c_vp, C.c_int64, c_vp, C.c_int32, c_vp, C.POINTER(C.c_int64), c_vp, c_vp]),
    "botgat_sample_neighbors": (C.c_int, [c_vp, C.c_int64, c_vp, C.c_int32, C.c_uint64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "botgat_block_workspace_bytes": (C.c_int64, [C.c_int64]),
    "botgat_block_compact": (C.c_int, [C.c_int64, C.c_int64, c_vp, C.c_int64, c_vp, c_vp, c_vp, C.POINTER(C.c_int64), c_vp,
                                       C.c_int, c_vp]),
    "botgat_edge_drop_workspace_bytes": (C.c_int64, [C.c_int64]),
    "botgat_edge_drop_draw": (C.c_int, [C.c_int64, C.c_int64, C.c_uint64, c_vp, c_vp, C.c_int, c_vp]),
    "botgat_edge_mlp_supported": (C.c_int, [C.c_int32, C.c_int32, C.c_int32]),
    "botgat_edge_mlp_workspace_floats": (C.c_int64, [C.c_int32, C.c_int32, C.c_int32]),
    "botgat_edge_mlp_forward": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.c_int32, c_vp, C.c_int64, c_vp, c_vp, c_vp, c_vp,
                                          C.c_int64, C.c_int, c_vp]),
    "botgat_edge_mlp_backward": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, C.c_int32, c_vp, C.c_int64, c_vp, c_vp, c_vp, c_vp,
                                           C.c_int64, c_vp, c_vp, c_vp, c_vp, C.c_int, c_vp]),
    "botgat_edge_proj_gw_blocks": (C.c_int, []),
    "botgat_edge_proj_forward": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, c_vp, C.c_int64, c_vp, c_vp, C.c_int64, C.c_int, c_vp]),
    "botgat_edge_proj_backward": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, c_vp, C.c_int64, c_vp, c_vp, C.c_int64, c_vp,
                                            C.c_int64, c_vp, c_vp, C.c_int, c_vp]),
    "botgat_gat_forward": (C.c_int, [c_vp, C.POINTER(FwdArgs), c_vp]),
    "botgat_gat_backward": (C.c_int, [c_vp, C.POINTER(BwdArgs), c_vp]),
    "botgat_partition_1d": (C.c_int, [c_vp, C.c_int32, c_i64p, c_vp]),
    "botgat_partition_extract": (C.c_int, [c_vp, C.c_int64, C.c_int64, c_vp, c_vp, c_vp, c_i64p, c_vp]),
    "botgat_rows_gather": (C.c_int, [c_vp, C.c_int64, C.c_int64, c_vp, C.c_int64, c_vp, c_vp]),
    "botgat_rows_scatter_add": (C.c_int, [c_vp, C.c_int64, C.c_int64, c_vp, C.c_int64, c_vp, c_vp]),
    "botgat_halo_pull": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(c_vp), C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int32, c_vp]),
    "botgat_halo_pull_reduce": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(c_vp), C.c_int64, C.c_int64, C.c_int64, C.c_int64, c_vp,
                                          C.c_int64, C.c_int32, c_vp]),
}

_lib = None


def load():
    """Load libbotgat.so (once) and bind every declared symbol.  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C bot_b200/csrc -j`.  bot_b200 has no CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    v = lib.botgat_abi_version()
    if v != ABI_VERSION:
        raise RuntimeError(f"libbotgat ABI version {v} != expected {ABI_VERSION}; rebuild")
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().botgat_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")


def ptr(t):
    """Device pointer of a tensor (or NULL for None)."""
    return None if t is None else C.c_void_p(t.data_ptr())
