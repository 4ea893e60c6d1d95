"""ctypes binding of libpetal_b200.so (include/petal_b200.h).  Fails loudly when the CUDA
library has not been built: there is no CPU fallback anywhere in this package."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PN_B200_LIB") or os.path.join(_HERE, "lib", "libpetal_b200.so")  # PN_B200_LIB: diagnostic builds

PN_OK, PN_EMPTY, PN_NOT_CONTIGUOUS, PN_BAD_ARG, PN_CUDA, PN_NCCL, PN_OOM = range(7)
PN_KIND_BALL, PN_KIND_VP = 0, 1
PN_F32, PN_F64 = 0, 1
PN_ALGO_AUTO, PN_ALGO_SIMT, PN_ALGO_TENSOR = 0, 1, 2
PN_FLAG_HOST_ONLY = 1
PN_BUILDER_AUTO, PN_BUILDER_HOST, PN_BUILDER_DEVICE = 0, 1, 2
PN_PRUNE_AUTO, PN_PRUNE_ON, PN_PRUNE_OFF = 0, 1, 2
PN_PARTITION_AUTO, PN_PARTITION_REFERENCE, PN_PARTITION_TWO_MEANS = 0, 1, 2

# every symbol include/petal_b200.h declares
EXPORTS = [
    "pn_last_error_message", "pn_abi_version", "pn_device_count",
    "pn_balltree_create_f32", "pn_balltree_create_f64", "pn_vptree_create_f32", "pn_vptree_create_f64",
    "pn_balltree_create_dev_f32", "pn_balltree_create_dev_f64", "pn_tree_destroy", "pn_tree_session",
    "pn_balltree_query_f32", "pn_balltree_query_f64",
    "pn_balltree_query_nearest_f32", "pn_balltree_query_nearest_f64",
    "pn_balltree_query_radius_f32", "pn_balltree_query_radius_f64",
    "pn_vptree_query_nearest_f32", "pn_vptree_query_nearest_f64",
    "pn_vptree_query_f32", "pn_vptree_query_f64", "pn_vptree_query_radius_f32", "pn_vptree_query_radius_f64",
    "pn_balltree_query_self_f32", "pn_balltree_query_self_f64", "pn_tree_query_self_dev",
    "pn_pairwise_f32", "pn_pairwise_f64",
    "pn_free", "pn_tree_query_knn_dev", "pn_tree_query_radius_dev", "pn_merge_topk_dev", "pn_merge_radius_dev",
    "pn_tree_get_info", "pn_tree_get_counters", "pn_tree_get_layout",
    "pn_comm_unique_id", "pn_comm_create", "pn_comm_create_all", "pn_comm_destroy", "pn_query_slice",
    "pn_sharded_query_knn_dev", "pn_tree_replicate",
    "pn_multi_balltree_create_f32", "pn_multi_balltree_query_f32", "pn_multi_balltree_query_radius_f32", "pn_multi_set_exchange", "pn_multi_get_stats", "pn_multi_destroy",
]
PN_SHARD_REPLICATE, PN_SHARD_BY_SUBTREE = 0, 1
PN_EXCHANGE_ALLGATHER, PN_EXCHANGE_SLICE, PN_EXCHANGE_PEER = 0, 1, 2
PN_UNIQUE_ID_BYTES = 128


class ShardStats(C.Structure):
    _fields_ = [("scan_ms", C.c_double), ("exchange_ms", C.c_double), ("merge_ms", C.c_double), ("total_ms", C.c_double),
                ("nccl_bytes_sent", C.c_uint64), ("nccl_calls", C.c_uint64), ("rows_out", C.c_uint64),
                ("n_chunks", C.c_uint32), ("peer_mib", C.c_uint32)]


class BuildOpts(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("device", C.c_int32), ("bucket_size", C.c_uint32),
                ("algo", C.c_uint32), ("host_threads", C.c_uint32), ("flags", C.c_uint32),
                ("shard_depth", C.c_uint32), ("shard_index", C.c_uint32), ("builder", C.c_uint32),
                ("prune", C.c_uint32), ("partition", C.c_uint32), ("reserved", C.c_uint32 * 5)]


class TreeInfo(C.Structure):
    _fields_ = [("n_points", C.c_uint64), ("n_points_total", C.c_uint64), ("dim", C.c_uint32),
                ("dim_padded", C.c_uint32), ("kind", C.c_uint32), ("dtype", C.c_uint32),
                ("n_levels", C.c_uint32), ("n_buckets", C.c_uint32), ("n_nodes", C.c_uint32),
                ("bucket_size_max", C.c_uint32), ("device", C.c_int32), ("algo", C.c_uint32),
                ("device_bytes", C.c_uint64), ("build_seconds", C.c_double),
                ("prune_seeded", C.c_uint32), ("prune_tiles", C.c_uint32), ("est_seed_candidates", C.c_double),
                ("est_tile_frac", C.c_double), ("est_group_tile_frac", C.c_double),
                ("tensor_partition", C.c_uint32), ("reserved0", C.c_uint32)]


class Counters(C.Structure):
    _fields_ = [("queries", C.c_uint64), ("pairs", C.c_uint64), ("filter_pairs", C.c_uint64),
                ("rerank_pairs", C.c_uint64), ("node_visits", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("device_ms", C.c_double), ("scan_ms", C.c_double), ("h2d_bytes", C.c_uint64),
                ("d2h_bytes", C.c_uint64)]


def _struct_dict(s):
    return {f: getattr(s, f) for f, _ in s._fields_ if not f.startswith("reserved")}


_lib = None


def lib():
    """The loaded shared library; raises if it is missing (build with __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: the CUDA extension is not built. Run `python -c 'import __graft_entry__ as g; "
            f"g.build()'` (or `make -C petal-neighbors_b200/csrc`). There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, sz, u64p = C.c_void_p, C.c_size_t, C.POINTER(C.c_uint64)
    L.pn_last_error_message.restype = C.c_char_p
    L.pn_abi_version.restype = C.c_int32
    L.pn_device_count.argtypes = [C.POINTER(C.c_int32)]
    for sfx, real in (("f32", C.c_float), ("f64", C.c_double)):
        pr = C.POINTER(real)
        for kind in ("balltree", "vptree"):
            f = getattr(L, f"pn_{kind}_create_{sfx}")
            f.restype = C.c_int32
            f.argtypes = [vp, sz, sz, sz, sz, C.POINTER(BuildOpts), C.POINTER(vp)]
        f = getattr(L, f"pn_balltree_create_dev_{sfx}")
        f.restype = C.c_int32
        f.argtypes = [vp, sz, sz, sz, C.POINTER(BuildOpts), C.POINTER(vp)]
        for kind in ("balltree", "vptree"):
            f = getattr(L, f"pn_{kind}_query_{sfx}")
            f.restype = C.c_int32
            f.argtypes = [vp, vp, sz, sz, sz, vp, vp]
            f = getattr(L, f"pn_{kind}_query_radius_{sfx}")
            f.restype = C.c_int32
            f.argtypes = [vp, vp, sz, sz, real, C.POINTER(u64p), C.POINTER(u64p)]
        for name in (f"pn_balltree_query_nearest_{sfx}", f"pn_vptree_query_nearest_{sfx}"):
            f = getattr(L, name)
            f.restype = C.c_int32
            f.argtypes = [vp, vp, sz, sz, vp, vp]
        f = getattr(L, f"pn_pairwise_{sfx}")
        f.restype = C.c_int32
        f.argtypes = [C.c_int32, vp, sz, sz, sz, vp]
        f = getattr(L, f"pn_balltree_query_self_{sfx}")
        f.restype = C.c_int32
        f.argtypes = [vp, sz, vp, vp]
    L.pn_tree_destroy.argtypes = [vp]
    L.pn_tree_destroy.restype = C.c_int32
    L.pn_tree_session.argtypes = [vp, C.POINTER(vp)]
    L.pn_tree_session.restype = C.c_int32
    L.pn_free.argtypes = [vp]
    L.pn_free.restype = None
    L.pn_tree_query_knn_dev.restype = C.c_int32
    L.pn_tree_query_knn_dev.argtypes = [vp, vp, sz, sz, sz, vp, vp, vp, C.c_int32]
    L.pn_tree_query_radius_dev.restype = C.c_int32
    L.pn_tree_query_radius_dev.argtypes = [vp, vp, sz, sz, C.c_double, vp, vp, sz, vp, C.c_int32]
    L.pn_tree_query_self_dev.restype = C.c_int32
    L.pn_tree_query_self_dev.argtypes = [vp, sz, vp, vp, vp, C.c_int32]
    L.pn_merge_topk_dev.restype = C.c_int32
    L.pn_merge_topk_dev.argtypes = [C.c_uint32, C.c_int32, vp, vp, sz, sz, sz, vp, vp, vp, C.c_int32]
    L.pn_merge_radius_dev.restype = C.c_int32
    L.pn_merge_radius_dev.argtypes = [C.c_int32, vp, vp, sz, sz, vp, vp, vp, C.c_int32]
    L.pn_tree_get_info.restype = C.c_int32
    L.pn_tree_get_info.argtypes = [vp, C.POINTER(TreeInfo)]
    L.pn_tree_get_counters.restype = C.c_int32
    L.pn_tree_get_counters.argtypes = [vp, C.POINTER(Counters)]
    L.pn_tree_get_layout.restype = C.c_int32
    L.pn_tree_get_layout.argtypes = [vp, vp, vp, vp, vp, vp, vp]
    L.pn_comm_unique_id.restype = C.c_int32
    L.pn_comm_unique_id.argtypes = [vp]
    L.pn_comm_create.restype = C.c_int32
    L.pn_comm_create.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32, C.POINTER(vp)]
    L.pn_comm_create_all.restype = C.c_int32
    L.pn_comm_create_all.argtypes = [C.POINTER(C.c_int32), C.c_int32, C.POINTER(vp)]
    L.pn_comm_destroy.restype = C.c_int32
    L.pn_comm_destroy.argtypes = [vp]
    L.pn_query_slice.restype = None
    L.pn_query_slice.argtypes = [sz, C.c_int32, C.c_int32, C.POINTER(sz), C.POINTER(sz)]
    L.pn_sharded_query_knn_dev.restype = C.c_int32
    L.pn_sharded_query_knn_dev.argtypes = [vp, vp, vp, sz, sz, sz, C.c_uint32, vp, vp, vp, C.POINTER(ShardStats)]
    L.pn_tree_replicate.restype = C.c_int32
    L.pn_tree_replicate.argtypes = [vp, vp, C.c_int32, C.POINTER(vp)]
    L.pn_multi_balltree_create_f32.restype = C.c_int32
    L.pn_multi_balltree_create_f32.argtypes = [C.POINTER(C.c_int32), C.c_int32, C.c_uint32, vp, sz, sz, sz, C.POINTER(BuildOpts), C.POINTER(vp)]
    L.pn_multi_balltree_query_f32.restype = C.c_int32
    L.pn_multi_balltree_query_f32.argtypes = [vp, vp, sz, sz, sz, vp, vp]
    L.pn_multi_balltree_query_radius_f32.restype = C.c_int32
    L.pn_multi_balltree_query_radius_f32.argtypes = [vp, vp, sz, sz, C.c_float, C.POINTER(u64p), C.POINTER(u64p)]
    L.pn_multi_set_exchange.restype = C.c_int32
    L.pn_multi_set_exchange.argtypes = [vp, C.c_uint32]
    L.pn_multi_get_stats.restype = C.c_int32
    L.pn_multi_get_stats.argtypes = [vp, C.POINTER(ShardStats), C.c_int32]
    L.pn_multi_destroy.restype = C.c_int32
    L.pn_multi_destroy.argtypes = [vp]
    _lib = L
    return L


def last_error() -> str:
    return lib().pn_last_error_message().decode("utf-8", "replace")
