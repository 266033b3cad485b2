"""ctypes binding of the C-ABI (include/smatrix.h, smatrix_batch.h, smatrix_b200.h).

This is the stub a Python binding of the reference would write; it contains no computation.
`load()` binds a shared library by path and declares every prototype; the default path is the
in-tree CUDA build and loading fails loudly if it is missing (there is no CPU fallback).
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# $SMATRIX_B200_LIB selects another build of the same library (A/B measurements of compile-time knobs)
DEFAULT_SO = os.environ.get("SMATRIX_B200_LIB") or os.path.join(HERE, "lib", "libsmatrix_b200.so")

u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)

# name -> (restype, argtypes); every symbol the three headers declare
PROTOTYPES = {
    # include/smatrix.h (reference src/smatrix.h:87-94)
    "smatrix_open": (C.c_void_p, [C.c_char_p]),
    "smatrix_close": (None, [C.c_void_p]),
    "smatrix_get": (C.c_uint32, [C.c_void_p, C.c_uint32, C.c_uint32]),
    "smatrix_set": (C.c_uint32, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]),
    "smatrix_incr": (C.c_uint32, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]),
    "smatrix_decr": (C.c_uint32, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32]),
    "smatrix_rowlen": (C.c_uint32, [C.c_void_p, C.c_uint32]),
    "smatrix_getrow": (C.c_uint32, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t]),
    # include/smatrix_batch.h
    "smatrix_incr_batch": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "smatrix_decr_batch": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "smatrix_set_batch": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "smatrix_incr_batch_out": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "smatrix_decr_batch_out": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "smatrix_set_batch_out": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "smatrix_get_batch": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "smatrix_rowlen_batch": (None, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "smatrix_getrow_batch": (C.c_uint64, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                          C.c_uint64]),
    "smatrix_cf_neighbors_batch": (C.c_uint64, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.c_uint64]),
    "smatrix_cf_topk_batch": (None, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p, C.c_void_p,
                                     C.c_void_p]),
    "smatrix_cf_recommend_batch": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    # include/smatrix_b200.h
    "smatrix_b200_open": (C.c_void_p, [C.c_char_p, C.c_int]),
    "smatrix_b200_open_arena": (C.c_void_p, [C.c_char_p, C.c_int, C.c_size_t]),
    "smatrix_b200_snapshot": (C.c_int, [C.c_void_p]),
    "smatrix_b200_device": (C.c_int, [C.c_void_p]),
    "smatrix_b200_stream": (C.c_void_p, [C.c_void_p]),
    "smatrix_b200_sync": (None, [C.c_void_p]),
    "smatrix_b200_timer_start": (None, [C.c_void_p]),
    "smatrix_b200_timer_stop_ms": (C.c_float, [C.c_void_p]),
    "smatrix_b200_stat": (C.c_uint64, [C.c_void_p, C.c_int]),
    "smatrix_b200_set_kernel_timing": (None, [C.c_void_p, C.c_int]),
    "smatrix_b200_set_get_slices": (None, [C.c_void_p, C.c_int]),
    "smatrix_b200_host_alloc": (C.c_void_p, [C.c_size_t]),
    "smatrix_b200_host_free": (None, [C.c_void_p]),
    "smatrix_b200_dev_alloc": (C.c_void_p, [C.c_void_p, C.c_size_t]),
    "smatrix_b200_dev_free": (None, [C.c_void_p, C.c_void_p]),
    "smatrix_b200_memcpy": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "smatrix_b200_memset0": (None, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "smatrix_b200_gen_c2_ops": (None, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_size_t, C.c_uint32,
                                       C.c_uint32, C.c_void_p, C.c_void_p]),
    "smatrix_b200_gen_c2_queries": (None, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_size_t,
                                           C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    "smatrix_b200_gen_c3_ops": (None, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_size_t, C.c_void_p, C.c_uint32,
                                       C.c_void_p, C.c_void_p]),
    "smatrix_b200_gen_c3_queries": (None, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint64, C.c_size_t, C.c_uint64,
                                           C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]),
    "smatrix_b200_gen_c4_lens": (None, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_size_t, C.c_void_p, C.c_uint32,
                                        C.c_void_p]),
    "smatrix_b200_gen_c4_ops": (None, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_size_t, C.c_void_p, C.c_uint32,
                                       C.c_void_p, C.c_void_p, C.c_void_p]),
    "smatrix_b200_probe_random_read": (C.c_double, [C.c_void_p, C.c_size_t, C.c_size_t, C.c_int]),
    "smatrix_b200_probe_random_atomic": (C.c_double, [C.c_void_p, C.c_size_t, C.c_size_t]),
    "smatrix_b200_partition_count": (None, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p]),
    "smatrix_b200_route_p2p": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32,
                                      C.c_void_p, C.c_uint32, C.c_void_p]),
    "smatrix_b200_ipc_export": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "smatrix_b200_ipc_open": (C.c_void_p, [C.c_void_p, C.c_void_p]),
    "smatrix_b200_ipc_close": (None, [C.c_void_p, C.c_void_p]),
    "smatrix_b200_gather": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "smatrix_b200_row_counts_batch": (None, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "smatrix_b200_scan_counts": (C.c_uint64, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "smatrix_b200_getrow_fill_at": (None, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "smatrix_b200_route_offsets": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p]),
    "smatrix_b200_pair_cols": (None, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "smatrix_b200_cf_scores_totals": (None, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                             C.c_void_p, C.c_void_p]),
    "smatrix_b200_topk_segments": (None, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32,
                                          C.c_void_p, C.c_void_p, C.c_void_p]),
    "smatrix_b200_basket_topk": (None, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "smatrix_b200_enable_peer": (C.c_int, [C.c_void_p, C.c_int]),
    "smatrix_b200_is_device_ptr": (C.c_int, [C.c_void_p, C.c_void_p]),
    "smatrix_b200_memcpy_async": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]),
    "smatrix_b200_lane_sync": (None, [C.c_void_p, C.c_int]),
    "smatrix_b200_apply_ordered": (None, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_size_t]),
    "smatrix_b200_apply_ordered_out": (None, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_size_t, C.c_void_p]),
    "smatrix_b200_owner": (C.c_uint32, [C.c_uint32, C.c_uint32]),
    "smatrix_b200_snap_extent": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "smatrix_b200_snap_rows_base": (C.c_uint64, [C.c_uint64]),
    "smatrix_b200_snap_layout": (C.c_int, [C.c_int, C.c_uint64, C.c_uint64]),
    "smatrix_b200_snap_write": (C.c_int, [C.c_void_p, C.c_int, C.c_uint64, C.c_uint64]),
    "smatrix_b200_snap_commit": (C.c_int, [C.c_char_p, C.c_char_p]),
    "smatrix_b200_load_begin": (C.c_void_p, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "smatrix_b200_load_next": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    "smatrix_b200_load_end": (None, [C.c_void_p]),
    "smatrix_b200_load_fixup": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
}

# include/smatrix_shard.h
PROTOTYPES.update({
    "smatrix_b200_shard_open": (C.c_void_p, [C.c_char_p, C.c_int, C.c_int, C.c_int]),
    "smatrix_b200_shard_open_arena": (C.c_void_p, [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_size_t]),
    "smatrix_b200_shard_open_file": (C.c_void_p, [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_size_t, C.c_char_p]),
    "smatrix_b200_shard_snapshot": (C.c_int, [C.c_void_p]),
    "smatrix_b200_shard_close": (None, [C.c_void_p]),
    "smatrix_b200_shard_local": (C.c_void_p, [C.c_void_p]),
    "smatrix_b200_shard_rank": (C.c_int, [C.c_void_p]),
    "smatrix_b200_shard_world": (C.c_int, [C.c_void_p]),
    "smatrix_b200_shard_reserve": (None, [C.c_void_p, C.c_size_t, C.c_size_t]),
    "smatrix_b200_shard_incr_batch": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]),
    "smatrix_b200_shard_decr_batch": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]),
    "smatrix_b200_shard_set_batch": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "smatrix_b200_shard_incr_batch_out": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "smatrix_b200_shard_decr_batch_out": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "smatrix_b200_shard_set_batch_out": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "smatrix_b200_shard_get_batch": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "smatrix_b200_shard_rowlen_batch": (None, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "smatrix_b200_shard_cf_neighbors_batch": (C.c_uint64, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                                          C.c_void_p, C.c_uint64]),
    "smatrix_b200_shard_cf_topk_batch": (None, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32, C.c_void_p,
                                                C.c_void_p, C.c_void_p]),
    "smatrix_b200_shard_cf_recommend_batch": (None, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint32,
                                                     C.c_void_p, C.c_void_p, C.c_void_p]),
    "smatrix_b200_shard_getrow_batch": (C.c_uint64, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                                    C.c_uint64]),
    "smatrix_b200_shard_stat": (C.c_uint64, [C.c_void_p, C.c_int]),
    "smatrix_b200_shard_stat_reset": (None, [C.c_void_p]),
    "smatrix_b200_shard_barrier": (None, [C.c_void_p]),
    "smatrix_b200_shard_sum": (C.c_uint64, [C.c_void_p, C.c_uint64]),
    "smatrix_b200_shard_max": (C.c_uint64, [C.c_void_p, C.c_uint64]),
})

STAT = {"rows": 0, "nnz": 1, "dir_cap": 2, "slab_bytes": 3, "device_bytes": 4, "launches": 5,
        "rounds": 6, "row_grows": 7, "dir_grows": 8, "kernel_ns": 9, "ns_partition": 10, "ns_upsert": 11,
        "ns_grow_plan": 12, "ns_slab": 13, "ns_migrate": 14, "ns_dir": 15, "value_sum": 16,
        "live_bucket_bytes": 17, "free_bytes": 18, "recycled": 19, "h2d_bytes": 20, "d2h_bytes": 21, "bucket_bytes": 22, "spilled": 23,
        "sliced_gets": 24, "wide_chunks": 25, "ns_alloc": 26, "allocs": 27,
        "topk_big": 28, "topk_passes": 29, "rec_big": 30}

_cache: dict[str, C.CDLL] = {}


def load(path: str | None = None) -> C.CDLL:
    path = os.path.abspath(path or DEFAULT_SO)
    lib = _cache.get(path)
    if lib is None:
        if not os.path.exists(path):
            raise ImportError(
                f"{path} not found: build the CUDA library first "
                "(python -m libsmatrix_b200.build). There is no CPU fallback.")
        lib = C.CDLL(path)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)  # AttributeError = a declared symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _cache[path] = lib
    return lib
