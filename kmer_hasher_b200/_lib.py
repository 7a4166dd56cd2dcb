"""ctypes binding of csrc/libkmergpu.so (the C ABI declared in include/kmergpu.h).

There is no fallback: if the shared library is missing, or no B200 is visible, every call
raises.  Nothing here imports the CPU oracle.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libkmergpu.so")

u64p = C.POINTER(C.c_uint64)
i32p = C.POINTER(C.c_int32)
vp = C.c_void_p

# every symbol include/kmergpu.h declares: name -> (restype, argtypes)
SIGNATURES = {
    "kmg_last_error": (C.c_char_p, []),
    "kmg_version": (C.c_int, []),
    "kmg_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "kmg_set_device": (C.c_int, [C.c_int]),
    "kmg_set_stream": (C.c_int, [vp]),
    "kmg_host_alloc": (vp, [C.c_size_t]),
    "kmg_host_free": (None, [vp]),
    "kmg_build": (C.c_int, [vp, C.c_int64, C.c_int, C.POINTER(vp)]),
    "kmg_build_ordered": (C.c_int, [vp, C.c_int64, C.c_int, C.c_int, C.POINTER(vp)]),
    "kmg_index_order": (C.c_int, [vp]),
    "kmg_free": (C.c_int, [vp]),
    "kmg_sizes": (C.c_int, [vp, u64p, u64p, u64p]),
    "kmg_index_k": (C.c_int, [vp]),
    "kmg_kmers_u64": (C.c_int, [vp, vp]),
    "kmg_kmers_ascii": (C.c_int, [vp, vp]),
    "kmg_counts": (C.c_int, [vp, vp]),
    "kmg_positions": (C.c_int, [vp, vp]),
    "kmg_pairs": (C.c_int, [vp, vp]),
    "kmg_pairs_chunk": (C.c_int, [vp, C.c_uint64, C.c_uint64, vp]),
    "kmg_query_begin": (C.c_int, [vp, vp, C.c_int64, C.c_int, C.POINTER(vp), u64p]),
    "kmg_query_begin_rc": (C.c_int, [vp, vp, C.c_int64, C.c_int, C.POINTER(vp), u64p]),
    "kmg_query_emit": (C.c_int, [vp, vp]),
    "kmg_query_emit_chunk": (C.c_int, [vp, C.c_uint64, C.c_uint64, vp]),
    "kmg_query_free": (C.c_int, [vp]),
    "kmg_join_begin": (C.c_int, [vp, vp, C.POINTER(vp), u64p]),
    "kmg_join_emit": (C.c_int, [vp, vp]),
    "kmg_join_emit_chunk": (C.c_int, [vp, C.c_uint64, C.c_uint64, vp]),
    "kmg_join_free": (C.c_int, [vp]),
    "kmg_query_dotplot": (C.c_int, [vp, vp, C.c_int64, C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_int,
                                    C.c_int64, C.c_int64, C.c_int, C.c_uint32, vp]),
    "kmg_join_dotplot": (C.c_int, [vp, vp, C.c_int64, C.c_int64, C.c_int, C.c_int64, C.c_int64, C.c_int, C.c_uint32, vp]),
    "kmg_shard_sample": (C.c_int, [vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, vp]),
    "kmg_shard_partition": (C.c_int, [vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int,
                                      u64p, C.c_int, vp, vp, u64p]),
    "kmg_build_records": (C.c_int, [vp, vp, C.c_int64, C.c_int, C.POINTER(vp)]),
    "kmg_query_records": (C.c_int, [vp, vp, vp, C.c_int64, C.POINTER(vp), u64p]),
    "kmg_shard_open": (C.c_int, [vp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.POINTER(vp)]),
    "kmg_shard_close": (C.c_int, [vp]),
    "kmg_shard_pack_bytes": (C.c_int, [C.c_int]),
    "kmg_shard_pack": (C.c_int, [vp, C.c_int64, C.c_int, C.c_int, C.c_int, vp]),
    "kmg_shard_open_packed": (C.c_int, [vp, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.POINTER(vp), vp]),
    "kmg_shard_set_mixed": (C.c_int, [vp, C.c_int]),
    "kmg_shard_windows": (C.c_int, [vp, C.POINTER(C.c_int64)]),
    "kmg_shard_sample_keys": (C.c_int, [vp, C.c_int, vp]),
    "kmg_shard_count": (C.c_int, [vp, vp, C.c_int, vp]),
    "kmg_shard_scatter": (C.c_int, [vp, vp, C.c_int, C.c_int, C.POINTER(vp), C.POINTER(vp), C.c_uint64, vp, C.c_int32, vp]),
    "kmg_build_received": (C.c_int, [vp, vp, C.c_uint64, vp, C.c_int, C.c_int, C.POINTER(vp)]),
    "kmg_query_received": (C.c_int, [vp, vp, vp, C.c_uint64, vp, C.c_int, C.POINTER(vp), u64p]),
    "kmg_shard_scatter_ranges": (C.c_int, [vp, C.c_int, C.c_int, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.c_uint64, C.c_int32]),
    "kmg_build_regions": (C.c_int, [vp, vp, C.c_uint64, C.c_int, vp, C.c_int, C.POINTER(vp)]),
    "kmg_query_regions": (C.c_int, [vp, vp, vp, C.c_uint64, C.c_int, vp, C.POINTER(vp), u64p]),
    "kmg_ipc_alloc": (C.c_int, [C.c_size_t, C.POINTER(vp), vp]),
    "kmg_ipc_free": (C.c_int, [vp]),
    "kmg_ipc_open": (C.c_int, [vp, C.POINTER(vp)]),
    "kmg_ipc_close": (C.c_int, [vp]),
    "kmg_profile_enable": (C.c_int, [C.c_int]),
    "kmg_profile_reset": (C.c_int, []),
    "kmg_profile_count": (C.c_int, []),
    "kmg_profile_get": (C.c_int, [C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_double), u64p, C.POINTER(C.c_double)]),
    "kmg_launch_count": (C.c_uint64, []),
    "kmg_selftest_lane_order": (C.c_int, [C.POINTER(C.c_uint32)]),
    "kmg_tune": (C.c_int, [C.c_char_p, C.c_int]),
    "kmg_count_new": (C.c_int, [C.c_int, C.c_int, C.POINTER(vp)]),
    "kmg_count_add": (C.c_int, [vp, vp, C.c_int64, C.c_int]),
    "kmg_count_sizes": (C.c_int, [vp, u64p, C.POINTER(C.c_int), C.POINTER(C.c_int), u64p]),
    "kmg_count_kmers_u64": (C.c_int, [vp, vp]),
    "kmg_count_kmers_ascii": (C.c_int, [vp, vp]),
    "kmg_count_matrix": (C.c_int, [vp, vp]),
    "kmg_count_positions": (C.c_int, [vp, vp]),
    "kmg_count_spectrum": (C.c_int, [vp, C.c_int, C.c_uint32, C.POINTER(C.c_double)]),
    "kmg_index_spectrum": (C.c_int, [vp, C.c_uint32, C.POINTER(C.c_double)]),
    "kmg_count_free": (C.c_int, [vp]),
    "kmg_count_depth": (C.c_int, [vp, vp, C.c_int64, C.c_int, vp]),
    "kmg_index_depth": (C.c_int, [vp, vp, C.c_int64, C.c_int, vp]),
    "kmg_reads_open": (C.c_int, [C.c_char_p, C.POINTER(vp)]),
    "kmg_reads_from_memory": (C.c_int, [vp, C.c_int64, C.POINTER(vp)]),
    "kmg_reads_count": (C.c_int, [vp, u64p, u64p]),
    "kmg_reads_record": (C.c_int, [vp, C.c_uint64, C.POINTER(C.c_int64), C.c_char_p, C.c_int]),
    "kmg_reads_sequence": (C.c_int, [vp, C.c_uint64, vp]),
    "kmg_build_record": (C.c_int, [vp, C.c_uint64, C.c_int, C.c_int, C.POINTER(vp)]),
    "kmg_count_add_reads": (C.c_int, [vp, vp, C.c_int]),
    "kmg_reads_free": (C.c_int, [vp]),
    "kmg_tune_get": (C.c_int64, [C.c_char_p, C.c_int64]),
    "kmg_trim": (C.c_int, []),
    "kmg_cached_bytes": (C.c_uint64, []),
    "kmg_positions_base": (C.c_int, [vp, C.c_uint64, vp]),
    "kmg_pairs_chunk_base": (C.c_int, [vp, C.c_uint64, C.c_uint64, C.c_uint64, vp]),
}

_lib = None


class KmgError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libkmergpu error {code}: {msg}")
        self.code = code


def load() -> C.CDLL:
    """dlopen libkmergpu.so and type every entry point. Loud failure if it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(libkmergpu is CUDA-only; there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        raise KmgError(rc, load().kmg_last_error().decode("utf-8", "replace"))
