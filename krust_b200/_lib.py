"""ctypes binding of include/kmerust_gpu.h.  Loads krust_b200/libkmerust_gpu.so and fails loudly when
it is missing: there is no CPU fallback anywhere in this package."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libkmerust_gpu.so")

KMG_ABI_VERSION = 1
KMG_OK, KMG_ERR_INVALID_K, KMG_ERR_INVALID_ARG, KMG_ERR_CUDA, KMG_ERR_OOM, KMG_ERR_TABLE_FULL, KMG_ERR_STATE, \
    KMG_ERR_IO, KMG_ERR_ABI, KMG_ERR_CAPACITY, KMG_ERR_PARSE = range(11)
KMG_FLAG_FORCE_HASH, KMG_FLAG_FORCE_DIRECT, KMG_FLAG_NO_PREAGG, KMG_FLAG_FORCE_PARTITIONED = 1, 2, 4, 8
KMG_TEXT_FASTA, KMG_TEXT_TSV, KMG_TEXT_JSON = 0, 1, 2
TEXT_SINK = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(C.c_uint8), C.c_size_t)


class KmgConfig(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("k", C.c_uint32), ("device", C.c_int32), ("flags", C.c_uint32),
                ("has_min_quality", C.c_uint8), ("min_quality", C.c_uint8), ("parts_log2", C.c_uint8), ("reserved", C.c_uint8 * 5),
                ("expected_distinct", C.c_uint64), ("batch_bases", C.c_uint64), ("stream", C.c_void_p)]


class KmgSummary(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("n_bases", C.c_uint64), ("n_windows", C.c_uint64),
                ("n_distinct", C.c_uint64), ("max_count", C.c_uint64), ("table_capacity", C.c_uint64),
                ("path", C.c_uint32), ("n_grows", C.c_uint32), ("kernel_ns", C.c_uint64), ("h2d_bytes", C.c_uint64),
                ("scan_ns", C.c_uint64), ("consolidate_ns", C.c_uint64)]


class KmgBatch(C.Structure):
    _fields_ = [("bases2bit", C.POINTER(C.c_uint64)), ("valid_bits", C.POINTER(C.c_uint32)),
                ("start_bits", C.POINTER(C.c_uint32)), ("capacity_bases", C.c_uint64), ("n_bases", C.c_uint64),
                ("n_records", C.c_uint64), ("slot", C.c_uint32)]


# name -> (restype, argtypes); also the list the "exports every declared symbol" test walks.
vp, u64, u32, i32 = C.c_void_p, C.c_uint64, C.c_uint32, C.c_int
SIGNATURES = {
    "kmg_abi_version": (u32, []),
    "kmg_status_string": (C.c_char_p, [i32]),
    "kmg_last_error": (C.c_char_p, [vp]),
    "kmg_create": (i32, [C.POINTER(KmgConfig), C.POINTER(vp)]),
    "kmg_destroy": (None, [vp]),
    "kmg_ctx_k": (u32, [vp]),
    "kmg_reset": (i32, [vp]),
    "kmg_count_ascii": (i32, [vp, vp, vp, vp, u64]),
    "kmg_count_fastx": (i32, [vp, vp, u64, i32, C.POINTER(u64)]),
    "kmg_fastx_stream_begin": (i32, [vp, i32, u64]),
    "kmg_fastx_stream_push": (i32, [vp, vp, u64]),
    "kmg_fastx_stream_end": (i32, [vp, C.POINTER(u64)]),
    "kmg_fastx_stream_rest": (i32, [vp, vp, u64, C.POINTER(u64)]),
    "kmg_acquire_batch": (i32, [vp, C.POINTER(KmgBatch)]),
    "kmg_submit_batch": (i32, [vp, C.POINTER(KmgBatch)]),
    "kmg_count_ascii_device": (i32, [vp, vp, vp, vp, u64, u64]),
    "kmg_insert_keys_device": (i32, [vp, vp, vp, u64]),
    "kmg_extract_keys_device": (i32, [vp, vp, vp, vp, u64, u64, u32, vp, u64, vp]),
    "kmg_owner_of": (u32, [u64, u32]),
    "kmg_partition_plan": (i32, [vp, u64, C.POINTER(u32), C.POINTER(u32)]),
    "kmg_adopt_coarse_device": (i32, [vp, vp, vp, u32, u64]),
    "kmg_shard_join": (i32, [vp, u32, u32, C.c_char_p, u64]),
    "kmg_shard_leave": (i32, [vp]),
    "kmg_shard_count_ascii_device": (i32, [vp, vp, vp, vp, u64, u64]),
    "kmg_shard_count_ascii": (i32, [vp, vp, vp, vp, u64]),
    "kmg_shard_count_fastx": (i32, [vp, vp, u64, i32, C.POINTER(u64)]),
    "kmg_shard_finalize": (i32, [vp, C.POINTER(KmgSummary)]),
    "kmg_shard_histogram": (i32, [vp, u64, vp, vp, u64, C.POINTER(u64)]),
    "kmg_shard_save_kmix": (i32, [vp, C.c_char_p, C.POINTER(u64)]),
    "kmg_shard_write_text": (i32, [vp, u64, i32, C.c_char_p, C.POINTER(u64), C.POINTER(u64)]),
    "kmg_shard_stats": (i32, [vp, C.POINTER(u64), C.POINTER(u64), C.POINTER(u64), C.POINTER(u64)]),
    "kmg_finalize": (i32, [vp, C.POINTER(KmgSummary)]),
    "kmg_export_counts": (i32, [vp, u64, i32, vp, vp, u64, C.POINTER(u64)]),
    "kmg_export_counts_device": (i32, [vp, u64, i32, vp, vp, u64, C.POINTER(u64)]),
    "kmg_export_shard": (i32, [vp, u64, i32, u64, u64, vp, vp, u64, C.POINTER(u64)]),
    "kmg_export_shard_device": (i32, [vp, u64, i32, u64, u64, vp, vp, u64, C.POINTER(u64)]),
    "kmg_histogram": (i32, [vp, u64, vp, vp, u64, C.POINTER(u64)]),
    "kmg_save_kmix": (i32, [vp, C.c_char_p]),
    "kmg_emit_text": (i32, [vp, u64, i32, vp, vp, C.POINTER(u64), C.POINTER(u64)]),
    "kmg_write_text": (i32, [vp, u64, i32, C.c_char_p, C.POINTER(u64), C.POINTER(u64)]),
    "kmg_kmix_begin": (i32, [C.c_char_p]),
    "kmg_save_kmix_shard": (i32, [vp, C.c_char_p, u64, C.POINTER(u64), C.POINTER(u32)]),
    "kmg_kmix_finish": (i32, [C.c_char_p, u32, vp, vp, u32]),
    "kmg_query_keys": (i32, [vp, vp, u64, vp]),
    "kmg_query_ascii": (i32, [vp, vp, u64, vp, C.POINTER(u64)]),
    "kmg_index_open": (i32, [C.c_char_p, C.c_int32, C.POINTER(vp)]),
    "kmg_progress": (i32, [vp, C.POINTER(u64), C.POINTER(u64)]),
    "kmg_kernel_launches": (u64, []),
    "kmg_phase_times": (i32, [vp, C.POINTER(u64)]),
    "kmg_synth_uniform_device": (i32, [vp, u64, u64, u64, vp]),
    "kmg_synth_reads_device": (i32, [vp, u64, u32, u64, u64, vp, vp]),
    "kmg_parse_fastx": (i32, [vp, u64, i32, vp, vp, vp, u64, C.POINTER(u64), C.c_char_p, C.c_size_t]),
}

_lib = None


def load():
    """Return the loaded library; raises if the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m krust_b200.build` (needs nvcc). "
                "krust_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if a declared symbol is not exported
            fn.restype = res
            fn.argtypes = args
        if L.kmg_abi_version() != KMG_ABI_VERSION:
            raise RuntimeError("libkmerust_gpu.so ABI version mismatch")
        _lib = L
    return _lib
