"""ctypes binding of libblu_consensus.so (C ABI: include/blu_consensus.h).

There is no Python or CPU implementation behind this module: if the CUDA library has not been built
(`python -c "import __graft_entry__ as g; g.build()"` or `make -C blutils_b200/csrc`) importing fails loudly."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BLU_CONSENSUS_LIB") or os.path.join(_HERE, "libblu_consensus.so")  # (override: tuning builds)
SYNTH_PATH = os.path.join(_HERE, "libblu_synth.so")

BLU_OK, BLU_ERR_IO, BLU_ERR_DATA, BLU_ERR_CUDA, BLU_ERR_ARG, BLU_ERR_UNSUPPORTED, BLU_ERR_INTERNAL = range(7)
BLU_CUTOFF_ABSENT = -(2 ** 31)


class blu_opts(C.Structure):
    _fields_ = [("device", C.c_int32), ("taxon", C.c_int32), ("strategy", C.c_int32), ("use_taxid", C.c_int32),
                ("has_custom", C.c_int32), ("custom", C.c_int32 * 8), ("chunk_bytes", C.c_uint64), ("flags", C.c_uint64), ("reserved", C.c_uint64 * 3)]


class blu_record(C.Structure):
    _fields_ = [("query_off", C.c_uint64), ("query_len", C.c_uint32), ("n_rows", C.c_uint32), ("keep_mask", C.c_uint64),
                ("perc_identity", C.c_double), ("bit_score", C.c_int64), ("ref_lineage", C.c_uint32), ("bean_base", C.c_uint32),
                ("n_beans", C.c_uint32), ("acc_base", C.c_uint32), ("status", C.c_uint8), ("single_match", C.c_uint8),
                ("mutated", C.c_uint8), ("reached_pos", C.c_int8), ("allowed_pos", C.c_int8), ("bean_level", C.c_int8),
                ("pad", C.c_uint8 * 2)]


class blu_bean(C.Structure):
    _fields_ = [("first_lineage", C.c_uint32), ("occurrences", C.c_uint32), ("acc_begin", C.c_uint32), ("n_acc", C.c_uint32)]


BLU_OPT_TEXT_REFS = 1


class blu_timings(C.Structure):
    _fields_ = [("ms_total_device", C.c_double), ("ms_tile_kernel", C.c_double), ("ms_longrun_kernel", C.c_double),
                ("ms_gather_kernel", C.c_double), ("ms_other", C.c_double), ("text_bytes", C.c_uint64), ("result_bytes", C.c_uint64),
                ("taxonomy_bytes", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("n_queries", C.c_uint64),
                ("n_rows", C.c_uint64), ("n_deferred_runs", C.c_uint64), ("n_kernel_launches", C.c_uint64), ("n_regrouped", C.c_uint64), ("n_tile_launches", C.c_uint64), ("reserved", C.c_uint64 * 2)]


# every symbol include/blu_consensus.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("blu_abi_version", C.c_int, []),
    ("blu_ctx_create", C.c_int, [C.POINTER(blu_opts), C.POINTER(C.c_void_p)]),
    ("blu_ctx_create_multi", C.c_int, [C.POINTER(blu_opts), C.POINTER(C.c_int), C.c_int, C.POINTER(C.c_void_p)]),
    ("blu_ctx_num_devices", C.c_int, [C.c_void_p]),
    ("blu_ctx_destroy", None, [C.c_void_p]),
    ("blu_last_error", C.c_char_p, [C.c_void_p]),
    ("blu_custom_cutoffs_from_file", C.c_int, [C.c_char_p, C.POINTER(blu_opts), C.c_char_p, C.c_size_t]),
    ("blu_taxonomy_load_json", C.c_int, [C.c_void_p, C.c_char_p]),
    ("blu_taxonomy_load_json_cached", C.c_int, [C.c_void_p, C.c_char_p, C.c_char_p, C.POINTER(C.c_int)]),
    ("blu_result_file_to_tabular", C.c_int, [C.c_char_p, C.c_char_p, C.c_int, C.c_char_p, C.c_char_p, C.c_size_t]),
    ("blu_taxonomy_load_arrays", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]),
    ("blu_consensus_run_host", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]),
    ("blu_consensus_run_device", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_void_p)]),
    ("blu_consensus_run_device_resident", C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_void_p)]),
    ("blu_result_device_text", C.c_void_p, [C.c_void_p, C.POINTER(C.c_uint64)]),
    ("blu_result_device_records", C.c_void_p, [C.c_void_p]),
    ("blu_result_device_beans", C.c_void_p, [C.c_void_p, C.POINTER(C.c_uint64)]),
    ("blu_result_device_accessions", C.c_void_p, [C.c_void_p, C.POINTER(C.c_uint64)]),
    ("blu_result_download", C.c_int, [C.c_void_p]),
    ("blu_consensus_run_file", C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p)]),
    ("blu_result_add_headers", C.c_int, [C.c_void_p, C.c_char_p, C.c_uint64]),
    ("blu_consensus_run_host_configs", C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]),
    ("blu_consensus_run_file_configs", C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_char_p, C.POINTER(C.c_void_p)]),
    ("blu_consensus_run_device_resident_configs", C.c_int,
     [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_uint64, C.c_void_p, C.POINTER(C.c_void_p)]),
    ("blu_result_num_queries", C.c_uint64, [C.c_void_p]),
    ("blu_result_num_records", C.c_uint64, [C.c_void_p]),
    ("blu_result_sort_by_query", C.c_int, [C.c_void_p, C.c_void_p]),
    ("blu_result_num_rows", C.c_uint64, [C.c_void_p]),
    ("blu_result_records", C.POINTER(blu_record), [C.c_void_p]),
    ("blu_result_beans", C.c_void_p, [C.c_void_p]),
    ("blu_result_accessions", C.c_void_p, [C.c_void_p]),
    ("blu_result_pool", C.c_void_p, [C.c_void_p, C.POINTER(C.c_uint64)]),
    ("blu_result_num_beans", C.c_uint64, [C.c_void_p]),
    ("blu_result_num_accessions", C.c_uint64, [C.c_void_p]),
    ("blu_result_checksum", C.c_uint64, [C.c_void_p]),
    ("blu_result_to_jsonl", C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]),
    ("blu_result_to_jsonl_head", C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]),
    ("blu_result_write", C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.c_char_p]),
    ("blu_result_write_tabular", C.c_int, [C.c_void_p, C.c_char_p, C.c_char_p]),
    ("blu_result_free", None, [C.c_void_p]),
    ("blu_free", None, [C.c_void_p]),
    ("blu_ctx_last_timings", C.c_int, [C.c_void_p, C.POINTER(blu_timings)]),
    ("blu_ctx_measure_h2d", C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_double)]),
    ("blu_ctx_measure_d2h", C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_double)]),
    ("blu_shard_cuts", C.c_int, [C.c_void_p, C.c_uint64, C.c_int, C.POINTER(C.c_uint64)]),
    ("blu_shard_cuts_file", C.c_int, [C.c_char_p, C.c_int, C.POINTER(C.c_uint64)]),
    ("blu_host_alloc", C.c_void_p, [C.c_uint64]),
    ("blu_host_free", None, [C.c_void_p]),
]

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} is missing: the CUDA extension has not been built and there is no fallback "
                              "(run `make -C blutils_b200/csrc` or __graft_entry__.build())")
        l = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(l, name)  # AttributeError if the .so does not export it
            fn.restype = res
            fn.argtypes = args
        if l.blu_abi_version() != 2:
            raise ImportError("libblu_consensus.so ABI version mismatch")
        _lib = l
    return _lib


_synth = None


def synth_lib():
    global _synth
    if _synth is None:
        if not os.path.exists(SYNTH_PATH):
            raise ImportError(f"{SYNTH_PATH} is missing (run `make -C blutils_b200/csrc`)")
        l = C.CDLL(SYNTH_PATH)
        l.blu_synth_create.restype = C.c_void_p
        l.blu_synth_create.argtypes = [C.c_uint64, C.c_uint64]
        l.blu_synth_destroy.argtypes = [C.c_void_p]
        l.blu_synth_num_taxa.restype = C.c_uint64
        l.blu_synth_num_taxa.argtypes = [C.c_void_p]
        l.blu_synth_lineages.restype = C.c_uint64
        l.blu_synth_lineages.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        l.blu_synth_write_json.restype = C.c_int
        l.blu_synth_write_json.argtypes = [C.c_void_p, C.c_char_p]
        l.blu_synth_hits.restype = C.c_int
        l.blu_synth_hits.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_int, C.c_uint32, C.c_int, C.c_void_p, C.c_uint64,
                                     C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        _synth = l
    return _synth
