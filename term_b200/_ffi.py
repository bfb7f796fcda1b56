"""ctypes binding of include/termgpu.h — the same stub a reference maintainer would write as a
`term-guard-gpu-sys` crate (see INTEGRATION.md). No torch types cross this boundary.

The library is built in-tree (term_b200/libtermgpu.so) by `__graft_entry__.build()` /
`make -C term_b200/csrc`; importing this module fails loudly if it is missing.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# TG_LIB selects another build of the same library (kernel-parameter sweeps on the GPU box); the product is libtermgpu.so
LIB_PATH = os.environ.get("TG_LIB") or os.path.join(_HERE, "libtermgpu.so")


class TermGpuError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"[{STATUS_NAMES.get(code, code)}] {message}")
        self.code = code
        self.message = message


STATUS_NAMES = {
    0: "TG_OK", 1: "TG_ERR_INVALID_ARG", 2: "TG_ERR_COLUMN_NOT_FOUND", 3: "TG_ERR_TYPE_MISMATCH",
    4: "TG_ERR_SECURITY", 5: "TG_ERR_UNSUPPORTED", 6: "TG_ERR_CUDA", 7: "TG_ERR_NCCL", 8: "TG_ERR_INTERNAL",
    9: "TG_ERR_TABLE_NOT_FOUND", 10: "TG_ERR_VALIDATION", 11: "TG_ERR_CONFIGURATION",
}
TG_ERR_SECURITY, TG_ERR_UNSUPPORTED, TG_ERR_CUDA, TG_ERR_VALIDATION, TG_ERR_CONFIGURATION = 4, 5, 6, 10, 11

# tg_dtype
TG_INT64, TG_FLOAT64, TG_UTF8, TG_INT32, TG_FLOAT32, TG_BOOL, TG_FP128 = 1, 2, 3, 4, 5, 6, 7
TG_PQ_INT96 = 8  # tg_table_append_parquet_chunk only: a Parquet INT96 timestamp chunk
# tg_constraint_status
TG_SUCCESS, TG_FAILURE, TG_SKIPPED = 0, 1, 2
TG_KEY_ROWS_DUPLICATE, TG_KEY_ROWS_FIRST, TG_KEY_ROWS_ORPHAN = 0, 1, 2  # tg_key_rows_kind


class tg_assertion(C.Structure):
    _fields_ = [("kind", C.c_int32), ("a", C.c_double), ("b", C.c_double)]


class tg_format_options(C.Structure):
    _fields_ = [("case_sensitive", C.c_int32), ("trim_before_check", C.c_int32), ("null_is_valid", C.c_int32)]


class tg_result(C.Structure):
    _fields_ = [("status", C.c_int32), ("has_metric", C.c_int32), ("metric", C.c_double),
                ("message", C.c_char_p), ("name", C.c_char_p), ("error_code", C.c_int32),
                ("reserved", C.c_int32)]


class tg_analyzer_result(C.Structure):
    _fields_ = [("u", C.c_uint64 * 4), ("f", C.c_double * 8), ("metric_kind", C.c_int32),
                ("error", C.c_int32), ("metric_double", C.c_double), ("metric_long", C.c_int64),
                ("metric_key", C.c_char_p), ("message", C.c_char_p)]


class tg_column_buffers(C.Structure):
    _fields_ = [("dtype", C.c_int32), ("n_rows", C.c_int64), ("values", C.c_void_p), ("offsets", C.c_void_p),
                ("validity", C.c_void_p), ("n_value_bytes", C.c_int64), ("null_count", C.c_int64)]


class tg_parquet_page(C.Structure):
    _fields_ = [("page_type", C.c_int32), ("version", C.c_int32), ("encoding", C.c_int32), ("definition_level_encoding", C.c_int32),
                ("num_values", C.c_int32), ("num_nulls", C.c_int32), ("uncompressed_bytes", C.c_int32), ("body_bytes", C.c_int32),
                ("definition_levels_bytes", C.c_int32), ("repetition_levels_bytes", C.c_int32), ("is_compressed", C.c_int32),
                ("reserved", C.c_int32), ("header_offset", C.c_int64), ("body_offset", C.c_int64)]


class tg_csv_format(C.Structure):
    _fields_ = [("delimiter", C.c_int32), ("quote", C.c_int32), ("escape", C.c_int32), ("comment", C.c_int32), ("terminator", C.c_int32),
                ("has_header", C.c_int32), ("null_regex", C.c_char_p)]


class tg_exec_stats(C.Structure):
    _fields_ = [("gpu_ms", C.c_double), ("scan_ms", C.c_double), ("string_ms", C.c_double),
                ("hash_ms", C.c_double), ("sketch_ms", C.c_double), ("bytes_scanned", C.c_uint64),
                ("launches", C.c_uint64), ("scan_passes", C.c_uint64), ("scan_min_tile_rows", C.c_uint64),
                ("scan_max_units", C.c_uint64), ("scan_smem_state", C.c_uint64)]


P = C.c_void_p
PP = C.POINTER(C.c_void_p)
STRS = C.POINTER(C.c_char_p)

# name -> (restype, argtypes); every symbol include/termgpu.h declares
SIGNATURES = {
    "tg_engine_create": (C.c_int, [C.c_int, PP]),
    "tg_engine_destroy": (None, [P]),
    "tg_last_error": (C.c_char_p, []),
    "tg_version": (C.c_char_p, []),
    "tg_engine_launch_count": (C.c_uint64, [P]),
    "tg_engine_stream": (C.c_void_p, [P]),
    "tg_engine_sync_copies": (C.c_int, [P]),
    "tg_table_create": (C.c_int, [P, C.c_char_p, PP]),
    "tg_table_drop": (C.c_int, [P, C.c_char_p]),
    "tg_table_lookup": (C.c_int, [P, C.c_char_p, PP]),
    "tg_table_num_rows": (C.c_int64, [P]),
    "tg_table_column_dtype": (C.c_int, [P, C.c_char_p, C.POINTER(C.c_int32)]),
    "tg_table_append_parquet_chunk": (C.c_int, [P, C.c_char_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_int64]),
    "tg_parquet_chunk_validity": (C.c_int64, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]),
    "tg_parquet_snappy_decompress": (C.c_int64, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64]),
    "tg_table_set_column_arrow_type": (C.c_int32, [C.c_void_p, C.c_char_p, C.c_char_p]),
    "tg_parquet_decode_to_plain": (C.c_int64, [C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int64]),
    "tg_parquet_page_decompress": (C.c_int64, [C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64]),
    "tg_parquet_inspect_chunk": (C.c_int32, [C.c_void_p, C.c_int64, C.POINTER(tg_parquet_page), C.c_int32]),
    "tg_table_column_buffers": (C.c_int, [P, C.c_char_p, C.c_char_p, C.POINTER(tg_column_buffers)]),
    "tg_table_append_host": (C.c_int, [P, C.c_char_p, C.c_int32, C.c_int64, P, P, P, C.c_int64]),
    "tg_table_adopt_device": (C.c_int, [P, C.c_char_p, C.c_int32, C.c_int64, P, P, P, C.c_int64]),
    "tg_table_append_arrow": (C.c_int, [P, P, P]),
    "tg_table_append_arrow_device": (C.c_int, [P, P, P]),
    "tg_table_append_csv": (C.c_int, [P, STRS, STRS, C.c_int32, P, C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_int64)]),
    "tg_csv_parse_value": (C.c_int, [C.c_char_p, P, C.c_int64, P, C.POINTER(C.c_int32)]),
    "tg_table_append_csv_format": (C.c_int, [P, STRS, STRS, C.c_int32, P, C.c_int64, C.POINTER(tg_csv_format), C.POINTER(C.c_int64)]),
    "tg_csv_split_host": (C.c_int, [C.POINTER(tg_csv_format), P, C.c_int64, P, C.POINTER(C.c_int64), P, C.POINTER(C.c_int64),
                                    C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "tg_table_partition_fingerprints": (C.c_int, [P, C.c_char_p, STRS, C.c_int32, C.c_int32, PP, C.POINTER(C.c_int64)]),
    "tg_table_partition_keys": (C.c_int, [P, C.c_char_p, C.c_char_p, C.c_int32, PP, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "tg_plan_create": (C.c_int, [PP]),
    "tg_plan_destroy": (None, [P]),
    "tg_plan_num_slots": (C.c_int32, [P]),
    "tg_plan_add_completeness": (C.c_int32, [P, STRS, C.c_int32, C.c_double, C.c_int32, C.c_int32]),
    "tg_plan_add_size": (C.c_int32, [P, tg_assertion]),
    "tg_plan_add_statistic": (C.c_int32, [P, C.c_char_p, C.c_int32, C.c_double, tg_assertion]),
    "tg_plan_add_multi_statistic": (C.c_int32, [P, C.c_char_p, C.POINTER(C.c_int32), C.POINTER(C.c_double),
                                                 C.POINTER(tg_assertion), C.c_int32]),
    "tg_plan_add_format": (C.c_int32, [P, C.c_char_p, C.c_int32, C.c_char_p, C.c_int32, C.c_double,
                                        C.POINTER(tg_format_options)]),
    "tg_plan_add_uniqueness": (C.c_int32, [P, STRS, C.c_int32, C.c_int32, C.c_double, tg_assertion, C.c_int32]),
    "tg_plan_add_correlation": (C.c_int32, [P, C.c_char_p, C.c_char_p, C.c_int32, tg_assertion]),
    "tg_plan_add_custom_sql": (C.c_int32, [P, C.c_char_p, C.c_char_p]),
    "tg_plan_add_foreign_key": (C.c_int32, [P, C.c_char_p, C.c_char_p, C.c_int32, C.c_int32]),
    "tg_plan_add_analyzer": (C.c_int32, [P, C.c_int32, C.c_char_p, C.c_char_p, C.c_char_p]),
    "tg_plan_add_kll": (C.c_int32, [P, C.c_char_p, C.c_int32, C.POINTER(C.c_double), C.c_int32]),
    "tg_plan_add_length": (C.c_int32, [P, C.c_char_p, C.c_int32, C.c_int64, C.c_int64]),
    "tg_plan_add_containment": (C.c_int32, [P, C.c_char_p, STRS, C.c_int32]),
    "tg_plan_add_non_negative": (C.c_int32, [P, C.c_char_p]),
    "tg_plan_add_approx_count_distinct": (C.c_int32, [P, C.c_char_p, tg_assertion]),
    "tg_plan_add_data_type": (C.c_int32, [P, C.c_char_p, C.c_int32, C.c_double]),
    "tg_plan_add_column_count": (C.c_int32, [P, tg_assertion]),
    "tg_plan_add_histogram": (C.c_int32, [P, C.c_char_p, C.c_int32]),
    "tg_plan_add_quantile": (C.c_int32, [P, C.c_char_p, C.c_int32, C.POINTER(C.c_double), C.POINTER(tg_assertion),
                                         C.c_int32, C.c_int32]),
    "tg_plan_add_grouped_completeness": (C.c_int32, [P, C.c_char_p, STRS, C.c_int32, C.c_int32, C.c_int32]),
    "tg_plan_add_value_histogram": (C.c_int32, [P, C.c_char_p]),
    "tg_plan_execute": (C.c_int, [P, P, C.c_char_p]),
    "tg_plan_execute_partial": (C.c_int, [P, P, C.c_char_p]),
    "tg_plan_request_row_mask": (C.c_int, [P, C.c_int32]),
    "tg_plan_export_row_mask": (C.c_int, [P, C.c_int32, P, P]),
    "tg_plan_request_key_rows": (C.c_int, [P, C.c_int32, C.c_int32]),
    "tg_plan_export_key_rows": (C.c_int, [P, C.c_int32, C.c_int32, P, P]),
    "tg_plan_partial_size": (C.c_int, [P, C.POINTER(C.c_size_t)]),
    "tg_plan_partial_export": (C.c_int, [P, P, C.c_size_t]),
    "tg_plan_partial_reset": (C.c_int, [P]),
    "tg_plan_partial_merge": (C.c_int, [P, P, C.c_size_t]),
    "tg_plan_finalize": (C.c_int, [P]),
    "tg_plan_num_aggregates": (C.c_int32, [P]),
    "tg_plan_aggregate_info": (C.c_int, [P, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_char_p)]),
    "tg_engine_mailbox_create": (C.c_int, [P, C.c_int32, C.c_int32, C.c_size_t, P]),
    "tg_engine_mailbox_open": (C.c_int, [P, P]),
    "tg_plan_exchange_and_finalize": (C.c_int, [P, P]),
    "tg_plan_exchange_ex": (C.c_int, [P, P, C.POINTER(C.c_int32)]),
    "tg_plan_execute_exchange": (C.c_int, [P, P, C.c_char_p, C.POINTER(C.c_int32)]),
    "tg_debug_sort_pairs": (C.c_int, [P, P, C.c_int64, C.c_int32, C.c_int32, P, P]),
    "tg_comm_unique_id": (C.c_int, [P]),
    "tg_comm_init": (C.c_int, [P, P, C.c_int32, C.c_int32]),
    "tg_comm_destroy": (C.c_int, [P]),
    "tg_comm_bytes_sent": (C.c_uint64, [P]),
    "tg_table_shuffle_column": (C.c_int, [P, C.c_char_p, C.c_char_p, C.c_char_p, C.c_int32, C.POINTER(C.c_int64)]),
    "tg_table_shuffle_fingerprints": (C.c_int, [P, C.c_char_p, STRS, C.c_int32, C.c_char_p, C.POINTER(C.c_int64)]),
    "tg_rank_begin": (C.c_int, [P, C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(C.c_int64)]),
    "tg_rank_local_sort": (C.c_int, [P]),
    "tg_rank_sample": (C.c_int32, [P, C.c_int32, C.POINTER(C.c_uint64)]),
    "tg_rank_split": (C.c_int, [P, C.POINTER(C.c_uint64), C.c_int32, C.POINTER(C.c_int64)]),
    "tg_rank_send_buffers": (C.c_int, [P, PP, PP, C.POINTER(C.c_int32)]),
    "tg_rank_recv_buffers": (C.c_int, [P, C.c_int64, PP, PP]),
    "tg_rank_recv_commit": (C.c_int, [P, C.c_int64]),
    "tg_rank_finish_x": (C.c_int, [P, C.c_uint64]),
    "tg_rank_finish_y": (C.c_int, [P, C.c_uint64, C.c_double, C.POINTER(C.c_uint64), C.POINTER(C.c_double)]),
    "tg_rank_abort": (C.c_int, [P]),
    "tg_rank_exchange": (C.c_int, [P, C.POINTER(C.c_int64), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_int32)]),
    "tg_plan_set_aggregate_partial": (C.c_int, [P, C.c_int32, C.POINTER(C.c_uint64), C.POINTER(C.c_double)]),
    "tg_plan_kll_levels": (C.c_int32, [P, C.c_int32, C.c_int32, C.POINTER(C.c_double), C.c_int32]),
    "tg_plan_histogram_pending": (C.c_int32, [P, C.POINTER(C.c_int32), C.c_int32]),
    "tg_plan_histogram_rebucket": (C.c_int, [P, P, C.c_char_p, C.c_int32, C.POINTER(C.c_uint64), C.c_int32]),
    "tg_plan_histogram_install": (C.c_int, [P, C.c_int32, C.POINTER(C.c_uint64), C.c_int32]),
    "tg_plan_analyzer_state_json": (C.c_int32, [P, C.c_int32, C.c_char_p, C.c_int32]),
    "tg_plan_redirect_aggregate": (C.c_int, [P, C.c_int32, C.c_int32, C.c_char_p]),
    "tg_plan_result": (C.c_int, [P, C.c_int32, C.POINTER(tg_result)]),
    "tg_plan_analyzer_result": (C.c_int, [P, C.c_int32, C.POINTER(tg_analyzer_result)]),
    "tg_plan_map_size": (C.c_int32, [P, C.c_int32]),
    "tg_plan_map_entry": (C.c_int, [P, C.c_int32, C.c_int32, C.POINTER(C.c_char_p), C.POINTER(C.c_double)]),
    "tg_plan_exec_stats": (C.c_int, [P, C.POINTER(tg_exec_stats)]),
    "tg_assertion_evaluate": (C.c_int32, [tg_assertion, C.c_double]),
    "tg_assertion_description": (C.c_int32, [tg_assertion, C.c_char_p, C.c_int32]),
    "tg_logical_evaluate": (C.c_int32, [C.c_int32, C.c_int32, C.POINTER(C.c_uint8), C.c_int32]),
    "tg_validate_identifier": (C.c_int, [C.c_char_p]),
    "tg_validate_regex_pattern": (C.c_int, [C.c_char_p]),
    "tg_validate_sql_expression": (C.c_int, [C.c_char_p]),
    "tg_format_pattern": (C.c_char_p, [C.c_int32, C.c_char_p, C.c_int32]),
    "tg_regex_host_match": (C.c_int32, [C.c_char_p, C.c_int32, P, C.c_int64, C.POINTER(C.c_int32)]),
    "tg_regex_dfa_size": (C.c_int32, [C.c_char_p, C.c_int32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "tg_format_f64": (C.c_int32, [C.c_double, C.c_char_p, C.c_int32]),
    "tg_format_f64_json": (C.c_int32, [C.c_double, C.c_char_p, C.c_int32]),
}

_lib = None


def lib():
    """Load libtermgpu.so (once). Raises if the CUDA extension has not been built: there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(termgpu has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def last_error():
    m = lib().tg_last_error()
    return m.decode("utf-8", "replace") if m else ""


def check(status):
    if status != 0:
        raise TermGpuError(status, last_error())


def check_slot(slot):
    if slot < 0:
        raise TermGpuError(-slot, last_error())
    return slot
