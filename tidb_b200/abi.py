"""ctypes mirror of include/tidbgpu.h — the C-ABI of libtidbgpu.so.

The structures here are byte-for-byte the ones a cgo shim would fill (INTEGRATION.md); the Python
host side exists only because this image has no Go toolchain.  Loading fails loudly when the CUDA
library has not been built: there is no CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TIDBGPU_LIB") or os.path.join(_HERE, "csrc", "libtidbgpu.so")   # TIDBGPU_LIB: A/B runs against another build of the same ABI

# ---- status codes (tg_status) -------------------------------------------------------------------
TG_OK, TG_ERR_INVALID, TG_ERR_UNSUPPORTED, TG_ERR_CUDA, TG_ERR_OOM = 0, 1, 2, 3, 4
TG_ERR_STATE, TG_ERR_CANCELLED, TG_ERR_OVERFLOW, TG_ERR_CAPACITY = 5, 6, 7, 8

# ---- enumerations copied from the reference (see tidbgpu.h for file:line) ------------------------
TYPE_TINY, TYPE_SHORT, TYPE_LONG, TYPE_FLOAT, TYPE_DOUBLE = 1, 2, 3, 4, 5
TYPE_TIMESTAMP, TYPE_LONGLONG, TYPE_INT24, TYPE_DATE, TYPE_DURATION = 7, 8, 9, 10, 11
TYPE_DATETIME, TYPE_YEAR, TYPE_NEWDECIMAL, TYPE_VARSTRING = 12, 13, 0xF6, 0xFD
FLAG_NOT_NULL, FLAG_UNSIGNED = 1 << 0, 1 << 5
JOIN_INNER, JOIN_LEFT_OUTER, JOIN_RIGHT_OUTER, JOIN_SEMI, JOIN_ANTI_SEMI = 0, 1, 2, 3, 4
JOIN_LEFT_OUTER_SEMI, JOIN_ANTI_LEFT_OUTER_SEMI = 5, 6
AGG_COUNT, AGG_SUM, AGG_AVG, AGG_MIN, AGG_MAX, AGG_FIRSTROW = 0, 1, 2, 3, 4, 5
AGGMODE_COMPLETE, AGGMODE_FINAL, AGGMODE_PARTIAL1, AGGMODE_PARTIAL2, AGGMODE_DEDUP = 0, 1, 2, 3, 4
CMP_LT, CMP_LE, CMP_GT, CMP_GE, CMP_EQ, CMP_NE = 0, 1, 2, 3, 4, 5
ARITH_PLUS, ARITH_MINUS, ARITH_MUL = 0, 1, 2


class TgColumn(C.Structure):
    _fields_ = [("length", C.c_int64), ("null_bitmap", C.c_void_p), ("offsets", C.c_void_p),
                ("data", C.c_void_p), ("elem_len", C.c_int32), ("reserved", C.c_int32)]


class TgChunk(C.Structure):
    _fields_ = [("ncols", C.c_int32), ("reserved", C.c_int32), ("cols", C.POINTER(TgColumn)),
                ("sel", C.c_void_p), ("nsel", C.c_int64)]


class TgMutColumn(C.Structure):
    _fields_ = [("null_bitmap", C.c_void_p), ("data", C.c_void_p), ("elem_len", C.c_int32),
                ("reserved", C.c_int32)]


class TgMutChunk(C.Structure):
    _fields_ = [("ncols", C.c_int32), ("reserved", C.c_int32), ("cols", C.POINTER(TgMutColumn)),
                ("capacity_rows", C.c_int64)]


class TgFilterItem(C.Structure):
    _fields_ = [("op", C.c_int32), ("lhs_col", C.c_int32), ("rhs_col", C.c_int32),
                ("is_real", C.c_int32), ("lhs_unsigned", C.c_int32), ("rhs_unsigned", C.c_int32),
                ("const_i64", C.c_int64), ("const_f64", C.c_double)]


class TgOtherItem(C.Structure):
    """tg_other_item: one CNF item of OtherCondition over the joined row (side 0 = left child, 1 = right, -1 = constant)"""
    _fields_ = [("op", C.c_int32), ("is_real", C.c_int32), ("lhs_side", C.c_int32), ("lhs_col", C.c_int32),
                ("rhs_side", C.c_int32), ("rhs_col", C.c_int32), ("lhs_unsigned", C.c_int32), ("rhs_unsigned", C.c_int32),
                ("const_i64", C.c_int64), ("const_f64", C.c_double)]


class TgJoinDesc(C.Structure):
    _fields_ = [("join_type", C.c_int32), ("build_is_right", C.c_int32),
                ("n_left_cols", C.c_int32), ("n_right_cols", C.c_int32),
                ("left_types", C.POINTER(C.c_int32)), ("left_flags", C.POINTER(C.c_uint32)),
                ("right_types", C.POINTER(C.c_int32)), ("right_flags", C.POINTER(C.c_uint32)),
                ("nkeys", C.c_int32), ("reserved0", C.c_int32),
                ("left_key_idx", C.POINTER(C.c_int32)), ("right_key_idx", C.POINTER(C.c_int32)),
                ("n_lused", C.c_int32), ("n_rused", C.c_int32),
                ("lused", C.POINTER(C.c_int32)), ("rused", C.POINTER(C.c_int32)),
                ("n_build_filter", C.c_int32), ("n_probe_filter", C.c_int32),
                ("build_filter", C.POINTER(TgFilterItem)), ("probe_filter", C.POINTER(TgFilterItem)),
                ("device", C.c_int32), ("reserved1", C.c_int32),
                ("stream", C.c_void_p), ("load_factor", C.c_double),
                ("n_other_cond", C.c_int32), ("reserved2", C.c_int32), ("other_cond", C.POINTER(TgOtherItem))]


class TgJoinStats(C.Structure):
    _fields_ = [("build_rows", C.c_int64), ("build_valid_keys", C.c_int64),
                ("table_slots", C.c_int64), ("distinct_keys", C.c_int64), ("max_dup", C.c_int64),
                ("probe_rows", C.c_int64), ("output_rows", C.c_int64),
                ("kernel_launches", C.c_int64), ("table_mode", C.c_int32), ("reserved", C.c_int32),
                ("build_ms", C.c_double), ("probe_ms", C.c_double),
                ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64)]


class TgSortItem(C.Structure):
    _fields_ = [("col", C.c_int32), ("desc", C.c_int32)]


class TgMailTargets(C.Structure):
    """tg_mail_targets: where this rank's mailbox word lives on every peer (tg_mail_signal)"""
    _fields_ = [("n", C.c_int32), ("pad", C.c_int32), ("slot", C.c_uint64 * 16)]


class TgAggFunc(C.Structure):
    _fields_ = [("name", C.c_int32), ("mode", C.c_int32), ("arg_col", C.c_int32),
                ("arg_type", C.c_int32), ("arg_flag", C.c_uint32), ("arg_col2", C.c_int32),
                ("arg_expr", C.c_int32), ("reserved", C.c_int32), ("arg_const", C.c_double)]


ARGEXPR_COL, ARGEXPR_MUL, ARGEXPR_MUL_CSUB = 0, 1, 2


class TgAggDesc(C.Structure):
    _fields_ = [("n_cols", C.c_int32), ("n_group_by", C.c_int32),
                ("col_types", C.POINTER(C.c_int32)), ("col_flags", C.POINTER(C.c_uint32)),
                ("group_by_cols", C.POINTER(C.c_int32)),
                ("n_funcs", C.c_int32), ("device", C.c_int32),
                ("funcs", C.POINTER(TgAggFunc)), ("stream", C.c_void_p),
                ("expected_groups", C.c_int64)]


class TgAggStats(C.Structure):
    _fields_ = [("input_rows", C.c_int64), ("groups", C.c_int64), ("table_slots", C.c_int64),
                ("kernel_launches", C.c_int64), ("update_ms", C.c_double),
                ("finalize_ms", C.c_double), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64)]


class TgSortDesc(C.Structure):
    _fields_ = [("n_cols", C.c_int32), ("n_items", C.c_int32),
                ("col_types", C.POINTER(C.c_int32)), ("col_flags", C.POINTER(C.c_uint32)),
                ("items", C.POINTER(TgSortItem)), ("device", C.c_int32), ("reserved", C.c_int32),
                ("stream", C.c_void_p), ("expected_rows", C.c_int64)]


class TgSortStats(C.Structure):
    _fields_ = [("input_rows", C.c_int64), ("digit_passes", C.c_int64), ("skipped_passes", C.c_int64),
                ("null_passes", C.c_int64), ("kernel_launches", C.c_int64), ("sort_ms", C.c_double),
                ("gather_ms", C.c_double), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64)]


def sort_desc(schema, by_items, device: int = 0, expected_rows: int = 0, stream=None):
    """tg_sort_desc for a child schema (FieldType list) and ORDER BY items [(column, desc)]; returns (desc, keep-alive)"""
    tps = (C.c_int32 * max(len(schema), 1))(*[t.tp for t in schema])
    fls = (C.c_uint32 * max(len(schema), 1))(*[t.flag for t in schema])
    items = (TgSortItem * max(len(by_items), 1))(*[TgSortItem(int(c), int(bool(d))) for c, d in by_items])
    d = TgSortDesc()
    d.n_cols, d.n_items = len(schema), len(by_items)
    d.col_types = C.cast(tps, C.POINTER(C.c_int32))
    d.col_flags = C.cast(fls, C.POINTER(C.c_uint32))
    d.items = C.cast(items, C.POINTER(TgSortItem))
    d.device, d.stream, d.expected_rows = device, stream, expected_rows
    return d, (tps, fls, items)


# every symbol include/tidbgpu.h declares; tests/test_abi_exports.py checks the .so exports them all
EXPORTED_SYMBOLS = [
    "tg_last_error", "tg_abi_version", "tg_device_count", "tg_device_info", "tg_fixed_len",
    "tg_host_alloc", "tg_host_free", "tg_dev_alloc", "tg_dev_free", "tg_memcpy_h2d", "tg_memcpy_d2h", "tg_memcpy_d2d_async",
    "tg_device_synchronize",
    "tg_chunk_wire_size", "tg_chunk_encode", "tg_chunk_decode", "tg_chunk_decode_into",
    "tg_join_supported", "tg_join_open", "tg_join_build_push", "tg_join_build_push_dev",
    "tg_join_build_finish", "tg_join_probe_push", "tg_join_probe_finish", "tg_join_next", "tg_join_next_wait", "tg_join_probe_rewind",
    "tg_join_close", "tg_join_probe_dev", "tg_join_probe_dev_seg", "tg_join_get_stats",
    "tg_agg_supported", "tg_agg_open", "tg_agg_push", "tg_agg_push_dev", "tg_agg_finish",
    "tg_agg_next", "tg_agg_close", "tg_agg_result_dev", "tg_agg_get_stats",
    "tg_vec_compare_int", "tg_vec_compare_real", "tg_vec_arith_int", "tg_vec_arith_real",
    "tg_vec_filter", "tg_topn",
    "tg_sort_supported", "tg_sort_open", "tg_sort_push", "tg_sort_push_dev", "tg_sort_finish", "tg_sort_next",
    "tg_sort_result_dev", "tg_sort_get_stats", "tg_sort_close", "tg_sort_key_host",
    "tg_partition_by_key", "tg_partition_of_key", "tg_partition_exchange", "tg_partition_exchange_cf", "tg_partition_exchange_cf_ex", "tg_partition_exchange_cf_spill", "tg_partition_count",
    "tg_mail_signal", "tg_mail_wait", "tg_peer_copy_regions",
    "tg_ipc_export", "tg_ipc_open", "tg_ipc_close",
]

_lib = None


class TgError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"tidbgpu error {code}: {msg}")
        self.code = code


def load_lib() -> C.CDLL:
    """Load libtidbgpu.so (built in-tree by tidb_b200/build.py).  No fallback: missing library is an error."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: run `python -m tidb_b200.build` (nvcc, sm_100a). "
            "There is no CPU fallback for the GPU operators.")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    lib.tg_last_error.restype = C.c_char_p
    lib.tg_partition_of_key.restype = C.c_int32
    lib.tg_partition_of_key.argtypes = [C.c_int64, C.c_int32]
    lib.tg_sort_key_host.argtypes = [C.c_int32, C.c_uint32, C.c_int32, C.c_uint64, C.POINTER(C.c_uint64)]
    _lib = lib
    return lib


def check(code: int) -> None:
    if code != 0:
        lib = load_lib()
        msg = lib.tg_last_error()
        raise TgError(code, msg.decode() if msg else "")
