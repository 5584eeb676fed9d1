"""CPU-side checks of the GPU sort (tg_sort_*, csrc/sort.cu): the planner gate answers without a device, opening a sort
without a device fails (no CPU fallback), the key normalizer — evaluated on the host by tg_sort_key_host, the same
__host__ __device__ function the kernels use — orders edge values exactly as the SortExec restatement does (ties included),
and the restatement reproduces the ORDER BY results transcribed from the reference."""
import ctypes as C
import json
import math
import os
import struct

import pytest

from tidb_b200 import abi
from tidb_b200.plan import FieldType
import sort_oracle as OS

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SORT_TYPES = [abi.TYPE_TINY, abi.TYPE_SHORT, abi.TYPE_INT24, abi.TYPE_LONG, abi.TYPE_LONGLONG, abi.TYPE_YEAR,
              abi.TYPE_DURATION, abi.TYPE_DOUBLE, abi.TYPE_DATE, abi.TYPE_DATETIME, abi.TYPE_TIMESTAMP]


@pytest.fixture(scope="module")
def lib():
    from tidb_b200 import build
    build.build()
    return abi.load_lib()


def _supported(lib, schema, by):
    d, keep = abi.sort_desc(schema, by)
    return lib.tg_sort_supported(C.byref(d))


def test_sort_gate_accepts_every_8_byte_type(lib):
    for tp in SORT_TYPES:
        for flag in (0, abi.FLAG_UNSIGNED, abi.FLAG_NOT_NULL):
            schema = [FieldType(tp, flag)] * 8 + [FieldType(abi.TYPE_LONGLONG, 0)]
            for n_items in range(1, 9):
                for desc in (False, True):
                    by = [(c, desc if c % 2 == 0 else not desc) for c in range(n_items)]
                    assert _supported(lib, schema, by) == abi.TG_OK, (tp, flag, n_items, desc)


def test_sort_gate_declines(lib):
    INT = FieldType(abi.TYPE_LONGLONG, 0)
    for tp in (abi.TYPE_FLOAT, abi.TYPE_NEWDECIMAL, abi.TYPE_VARSTRING):
        assert _supported(lib, [INT, FieldType(tp, 0)], [(1, False)]) == abi.TG_ERR_UNSUPPORTED   # as an item
        assert _supported(lib, [INT, FieldType(tp, 0)], [(0, False)]) == abi.TG_ERR_UNSUPPORTED   # as a payload column
    assert _supported(lib, [INT] * 9, [(c, False) for c in range(9)]) == abi.TG_ERR_UNSUPPORTED   # > 8 items
    assert _supported(lib, [INT] * 2, []) == abi.TG_ERR_UNSUPPORTED
    assert _supported(lib, [INT] * 17, [(0, False)]) == abi.TG_ERR_UNSUPPORTED                      # > TG_MAX_COLS
    assert _supported(lib, [INT] * 2, [(2, False)]) == abi.TG_ERR_INVALID                           # column out of range
    assert _supported(lib, [INT] * 2, [(-1, True)]) == abi.TG_ERR_INVALID
    assert lib.tg_sort_supported(None) == abi.TG_ERR_INVALID


def test_sort_open_without_device_fails(lib):
    if lib.tg_device_count() > 0:
        pytest.skip("a CUDA device is present")
    d, keep = abi.sort_desc([FieldType(abi.TYPE_LONGLONG, 0)], [(0, False)])
    h = C.c_void_p()
    assert lib.tg_sort_open(C.byref(d), C.byref(h)) == abi.TG_ERR_CUDA
    assert b"no CPU fallback" in lib.tg_last_error()
    assert not h.value


def _dbl_bits(x: float) -> int:
    return struct.unpack("<Q", struct.pack("<d", x))[0]


def _bits_dbl(u: int) -> float:
    return struct.unpack("<d", struct.pack("<Q", u))[0]


I64_MIN, I64_MAX, U64_MAX = -(1 << 63), (1 << 63) - 1, (1 << 64) - 1
TIME_WORDS = [0x19A2_8000_0000_0000 | f for f in (0, 1, 6, 0xF)] + [0x19A2_8000_0000_0010 | f for f in (0, 3)] + [0, 0xF, U64_MAX]
EDGES = {
    "int": (abi.TYPE_LONGLONG, 0, [I64_MIN, I64_MIN + 1, -1, 0, 1, I64_MAX, I64_MAX - 1, -1, 0]),
    "duration": (abi.TYPE_DURATION, 0, [I64_MIN, -86400_000000, -1, 0, 1, 838 * 3600_000000, I64_MAX, 0]),
    "uint": (abi.TYPE_LONGLONG, abi.FLAG_UNSIGNED, [0, 1, I64_MAX, 1 << 63, U64_MAX, U64_MAX - 1, 0]),
    "real": (abi.TYPE_DOUBLE, 0, [0.0, -0.0, math.inf, -math.inf, 1.0, -1.0, 5e-324, -5e-324, 2.2250738585072014e-308,
                                  1.7976931348623157e308, -1.7976931348623157e308, _bits_dbl(0x7FF8000000000000),
                                  _bits_dbl(0x7FF0000000000001), _bits_dbl(0xFFF8000000000123), _bits_dbl(0xFFFFFFFFFFFFFFFF)]),
    "time": (abi.TYPE_DATETIME, 0, TIME_WORDS),
}


def _raw(v, kind):
    return _dbl_bits(v) if kind == "real" else v % (1 << 64)


def _canon(v, kind):
    """the class of values the comparator calls equal"""
    if v is None:
        return ("null",)
    if kind == "real":
        return ("nan",) if math.isnan(v) else (v + 0.0,)
    return (OS.comparable(v, kind),)


@pytest.mark.parametrize("kind", sorted(EDGES))
@pytest.mark.parametrize("desc", [False, True])
def test_sort_key_matches_oracle(lib, kind, desc):
    tp, flag, vals = EDGES[kind]
    vals = list(vals) + [None, None]
    keyed = []
    for v in vals:
        k = C.c_uint64(0)
        if v is None:
            keyed.append(((1 if desc else 0), 0, v))   # the NULL pass: NULLs first ascending, last descending
            continue
        assert lib.tg_sort_key_host(tp, flag, int(desc), C.c_uint64(_raw(v, kind)), C.byref(k)) == abi.TG_OK
        keyed.append(((0 if desc else 1), k.value, v))
    by_key = [v for _, _, v in sorted(keyed, key=lambda t: (t[0], t[1]))]
    exp = [r[0] for r in OS.sort_rows([(v,) for v in vals], [kind], [(0, desc)])]
    assert [_canon(v, kind) for v in by_key] == [_canon(v, kind) for v in exp]
    # ties: two values get the same key exactly when the comparator calls them equal
    for a in keyed:
        for b in keyed:
            assert ((a[0], a[1]) == (b[0], b[1])) == (_canon(a[2], kind) == _canon(b[2], kind)), (a, b)


def test_sort_key_host_declines_unsupported_types(lib):
    k = C.c_uint64(0)
    for tp in (abi.TYPE_FLOAT, abi.TYPE_NEWDECIMAL, abi.TYPE_VARSTRING):
        assert lib.tg_sort_key_host(tp, 0, 0, C.c_uint64(1), C.byref(k)) == abi.TG_ERR_UNSUPPORTED
    assert lib.tg_sort_key_host(abi.TYPE_LONGLONG, 0, 0, C.c_uint64(1), None) == abi.TG_ERR_INVALID


def _golden_cases():
    return json.load(open(os.path.join(ROOT, "tests", "golden", "sort_cases.json")))["cases"]


@pytest.mark.parametrize("case", _golden_cases(), ids=lambda c: c["name"])
def test_sort_oracle_reproduces_reference_results(case):
    rows = [tuple(r) for r in case["rows"]]
    got = OS.sort_rows(rows, case["kinds"], [(c, d) for c, d in case["by_items"]])
    assert [[r[c] for c in case["select"]] for r in got] == case["expected"]


def test_sort_oracle_time_and_duration_kinds():
    # fsp bits do not order time words; DURATION is signed
    rows = [(0x1000 | 5,), (0x1000,), (0x0FF0 | 0xF,), (0x2000,)]
    assert OS.sort_rows(rows, ["time"], [(0, False)]) == [(0x0FF0 | 0xF,), (0x1000 | 5,), (0x1000,), (0x2000,)]
    assert OS.sort_rows([(1,), (-5,), (None,), (0,)], ["duration"], [(0, True)]) == [(1,), (0,), (-5,), (None,)]
