"""SortExec on the device (tg_sort_*, csrc/sort.cu) against the restatement of sortexec.SortExec's order
(tests/sort_oracle.py over oracle/topn.py's comparator), through the executor shim and the C ABI.  Ties are unordered in
the reference (sort.Slice), so outputs are compared on their ORDER BY values position by position and, inside each run of
tied keys, as a multiset of whole rows — never on the device sort's (stable) tie order."""
import ctypes as C
import json
import math
import os
import struct
from itertools import groupby

import numpy as np
import pytest

from tidb_b200 import abi
from tidb_b200.chunk import Chunk, Column, MutChunk
from tidb_b200.executor import MockDataSource, SortExec, drain
from tidb_b200.plan import FieldType
import sort_oracle as OS

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INT = FieldType(abi.TYPE_LONGLONG, 0)
UINT = FieldType(abi.TYPE_LONGLONG, abi.FLAG_UNSIGNED)
DBL = FieldType(abi.TYPE_DOUBLE, 0)
DT = FieldType(abi.TYPE_DATETIME, 0)
DUR = FieldType(abi.TYPE_DURATION, 0)
KIND = {id(INT): "int", id(UINT): "uint", id(DBL): "real", id(DT): "time", id(DUR): "duration"}


def _rows(chunks):
    out = []
    for c in chunks:
        cols = [(col.data, col.nulls()) for col in c.columns]
        for i in range(c.num_rows()):
            out.append(tuple(None if nl[i] else v[i].item() for v, nl in cols))
    return out


def _canon(v, kind):
    if v is None:
        return ("null",)
    if kind == "real":
        return ("nan",) if math.isnan(v) else (v + 0.0,)
    return (OS.comparable(v, kind),)


def _exact(v):
    return None if v is None else (struct.pack("<d", v) if isinstance(v, float) else v)


def _check(got, rows, kinds, by):
    exp = OS.sort_rows(rows, kinds, by)
    assert len(got) == len(exp)
    key = lambda r: tuple(_canon(r[c], kinds[c]) for c, _ in by)
    gk, ek = [key(r) for r in got], [key(r) for r in exp]
    assert gk == ek                                           # the same ORDER BY values at every position
    pos = 0
    for k, grp in groupby(range(len(gk)), key=lambda i: gk[i]):   # each run of tied keys holds the same rows
        idx = list(grp)
        g = sorted(repr(tuple(_exact(v) for v in got[i])) for i in idx)
        e = sorted(repr(tuple(_exact(v) for v in exp[i])) for i in idx)
        assert g == e, k
        pos += len(idx)
    return exp


def _run(tbl_chunks, schema, by, required_rows=1024):
    e = SortExec(MockDataSource(schema, tbl_chunks), by)
    e.open()
    out = []
    try:
        while True:
            c = e.next(required_rows)
            if c.num_rows() == 0:
                break
            assert c.num_rows() <= required_rows
            out.append(c)
        stats = e.stats()
    finally:
        e.close()
    return _rows(out), stats


def _golden_cases():
    return json.load(open(os.path.join(ROOT, "tests", "golden", "sort_cases.json")))["cases"]


@pytest.mark.parametrize("case", _golden_cases(), ids=lambda c: c["name"])
def test_sort_goldens(case):
    schema = [FieldType(getattr(abi, "TYPE_" + t), 0) for t in case["types"]]
    n = len(case["rows"])
    cols = []
    for c in range(len(schema)):
        vals = [r[c] for r in case["rows"]]
        nulls = np.array([v is None for v in vals])
        cols.append(Column(np.array([0 if v is None else v for v in vals], dtype=np.int64), nulls if nulls.any() else None))
    got, _ = _run(Chunk(cols).split(2), schema, [(c, d) for c, d in case["by_items"]], required_rows=3)
    assert len(got) == n
    assert [[r[c] for c in case["select"]] for r in got] == case["expected"]


def test_sort_empty_and_one_row():
    got, st = _run([], [INT, DBL], [(0, False)])
    assert got == [] and st.input_rows == 0
    one = Chunk([Column(np.array([7], dtype=np.int64)), Column(np.array([1.5]), np.array([True]))])
    got, _ = _run([one], [INT, DBL], [(1, True), (0, False)])
    assert got == [(7, None)]


def test_sort_all_null_column():
    n = 5000
    rng = np.random.default_rng(1)
    a = rng.integers(-50, 50, n).astype(np.int64)
    tbl = Chunk([Column(np.zeros(n, dtype=np.int64), np.ones(n, dtype=bool)), Column(a)])
    rows = _rows([tbl])
    for by in ([(0, False), (1, True)], [(0, True), (1, False)]):
        got, st = _run(tbl.split(1024), [INT, INT], by)
        _check(got, rows, ["int", "int"], by)
        assert st.null_passes == 0          # every row is NULL: the NULL-flag histogram has one bin


def test_sort_constant_key_skips_every_digit_pass():
    n = 70_000
    tbl = Chunk([Column(np.full(n, -123456789, dtype=np.int64)), Column(np.arange(n, dtype=np.int64))])
    got, st = _run(tbl.split(1024), [INT, INT], [(0, True)])
    assert st.digit_passes == 0 and st.skipped_passes == 8 and st.null_passes == 0
    assert sorted(r[1] for r in got) == list(range(n)) and all(r[0] == -123456789 for r in got)


def test_sort_low_16_bit_keys_run_two_passes():
    n = 300_000
    rng = np.random.default_rng(2)
    k = rng.integers(0, 1 << 16, n).astype(np.int64)
    tbl = Chunk([Column(k), Column(rng.random(n))])
    got, st = _run(tbl.split(1024), [INT, DBL], [(0, False)])
    assert st.digit_passes == 2 and st.skipped_passes == 6
    assert [r[0] for r in got] == sorted(k.tolist())
    assert sorted((r[0], r[1]) for r in got) == sorted(zip(k.tolist(), tbl.columns[1].data.tolist()))


def _random_table(n, seed):
    rng = np.random.default_rng(seed)
    a = rng.integers(-1000, 1000, n).astype(np.int64); an = rng.random(n) < 0.01                         # heavy ties
    u = rng.integers(0, 1 << 63, n).astype(np.int64) * 2 + rng.integers(0, 2, n); un = rng.random(n) < 0.01   # full uint64
    x = np.floor(rng.random(n) * 2000) / 4 - 250; xn = rng.random(n) < 0.01
    special = rng.random(n)
    x[special < 0.01] = np.nan
    x[(special >= 0.01) & (special < 0.02)] = -0.0
    x[(special >= 0.02) & (special < 0.025)] = np.inf
    x[(special >= 0.025) & (special < 0.03)] = -np.inf
    nan_payload = np.where(rng.random(n) < 0.5, 0x7FF8000000000001, 0xFFF8000000000ABC).astype(np.uint64).view(np.float64)
    x = np.where(np.isnan(x), nan_payload, x)
    days = rng.integers(0, 300, n).astype(np.int64)                                                      # time words, fsp bits vary
    t = ((days << 24) | (rng.integers(0, 4, n).astype(np.int64) << 4) | rng.integers(0, 16, n)).astype(np.int64); tn = rng.random(n) < 0.01
    d = rng.integers(-5, 5, n).astype(np.int64) * 1_000_000; dn = rng.random(n) < 0.01                  # DURATION
    return [Column(a, an), Column(u, un), Column(x, xn), Column(t, tn), Column(d, dn), Column(np.arange(n, dtype=np.int64))]


def _with_sel(cols, n, rng, chunk=1024):
    """cut into chunks of `chunk` selected rows, each carrying a sel vector over extra physical rows"""
    out, pos = [], 0
    while pos < n:
        take = min(chunk, n - pos)
        phys = take + int(rng.integers(0, 200))
        sel = np.sort(rng.choice(phys, take, replace=False)).astype(np.int64)
        pc = []
        for col in cols:
            v = np.zeros(phys, dtype=col.data.dtype); v[sel] = col.data[pos:pos + take]
            v[np.setdiff1d(np.arange(phys), sel)] = col.data[pos] if take else 0    # garbage rows outside sel
            nl = None
            if col.null_bitmap is not None:
                nl = np.ones(phys, dtype=bool); nl[sel] = col.nulls()[pos:pos + take]
            pc.append(Column(v, nl))
        out.append(Chunk(pc, sel))
        pos += take
    return out


SCHEMA6 = [INT, UINT, DBL, DT, DUR, INT]
KINDS6 = ["int", "uint", "real", "time", "duration", "int"]


@pytest.mark.parametrize("by", [[(0, False)], [(2, True), (0, False)], [(3, False), (1, True), (4, False)],
                                [(4, True), (2, False), (0, True), (3, True)]])
def test_sort_random_vs_oracle(by):
    n = 200_000
    cols = _random_table(n, 70 + len(by))
    rows = _rows([Chunk(cols)])
    chunks = _with_sel(cols, n, np.random.default_rng(len(by)))
    got, st = _run(chunks, SCHEMA6, by, required_rows=333)
    assert st.input_rows == n
    _check(got, rows, KINDS6, by)


def _open(schema, by):
    lib = abi.load_lib()
    d, keep = abi.sort_desc(schema, by)
    h = C.c_void_p()
    abi.check(lib.tg_sort_open(C.byref(d), C.byref(h)))
    return lib, h


def test_sort_state_errors():
    lib, h = _open([INT], [(0, False)])
    ck = Chunk([Column(np.array([3, 1, 2], dtype=np.int64))])
    cs = ck.to_struct()
    abi.check(lib.tg_sort_push(h, C.byref(cs)))
    out = MutChunk([8], 8)
    n = C.c_int64(0)
    assert lib.tg_sort_next(h, C.byref(out.struct), 8, C.byref(n)) == abi.TG_ERR_STATE
    abi.check(lib.tg_sort_finish(h))
    assert lib.tg_sort_push(h, C.byref(cs)) == abi.TG_ERR_STATE
    abi.check(lib.tg_sort_next(h, C.byref(out.struct), 8, C.byref(n)))
    assert n.value == 3 and out.data[0][:3].tolist() == [1, 2, 3]
    abi.check(lib.tg_sort_next(h, C.byref(out.struct), 8, C.byref(n)))
    assert n.value == 0
    assert lib.tg_sort_close(h) == abi.TG_OK
    assert lib.tg_sort_close(h) == abi.TG_OK
    assert lib.tg_sort_next(h, C.byref(out.struct), 8, C.byref(n)) == abi.TG_ERR_CANCELLED


def test_sort_several_device_chunks_and_host_chunks():
    # a device chunk is sorted in place when it is the only input; more pieces are appended (bitmaps at unaligned bit
    # offsets, columns that gain a bitmap late) — checked through tg_sort_next against the oracle
    import torch
    from tidb_b200.device import dev_chunk
    from tidb_b200.chunk import pack_not_null_bitmap
    rng = np.random.default_rng(5)
    lib, h = _open([INT, DBL, INT], [(1, True), (0, False)])
    rows, keep = [], []
    for i, m in enumerate((1001, 5003, 777, 64)):
        a = rng.integers(-20, 20, m).astype(np.int64)
        x = np.floor(rng.random(m) * 8) - 4; xn = rng.random(m) < 0.1 if i != 0 else None
        p = np.arange(m, dtype=np.int64) + 100000 * i
        if i == 2:   # a host chunk with a sel vector in the middle
            ck = Chunk([Column(a), Column(x, xn), Column(p)], np.arange(0, m, 2))
            cs = ck.to_struct(); keep.append(ck)
            abi.check(lib.tg_sort_push(h, C.byref(cs)))
            rows += _rows([Chunk([Column(a[::2]), Column(x[::2], xn[::2]), Column(p[::2])])])
            continue
        t = [torch.from_numpy(a).cuda(), torch.from_numpy(x).cuda(), torch.from_numpy(p).cuda()]
        nb = [None, torch.from_numpy(pack_not_null_bitmap(xn)).cuda() if xn is not None else None, None]
        ck = dev_chunk(t, nb); keep.append(ck)
        abi.check(lib.tg_sort_push_dev(h, C.byref(ck)))
        rows += _rows([Chunk([Column(a), Column(x, xn), Column(p)])])
    abi.check(lib.tg_sort_finish(h))
    got = []
    out = MutChunk([8, 8, 8], 500, [np.int64, np.float64, np.int64])
    n = C.c_int64(0)
    while True:
        abi.check(lib.tg_sort_next(h, C.byref(out.struct), 333, C.byref(n)))
        if n.value == 0:
            break
        cols = out.columns(n.value)
        got += [tuple(None if cols[c][1][i] else cols[c][0][i].item() for c in range(3)) for i in range(n.value)]
    lib.tg_sort_close(h)
    _check(got, rows, ["int", "real", "int"], [(1, True), (0, False)])


def _d2h(ptr, nbytes, dtype):
    from tidb_b200.device import fetch_device
    return fetch_device(ptr, nbytes).view(dtype)


def test_sort_device_resident_100m():
    # ORDER BY k ASC, x DESC (x nullable DOUBLE with NaN and -0.0) over 100 M device-resident rows, two payload columns
    import torch
    from tidb_b200.device import DeviceSort
    from tidb_b200.chunk import pack_not_null_bitmap, unpack_nulls
    n = 100_000_000
    rng = np.random.default_rng(11)
    k = rng.integers(0, 1 << 20, n).astype(np.int64)
    x = np.floor(rng.random(n) * 64) - 32
    sp = rng.random(n)
    x[sp < 0.001] = np.nan
    x[(sp >= 0.001) & (sp < 0.01)] = -0.0
    xn = rng.random(n) < 0.01
    rid = np.arange(n, dtype=np.int64)
    p1 = rng.integers(-(1 << 62), 1 << 62, n).astype(np.int64)
    t = [torch.from_numpy(c).cuda() for c in (k, x, rid, p1)]
    nb = [None, torch.from_numpy(pack_not_null_bitmap(xn)).cuda(), None, None]
    s = DeviceSort([INT, DBL, INT, INT], [(0, False), (1, True)], expected_rows=n)
    s.push(t, nb)
    rows, ptrs, nptrs = s.finish()
    assert rows == n and nptrs[0] == 0 and nptrs[1] != 0 and nptrs[2] == 0
    ok = _d2h(ptrs[0], n * 8, np.int64); ox = _d2h(ptrs[1], n * 8, np.float64)
    orid = _d2h(ptrs[2], n * 8, np.int64); op1 = _d2h(ptrs[3], n * 8, np.int64)
    oxn = unpack_nulls(_d2h(nptrs[1], (n + 7) // 8, np.uint8), n)
    s.close()
    del t, nb
    # a permutation of the input rows: the row ids are each present once and every column matches its row
    seen = np.zeros(n, dtype=bool); seen[orid] = True
    assert seen.all()
    assert np.array_equal(ok, k[orid]) and np.array_equal(op1, p1[orid]) and np.array_equal(oxn, xn[orid])
    assert np.array_equal(ox.view(np.uint64)[~oxn], x.view(np.uint64)[orid][~oxn])
    # adjacent rows are in order: k ascending; within equal k, x descending with NULL last, NaN after every number,
    # -0.0 == +0.0
    assert (np.diff(ok) >= 0).all()
    same = ok[1:] == ok[:-1]
    an, bn = oxn[:-1], oxn[1:]
    a, b = ox[:-1], ox[1:]
    anan, bnan = np.isnan(a) & ~an, np.isnan(b) & ~bn
    bad = same & an & ~bn                                               # NULL before a value
    bad |= same & ~an & ~bn & anan & ~bnan                              # NaN before a number
    bad |= same & ~an & ~bn & ~anan & ~bnan & (a < b)                   # ascending numbers
    assert not bad.any()
    # tie groups: the ORDER BY values at every position equal those of an independent lexsort of the input
    xc = np.where(np.isnan(x), -np.inf, x) + 0.0                       # NaN below every number; -0.0 -> 0.0
    rank = np.where(xn, 2, np.where(np.isnan(x), 1, 0))                # DESC: numbers, then NaN, then NULL
    order = np.lexsort((-np.where(xn | np.isnan(x), 0.0, xc), rank, k))
    assert np.array_equal(k[order], ok)
    assert np.array_equal(rank[order], np.where(oxn, 2, np.where(np.isnan(ox), 1, 0)))
    val = lambda arr, m: np.where(m, 0.0, arr + 0.0)
    assert np.array_equal(val(x[order], xn[order] | np.isnan(x[order])), val(ox, oxn | np.isnan(ox)))
