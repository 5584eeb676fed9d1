"""Host-side mirror of the reference's executor interface for the GPU operators.

The reference's contract is exec.Executor (pkg/executor/internal/exec/executor.go:51-77):
Open(ctx) / Next(ctx, req *chunk.Chunk) / Close(), children pulled with exec.Next(ctx, child, chk),
zero rows = EOF.  A cgo shim implementing that interface forwards to the C-ABI exactly like the
classes below do (INTEGRATION.md shows the Go source); they exist in Python only because this image
has no Go toolchain.  Names follow the reference: MockDataSource (internal/testutil/testutil.go:63),
HashJoinV2Exec (join/hash_join_v2.go:608), HashAggExec (aggregate/agg_hash_executor.go:93), SortExec
(sortexec/sort.go:43).

There is no CPU fallback: every operator fails if libtidbgpu.so is missing or no CUDA device exists.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence

import numpy as np

from . import abi
from .chunk import Chunk, Column, MutChunk
from .plan import AggPlan, FieldType, JoinPlan

MAX_CHUNK_SIZE = 1024  # tidb_max_chunk_size default (vardef/tidb_vars.go:1464)


def np_dtype_of(t: FieldType):
    if t.tp == abi.TYPE_DOUBLE:
        return np.float64
    if t.tp == abi.TYPE_FLOAT:
        return np.float32
    return np.int64   # unsigned columns keep their bit pattern (chunk.Column stores raw 8 bytes)


class Executor:
    """exec.Executor: open → next* → close.  next() returns a Chunk; 0 rows means EOF."""

    def __init__(self, schema: Sequence[FieldType], children: Sequence["Executor"] = ()):
        self.schema = list(schema)
        self.children = list(children)

    def open(self) -> None:            # BaseExecutorV2.Open executor.go:301: open the children first
        for c in self.children:
            c.open()

    def next(self, required_rows: int = MAX_CHUNK_SIZE) -> Chunk:
        raise NotImplementedError

    def close(self) -> None:
        for c in self.children:
            c.close()

    def empty_chunk(self) -> Chunk:
        return Chunk([Column(np.zeros(0, dtype=np_dtype_of(t))) for t in self.schema])


class MockDataSource(Executor):
    """Replays pre-generated chunks: the fake backend of every operator test / benchmark
    (pkg/executor/internal/testutil/testutil.go:63 MockDataSource, :269 BuildMockDataSource)."""

    def __init__(self, schema: Sequence[FieldType], chunks: Sequence[Chunk]):
        super().__init__(schema)
        self.chunks = list(chunks)
        self._pos = 0

    def open(self) -> None:
        self._pos = 0

    def next(self, required_rows: int = MAX_CHUNK_SIZE) -> Chunk:
        if self._pos >= len(self.chunks):
            return self.empty_chunk()
        c = self.chunks[self._pos]
        self._pos += 1
        return c


def _out_chunk(schema: Sequence[FieldType], capacity: int) -> MutChunk:
    dts = [np_dtype_of(t) for t in schema]
    return MutChunk([np.dtype(d).itemsize for d in dts], capacity, dts)


class HashJoinExec(Executor):
    """GPU replacement of join.HashJoinV2Exec behind the same Open/Next/Close surface.

    Build side is a pipeline breaker (fetchAndBuildHashTable hash_join_v2.go:1266): the first Next drains
    the build child into tg_join_build_push and calls tg_join_build_finish.  The probe side streams:
    Next pulls probe chunks (fetchProbeSideChunks hash_join_base.go:161) into tg_join_probe_push until
    tg_join_next has rows to hand out (hash_join_v2.go:1176-1186)."""

    def __init__(self, plan: JoinPlan, left: Executor, right: Executor):
        super().__init__(plan.out_schema(), [left, right])
        self.plan = plan
        self.build_child, self.probe_child = (right, left) if plan.build_is_right else (left, right)
        self._h = C.c_void_p()
        self._lib = None
        self._prepared = False
        self._probe_done = False
        self._out: Optional[MutChunk] = None

    def open(self) -> None:
        super().open()
        self._lib = abi.load_lib()
        desc, self._keep = self.plan.to_struct()
        self._h = C.c_void_p()
        abi.check(self._lib.tg_join_open(C.byref(desc), C.byref(self._h)))
        self._prepared = False
        self._probe_done = False

    def _build(self) -> None:
        while True:
            chk = self.build_child.next(MAX_CHUNK_SIZE)
            if chk.num_rows() == 0:
                break
            cs = chk.to_struct()
            abi.check(self._lib.tg_join_build_push(self._h, C.byref(cs)))
        abi.check(self._lib.tg_join_build_finish(self._h))
        self._prepared = True

    def next(self, required_rows: int = MAX_CHUNK_SIZE) -> Chunk:
        if not self._h:
            raise RuntimeError("next before open")
        if not self._prepared:
            self._build()
        if self._out is None or self._out.capacity < required_rows:
            self._out = _out_chunk(self.schema, max(required_rows, 8))
        n = C.c_int64(0)
        while True:
            abi.check(self._lib.tg_join_next(self._h, C.byref(self._out.struct), C.c_int64(required_rows), C.byref(n)))
            if n.value > 0 or self._probe_done:
                break
            chk = self.probe_child.next(MAX_CHUNK_SIZE)
            if chk.num_rows() == 0:
                abi.check(self._lib.tg_join_probe_finish(self._h))
                self._probe_done = True
            else:
                cs = chk.to_struct()
                abi.check(self._lib.tg_join_probe_push(self._h, C.byref(cs)))
        cols = self._out.columns(n.value)
        return Chunk([Column(v, nl if nl.any() else None) for v, nl in cols])

    def stats(self) -> abi.TgJoinStats:
        s = abi.TgJoinStats()
        abi.check(self._lib.tg_join_get_stats(self._h, C.byref(s)))
        return s

    def close(self) -> None:
        if self._h:
            self._lib.tg_join_close(self._h)
            self._h = C.c_void_p()
        super().close()


class HashAggExec(Executor):
    """GPU replacement of aggregate.HashAggExec.  Output schema: one column per aggregate function in
    descriptor order (group columns are emitted through firstrow() funcs, as the reference's plans do)."""

    def __init__(self, plan: AggPlan, child: Executor, out_schema: Optional[Sequence[FieldType]] = None):
        super().__init__(out_schema or [self._ret_type(plan, f) for f in plan.funcs], [child])
        self.plan = plan
        self._h = C.c_void_p()
        self._lib = None
        self._prepared = False
        self._out: Optional[MutChunk] = None

    @staticmethod
    def _ret_type(plan: AggPlan, f) -> FieldType:
        if f.name == abi.AGG_COUNT:
            return FieldType(abi.TYPE_LONGLONG, abi.FLAG_NOT_NULL)
        if f.name in (abi.AGG_SUM, abi.AGG_AVG):
            return FieldType(abi.TYPE_DOUBLE, 0)
        return FieldType(plan.col_types[f.arg_col].tp, plan.col_types[f.arg_col].flag & ~abi.FLAG_NOT_NULL)

    def open(self) -> None:
        super().open()
        self._lib = abi.load_lib()
        desc, self._keep = self.plan.to_struct()
        self._h = C.c_void_p()
        abi.check(self._lib.tg_agg_open(C.byref(desc), C.byref(self._h)))
        self._prepared = False

    def next(self, required_rows: int = MAX_CHUNK_SIZE) -> Chunk:
        if not self._prepared:
            child = self.children[0]
            while True:   # fetchChildData agg_hash_executor.go:449
                chk = child.next(MAX_CHUNK_SIZE)
                if chk.num_rows() == 0:
                    break
                cs = chk.to_struct()
                abi.check(self._lib.tg_agg_push(self._h, C.byref(cs)))
            abi.check(self._lib.tg_agg_finish(self._h))
            self._prepared = True
        if self._out is None or self._out.capacity < required_rows:
            self._out = _out_chunk(self.schema, max(required_rows, 8))
        n = C.c_int64(0)
        abi.check(self._lib.tg_agg_next(self._h, C.byref(self._out.struct), C.c_int64(required_rows), C.byref(n)))
        cols = self._out.columns(n.value)
        return Chunk([Column(v, nl if nl.any() else None) for v, nl in cols])

    def stats(self) -> abi.TgAggStats:
        s = abi.TgAggStats()
        abi.check(self._lib.tg_agg_get_stats(self._h, C.byref(s)))
        return s

    def close(self) -> None:
        if self._h:
            self._lib.tg_agg_close(self._h)
            self._h = C.c_void_p()
        super().close()


# ---------------------------------------------------------------------------------------------------------------
# SelectionExec / ProjectionExec: the two operators that call the VecEval layer around joins and aggregates
# ---------------------------------------------------------------------------------------------------------------
def _concat_chunks(chunks: Sequence[Chunk]) -> Chunk:
    """child chunks -> one dense chunk (sel vectors applied), the batch a device call works on"""
    cols = []
    for c in range(chunks[0].num_cols()):
        vals, nls, any_null = [], [], False
        for ck in chunks:
            col = ck.columns[c]
            idx = ck.sel if ck.sel is not None else slice(None)
            vals.append(col.data[idx])
            nl = col.nulls()[idx]
            any_null |= bool(nl.any())
            nls.append(nl)
        cols.append(Column(np.concatenate(vals), np.concatenate(nls) if any_null else None))
    return Chunk(cols)


class SelectionExec(Executor):
    """GPU replacement of executor.SelectionExec (pkg/executor/select.go:746-785): pulls child chunks, evaluates the
    CNF filter list with expression.VectorizedFilter semantics (chunk_executor.go:413: a row is selected iff every item is
    non-NULL true) on the device (tg_vec_filter) and hands the selected rows on, at most `required_rows` per Next.
    Child chunks are batched (`batch_rows`) so that one launch filters many 1024-row chunks."""

    def __init__(self, child: Executor, filters: Sequence, device: int = 0, batch_rows: int = 64 * MAX_CHUNK_SIZE):
        super().__init__(child.schema, [child])
        self.filters, self.device, self.batch_rows = list(filters), device, batch_rows
        self._lib = None
        self._pending: List[Chunk] = []     # selected rows not handed out yet
        self._eof = False
        self.launches = 0

    def open(self) -> None:
        super().open()
        self._lib = abi.load_lib()
        if self._lib.tg_device_count() <= 0:
            raise RuntimeError("SelectionExec: no CUDA device (the GPU operators have no CPU fallback)")
        self._pending, self._eof = [], False

    def _fill(self) -> None:
        from .plan import filter_array
        batch, rows = [], 0
        while rows < self.batch_rows:
            chk = self.children[0].next(MAX_CHUNK_SIZE)
            if chk.num_rows() == 0:
                self._eof = True
                break
            batch.append(chk); rows += chk.num_rows()
        if not batch:
            return
        dense = _concat_chunks(batch)
        n = dense.num_rows()
        selected = np.zeros(n, dtype=np.uint8)
        nsel = C.c_int64(0)
        cs = dense.to_struct()
        arr = filter_array(self.filters)
        abi.check(self._lib.tg_vec_filter(self.device, 0, C.byref(cs), arr, len(self.filters), selected.ctypes.data_as(C.c_void_p), C.byref(nsel), None))
        self.launches += 1
        keep = selected.astype(bool)
        assert int(keep.sum()) == nsel.value
        if nsel.value:
            self._pending.append(Chunk([Column(c.data[keep], c.nulls()[keep] if c.nulls().any() else None) for c in dense.columns]))

    def next(self, required_rows: int = MAX_CHUNK_SIZE) -> Chunk:
        while not self._pending and not self._eof:
            self._fill()
        if not self._pending:
            return self.empty_chunk()
        head = self._pending[0]
        if head.num_rows() <= required_rows:
            self._pending.pop(0)
            return head
        out = Chunk([Column(c.data[:required_rows], c.nulls()[:required_rows] if c.nulls().any() else None) for c in head.columns])
        self._pending[0] = Chunk([Column(c.data[required_rows:], c.nulls()[required_rows:] if c.nulls().any() else None) for c in head.columns])
        return out


class ProjectionExec(Executor):
    """GPU replacement of executor.ProjectionExec (pkg/executor/projection.go:450-483 -> EvaluatorSuite.Run,
    expression/evaluator.go:128): plain column references are passed through (the reference SWAPS them, ColumnSwapHelper),
    scalar functions are evaluated column-at-a-time by the VecEval kernels (tg_vec_arith_* / tg_vec_compare_*), constants
    are scalars (the reference materialises them as columns, vectorized.go:23).  Errors keep the reference's meaning:
    overflow on a non-NULL row fails the Next call (types.ErrOverflow <-> TG_ERR_OVERFLOW)."""

    def __init__(self, child: Executor, exprs: Sequence, device: int = 0, batch_rows: int = 64 * MAX_CHUNK_SIZE):
        from .plan import Expr
        self.exprs = list(exprs)
        super().__init__([e.ret_type(child.schema) for e in self.exprs], [child])
        self.device, self.batch_rows = device, batch_rows
        self._lib = None
        self._pending: List[Chunk] = []
        self._eof = False
        self.launches = 0

    def open(self) -> None:
        super().open()
        self._lib = abi.load_lib()
        if self._lib.tg_device_count() <= 0:
            raise RuntimeError("ProjectionExec: no CUDA device (the GPU operators have no CPU fallback)")
        self._pending, self._eof = [], False

    def _eval(self, e, chk: Chunk) -> Column:
        from .plan import ColRef, Const, ScalarFunc
        if isinstance(e, ColRef):
            return chk.columns[e.idx]
        if isinstance(e, Const):
            raise abi.TgError(abi.TG_ERR_UNSUPPORTED, "a bare constant projection is not offloaded")
        assert isinstance(e, ScalarFunc)
        a, b = e.args
        n = chk.num_rows()
        if isinstance(a, Const):
            raise abi.TgError(abi.TG_ERR_UNSUPPORTED, "constant on the left of a scalar function is not offloaded (the planner folds or swaps it)")
        ca = self._eval(a, chk)
        cb = None if isinstance(b, Const) else self._eval(b, chk)
        real = e.is_real
        res = np.zeros(n, dtype=np.float64 if (real and e.kind == "arith") else np.int64)
        nulls = np.zeros((n + 7) // 8, dtype=np.uint8)
        sa = ca.to_struct(); sb = cb.to_struct() if cb is not None else None
        pb = C.byref(sb) if sb is not None else None
        rp, np_ = res.ctypes.data_as(C.c_void_p), nulls.ctypes.data_as(C.c_void_p)
        k = b.value if isinstance(b, Const) else 0
        if e.kind == "arith" and real:
            rc = self._lib.tg_vec_arith_real(self.device, 0, e.op, C.byref(sa), pb, C.c_double(float(k)), rp, np_, None)
        elif e.kind == "arith":
            rc = self._lib.tg_vec_arith_int(self.device, 0, e.op, int(e.a_unsigned), int(e.b_unsigned), C.byref(sa), pb, C.c_int64(int(k)), rp, np_, None)
        elif real:
            rc = self._lib.tg_vec_compare_real(self.device, 0, e.op, C.byref(sa), pb, C.c_double(float(k)), rp, np_, None)
        else:
            rc = self._lib.tg_vec_compare_int(self.device, 0, e.op, int(e.a_unsigned), int(e.b_unsigned), C.byref(sa), pb, C.c_int64(int(k)), rp, np_, None)
        abi.check(rc)
        self.launches += 1
        isnull = np.unpackbits(nulls, bitorder="little")[:n] == 0
        return Column(res, isnull if isnull.any() else None)

    def next(self, required_rows: int = MAX_CHUNK_SIZE) -> Chunk:
        while not self._pending and not self._eof:
            batch, rows = [], 0
            while rows < self.batch_rows:
                chk = self.children[0].next(MAX_CHUNK_SIZE)
                if chk.num_rows() == 0:
                    self._eof = True
                    break
                batch.append(chk); rows += chk.num_rows()
            if batch:
                dense = _concat_chunks(batch)
                self._pending.append(Chunk([self._eval(e, dense) for e in self.exprs]))
        if not self._pending:
            return self.empty_chunk()
        head = self._pending[0]
        if head.num_rows() <= required_rows:
            self._pending.pop(0)
            return head
        out = Chunk([Column(c.data[:required_rows], c.nulls()[:required_rows] if c.nulls().any() else None) for c in head.columns])
        self._pending[0] = Chunk([Column(c.data[required_rows:], c.nulls()[required_rows:] if c.nulls().any() else None) for c in head.columns])
        return out


class TopNExec(Executor):
    """GPU replacement of sortexec.TopNExec (pkg/executor/sortexec/topn.go:74; Next :230 executeTopN): a pipeline breaker that
    drains the child, selects rows [offset, offset + count) in ORDER BY order on the device (tg_topn: rank pass, radix
    select, gather) and hands them out chunk by chunk.  by_items = [(column, desc)]."""

    def __init__(self, child: Executor, by_items: Sequence, offset: int, count: int, device: int = 0):
        super().__init__(child.schema, [child])
        self.by_items, self.offset, self.count, self.device = list(by_items), int(offset), int(count), device
        self._result: Optional[Chunk] = None
        self._pos = 0

    def open(self) -> None:
        super().open()
        self._lib = abi.load_lib()
        self._result, self._pos = None, 0

    def _execute(self) -> None:
        chunks = []
        while True:
            chk = self.children[0].next(MAX_CHUNK_SIZE)
            if chk.num_rows() == 0:
                break
            chunks.append(chk)
        if not chunks or self.count == 0:
            self._result = self.empty_chunk()
            return
        dense = _concat_chunks(chunks)
        out = _out_chunk(self.schema, max(self.count, 8))
        items = (abi.TgSortItem * len(self.by_items))(*[abi.TgSortItem(c, int(bool(d))) for c, d in self.by_items])
        tps = (C.c_int32 * len(self.schema))(*[t.tp for t in self.schema])
        fls = (C.c_uint32 * len(self.schema))(*[t.flag for t in self.schema])
        n = C.c_int64(0)
        cs = dense.to_struct()
        abi.check(self._lib.tg_topn(self.device, 0, C.byref(cs), tps, fls, items, len(self.by_items), C.c_int64(self.offset), C.c_int64(self.count),
                                    C.byref(out.struct), C.byref(n), None))
        self._result = Chunk([Column(v.copy(), nl.copy() if nl.any() else None) for v, nl in out.columns(n.value)])

    def next(self, required_rows: int = MAX_CHUNK_SIZE) -> Chunk:
        if self._result is None:
            self._execute()
        lo, hi = self._pos, min(self._pos + required_rows, self._result.num_rows())
        self._pos = hi
        if hi <= lo:
            return self.empty_chunk()
        return Chunk([Column(c.data[lo:hi], c.nulls()[lo:hi] if c.nulls().any() else None) for c in self._result.columns])


class SortExec(Executor):
    """GPU replacement of sortexec.SortExec (pkg/executor/sortexec/sort.go:43) for ORDER BY without LIMIT: a pipeline
    breaker.  Open opens a tg_sort handle (sort.go:155); the first Next pushes every child chunk, sel vectors included
    (fetchChunks sort.go:526), and sorts on the device (tg_sort_finish); each Next then returns at most `required_rows`
    rows of the child's schema in ORDER BY order (sort.go:265).  by_items = [(column, desc)], plain column references."""

    def __init__(self, child: Executor, by_items: Sequence, device: int = 0):
        super().__init__(child.schema, [child])
        self.by_items, self.device = [(int(c), bool(d)) for c, d in by_items], device
        self._h = C.c_void_p()
        self._lib = None
        self._prepared = False
        self._out: Optional[MutChunk] = None

    def open(self) -> None:
        super().open()
        self._lib = abi.load_lib()
        desc, keep = abi.sort_desc(self.schema, self.by_items, self.device)
        self._h = C.c_void_p()
        abi.check(self._lib.tg_sort_open(C.byref(desc), C.byref(self._h)))
        self._prepared = False

    def next(self, required_rows: int = MAX_CHUNK_SIZE) -> Chunk:
        if not self._h:
            raise RuntimeError("next before open")
        if not self._prepared:
            while True:
                chk = self.children[0].next(MAX_CHUNK_SIZE)
                if chk.num_rows() == 0:
                    break
                cs = chk.to_struct()
                abi.check(self._lib.tg_sort_push(self._h, C.byref(cs)))
            abi.check(self._lib.tg_sort_finish(self._h))
            self._prepared = True
        if self._out is None or self._out.capacity < required_rows:
            self._out = _out_chunk(self.schema, max(required_rows, 8))
        n = C.c_int64(0)
        abi.check(self._lib.tg_sort_next(self._h, C.byref(self._out.struct), C.c_int64(required_rows), C.byref(n)))
        cols = self._out.columns(n.value)
        return Chunk([Column(v, nl if nl.any() else None) for v, nl in cols])

    def stats(self) -> abi.TgSortStats:
        s = abi.TgSortStats()
        abi.check(self._lib.tg_sort_get_stats(self._h, C.byref(s)))
        return s

    def close(self) -> None:
        if self._h:
            self._lib.tg_sort_close(self._h)
            self._h = C.c_void_p()
        super().close()


def drain(e: Executor, required_rows: int = MAX_CHUNK_SIZE) -> List[Chunk]:
    """open → next until EOF → close, like the reference's test helpers."""
    e.open()
    out = []
    try:
        while True:
            c = e.next(required_rows)
            if c.num_rows() == 0:
                break
            out.append(c)
    finally:
        e.close()
    return out
