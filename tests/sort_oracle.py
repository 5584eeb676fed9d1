"""TEST INFRASTRUCTURE (oracle): CPU restatement of SortExec's row order (ORDER BY without LIMIT), used only by tests.

SortExec.lessRow (pkg/executor/sortexec/sort.go:804) compares rows item by item with the same CompareFuncs as TopNExec, so
this is oracle/topn.py's comparator over every row (offset 0, count = all rows) — not a second comparator.  It adds the two
8-byte kinds TopN's restatement does not name:
  "time"     DATE / DATETIME / TIMESTAMP: cmpTime -> Time.Compare (types/core_time.go:256) compares the calendar fields and
             microseconds, i.e. the packed CoreTime word (types/time.go:235-251) without its 4 fsp bits, as uint64;
  "duration" cmpDuration = cmp.Compare(int64) (util/chunk/compare.go:138): "int".
Ties keep no particular order in the reference (sort.Slice / slices.SortFunc, sort_partition.go:153,
parallel_sort_worker.go:175): compare ORDER BY values per position and tie groups as multisets, never row identity.
"""
from __future__ import annotations

import os
import sys
from typing import List, Sequence, Tuple

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
import topn as _topn   # noqa: E402

TIME_FSP_MASK = ~0xF & ((1 << 64) - 1)


def _topn_kind(kind: str) -> str:
    return {"time": "uint", "duration": "int"}.get(kind, kind)


def comparable(v, kind: str):
    """the value the comparator orders by (None stays None)"""
    if v is None:
        return None
    if kind == "time":
        return (v % (1 << 64)) & TIME_FSP_MASK
    return v


def sort_rows(rows: Sequence[Tuple], kinds: Sequence[str], by_items: Sequence[Tuple[int, bool]]) -> List[Tuple]:
    """rows: tuples with None for NULL; kinds[c] in {"int", "uint", "real", "time", "duration"}; by_items: (column, desc).
    Returns the rows (unchanged values) in ORDER BY order."""
    keyed = [(tuple(comparable(v, kinds[c]) for c, v in enumerate(r)), i) for i, r in enumerate(rows)]
    ordered = _topn.topn_rows([k + (i,) for k, i in keyed], [_topn_kind(k) for k in kinds] + ["int"], by_items, 0, len(rows))
    return [rows[r[-1]] for r in ordered]
