"""Device-resident ("synthetic columnar") entry points: columns live in HBM as torch tensors, the
operators run through the same C-ABI handles (tg_join_build_push_dev / tg_join_probe_dev /
tg_agg_push_dev / tg_sort_push_dev).  torch is plumbing here — device memory, streams, torch.distributed — never compute.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import torch

from . import abi
from .plan import AggPlan, JoinPlan


def dev_chunk(cols: Sequence[torch.Tensor], nulls: Optional[Sequence[Optional[torch.Tensor]]] = None):
    """tg_chunk whose pointers are device addresses of 1-D int64/float64/float32 CUDA tensors."""
    n = len(cols)
    arr = (abi.TgColumn * max(n, 1))()
    for i, t in enumerate(cols):
        assert t.is_cuda and t.dim() == 1 and t.is_contiguous()
        arr[i].length = t.numel()
        arr[i].data = t.data_ptr()
        arr[i].elem_len = t.element_size()
        arr[i].offsets = None
        nb = nulls[i] if nulls is not None else None
        arr[i].null_bitmap = nb.data_ptr() if nb is not None else None
    s = abi.TgChunk()
    s.ncols = n
    s.cols = C.cast(arr, C.POINTER(abi.TgColumn))
    s.sel = None
    s.nsel = 0
    s._keep = (arr, list(cols), list(nulls) if nulls is not None else None)
    return s


class DeviceJoin:
    """One tg_join handle driven with device-resident chunks."""

    def __init__(self, plan: JoinPlan):
        self.lib = abi.load_lib()
        self.plan = plan
        desc, self._keep = plan.to_struct()
        self.h = C.c_void_p()
        abi.check(self.lib.tg_join_open(C.byref(desc), C.byref(self.h)))
        self.n_out = len(plan.out_schema())

    def build(self, cols: Sequence[torch.Tensor], nulls=None) -> None:
        ck = dev_chunk(cols, nulls)
        abi.check(self.lib.tg_join_build_push_dev(self.h, C.byref(ck)))
        abi.check(self.lib.tg_join_build_finish(self.h))

    def probe(self, cols: Sequence[torch.Tensor], nulls=None, sync: bool = True) -> Tuple[Optional[int], List[int], List[int]]:
        """-> (rows or None when sync=False, device pointers of the output columns, of their null bitmaps)"""
        ck = dev_chunk(cols, nulls)
        out_cols = (C.c_void_p * self.n_out)()
        out_nulls = (C.c_void_p * self.n_out)()
        rows = C.c_int64(0)
        abi.check(self.lib.tg_join_probe_dev(self.h, C.byref(ck), C.byref(rows) if sync else None, out_cols, out_nulls))
        return (rows.value if sync else None), [p or 0 for p in out_cols], [p or 0 for p in out_nulls]

    def probe_segments(self, cols: Sequence[torch.Tensor], seg_cnt: torch.Tensor, seg_cap: int, sync: bool = True):
        """cols hold len(seg_cnt) segments of seg_cap rows each, segment s valid for its first seg_cnt[s] rows (the shape a
        count-free exchange delivers, parallel.py:SegmentExchange).  Same return value as probe()."""
        ck = dev_chunk(cols, None)
        out_cols = (C.c_void_p * self.n_out)()
        out_nulls = (C.c_void_p * self.n_out)()
        rows = C.c_int64(0)
        abi.check(self.lib.tg_join_probe_dev_seg(self.h, C.byref(ck), C.c_void_p(seg_cnt.data_ptr()), C.c_int32(seg_cnt.numel()), C.c_int64(seg_cap),
                                                 C.byref(rows) if sync else None, out_cols, out_nulls))
        return (rows.value if sync else None), [p or 0 for p in out_cols], [p or 0 for p in out_nulls]

    def stats(self) -> abi.TgJoinStats:
        s = abi.TgJoinStats()
        abi.check(self.lib.tg_join_get_stats(self.h, C.byref(s)))
        return s

    def close(self) -> None:
        if self.h:
            self.lib.tg_join_close(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DeviceAgg:
    def __init__(self, plan: AggPlan):
        self.lib = abi.load_lib()
        self.plan = plan
        desc, self._keep = plan.to_struct()
        self.h = C.c_void_p()
        abi.check(self.lib.tg_agg_open(C.byref(desc), C.byref(self.h)))
        self.n_out = len(plan.funcs)

    def push(self, cols: Sequence[torch.Tensor], nulls=None) -> None:
        ck = dev_chunk(cols, nulls)
        abi.check(self.lib.tg_agg_push_dev(self.h, C.byref(ck)))

    def finish(self) -> Tuple[int, List[int], List[int]]:
        abi.check(self.lib.tg_agg_finish(self.h))
        out_cols = (C.c_void_p * self.n_out)()
        out_nulls = (C.c_void_p * self.n_out)()
        rows = C.c_int64(0)
        abi.check(self.lib.tg_agg_result_dev(self.h, C.byref(rows), out_cols, out_nulls))
        return rows.value, [p or 0 for p in out_cols], [p or 0 for p in out_nulls]

    def stats(self) -> abi.TgAggStats:
        s = abi.TgAggStats()
        abi.check(self.lib.tg_agg_get_stats(self.h, C.byref(s)))
        return s

    def close(self) -> None:
        if self.h:
            self.lib.tg_agg_close(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DeviceSort:
    """One tg_sort handle driven with device-resident chunks (tg_sort_push_dev; the columns are borrowed until finish)."""

    def __init__(self, schema, by_items, device: int = 0, expected_rows: int = 0, stream: Optional[int] = None):
        self.lib = abi.load_lib()
        desc, self._keep = abi.sort_desc(schema, by_items, device, expected_rows, stream)
        self.h = C.c_void_p()
        abi.check(self.lib.tg_sort_open(C.byref(desc), C.byref(self.h)))
        self.n_out = len(schema)
        self._pushed = []

    def push(self, cols: Sequence[torch.Tensor], nulls=None) -> None:
        ck = dev_chunk(cols, nulls)
        abi.check(self.lib.tg_sort_push_dev(self.h, C.byref(ck)))
        self._pushed.append(ck)

    def finish(self) -> Tuple[int, List[int], List[int]]:
        """-> (rows, device pointers of the sorted columns, of their null bitmaps or 0)"""
        abi.check(self.lib.tg_sort_finish(self.h))
        self._pushed = []
        out_cols = (C.c_void_p * self.n_out)()
        out_nulls = (C.c_void_p * self.n_out)()
        rows = C.c_int64(0)
        abi.check(self.lib.tg_sort_result_dev(self.h, C.byref(rows), out_cols, out_nulls))
        return rows.value, [p or 0 for p in out_cols], [p or 0 for p in out_nulls]

    def stats(self) -> abi.TgSortStats:
        s = abi.TgSortStats()
        abi.check(self.lib.tg_sort_get_stats(self.h, C.byref(s)))
        return s

    def close(self) -> None:
        if self.h:
            self.lib.tg_sort_close(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def fetch_device(ptr: int, nbytes: int, device: int = 0):
    """Copy `nbytes` from a raw device pointer into a numpy uint8 array (tests / verification)."""
    import numpy as np
    out = np.empty(nbytes, dtype=np.uint8)
    if nbytes:
        abi.check(abi.load_lib().tg_memcpy_d2h(device, out.ctypes.data_as(C.c_void_p), C.c_void_p(ptr), C.c_size_t(nbytes)))
    return out
