#!/usr/bin/env python
"""GPU sort (tg_sort_*, csrc/sort.cu) on device-resident data: ORDER BY without LIMIT over 100 M rows from a fixed seed.

    (a) one full-range int64 key + 3 payload columns            every digit pass runs
    (b) the same with keys in [0, 2^20)                         digit passes 3..7 are skipped
    (c) ORDER BY date-like int, nullable DOUBLE DESC + 2 payload columns   (Q3-style: few distinct dates, ties broken by the
        second item; one NULL-flag pass)
Each case is timed with CUDA events around push + finish (the radix sort and the gather of every column) after warm-up,
next to a torch arm on the same data: torch.sort(stable=True) per item (least significant first) + index_select of the
columns, whose ORDER BY values must equal ours.  Inputs are 0.8 GB per column, far above the 126 MB L2.  One JSON line per
case with the card name and power limit read in the same run, the passes run and skipped, the modelled bytes per row and
the fraction of the HBM peak for the modelled bytes and for the lower bound of 16 B per row and column (read + write once)."""
import argparse, json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from bench import peaks
from tidb_b200 import abi
from tidb_b200.chunk import pack_not_null_bitmap, unpack_nulls
from tidb_b200.device import DeviceSort, fetch_device
from tidb_b200.plan import FieldType

ap = argparse.ArgumentParser()
ap.add_argument("--rows", type=int, default=100_000_000)
ap.add_argument("--steps", type=int, default=5)
ap.add_argument("--warmup", type=int, default=2)
ap.add_argument("--cases", default="abc")
ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
a = ap.parse_args()
assert torch.cuda.is_available(), "bench_sort needs a CUDA device"
dev = torch.device("cuda", 0)
peak, peak_src = peaks()
q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip()
card = dict(zip(("name", "power_limit", "sm_max_clock"), [s.strip() for s in q.split(",")])) if q else {"name": torch.cuda.get_device_name(0)}
stream = torch.cuda.Stream(device=dev)
fout = None
if a.out:
    os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
    fout = open(a.out, "a")
INT, DBL = FieldType(abi.TYPE_LONGLONG, 0), FieldType(abi.TYPE_DOUBLE, 0)
n = a.rows


def model_bytes(items, ncols, nullable_items, nullable_cols, digit_passes, null_passes):
    """first-order HBM bytes per row of the algorithm as implemented; a random 8-byte (or bitmap) read costs a 32 B sector"""
    b = 16                                    # key pass of the last item: read the column, write the keys
    b += 44 * (items - 1)                     # key pass of every other item: read the row id, gather the value, write the key
    b += 44 * nullable_items                  # NULL-flag key pass: row id, bitmap sector, key
    passes = digit_passes + null_passes
    b += 24 * passes - (4 if passes else 0)   # scatter: key + row id in and out (the first pass reads no row id)
    b += 4 + 40 * ncols + 32 * nullable_cols  # gather: final row ids, per column one sector in + 8 B out, bitmap sectors
    return b


def timed(fn, prep=lambda: None, done=lambda: None):
    """CUDA events around fn() on `stream`; prep() / done() run outside the timed region (handle open / close)"""
    ts, r = [], None
    for it in range(a.warmup + a.steps):
        prep()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            r = fn()
            e1.record(stream)
        stream.synchronize()
        if it >= a.warmup:
            ts.append(e0.elapsed_time(e1))
        if it < a.warmup + a.steps - 1:
            done()
    return ts, r


def view(p, dt):
    class _A:
        pass
    o = _A()
    o.__cuda_array_interface__ = {"shape": (n,), "typestr": dt, "data": (p, False), "version": 3}
    return torch.as_tensor(o, device=dev)


g = torch.Generator(device=dev)
g.manual_seed(2024)
with torch.cuda.stream(stream):
    full = torch.randint(-(1 << 63), (1 << 63) - 1, (n,), device=dev, generator=g, dtype=torch.int64)
    pays = [torch.randint(-(1 << 62), 1 << 62, (n,), device=dev, generator=g, dtype=torch.int64) for _ in range(3)]
    dates = torch.randint(8035, 10441, (n,), device=dev, generator=g, dtype=torch.int64)       # ~2406 days, like o_orderdate
    x = torch.floor(torch.rand(n, device=dev, generator=g, dtype=torch.float64) * 1e6) / 100
    xnull = torch.rand(n, device=dev, generator=g) < 0.01
stream.synchronize()
xbitmap = torch.from_numpy(pack_not_null_bitmap(xnull.cpu().numpy())).to(dev)

cases = {
    "a": ("(a) int64 full range ASC + 3 payload", [full] + pays, [None] * 4, [INT] * 4, [(0, False)]),
    "b": ("(b) int64 in [0, 2^20) ASC + 3 payload", [full & ((1 << 20) - 1)] + pays, [None] * 4, [INT] * 4, [(0, False)]),
    "c": ("(c) date-like int ASC, nullable DOUBLE DESC + 2 payload", [dates, x] + pays[:2], [None, xbitmap, None, None],
          [INT, DBL, INT, INT], [(0, False), (1, True)]),
}

for name in a.cases:
    label, cols, nulls, schema, by = cases[name]
    state = {}

    def open_sort():
        state["sort"] = DeviceSort(schema, by, expected_rows=n, stream=stream.cuda_stream)

    def ours():
        state["sort"].push(cols, nulls)
        rows, state["ptrs"], state["nptrs"] = state["sort"].finish()
        return rows

    def torch_arm():
        perm = None
        for c, desc in reversed(by):       # LSD over the items with stable sorts
            k = cols[c] if perm is None else cols[c].index_select(0, perm)
            if schema[c].tp == abi.TYPE_DOUBLE:
                nl = xnull if perm is None else xnull.index_select(0, perm)
                k = torch.where(nl, torch.full_like(k, -float("inf")), k)   # NULL below every value (the data has no -inf)
            idx = torch.sort(k, stable=True, descending=desc).indices
            perm = idx if perm is None else perm.index_select(0, idx)
        return [c.index_select(0, perm) for c in cols], perm

    ts, rows = timed(ours, open_sort, lambda: state["sort"].close())
    tts, (tcols, tperm) = timed(torch_arm)
    assert rows == n
    st = state["sort"].stats()
    # our ORDER BY values equal the torch arm's
    for c, desc in by:
        got = view(state["ptrs"][c], "<f8" if schema[c].tp == abi.TYPE_DOUBLE else "<i8")
        if state["nptrs"][c]:
            tn = xnull.index_select(0, tperm)
            on = torch.from_numpy(unpack_nulls(fetch_device(state["nptrs"][c], (n + 7) // 8), n)).to(dev)
            assert torch.equal(on, tn), f"{label}: NULL positions differ from the torch arm"
            assert torch.equal(torch.where(on, 0.0, got), torch.where(tn, 0.0, tcols[c])), f"{label}: values differ"
        else:
            assert torch.equal(got, tcols[c]), f"{label}: key sequence differs from the torch arm"
    state["sort"].close()
    ms, tms = min(ts), min(tts)
    nullable = sum(1 for v in nulls if v is not None)
    nullable_items = sum(1 for c, _ in by if nulls[c] is not None)
    bpr = model_bytes(len(by), len(cols), nullable_items, nullable, st.digit_passes, st.null_passes)
    min_bpr = 16 * len(cols)
    rec = dict(case=label, rows=n, items=len(by), cols=len(cols), card=card, ms_min=ms, ms_median=sorted(ts)[len(ts) // 2], ms_all=ts,
               sort_ms=st.sort_ms, gather_ms=st.gather_ms, digit_passes=st.digit_passes, skipped_passes=st.skipped_passes,
               null_passes=st.null_passes, launches=st.kernel_launches, model_bytes_per_row=bpr,
               model_gbs=bpr * n / ms / 1e6, model_frac=bpr * n / ms / 1e6 / peak, min_bytes_per_row=min_bpr,
               min_frac=min_bpr * n / ms / 1e6 / peak, peak_gbs=peak, peak_src=peak_src, torch_ms_min=tms,
               torch_ms_all=tts, speedup_vs_torch=tms / ms, steps=a.steps, warmup=a.warmup)
    print(json.dumps(rec))
    if fout:
        fout.write(json.dumps(rec) + "\n")
        fout.flush()
