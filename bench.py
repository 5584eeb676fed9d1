#!/usr/bin/env python
"""bench.py — hash-join probe rows/sec (BASELINE.json metric) on 1..N B200s.

  python bench.py --gpus 1 --steps K --warmup W                       (N = 1)
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...   (N > 1)
  python bench.py --impl reference ...      the reference algorithm's CPU restatement on the host cores

N = 1 workload = BASELINE.json configs[1]: hash join 100M ⋈ 10M int64 keys, 8-byte payload, 100 % match,
output (probe.k, probe.v, build.k, build.v).  A step = one pass of the probe over the whole 100M-row
probe side against the already built table:
  value : columns resident in HBM, kernel-only (tg_join_probe_dev), CUDA events on the launch stream
  e2e   : the same probe through the host-facing C-ABI (tg_join_probe_push / tg_join_next) with pinned HOST
          buffers, host→device and device→host copies inside the timed region
N > 1 (weak scaling, per-GPU work fixed) = BASELINE.json configs[4] divided by 8: every rank owns 12.5M build +
125M probe rows (N = 8: the 1B x 100M join) whose keys are uniform over the GLOBAL key set, so a key-hash
repartition is mandatory: build side repartitioned once (untimed, like the build itself), every timed step =
regroup the probe columns by destination GPU + move them over NVLink + shard-local probe (L2 partition pass +
segment probe).  tidb_b200/parallel.py:MailboxExchange: a kernel regroups 1024-row tiles by destination with bulk stores (into a
local staging copy of the region layout, or straight into a peer), copy engines move the staged regions over NVLink
under the probe of the previous step, and the only synchronisation is device-side mailboxes (peer stores + spinning
loads): no NCCL collective and no host wait inside a step.  All SM kernels of a rank run on ONE stream in the order
regroup(k+1), probe(k) (two receive sets), the way a stream of probe batches is processed.  The timed region holds exactly K exchanges and K probes (the pipeline is empty at
both events: barrier + synchronize before, the last probe's completion after).  --exchange auto times the
candidate transports for a few untimed steps and keeps the fastest (reported in config).

Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np

ODD = 0x9E3779B97F4A7C15 - (1 << 64)   # odd 64-bit multiplier (as int64): a bijection, keys are unique but not dense
BYTES_PER_PROBE_ROW = 64                # SURVEY §8(d): 16 read + 16 gathered + 32 written at 100 % match


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    NVML_REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def start(self):
        # NVML polled every 2 ms from a thread (the default timed region is ~40 ms: an nvidia-smi child process would deliver its
        # first sample after the region has ended); nvidia-smi -lms stays as the fall-back when NVML cannot be used
        self.samples, self._halt, self.nv = [], threading.Event(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            try:
                import torch
                u = str(torch.cuda.get_device_properties(self.idx).uuid)
                u = u if u.startswith("GPU-") else "GPU-" + u
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(u)
                except Exception:
                    h = pynvml.nvmlDeviceGetHandleByUUID(u.encode())
            except Exception:
                h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))     # fails here, not in the thread, if unsupported
            self.nv = (pynvml, h)
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll(self):
        pynvml, h = self.nv
        while not self._halt.is_set():
            try:
                sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                try:
                    r = int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                except Exception:
                    r = int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                self.samples.append((sm, r))
            except Exception:
                pass
            time.sleep(0.002)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if getattr(self, "nv", None):
            self._halt.set()
            self.t.join(timeout=1)
            sm = [a for a, _ in self.samples]
            bits = 0
            for _, r in self.samples:
                bits |= r
            return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": self.mx, "samples": len(sm),
                    "reasons": sorted(nm for bit, nm in self.NVML_REASONS if bits & bit), "source": "nvml, 2 ms period, timed region only"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def make_plan(device: int, stream: int):
    from tidb_b200 import abi
    from tidb_b200.plan import FieldType, JoinPlan
    INT = FieldType(abi.TYPE_LONGLONG, abi.FLAG_NOT_NULL)
    # probe = left child, build = right child (RightAsBuildSide), all columns used (benchmark_test.go:722-729)
    return JoinPlan(abi.JOIN_INNER, [INT, INT], [INT, INT], [0], [0], build_is_right=True, device=device, stream=stream)


def gen_local(torch, dev, rank, world, n_build, n_probe):
    """Synthetic fixed-width columns, generated on the device (seeds 42/43 per BASELINE.md)."""
    g = torch.Generator(device=dev); g.manual_seed(42 + 1000 * rank)
    ids = torch.randperm(n_build, device=dev, generator=g, dtype=torch.int64) + rank * n_build
    bk = ids * ODD                                   # wraps mod 2^64: unique, scattered keys
    bv = ids * 7
    g.manual_seed(43 + 1000 * rank)
    pid = torch.randint(0, n_build * world, (n_probe,), device=dev, generator=g, dtype=torch.int64)
    pk = pid * ODD
    pv = torch.arange(n_probe, device=dev, dtype=torch.int64) + rank * n_probe
    return bk, bv, pk, pv


DUMP_ROWS = 1 << 19    # rows kept from a larger output: 8 float64 arrays of 4 MiB at most (4 int64 join columns)


def dump_outputs(out_dir, cols, order_by):
    """--dump-outputs: write the result columns of one step (name -> 1-D int64/float64 CUDA tensor, all of one length) as
    out_dir/<name>.npy, so that two builds can be compared output for output.  The kernels emit rows in no fixed order, so
    rows are first sorted by cols[order_by], which is unique per output row; an output longer than DUMP_ROWS is cut to a
    fixed, seeded sample of DUMP_ROWS rows.  float64 columns are stored as they are; an int64 column, which float64 cannot
    hold exactly, as two exact float64 arrays <name>_hi (bits 63..32, signed) and <name>_lo (bits 31..0)."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    order = torch.sort(cols[order_by], stable=True).indices
    if order.numel() > DUMP_ROWS:
        pick = np.sort(np.random.default_rng(0).choice(order.numel(), DUMP_ROWS, replace=False))
        order = order[torch.from_numpy(pick).to(order.device)]
    for name, t in cols.items():
        v = t[order]
        parts = {name: v} if v.dtype == torch.float64 else {name + "_hi": (v >> 32).double(), name + "_lo": (v & 0xFFFFFFFF).double()}
        for part, a in parts.items():
            np.save(os.path.join(out_dir, part + ".npy"), a.cpu().numpy())


# ---------------------------------------------------------------------------------------------------------
# CPU legs (oracle): the only place bench.py touches oracle/
# ---------------------------------------------------------------------------------------------------------
def host_threads():
    """threads the CPU baseline may really use: CPUs in the affinity mask, capped by a cgroup CPU quota when one is set
    (os.cpu_count() reports the machine, not the container)"""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]) + 0.999)))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, (q + per - 1) // per))
            break
        except Exception:
            continue
    return max(1, n)


def cpu_probe_rate(bk, bv, pk, pv, sample_rows, threads, steps, warmup):
    """Probe rows/s of the reference algorithm's restatement (oracle/join.cpp) on `threads` host threads:
    full build, probe of the first `sample_rows` probe rows fed as 1024-row chunks."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    from tidb_b200.chunk import Chunk, Column, chunk_array
    plan = make_plan(0, 0)
    j = O.OracleJoin(plan, threads)
    build_chunks = Chunk([Column(bk), Column(bv)]).split(1024)
    j.build(build_chunks)
    pchunks = Chunk([Column(pk[:sample_rows]), Column(pv[:sample_rows])]).split(1024)
    parr = chunk_array(pchunks)
    times = []
    rows = 0
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        rows = j.probe(parr, len(pchunks))
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    bsec = j.stat("build_seconds")
    j.close()
    return sample_rows / (sum(times) / len(times)), (sum(times) / len(times)) * 1e3, rows, bsec


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # the same workload as the GPU arm at this N: configs[1] on one GPU, configs[4] / 8 per GPU otherwise — the CPU arm is ONE
    # host process, so it builds the GLOBAL table (12.5 M x N rows) and probes a bounded sample of the global probe side
    world = max(1, int(args.gpus))
    per_gpu = args.build_rows is None and args.probe_rows is None and world > 1
    if args.build_rows is None:
        args.build_rows = 10_000_000 if world == 1 else 12_500_000 * world
    if args.probe_rows is None:
        args.probe_rows = 100_000_000 if world == 1 else 125_000_000 * world
    note_mem = None
    try:
        import psutil
        need = args.build_rows * 160          # numpy inputs + row store + hash values + tables of the restatement, generously
        if psutil.virtual_memory().available < need:
            note_mem = f"host memory too small for the {args.build_rows}-row build of this configuration: built 10000000 rows instead"
            args.build_rows = 10_000_000
    except Exception:
        pass
    nb, sample = args.build_rows, min(args.probe_rows, args.ref_sample_rows)
    rng = np.random.default_rng(42)
    ids = rng.permutation(nb).astype(np.int64)
    bk = ids * np.int64(ODD); bv = ids * 7
    rng = np.random.default_rng(43)
    pk = rng.integers(0, nb, sample).astype(np.int64) * np.int64(ODD)
    pv = np.arange(sample, dtype=np.int64)
    threads = host_threads()
    rate, ms, rows, bsec = cpu_probe_rate(bk, bv, pk, pv, sample, threads, args.steps, args.warmup)
    assert rows == sample
    line = {
        "impl": "reference", "metric": "hash-join probe rows/sec", "value": rate, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": (f"hash join {args.probe_rows}x{nb} int64 keys, 8-byte payload, 100% match (BASELINE configs[1])" if world == 1 else
                                f"hash join {args.probe_rows}x{nb} int64 keys (the GPU arm's partitioned join over {world} GPUs, "
                                f"{args.probe_rows // world}x{nb // world} per GPU), 8-byte payload, 100% match, in ONE host process "
                                f"(BASELINE configs[4] / 8 per GPU" + ("" if world != 8 else " = the 1Bx100M join") + ")"),
                   "note": "CPU restatement of TiDB's HashJoinV2 algorithm (oracle/join.cpp), NOT the Go binary: no Go toolchain in this image"
                           + ("; " + note_mem if note_mem else "")},
        "cpu_baseline": {"value": rate, "unit": "rows/s", "cores": threads, "kind": "port",
                         "sample": f"full {nb}-row build ({bsec:.2f}s, untimed) + probe of {sample} rows as 1024-row chunks per step"},
        "e2e": {"value": rate, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
def run_gpu(args):
    # the exchange keeps up to 16 copy streams + compute + NCCL busy: more hardware work queues than the default 8, or streams
    # that share a queue serialise behind each other (must be set before the CUDA context exists)
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
    import torch
    import torch.distributed as dist
    from tidb_b200 import abi
    from tidb_b200.device import DeviceJoin, dev_chunk, fetch_device

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = abi.load_lib()
    assert lib.tg_device_count() > 0
    stream = torch.cuda.Stream(device=dev)
    if args.build_rows is None:
        args.build_rows = 10_000_000 if world == 1 else 12_500_000
    if args.probe_rows is None:
        args.probe_rows = 100_000_000 if world == 1 else 125_000_000
    nb, npb = args.build_rows, args.probe_rows
    hbm_peak, peak_src = peaks()

    with torch.cuda.stream(stream):
        bk, bv, pk, pv = gen_local(torch, dev, rank, world, nb, npb)
    stream.synchronize()
    plan = make_plan(local, stream.cuda_stream)
    launches_extra = 0

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- build side (untimed): repartition by key hash when N > 1, then build the local table ---------
    xch_b = xch_p = xseg = None
    xstream = None
    xchunks = max(1, args.xchunks) if world > 1 else 1
    if world > 1:
        from tidb_b200.parallel import KeyExchange
        xstream = torch.cuda.Stream(device=dev)
        # receive capacity: expected rows + 2 % (uniform hash; a skewed key set would need a count-then-allocate round)
        with torch.cuda.stream(stream):
            xch_b = KeyExchange(rank, world, local, stream, 2, int(nb * 1.02) + 4096, "nccl" if args.exchange == "nccl" else "p2p")
        with torch.cuda.stream(xstream):
            # the probe side is exchanged in `xchunks` pieces through two alternating sets of receive buffers, so that the
            # NVLink scatter of piece c+1 overlaps the probe kernel of piece c
            xch_p = ([KeyExchange(rank, world, local, xstream, 2, int(npb / xchunks * 1.03) + 8192, args.exchange) for _ in range(2 if xchunks > 1 else 1)]
                     if args.exchange in ("p2p", "nccl") else [])
        if args.exchange in ("mail", "mail-dma", "mail-hybrid", "mail-smcopy", "auto"):
            pass   # created below (after the build side's exchange), possibly several candidates
        elif args.exchange == "cf":
            from tidb_b200.parallel import SegmentExchange
            xs = xstream if args.overlap else stream
            with torch.cuda.stream(xs):
                xseg = SegmentExchange(rank, world, local, xs, 2, npb, dma=bool(args.dma))
        # leave room on every SM for the scatter CTAs next to the persistent probe CTAs
        if xchunks > 1:
            os.environ.setdefault("TG_PROBE_CTAS_PER_SM", "2")

    join = DeviceJoin(plan)
    with torch.cuda.stream(stream):
        if world > 1:
            lbk, lbv = xch_b.exchange(bk, [bk, bv])
        else:
            lbk, lbv = bk, bv
        join.build([lbk, lbv])
    bstats = join.stats()

    # ---- one step ------------------------------------------------------------------------------------------
    bounds = [(npb * c // xchunks, npb * (c + 1) // xchunks) for c in range(xchunks)]
    done_ev = [None, None]

    def dview(p, n):
        class _A:   # __cuda_array_interface__ wrapper for a library-owned device buffer (verification only, no copy)
            pass
        a = _A()
        a.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i8", "data": (p, False), "version": 3}
        return torch.as_tensor(a, device=dev)

    def check_piece(cols, rows):
        """size-independent properties of one probe result: equal keys, payload belongs to the key; returns checksums of
        the probe row ids (every probe row must appear exactly once overall)"""
        o_pk, o_pv, o_bk, o_bv = [dview(p, rows) for p in cols]
        assert bool((o_pk == o_bk).all()), "joined rows must carry equal keys"
        assert bool((o_bv * ODD == o_bk * 7).all()), "build payload does not belong to the matched key"   # bv = 7*id, bk = id*ODD
        return torch.stack([o_pv.sum(), (o_pv * o_pv).sum()])

    TRACE = [] if os.environ.get("BENCH_TRACE") else None
    last_cols = []    # N = 1: device pointers of the latest step's output columns (valid until the next probe call)

    # ---- N > 1, mailbox exchange: candidates and (for --exchange auto) an untimed calibration -----------------------
    xmail = None
    mail_choice = None
    mail_timings = {}
    MAIL_CANDIDATES = {"mail": dict(dma=False, ctas_per_sm=args.scatter_ctas), "mail-dma": dict(dma=True, ctas_per_sm=args.scatter_ctas, copy_streams=args.copy_streams, direct_peers=args.direct_peers),
                       "mail-smcopy": dict(dma=True, ctas_per_sm=args.scatter_ctas, sm_copy=True, sm_copy_ctas=args.sm_copy_ctas),
                       "mail-hybrid": dict(dma=True, ctas_per_sm=args.scatter_ctas, copy_streams=args.copy_streams, direct_peers=1)}   # measured at 8 GPUs: 1 direct peer 4.07 ms, 2: 4.21, 3: 4.42, 0 (copy engines only): 4.69

    def mail_step(xm, sync: bool):
        """ALL SM kernels of a rank on ONE stream, in the order regroup(k+1), probe(k): the shared-memory-heavy scatter never
        shares an SM with the L1-hungry probe kernel.  With dma the copy engines move step k+1 over NVLink under probe(k);
        without it the scatter stores into the peers itself (NVLink-bound at N = 8, no overlap)."""
        def mark(name):
            if TRACE is not None:
                e = torch.cuda.Event(enable_timing=True); e.record(stream); TRACE.append((name, e))
        with torch.cuda.stream(stream):
            if not getattr(xm, "_primed", False):
                xm.send(pk, [pk, pv], stream)      # pipeline prologue: step 0
                xm._primed = True
            mark("step begin")
            xm.send(pk, [pk, pv], stream)          # step k+1
            mark("regroup(k+1) done")
            cols_in, seg_cnt, cap, s_, ep = xm.recv(stream)
            mark("counts(k) arrived")
            rows, cols, _ = join.probe_segments(cols_in, seg_cnt, cap, sync=sync)
            mark("probe(k) done")
            out = (rows, check_piece(cols, rows)) if sync else (None, None)
            xm.release(stream, s_, ep)     # the probe has consumed receive set s_: the senders may overwrite it
        return out

    def mail_drain(xm):
        """before the closing event: the transfer of the step sent last must have left this rank (its regroup already ran)"""
        if xm.last_transfer is not None:
            stream.wait_event(xm.last_transfer)

    if world > 1 and args.exchange in ("mail", "mail-dma", "mail-hybrid", "mail-smcopy", "auto"):
        from tidb_b200.parallel import MailboxExchange
        names = ["mail-dma", "mail-hybrid", "mail"] if args.exchange == "auto" else [args.exchange]   # mail-smcopy measured slower (4.75 vs 3.45 ms at N = 2): explicit only
        timings = {}
        for nm in names:
            xm = MailboxExchange(rank, world, local, xstream, 2, npb, slack=args.slack, **MAIL_CANDIDATES[nm])
            if len(names) > 1:
                for _ in range(2):
                    mail_step(xm, False)
                barrier()
                c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                with torch.cuda.stream(stream):
                    c0.record(stream); xstream.wait_event(c0)
                    for _ in range(4):
                        mail_step(xm, False)
                    mail_drain(xm)
                    c1.record(stream)
                stream.synchronize(); xm.check()
                tt = torch.tensor([c0.elapsed_time(c1) / 4], dtype=torch.float64, device=dev)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)      # every rank sees the same numbers -> the same choice
                timings[nm] = float(tt.item())
                xm.close()
        if len(names) > 1:
            mail_choice = min(timings, key=timings.get)
            xmail = MailboxExchange(rank, world, local, xstream, 2, npb, slack=args.slack, **MAIL_CANDIDATES[mail_choice])
        else:
            mail_choice, xmail = names[0], xm
        mail_timings = timings

    def step(sync: bool):
        """sync=True is the verifying pass: returns (rows, checksums)"""
        if world == 1:
            rows, cols, _ = join.probe([pk, pv], sync=sync)
            last_cols[:] = cols
            return (rows, check_piece(cols, rows)) if sync else (None, None)
        if xmail is not None:
            return mail_step(xmail, sync)
        if xseg is not None:
            # count-free exchange: scatter into the peers' regions -> all-gather of the counts (the barrier) -> segmented
            # probe; everything is enqueued on `stream`, the host never waits inside a step
            # Two streams when --overlap: the NVLink-bound scatter of this step runs under the probe of the previous step;
            # only the all-gather (which releases the peers into the step that reuses the buffer set still being probed)
            # waits for that probe.  Without --overlap both streams are the same one and the waits are no-ops.
            xs = xseg.stream
            prev = done_ev[0]
            if args.overlap >= 2 and xseg.dma:
                # three-deep: regroup step k+1 | copy engines move step k (NVLink) | probe step k-1
                cols_in, seg_cnt, cap, got = xseg.exchange_async(pk, [pk, pv], prev_probe_done=prev, prev2_probe_done=done_ev[1])
                with torch.cuda.stream(stream):
                    stream.wait_event(got)
                    rows, cols, _ = join.probe_segments(cols_in, seg_cnt, cap, sync=sync)
                    ev = torch.cuda.Event(); ev.record(stream); done_ev[1] = done_ev[0]; done_ev[0] = ev
                    return (rows, check_piece(cols, rows)) if sync else (None, None)
            with torch.cuda.stream(xs):
                if prev is not None and (sync or not args.overlap):
                    xs.wait_event(prev)
                cols_in, seg_cnt, cap = xseg.exchange(pk, [pk, pv], before_gather=(lambda: xs.wait_event(prev)) if prev is not None else None, trace=TRACE)
                got = torch.cuda.Event(); got.record(xs)
            with torch.cuda.stream(stream):
                stream.wait_event(got)
                if TRACE is not None:
                    e = torch.cuda.Event(enable_timing=True); e.record(stream); TRACE.append(("probe start", e))
                rows, cols, _ = join.probe_segments(cols_in, seg_cnt, cap, sync=sync)
                ev = torch.cuda.Event(enable_timing=TRACE is not None); ev.record(stream); done_ev[0] = ev
                if TRACE is not None:
                    TRACE.append(("probe end", ev))
                return (rows, check_piece(cols, rows)) if sync else (None, None)
        total, chk = 0, torch.zeros(2, dtype=torch.int64, device=dev)
        for c, (lo, hi) in enumerate(bounds):
            x = xch_p[c % len(xch_p)]
            if done_ev[c % 2] is not None:
                done_ev[c % 2].synchronize()          # my probe of the piece that used this buffer set has finished
            with torch.cuda.stream(xstream):
                lpk, lpv = x.exchange(pk[lo:hi], [pk[lo:hi], pv[lo:hi]])    # returns after the closing barrier: data has landed
            with torch.cuda.stream(stream):
                rows, cols, _ = join.probe([lpk, lpv], sync=sync)
                if sync:
                    total += rows
                    chk += check_piece(cols, rows)
                ev = torch.cuda.Event(); ev.record(stream); done_ev[c % 2] = ev
        return (total, chk) if sync else (None, None)

    with torch.cuda.stream(stream):
        for _ in range(args.warmup):
            step(False)
        # correctness of the timed configuration: bit-exact output row count, per-row invariants, checksum of checksums
        rows, chk = step(True)
        total_rows = torch.tensor([rows], dtype=torch.int64, device=dev)
        pvs = torch.stack([pv.sum(), (pv * pv).sum()])
        if world > 1:
            dist.all_reduce(total_rows); dist.all_reduce(chk); dist.all_reduce(pvs)
        assert int(total_rows.item()) == npb * world, f"output rows {int(total_rows.item())} != {npb * world}"
        assert torch.equal(chk, pvs), "every probe row must appear exactly once in the output (100% match, unique build keys)"
    stream.synchronize()

    # ---- timed region: value (device resident) ----------------------------------------------------------------
    sampler = ClockSampler(local)
    l0 = join.stats().kernel_launches
    lx0 = (sum(x.launches for x in xch_p) if xch_p else 0) + (xseg.launches if xseg else 0) + (xmail.launches if xmail else 0)
    barrier()
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        ev0.record(stream)
        if xstream is not None:
            xstream.wait_event(ev0)
        for _ in range(args.steps):
            step(False)
        if xmail is not None:
            mail_drain(xmail)
        ev1.record(stream)
    stream.synchronize()
    barrier()
    if TRACE and rank == 0:
        t0 = ev0
        for name, e in TRACE[-(4 if xmail is not None else 7) * min(args.steps, 4):]:
            print(f"[trace] {t0.elapsed_time(e):9.3f} ms  {name}", file=sys.stderr)
    clocks = sampler.stop() if rank == 0 else None
    ms_total = ev0.elapsed_time(ev1)
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    launches_extra = (sum(x.launches for x in xch_p) if xch_p else 0) + (xseg.launches if xseg else 0) + (xmail.launches if xmail else 0)
    if xseg is not None:
        xseg.check_overflow()
    if xmail is not None:
        xmail.check()
    launches = (join.stats().kernel_launches - l0) + (launches_extra - lx0)
    value = npb * world / (ms_step * 1e-3)

    # kernel-only duration for the roofline at N = 1 (the step IS the probe kernel + an 8-byte memset)
    roof = None
    traffic = args.ncu_traffic_bytes
    if traffic is None:
        try:   # per-launch DRAM bytes of the committed ncu --set full capture of this kernel
            traffic = float(json.load(open(os.path.join(ROOT, "profiles", "r2_pipeline_traffic.json" if os.environ.get("TG_PROBE_PARTITION", "1") == "1" else "r1_probe_final_traffic.json")))["dram_bytes_per_launch"])
        except Exception:
            traffic = None
    if world == 1:
        achieved = BYTES_PER_PROBE_ROW * npb / (ms_step * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "traffic": traffic, "peak_source": peak_src,
                "kernel": ("k_partition_scatter_bulk<1,2,4> + k_probe_inner_u1_seg_lean<1,2,1,0> (L2 partition pass + segment probe: one step; frac is over the WHOLE step)"
                           if os.environ.get("TG_PROBE_PARTITION", "1") == "1" else "k_probe_inner_u1_w<4,1,2,1>"),
                "algorithmic_bytes_per_launch": BYTES_PER_PROBE_ROW * npb,
                "read_only_frac": 32 * npb / (ms_step * 1e-3) / 1e9 / hbm_peak}

    else:
        # N GPUs: same algorithmic bytes per probe row, denominator = N x the per-GPU peak (SURVEY 8d); the exchange adds
        # NVLink payload = 16 B x (N-1)/N of the rows, per direction per GPU
        achieved = BYTES_PER_PROBE_ROW * npb * world / (ms_step * 1e-3) / 1e9
        nvl = 16.0 * npb * (world - 1) / world / (ms_step * 1e-3) / 1e9
        roof = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak * world, "unit": "GB/s", "frac": achieved / (hbm_peak * world),
                "traffic": None, "peak_source": peak_src + f" x {world} GPUs",
                "kernel": "per rank and step: k_partition_scatter_bulk<0,2,4> (repartition + NVLink bulk stores) | k_partition_scatter_bulk<1,2,4> + k_probe_inner_u1_seg_lean<1,2,1,0> (L2 pass + segment probe)",
                "algorithmic_bytes_per_launch": BYTES_PER_PROBE_ROW * npb * world,
                "nvlink": {"payload_gbs_per_direction_per_gpu": nvl, "reference_gbs": 770.0, "frac": nvl / 770.0,
                           "note": "16 B per exchanged row; reference = measured peer-copy bandwidth per direction (B200_PROFILING.md)"}}

    if args.dump_outputs:
        # the last timed step's result, still in the join's output buffers; it probed the same inputs as the verifying
        # step, whose output row count `rows` was checked above
        with torch.cuda.stream(stream):
            dump_outputs(args.dump_outputs, {name: dview(p, rows) for name, p in
                                             zip(("probe_key", "probe_payload", "build_key", "build_payload"), last_cols)}, "probe_payload")
        stream.synchronize()

    # ---- side line (N = 1): the 50 % match variant of the same workload (SURVEY 8d input 2) ---------------------------
    side50 = None
    if world == 1 and not args.skip_side:
        with torch.cuda.stream(stream):
            g2 = torch.Generator(device=dev); g2.manual_seed(4343)
            pk2 = torch.randint(0, 2 * nb, (npb,), device=dev, generator=g2, dtype=torch.int64) * ODD      # uniform over twice the key range
            rows2, cols2, _ = join.probe([pk2, pv], sync=True)
            o_pk, o_pv, o_bk, o_bv = [dview(p, rows2) for p in cols2]
            assert bool((o_pk == o_bk).all()) and bool((o_bv * ODD == o_bk * 7).all())
            assert bool((pk2[o_pv] == o_pk).all()), "output rows must carry their own probe key"
            # bit-exact row count: a probe key matches iff its id (key * ODD^-1 mod 2^64) is below nb; ids were drawn directly
            g2.manual_seed(4343)
            ids2 = torch.randint(0, 2 * nb, (npb,), device=dev, generator=g2, dtype=torch.int64)
            assert rows2 == int((ids2 < nb).sum().item()), "50 % match: output row count differs from the number of matching probe keys"
            del ids2
            for _ in range(3):
                join.probe([pk2, pv], sync=False)
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record(stream)
            for _ in range(args.steps):
                join.probe([pk2, pv], sync=False)
            s1.record(stream)
        stream.synchronize()
        ms2 = s0.elapsed_time(s1) / args.steps
        b2 = 16 * npb + 16 * rows2 + 32 * rows2
        side50 = {"workload": "same join, probe keys uniform over twice the build key range (50 % match)", "ms_per_step": ms2, "value": npb / (ms2 * 1e-3),
                  "unit": "rows/s", "output_rows": rows2, "algorithmic_bytes": b2, "achieved_gbs": b2 / (ms2 * 1e-3) / 1e9, "frac": b2 / (ms2 * 1e-3) / 1e9 / hbm_peak}
        del pk2

    # ---- e2e: host buffers through tg_join_probe_push / tg_join_next (N = 1 path; per rank at N > 1) ---------
    e2e = None
    if not args.skip_e2e:
        if world == 1:
            e2e = run_e2e(args, lib, abi, torch, dev, local, rank, world, bk, bv, pk, pv, barrier)
            # side figure: the parent operator does not read build.k (it equals probe.k) -> RUsed = [build.v], 3 output columns
            e2e["pruned_3_columns"] = run_e2e(args, lib, abi, torch, dev, local, rank, world, bk, bv, pk, pv, barrier, rused=[1])
        else:
            e2e = (run_e2e_mail(args, torch, dist, dev, stream, xstream, rank, world, pk, pv, xmail, join, barrier, dview) if xmail is not None else
                   run_e2e_multi(args, torch, dist, dev, stream, xstream, rank, world, pk, pv, xch_p, bounds, join, barrier))

    # ---- CPU baseline (rank 0, N = 1 only): bounded sample on the box's host cores ------------------------------
    cpu = None
    if world == 1 and not args.skip_cpu:
        sample = min(npb, args.cpu_sample_rows)
        threads = host_threads()
        rate, ms, rows_c, bsec = cpu_probe_rate(bk.cpu().numpy(), bv.cpu().numpy(), pk[:sample].cpu().numpy(), pv[:sample].cpu().numpy(),
                                                sample, threads, 2, 1)
        assert rows_c == sample
        cpu = {"value": rate, "unit": "rows/s", "cores": threads, "kind": "port",
               "sample": f"full {nb}-row build ({bsec:.2f}s, untimed) + probe of the first {sample} probe rows as 1024-row chunks, mean of 2 after 1 warm-up; "
                         "oracle/join.cpp restates TiDB's HashJoinV2 (not the Go binary)"}
        if threads > 5:
            # the reference's own default: tidb_executor_concurrency = 5 (SURVEY §8d asks for both figures)
            s5 = min(sample, 2_000_000)
            r5, _, rows5, _ = cpu_probe_rate(bk.cpu().numpy(), bv.cpu().numpy(), pk[:s5].cpu().numpy(), pv[:s5].cpu().numpy(), s5, 5, 2, 1)
            assert rows5 == s5
            cpu["value_at_reference_default_concurrency_5"] = r5

    if rank == 0:
        line = {
            "metric": "hash-join probe rows/sec", "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64", "data": "synthetic",
            "config": {"workload": (f"hash join {npb}x{nb} int64 keys, 8-byte payload, 100% match, output 4 columns (BASELINE configs[1])" if world == 1 else
                                    f"partitioned hash join {npb * world}x{nb * world} int64 keys over {world} GPUs ({npb}x{nb} per GPU, keys uniform over the global key set), "
                                    f"8-byte payload, 100% match, output 4 columns, key-hash exchange over NVLink every step (BASELINE configs[4] / 8 per GPU" + ("" if world != 8 else " = the 1Bx100M join") + ")"),
                       "l2": "inputs larger than L2 (1.6 GB probe columns + 3.2 GB output + %.0f MB table per step vs 126 MB L2)" % (bstats.table_slots * 16 / 1e6),
                       "table": {"slots": bstats.table_slots, "mode": bstats.table_mode, "distinct_keys": bstats.distinct_keys, "build_ms": bstats.build_ms},
                       "exchange": "none" if world == 1 else {"mail": f"MailboxExchange ({mail_choice}): k_partition_scatter_bulk appends to this rank's fixed-capacity region on every peer with bulk stores over NVLink (tg_partition_exchange_cf_ex), counts and buffer-reuse ACKs through device mailboxes (tg_mail_signal / tg_mail_wait): no NCCL, no copy engine, no host wait in a step; exchange stream one step ahead of the probe stream; segmented probe (tg_join_probe_dev_seg)",
                                                                    "cf": "count-free: k_partition_scatter_bulk appends to this rank's fixed-capacity region on every peer over NVLink (tg_partition_exchange_cf), one all-gather of the counts per step, segmented probe (tg_join_probe_dev_seg)",
                                                                    "p2p": "k_partition_scatter storing into peer receive buffers over NVLink (tg_partition_exchange), counts all-gathered through the host",
                                                                    "nccl": "tg_partition_by_key + NCCL all_to_all_single per column"}["mail" if xmail is not None else args.exchange],
                       "exchange_calibration_ms": mail_timings or None},
            "clocks": clocks, "gpu_launches": int(launches), "e2e": e2e,
        }
        if roof:
            line["roofline"] = roof
        if side50:
            line["side_match_50"] = side50
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line))
    join.close()
    if world > 1:
        if xmail is not None:
            xmail.close()
        xch_b.close()
        for x in xch_p:
            x.close()
        dist.barrier()
        dist.destroy_process_group()


def run_e2e(args, lib, abi, torch, dev, local, rank, world, bk, bv, pk, pv, barrier, rused=None):
    """The probe through the host-facing C-ABI: pinned host columns in, pinned host columns out.
    rused = RUsed of the plan (None = all build columns, the reference harness; [1] = the parent does not read the build
    key, which equals the probe key: column pruning, builder.go:1868-1871)."""
    from tidb_b200.plan import JoinPlan
    nb, npb = bk.numel(), pk.numel()
    chunk_rows = args.e2e_chunk_rows

    def pinned(nbytes):
        p = C.c_void_p()
        abi.check(lib.tg_host_alloc(C.c_size_t(nbytes), C.byref(p)))
        return p

    def np_view(p, n):
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_int64)), shape=(n,))

    # the rank's own shard as host columns (what a TableReader would hand to the executor)
    hp = [pinned(npb * 8) for _ in range(2)]
    hb = [pinned(nb * 8) for _ in range(2)]
    for p, t in zip(hp, (pk, pv)):
        np_view(p, npb)[:] = t.cpu().numpy()
    for p, t in zip(hb, (bk, bv)):
        np_view(p, nb)[:] = t.cpu().numpy()
    n_out = 2 + (2 if rused is None else len(rused))
    out = [pinned(chunk_rows * 8) for _ in range(n_out)]
    plan = make_plan(local, 0)
    plan.rused = rused
    desc, keep = plan.to_struct()
    h = C.c_void_p()
    abi.check(lib.tg_join_open(C.byref(desc), C.byref(h)))

    def host_chunk(ptrs, lo, n):
        arr = (abi.TgColumn * 2)()
        for i, p in enumerate(ptrs):
            arr[i].length = n; arr[i].data = p.value + lo * 8; arr[i].elem_len = 8
        ck = abi.TgChunk(); ck.ncols = 2; ck.cols = C.cast(arr, C.POINTER(abi.TgColumn)); ck._keep = arr
        return ck

    for lo in range(0, nb, chunk_rows):
        ck = host_chunk(hb, lo, min(chunk_rows, nb - lo))
        abi.check(lib.tg_join_build_push(h, C.byref(ck)))
    abi.check(lib.tg_join_build_finish(h))
    mc = (abi.TgMutColumn * n_out)()
    for i in range(n_out):
        mc[i].data = out[i].value; mc[i].null_bitmap = None; mc[i].elem_len = 8
    mch = abi.TgMutChunk(); mch.ncols = n_out; mch.cols = C.cast(mc, C.POINTER(abi.TgMutColumn)); mch.capacity_rows = chunk_rows

    def one_pass():
        """a fresh probe of the whole probe side.  Two host threads, like the reference's probe fetcher goroutine and
        the consumer of joinResultCh: one pushes the pinned probe chunks (H2D + kernels), the other sits in
        tg_join_next_wait and receives the joined columns (D2H) — PCIe runs full duplex."""
        err = []

        def pusher():
            try:
                for lo in range(0, npb, chunk_rows):
                    ck = host_chunk(hp, lo, min(chunk_rows, npb - lo))
                    abi.check(lib.tg_join_probe_push(h, C.byref(ck)))
                abi.check(lib.tg_join_probe_finish(h))
            except Exception as e:   # noqa: BLE001
                err.append(e)
                lib.tg_join_probe_finish(h)

        th = threading.Thread(target=pusher)
        th.start()
        got = 0
        n = C.c_int64(0)
        while True:
            abi.check(lib.tg_join_next_wait(h, C.byref(mch), C.c_int64(chunk_rows), C.byref(n)))
            if n.value == 0:
                break
            got += n.value
        th.join()
        if err:
            raise err[0]
        abi.check(lib.tg_join_probe_rewind(h))
        return got

    for _ in range(max(1, args.warmup // 2)):
        assert one_pass() == npb
    barrier()
    t0 = time.perf_counter()
    steps = max(1, args.steps // 2)
    for _ in range(steps):
        got = one_pass()
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    assert got == npb
    st = abi.TgJoinStats()
    abi.check(lib.tg_join_get_stats(h, C.byref(st)))
    lib.tg_join_close(h)
    for p in hp + hb + out:
        lib.tg_host_free(p)
    tt = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    sec_step = float(tt.item()) / steps
    return {"value": npb * world / sec_step, "unit": "rows/s", "h2d_bytes_per_step": 16 * npb, "d2h_bytes_per_step": 8 * n_out * npb,
            "output_columns": n_out, "pcie_d2h_gbs": 8 * n_out * npb / sec_step / 1e9, "pcie_h2d_gbs": 16 * npb / sec_step / 1e9,
            "ms_per_step": sec_step * 1e3, "steps": steps, "chunk_rows": chunk_rows,
            "path": "thread A: tg_join_probe_push(host pinned 4M-row chunks) -> kernels; thread B: tg_join_next_wait -> D2H into host pinned buffers",
            "timing": "host wall clock around the passes, device synchronised on both sides (host work is part of the path)"}


def run_e2e_multi(args, torch, dist, dev, stream, xstream, rank, world, pk, pv, xch, bounds, join, barrier):
    """N > 1 end to end: every rank's probe shard starts in pinned HOST memory; a step = per piece: H2D, key-hash
    exchange over NVLink, shard-local probe, D2H of the joined columns into pinned host memory."""
    npb = pk.numel()
    hk = torch.empty(npb, dtype=torch.int64, pin_memory=True); hk.copy_(pk)
    hv = torch.empty(npb, dtype=torch.int64, pin_memory=True); hv.copy_(pv)
    piece = max(hi - lo for lo, hi in bounds)
    cap = int(piece * 1.03) + 8192
    hout = [torch.empty(cap, dtype=torch.int64, pin_memory=True) for _ in range(4)]
    dk = [torch.empty(piece, dtype=torch.int64, device=dev) for _ in range(2)]
    dv = [torch.empty(piece, dtype=torch.int64, device=dev) for _ in range(2)]

    def one_pass():
        total = 0
        for c, (lo, hi) in enumerate(bounds):
            x = xch[c % len(xch)]
            n = hi - lo
            with torch.cuda.stream(xstream):
                dk[c % 2][:n].copy_(hk[lo:hi], non_blocking=True); dv[c % 2][:n].copy_(hv[lo:hi], non_blocking=True)
                lpk, lpv = x.exchange(dk[c % 2][:n], [dk[c % 2][:n], dv[c % 2][:n]])
            with torch.cuda.stream(stream):
                rows, cols, _ = join.probe([lpk, lpv], sync=True)
                for i, p in enumerate(cols):
                    hout[i][:rows].copy_(x._view(p, rows), non_blocking=True)
            stream.synchronize()
            total += rows
        return total

    steps = max(1, args.steps // 2)
    for _ in range(2):
        rows = one_pass()
    tot = torch.tensor([rows], dtype=torch.int64, device=dev); dist.all_reduce(tot)
    assert int(tot.item()) == npb * world
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        one_pass()
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    tt = torch.tensor([dt], dtype=torch.float64, device=dev)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    sec_step = float(tt.item()) / steps
    return {"value": npb * world / sec_step, "unit": "rows/s", "h2d_bytes_per_step": 16 * npb * world, "d2h_bytes_per_step": 32 * npb * world,
            "ms_per_step": sec_step * 1e3, "steps": steps,
            "path": "per rank and piece: pinned host shard -> H2D -> key-hash exchange over NVLink -> tg_join_probe_dev -> D2H of the 4 joined columns into pinned host memory",
            "timing": "host wall clock, max over ranks, device synchronised on both sides"}


def run_e2e_mail(args, torch, dist, dev, stream, xstream, rank, world, pk, pv, xm, join, barrier, dview):
    """N > 1 end to end through the SAME exchange the device-resident number uses: every rank's probe shard starts in pinned
    HOST memory; a step = H2D of the shard (exchange stream), MailboxExchange.send, segmented probe, D2H of the joined
    columns into pinned host memory.  The exchange stream works on step k+1 (H2D + NVLink) while the probe stream
    finishes step k (probe + D2H): two device input sets."""
    npb = pk.numel()
    hk = torch.empty(npb, dtype=torch.int64, pin_memory=True); hk.copy_(pk)
    hv = torch.empty(npb, dtype=torch.int64, pin_memory=True); hv.copy_(pv)
    cap_out = int(npb * 1.06) + 65536
    hout = [torch.empty(cap_out, dtype=torch.int64, pin_memory=True) for _ in range(4)]
    dk = [torch.empty(npb, dtype=torch.int64, device=dev) for _ in range(2)]
    dv = [torch.empty(npb, dtype=torch.int64, device=dev) for _ in range(2)]
    probed = [None, None]

    def enqueue_send(i):
        with torch.cuda.stream(xstream):
            if probed[i % 2] is not None:
                xstream.wait_event(probed[i % 2])     # (the scatter of step i-2 read this input set on xstream itself; nothing else reads it)
            dk[i % 2].copy_(hk, non_blocking=True); dv[i % 2].copy_(hv, non_blocking=True)
            xm.send(dk[i % 2], [dk[i % 2], dv[i % 2]])

    def one_pass(steps):
        total = 0
        enqueue_send(0)
        for i in range(steps):
            if i + 1 < steps:
                enqueue_send(i + 1)
            with torch.cuda.stream(stream):
                cols_in, seg_cnt, cap, s_, ep = xm.recv(stream)
                rows, cols, _ = join.probe_segments(cols_in, seg_cnt, cap, sync=True)
                xm.release(stream, s_, ep)
                for c, p in enumerate(cols):
                    hout[c][:rows].copy_(dview(p, rows), non_blocking=True)
                ev = torch.cuda.Event(); ev.record(stream); probed[i % 2] = ev
            stream.synchronize()       # the consumer owns the host buffers before the next step overwrites them
            total = rows
        return total

    steps = max(2, args.steps // 2)
    with torch.cuda.stream(stream):
        xm.discard_outstanding(stream)      # the device-resident loop keeps one step in flight
    xm._primed = False
    rows = one_pass(2)
    tot = torch.tensor([rows], dtype=torch.int64, device=dev); dist.all_reduce(tot)
    assert int(tot.item()) == npb * world
    barrier()
    t0 = time.perf_counter()
    one_pass(steps)
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    tt = torch.tensor([dt], dtype=torch.float64, device=dev)
    dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    xm.check()
    sec_step = float(tt.item()) / steps
    return {"value": npb * world / sec_step, "unit": "rows/s", "h2d_bytes_per_step": 16 * npb * world, "d2h_bytes_per_step": 32 * npb * world,
            "ms_per_step": sec_step * 1e3, "steps": steps,
            "path": "per rank: pinned host shard -> H2D -> MailboxExchange (the exchange `value` times) -> tg_join_probe_dev_seg -> D2H of the 4 joined columns into pinned host memory; exchange stream one step ahead",
            "timing": "host wall clock, max over ranks, device synchronised on both sides"}


# ---------------------------------------------------------------------------------------------------------
# --workload agg: BASELINE configs[2], HashAgg SUM/COUNT GROUP BY int64, 100M rows / 1M groups, 1 GPU
# ---------------------------------------------------------------------------------------------------------
def run_agg(args):
    """Same JSON contract as the join line, metric = aggregated input rows/sec.  A step = one whole aggregation (table
    init + update + finalize) of the 100M-row batch.  roofline: 16.24 algorithmic bytes per row (SURVEY 8d) over the HBM peak,
    plus the measured L2-operation floor of this access pattern (profiles/r2_agg_lab.md) as `l2_op_floor_ms`."""
    os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
    import torch
    from tidb_b200 import abi
    from tidb_b200.chunk import Chunk, Column
    from tidb_b200.device import DeviceAgg
    from tidb_b200.plan import AggFunc, AggPlan, FieldType
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    n, G = args.agg_rows, args.agg_groups
    hbm_peak, peak_src = peaks()
    stream = torch.cuda.Stream(device=dev)
    INT = FieldType(abi.TYPE_LONGLONG, abi.FLAG_NOT_NULL); DBL = FieldType(abi.TYPE_DOUBLE, abi.FLAG_NOT_NULL)
    with torch.cuda.stream(stream):
        g = torch.Generator(device=dev); g.manual_seed(44)
        keys = torch.randint(0, G, (n,), device=dev, generator=g, dtype=torch.int64)
        x = torch.floor(torch.rand(n, device=dev, generator=g, dtype=torch.float64) * 1e7)
    stream.synchronize()
    funcs = [AggFunc(abi.AGG_FIRSTROW, 0), AggFunc(abi.AGG_SUM, 1, abi.TYPE_DOUBLE), AggFunc(abi.AGG_COUNT, 1, abi.TYPE_DOUBLE)]
    plan = AggPlan([INT, DBL], [0], funcs, stream=stream.cuda_stream, expected_groups=G)

    def view(p, m, dt):
        class _A:
            pass
        o = _A(); o.__cuda_array_interface__ = {"shape": (m,), "typestr": dt, "data": (p, False), "version": 3}
        return torch.as_tensor(o, device=dev)

    kept = []    # --dump-outputs: (handle, rows, result column pointers) of the last timed step, closed once written out

    def one(verify=False, keep=False):
        agg = DeviceAgg(plan)
        with torch.cuda.stream(stream):
            agg.push([keys, x])
            rows, cols, _ = agg.finish()
            if verify:   # COUNT bit-exact, SUM within 1e-6 relative against plain reductions of the same columns
                gk, s_, c_ = view(cols[0], rows, "<i8"), view(cols[1], rows, "<f8"), view(cols[2], rows, "<i8")
                assert rows == G and torch.equal(torch.sort(gk).values, torch.arange(G, device=dev))
                assert torch.equal(c_, torch.bincount(keys, minlength=G)[gk])
                exp = torch.zeros(G, dtype=torch.float64, device=dev).scatter_add_(0, keys, x)
                assert torch.allclose(s_, exp[gk], rtol=1e-6, atol=0)
        st = agg.stats()
        if keep:
            kept.append((agg, rows, cols))
        else:
            agg.close()
        return st
    for _ in range(max(3, args.warmup) - 1):
        one()
    one(verify=True)
    sampler = ClockSampler(0); sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    with torch.cuda.stream(stream):
        e0.record(stream)
    for i in range(args.steps):
        launches += one(keep=bool(args.dump_outputs) and i == args.steps - 1).kernel_launches
    with torch.cuda.stream(stream):
        e1.record(stream)
    stream.synchronize()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1) / args.steps
    if kept:
        agg, rows, cols = kept.pop()
        with torch.cuda.stream(stream):
            dump_outputs(args.dump_outputs, {"group_key": view(cols[0], rows, "<i8"), "sum": view(cols[1], rows, "<f8"),
                                             "count": view(cols[2], rows, "<i8")}, "group_key")
        stream.synchronize()
        agg.close()
    # e2e: host chunks through tg_agg_push / tg_agg_next (pinned host memory in, host result out)
    e2e = None
    if not args.skip_e2e:
        from tidb_b200.executor import HashAggExec, MockDataSource, drain
        hk = torch.empty(n, dtype=torch.int64, pin_memory=True); hk.copy_(keys)
        hx = torch.empty(n, dtype=torch.float64, pin_memory=True); hx.copy_(x)
        chunks = Chunk([Column(hk.numpy()), Column(hx.numpy())]).split(args.e2e_chunk_rows)
        hplan = AggPlan([INT, DBL], [0], funcs, expected_groups=G)
        drain(HashAggExec(hplan, MockDataSource(hplan.col_types, chunks)), 1 << 20)
        t0 = time.perf_counter(); reps = max(1, args.steps // 3)
        for _ in range(reps):
            out = drain(HashAggExec(hplan, MockDataSource(hplan.col_types, chunks)), 1 << 20)
        dt = (time.perf_counter() - t0) / reps
        assert sum(c.num_rows() for c in out) == G
        e2e = {"value": n / dt, "unit": "rows/s", "h2d_bytes_per_step": 16 * n, "d2h_bytes_per_step": 24 * G, "ms_per_step": dt * 1e3,
               "path": "pinned host columns in 4M-row chunks -> tg_agg_push (H2D + update) -> tg_agg_finish -> tg_agg_next (D2H of the 3 result columns)"}
    # CPU baseline: the oracle's HashAgg restatement on a bounded sample, at the reference's default concurrency (5) and on all threads
    cpu = None
    if not args.skip_cpu:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as O
        sample = min(n, args.cpu_sample_rows)
        hk_s, hx_s = keys[:sample].cpu().numpy(), x[:sample].cpu().numpy()
        ch = Chunk([Column(hk_s), Column(hx_s)]).split(1024)
        threads = host_threads()
        res = {}
        for conc in sorted({5, threads}):
            oa = O.OracleAgg(AggPlan([INT, DBL], [0], funcs), conc, conc)
            t0 = time.perf_counter(); oa.run(ch); dt = time.perf_counter() - t0
            oa.close()
            res[conc] = sample / dt
        cpu = {"value": res[threads], "unit": "rows/s", "cores": threads, "kind": "port",
               "sample": f"first {sample} rows as 1024-row chunks (groups seen: up to {G}); oracle/agg.cpp restates TiDB's HashAggExec partial/final workers (not the Go binary)",
               "value_at_reference_default_concurrency_5": res.get(5)}
    alg = 16 * n + 24 * G
    line = {"metric": "hash-agg input rows/sec", "value": n / (ms * 1e-3), "unit": "rows/s", "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"HashAggExec SUM/COUNT GROUP BY int64, {n} rows / {G} groups, 1 GPU (BASELINE configs[2])",
                       "l2": "inputs (1.6 GB) larger than L2; the group table (48 MB) is L2 resident by design"},
            "clocks": clocks, "gpu_launches": int(launches), "e2e": e2e,
            "roofline": {"bound": "hbm", "achieved": alg / (ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s", "frac": alg / (ms * 1e-3) / 1e9 / hbm_peak,
                         "traffic": None, "peak_source": peak_src, "kernel": "k_agg_init + k_agg_update2<false> + k_agg_count + k_agg_finalize (one step)",
                         "algorithmic_bytes_per_launch": alg,
                         "l2_op_floor_ms": 1.572 * n / 1e8, "frac_of_l2_op_floor": (1.572 * n / 1e8) / ms,
                         "note": "the table lives in L2: one key gather + two 64-bit REDs per row cost 1.572 ms per 100 M rows on this chip (tools/scratch/agg_lab.cu, profiles/r2_agg_lab.md)"}}
    if cpu:
        line["cpu_baseline"] = cpu
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="join", choices=["join", "agg"], help="join = the headline (BASELINE configs[1] / configs[4]); agg = BASELINE configs[2] on one GPU")
    ap.add_argument("--agg-rows", type=int, default=100_000_000)
    ap.add_argument("--agg-groups", type=int, default=1_000_000)
    ap.add_argument("--build-rows", type=int, default=None, help="per GPU; default 10M at N=1 (configs[1]), 12.5M at N>1 (configs[4] / 8)")
    ap.add_argument("--probe-rows", type=int, default=None, help="per GPU; default 100M at N=1, 125M at N>1")
    ap.add_argument("--cpu-sample-rows", type=int, default=8_000_000)
    ap.add_argument("--ref-sample-rows", type=int, default=8_000_000)
    ap.add_argument("--e2e-chunk-rows", type=int, default=4 << 20)
    ap.add_argument("--exchange", default="auto", choices=["mail", "mail-dma", "mail-hybrid", "mail-smcopy", "auto", "cf", "p2p", "nccl"],
                    help="N>1 probe-side exchange, all count-free with device mailboxes (no NCCL / host wait in a step): mail = the regroup kernel stores into the peers "
                         "itself; mail-dma = copy engines move the staged regions; mail-hybrid = copy engines + one direct peer; mail-smcopy = an SM copy kernel next to "
                         "the probe; auto (default) = time mail-dma / mail-hybrid / mail for a few untimed steps and keep the fastest.  cf = round-1 exchange (NCCL "
                         "all-gather per step); p2p = counted peer stores; nccl = local scatter + all_to_all")
    ap.add_argument("--slack", type=float, default=1.03, help="N>1, mailbox exchange: receive-region capacity = expected share x slack + 8192 rows (uniform keys: 3 %% is > 100 sigma)")
    ap.add_argument("--sm-copy-ctas", type=int, default=0, help="N>1, mail-smcopy: 128-thread CTAs of the region copy kernel (0 = one per SM)")
    ap.add_argument("--direct-peers", type=int, default=0, help="N>1, mail-dma: peers (ring order) whose rows the regroup kernel stores directly over NVLink; the rest go through the copy engines (mail-hybrid = (N-1)//3)")
    ap.add_argument("--copy-streams", type=int, default=0, help="N>1, mail-dma: streams the peer copies are spread over (0 = one per copy, at most 16)")
    ap.add_argument("--scatter-ctas", type=int, default=0, help="N>1, --exchange mail: cap on the exchange kernel's CTAs per SM (0 = as many as fit)")
    ap.add_argument("--overlap", type=int, default=2, help="N>1, --exchange cf: 1: run the exchange of step k+1 on a second stream under the probe of step k; 2: additionally a transfer stream, so regroup / NVLink copy / probe work on three consecutive steps")
    ap.add_argument("--dma", type=int, default=1, help="N>1, --exchange cf: regroup locally, let copy engines move the regions over NVLink")
    ap.add_argument("--xchunks", type=int, default=1, help="N>1: pieces the probe side is exchanged in (overlap with the probe kernel)")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-side", action="store_true", help="skip the 50 %% match side line (N = 1)")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--ncu-traffic-bytes", type=float, default=None, help="dram bytes per launch from the committed ncu capture")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the output columns of the last one as DIR/<name>.npy (float64; rows in a canonical "
                         f"order, a seeded sample of {DUMP_ROWS} rows of a larger output; GPU arm, one GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.gpus != 1):
        ap.error("--dump-outputs needs --impl b200 and --gpus 1")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "agg":
        run_agg(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
