// agg.cu — tg_agg_*: GPU hash aggregation behind HashAggExec's Open/Next/Close contract
// (pkg/executor/aggregate/agg_hash_executor.go:93, :237, :441, :164).
//
// What the kernels replace:
//   GetGroupKey + getPartialResultsOfEachRow + per-row af.UpdatePartialResult
//     (agg_util.go:106, agg_hash_partial_worker.go:219, :256)         → k_agg_update / k_agg_update_nogroup
//   HashAggFinalWorker merge + AppendFinalResult2Chunk (agg_hash_final_worker.go:73, :121;
//     func_sum.go:80, func_avg.go:332, func_count.go:43)              → k_agg_finalize
// There is no partial/final split on one GPU: every row updates the single device-resident group table
// with atomics (the 1M-group table of config 3 is 32–48 MB and lives in the 126 MB L2).
//
// Layout: structure-of-arrays open-addressing table — keys[S+2] (int64, sentinel = empty), rows[S+2]
// (group row count), and one or two 8-byte state arrays per aggregate.  Slot S holds the NULL group
// (NULL group keys DO form a group: codec.go:1766), slot S+1 the group whose key equals the sentinel.
#include <memory>
#include <algorithm>
#include "common.cuh"
#include "tma.cuh"

namespace tg {

#define TG_MAX_AGG 12
enum { GK_I64 = 0, GK_F64 = 1, GK_NONE = 2 };

struct AggFuncDev {
  int32_t name;         // TG_AGG_*
  int32_t arg_col;      // -1: COUNT(*)
  int32_t is_real;
  int32_t is_unsigned;
  int32_t s0, s1;       // state array indices (-1 = unused): s0 value (sum / min / max / count), s1 non-NULL count
  int32_t final_mode;   // TG_AGGMODE_FINAL: inputs are partial results
  int32_t arg_col2;
  int32_t arg_expr;     // TG_ARGEXPR_*
  int32_t pad;
  double arg_const;
};
struct AggSpec { int32_t n; int32_t pad; unsigned long long* err; AggFuncDev f[TG_MAX_AGG]; };

// argument of SUM / AVG as a double: a plain column or the fused scalar expression; false = NULL.  A non-finite
// intermediate on a non-NULL row raises *spec.err (types.ErrOverflow: builtin_arithmetic_vec.go:51-58, :312-318)
__device__ __forceinline__ bool agg_arg_real(const AggSpec& spec, const AggFuncDev& f, const DevCols& cols, int64_t row, double& v) {
  const uint8_t* nb = cols.nulls[f.arg_col];
  if (nb && !bit_not_null(nb, row)) return false;
  const double a = __longlong_as_double((long long)__ldcs(reinterpret_cast<const unsigned long long*>(cols.data[f.arg_col]) + row));
  if (f.arg_expr == TG_ARGEXPR_COL) { v = a; return true; }
  const uint8_t* nb2 = cols.nulls[f.arg_col2];
  if (nb2 && !bit_not_null(nb2, row)) return false;
  const double b = __longlong_as_double((long long)__ldcs(reinterpret_cast<const unsigned long long*>(cols.data[f.arg_col2]) + row));
  const double t = f.arg_expr == TG_ARGEXPR_MUL_CSUB ? __dsub_rn(f.arg_const, b) : b;
  const double r = __dmul_rn(a, t);     // separate roundings, like the two builtins (no fused multiply-add)
  if (!isfinite(t) || !isfinite(r)) atomicExch(spec.err, 1ull);
  v = r;
  return true;
}
#define TG_MAX_GROUP_COLS 4
struct AggTable {
  long long* keys;                       // single GROUP BY column: the key itself (kEmptyKey = unoccupied)
  unsigned long long* rows;
  unsigned long long* state[2 * TG_MAX_AGG];
  unsigned long long nslots;
  // several GROUP BY columns (GetGroupKey concatenates their encodings, agg_util.go:106 / codec.go:1761): a slot is claimed
  // through its 64-bit TAG word (0 empty, hash|1 being written, hash|3 published) and holds nkw key words — one per
  // column (NULL stored as 0) plus, when a column is nullable, a word with the columns' NULL bits
  unsigned long long* tags;
  long long* keyw[TG_MAX_GROUP_COLS + 1];
  int32_t nkw;
  // element stride of every array above, in 8-byte words: 1 = structure of arrays (single-key tables: hot groups live in
  // L2 and same-sector atomics would serialise, profiles/r2_agg_lab.md); multi-key tables are ARRAY OF RECORDS
  // [tag | key words | rows | states], padded to 32 bytes: their groups are mostly cold (Q3: 2.4 rows per group, a 1.4 GB
  // table), and a row should touch one or two DRAM sectors instead of one per array
  uint32_t stride;
};
struct GroupKey { const void* data; const uint8_t* nulls; int32_t kind; int32_t pad; };
struct GroupKeys { int32_t n, nkw; const void* data[TG_MAX_GROUP_COLS]; const uint8_t* nulls[TG_MAX_GROUP_COLS]; int32_t kind[TG_MAX_GROUP_COLS]; };

// order-preserving map double → u64 so that MIN/MAX(double) can use integer atomics
__device__ __forceinline__ unsigned long long f64_to_ordered(double d) {
  unsigned long long u = (unsigned long long)__double_as_longlong(d);
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double ordered_to_f64(unsigned long long u) {
  u = (u >> 63) ? (u & 0x7fffffffffffffffull) : ~u;
  return __longlong_as_double((long long)u);
}
__device__ __forceinline__ unsigned long long i64_to_ordered(long long v) { return (unsigned long long)v ^ 0x8000000000000000ull; }

__global__ void k_agg_init(AggTable t, AggSpec spec, unsigned long long n_total) {
  unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
  unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  for (; i < n_total; i += stride) {
    if (t.nkw) { t.tags[(size_t)i * t.stride] = 0; for (int j = 0; j < t.nkw; j++) t.keyw[j][(size_t)i * t.stride] = 0; }
    else t.keys[i] = kEmptyKey;
    t.rows[(size_t)i * t.stride] = 0;
    for (int k = 0; k < spec.n; k++) {
      const AggFuncDev& f = spec.f[k];
      if (f.s0 >= 0) {
        unsigned long long init = 0;
        if (f.name == TG_AGG_MIN) init = ~0ull;          // ordered domain: larger than everything
        t.state[f.s0][(size_t)i * t.stride] = init;
      }
      if (f.s1 >= 0) t.state[f.s1][(size_t)i * t.stride] = 0;
    }
  }
}

__device__ __forceinline__ void agg_apply(const AggTable& t, const AggSpec& spec, const DevCols& cols, int64_t row,
                                          unsigned long long s) {
  atomicAdd(&t.rows[(size_t)s * t.stride], 1ull);
  for (int k = 0; k < spec.n; k++) {
    const AggFuncDev& f = spec.f[k];
    if (f.arg_col < 0 || f.s0 < 0) continue;   // COUNT(*) and NOT NULL COUNT(x) read rows[]; FIRSTROW reads the key
    const uint8_t* nb = cols.nulls[f.arg_col];
    if (nb && !bit_not_null(nb, row)) continue;
    switch (f.name) {
      case TG_AGG_COUNT:
        if (f.final_mode) atomicAdd(&t.state[f.s0][(size_t)s * t.stride], reinterpret_cast<const unsigned long long*>(cols.data[f.arg_col])[row]);
        else atomicAdd(&t.state[f.s0][(size_t)s * t.stride], 1ull);
        break;
      case TG_AGG_SUM: {
        double v;
        if (!agg_arg_real(spec, f, cols, row, v)) break;
        atomicAdd(reinterpret_cast<double*>(&t.state[f.s0][(size_t)s * t.stride]), v);
        if (f.s1 >= 0) atomicAdd(&t.state[f.s1][(size_t)s * t.stride], 1ull);
        break;
      }
      case TG_AGG_AVG:
        if (f.final_mode) {   // args: count column, sum column (func_avg.go:405)
          const uint8_t* nb2 = cols.nulls[f.arg_col2];
          if (nb2 && !bit_not_null(nb2, row)) break;
          atomicAdd(reinterpret_cast<double*>(&t.state[f.s0][(size_t)s * t.stride]), reinterpret_cast<const double*>(cols.data[f.arg_col2])[row]);
          atomicAdd(&t.state[f.s1][(size_t)s * t.stride], reinterpret_cast<const unsigned long long*>(cols.data[f.arg_col])[row]);
        } else {
          double v;
          if (!agg_arg_real(spec, f, cols, row, v)) break;
          atomicAdd(reinterpret_cast<double*>(&t.state[f.s0][(size_t)s * t.stride]), v);
          if (f.s1 >= 0) atomicAdd(&t.state[f.s1][(size_t)s * t.stride], 1ull);
        }
        break;
      case TG_AGG_MIN: case TG_AGG_MAX: {
        unsigned long long v;
        if (f.is_real) v = f64_to_ordered(reinterpret_cast<const double*>(cols.data[f.arg_col])[row]);
        else if (f.is_unsigned) v = reinterpret_cast<const unsigned long long*>(cols.data[f.arg_col])[row];
        else v = i64_to_ordered(reinterpret_cast<const long long*>(cols.data[f.arg_col])[row]);
        if (f.name == TG_AGG_MIN) atomicMin(&t.state[f.s0][(size_t)s * t.stride], v); else atomicMax(&t.state[f.s0][(size_t)s * t.stride], v);
        if (f.s1 >= 0) atomicAdd(&t.state[f.s1][(size_t)s * t.stride], 1ull);
        break;
      }
      default: break;
    }
  }
}

// One thread per row: find-or-insert the group slot, then atomics.  Rows whose NEW key would push the
// table past max_fill are deferred (bit set in `deferred`) so the host can grow the table and re-run
// them; `only` restricts a re-run to those rows.
__global__ void __launch_bounds__(256)
k_agg_update(GroupKey gk, DevCols cols, int64_t n, AggTable t, AggSpec spec, unsigned long long max_fill,
             unsigned long long* fill, uint32_t* deferred, const uint32_t* only, unsigned long long* n_deferred) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    if (only && !((only[i >> 5] >> (i & 31)) & 1u)) continue;
    unsigned long long s;
    bool is_null = gk.nulls && !bit_not_null(gk.nulls, i);
    if (is_null) s = t.nslots;
    else {
      long long k;
      if (gk.kind == GK_I64) k = reinterpret_cast<const long long*>(gk.data)[i];
      else {
        double d = reinterpret_cast<const double*>(gk.data)[i];
        if (d == 0) d = 0;   // -0 and +0 encode to the same group key (codec float.go:23)
        k = __double_as_longlong(d);
      }
      if (k == kEmptyKey) s = t.nslots + 1;
      else {
        s = slot_of(mix64((uint64_t)k), t.nslots);
        bool defer = false;
        // No global fill counter: one atomic per NEW key on a single address serialised at ~3 ns each (1 M groups =
        // 3 ms, twice the rest of the kernel).  A probe sequence longer than `max_fill` steps means the table is
        // overfull: the row is deferred and the host grows the table.
        unsigned int steps = 0;
        for (;;) {
          long long cur = *reinterpret_cast<volatile long long*>(&t.keys[s]);
          if (cur == k) break;
          if (cur == kEmptyKey) {
            unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long*>(&t.keys[s]), (unsigned long long)kEmptyKey,
                                               (unsigned long long)k);
            if (old == (unsigned long long)kEmptyKey || old == (unsigned long long)k) break;
          }
          if (++steps > (unsigned int)max_fill) { defer = true; break; }
          if (++s == t.nslots) s = 0;
        }
        if (defer) {
          atomicOr(&deferred[i >> 5], 1u << (i & 31));
          atomicAdd(n_deferred, 1ull);
          continue;
        }
      }
    }
    agg_apply(t, spec, cols, i, s);
  }
}

// no GROUP BY: one group.  Warp-shuffle partial reduction, then one atomic per warp and aggregate.
__global__ void __launch_bounds__(256)
k_agg_update_nogroup(DevCols cols, int64_t n, AggTable t, AggSpec spec) {
  int64_t i0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int lane = threadIdx.x & 31;
  unsigned long long my_rows = 0;
  for (int64_t i = i0; i < n; i += stride) my_rows++;
  for (int o = 16; o; o >>= 1) my_rows += __shfl_xor_sync(0xffffffffu, my_rows, o);
  if (lane == 0 && my_rows) atomicAdd(&t.rows[t.nslots], my_rows);
  for (int k = 0; k < spec.n; k++) {
    const AggFuncDev& f = spec.f[k];
    if (f.arg_col < 0 || f.s0 < 0) continue;
    const uint8_t* nb = cols.nulls[f.arg_col];
    double fs = 0; unsigned long long cnt = 0, ext = f.name == TG_AGG_MIN ? ~0ull : 0ull, isum = 0;
    for (int64_t i = i0; i < n; i += stride) {
      if (nb && !bit_not_null(nb, i)) continue;
      if (f.name == TG_AGG_AVG && f.final_mode) {
        const uint8_t* nb2 = cols.nulls[f.arg_col2];
        if (nb2 && !bit_not_null(nb2, i)) continue;
        fs += reinterpret_cast<const double*>(cols.data[f.arg_col2])[i];
        cnt += reinterpret_cast<const unsigned long long*>(cols.data[f.arg_col])[i];
        continue;
      }
      if ((f.name == TG_AGG_SUM || f.name == TG_AGG_AVG) && f.arg_expr) {
        double v;
        if (!agg_arg_real(spec, f, cols, i, v)) continue;
        cnt++; fs += v;
        continue;
      }
      cnt++;
      if (f.name == TG_AGG_SUM || f.name == TG_AGG_AVG) fs += reinterpret_cast<const double*>(cols.data[f.arg_col])[i];
      else if (f.name == TG_AGG_COUNT) { if (f.final_mode) isum += reinterpret_cast<const unsigned long long*>(cols.data[f.arg_col])[i]; else isum++; }
      else {
        unsigned long long v;
        if (f.is_real) v = f64_to_ordered(reinterpret_cast<const double*>(cols.data[f.arg_col])[i]);
        else if (f.is_unsigned) v = reinterpret_cast<const unsigned long long*>(cols.data[f.arg_col])[i];
        else v = i64_to_ordered(reinterpret_cast<const long long*>(cols.data[f.arg_col])[i]);
        ext = f.name == TG_AGG_MIN ? (v < ext ? v : ext) : (v > ext ? v : ext);
      }
    }
    for (int o = 16; o; o >>= 1) {
      fs += __shfl_xor_sync(0xffffffffu, fs, o);
      cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
      isum += __shfl_xor_sync(0xffffffffu, isum, o);
      unsigned long long e2 = __shfl_xor_sync(0xffffffffu, ext, o);
      ext = f.name == TG_AGG_MIN ? (e2 < ext ? e2 : ext) : (e2 > ext ? e2 : ext);
    }
    if (lane == 0 && cnt) {
      unsigned long long s = t.nslots;
      if (f.name == TG_AGG_SUM || f.name == TG_AGG_AVG) atomicAdd(reinterpret_cast<double*>(&t.state[f.s0][s]), fs);
      else if (f.name == TG_AGG_COUNT) atomicAdd(&t.state[f.s0][s], isum);
      else if (f.name == TG_AGG_MIN) atomicMin(&t.state[f.s0][s], ext);
      else atomicMax(&t.state[f.s0][s], ext);
      if (f.s1 >= 0 && !(f.name == TG_AGG_COUNT)) atomicAdd(&t.state[f.s1][s], cnt);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Two-phase path for low-cardinality GROUP BY (the reference's own benchmark uses NDV 1000, benchmark_test.go:224): the
// same partial → final split as HashAggPartialWorker / HashAggFinalWorker (agg_hash_partial_worker.go:256,
// agg_hash_final_worker.go:73), with a CTA playing the partial worker.  Each CTA aggregates its rows into a
// shared-memory table (2048-4096 slots + the NULL and sentinel groups); rows whose new key does not fit are
// deferred to the global kernel.  At the end the CTA emits its partial results, and k_agg_merge folds them into the
// global table (MergePartialResult semantics) with the usual grow-and-retry protocol.
// ---------------------------------------------------------------------------------------------------------------
#define AGG_LOCAL_SLOTS_MAX 4096   // per-CTA table: 4096 slots with <= 1 state array, 2048 otherwise (about 96 KB, 2 CTAs per SM)
#define AGG_LOCAL_MAX_STATES 4
struct AggPartials {   // columnar partial results, capacity = gridDim.x * (local_slots / 2 + 2)
  long long* keys;
  unsigned char* kind;                 // 0 regular key, 1 NULL group, 2 sentinel-valued key
  unsigned long long* rows;
  unsigned long long* state[AGG_LOCAL_MAX_STATES];
  unsigned long long* count;           // number of tuples emitted
};

__global__ void __launch_bounds__(256)
k_agg_update_local(GroupKey gk, DevCols cols, int64_t row_lo, int64_t row_hi, AggSpec spec, int nstates, int local_slots,
                   AggPartials out, uint32_t* deferred, unsigned long long* n_deferred) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int LS = local_slots, NT = local_slots + 2;
  const unsigned int max_local_fill = (unsigned int)(local_slots / 2);
  AggTable lt;
  lt.stride = 1; lt.nkw = 0; lt.tags = nullptr;
  lt.nslots = (unsigned long long)LS;
  lt.keys = reinterpret_cast<long long*>(smem_raw);
  lt.rows = reinterpret_cast<unsigned long long*>(smem_raw) + NT;
  for (int s = 0; s < nstates; s++) lt.state[s] = reinterpret_cast<unsigned long long*>(smem_raw) + (size_t)NT * (2 + s);
  __shared__ unsigned int s_fill;
  for (int i = threadIdx.x; i < NT; i += blockDim.x) {
    lt.keys[i] = kEmptyKey; lt.rows[i] = 0;
    for (int k = 0; k < spec.n; k++) {
      const AggFuncDev& f = spec.f[k];
      if (f.s0 >= 0) lt.state[f.s0][i] = f.name == TG_AGG_MIN ? ~0ull : 0ull;
      if (f.s1 >= 0) lt.state[f.s1][i] = 0;
    }
  }
  if (threadIdx.x == 0) s_fill = 0;
  __syncthreads();
  unsigned long long my_deferred = 0;
  for (int64_t i = row_lo + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < row_hi; i += (int64_t)gridDim.x * blockDim.x) {
    unsigned long long s;
    bool is_null = gk.nulls && !bit_not_null(gk.nulls, i);
    bool defer = false;
    if (is_null) s = LS;
    else {
      long long k;
      if (gk.kind == GK_I64) k = reinterpret_cast<const long long*>(gk.data)[i];
      else { double d = reinterpret_cast<const double*>(gk.data)[i]; if (d == 0) d = 0; k = __double_as_longlong(d); }
      if (k == kEmptyKey) s = LS + 1;
      else {
        s = slot32(mix64((uint64_t)k), (uint32_t)LS);
        for (;;) {
          long long cur = *reinterpret_cast<volatile long long*>(&lt.keys[s]);
          if (cur == k) break;
          if (cur == kEmptyKey) {
            unsigned int f = atomicAdd(&s_fill, 1u);
            if (f >= max_local_fill) { atomicSub(&s_fill, 1u); defer = true; break; }
            unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long*>(&lt.keys[s]), (unsigned long long)kEmptyKey, (unsigned long long)k);
            if (old == (unsigned long long)kEmptyKey) break;
            atomicSub(&s_fill, 1u);
            if (old == (unsigned long long)k) break;
          }
          if (++s == (unsigned long long)LS) s = 0;
        }
      }
    }
    if (defer) { atomicOr(&deferred[i >> 5], 1u << (i & 31)); my_deferred++; continue; }
    agg_apply(lt, spec, cols, i, s);
  }
  for (int o = 16; o; o >>= 1) my_deferred += __shfl_xor_sync(0xffffffffu, my_deferred, o);
  if ((threadIdx.x & 31) == 0 && my_deferred) atomicAdd(n_deferred, my_deferred);
  __syncthreads();
  // emit the partial results of this CTA
  for (int i = threadIdx.x; i < NT; i += blockDim.x) {
    bool occ = i < LS ? lt.keys[i] != kEmptyKey : lt.rows[i] != 0;
    if (!occ) continue;
    unsigned long long o = atomicAdd(out.count, 1ull);
    out.keys[o] = i < LS ? lt.keys[i] : 0;
    out.kind[o] = i < LS ? 0 : (i == LS ? 1 : 2);
    out.rows[o] = lt.rows[i];
    for (int s = 0; s < nstates; s++) out.state[s][o] = lt.state[s][i];
  }
}

// fold partial results into the global table; same deferral protocol as k_agg_update
__global__ void __launch_bounds__(256)
k_agg_merge(AggPartials in, int64_t m, AggTable t, AggSpec spec, unsigned long long max_fill, unsigned long long* fill,
            uint32_t* deferred, const uint32_t* only, unsigned long long* n_deferred) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < m; i += stride) {
    if (only && !((only[i >> 5] >> (i & 31)) & 1u)) continue;
    unsigned long long s;
    if (in.kind[i] == 1) s = t.nslots;
    else if (in.kind[i] == 2) s = t.nslots + 1;
    else {
      long long k = in.keys[i];
      s = slot_of(mix64((uint64_t)k), t.nslots);
      bool defer = false;
      unsigned int steps = 0;
      for (;;) {
        long long cur = *reinterpret_cast<volatile long long*>(&t.keys[s]);
        if (cur == k) break;
        if (cur == kEmptyKey) {
          unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long*>(&t.keys[s]), (unsigned long long)kEmptyKey, (unsigned long long)k);
          if (old == (unsigned long long)kEmptyKey || old == (unsigned long long)k) break;
        }
        if (++steps > (unsigned int)max_fill) { defer = true; break; }
        if (++s == t.nslots) s = 0;
      }
      if (defer) { atomicOr(&deferred[i >> 5], 1u << (i & 31)); atomicAdd(n_deferred, 1ull); continue; }
    }
    atomicAdd(&t.rows[s], in.rows[i]);
    for (int k = 0; k < spec.n; k++) {
      const AggFuncDev& f = spec.f[k];
      if (f.s0 >= 0) {
        unsigned long long v = in.state[f.s0][i];
        switch (f.name) {
          case TG_AGG_COUNT: atomicAdd(&t.state[f.s0][s], v); break;                                                  // countPartial merge func_count.go:481
          case TG_AGG_SUM: case TG_AGG_AVG: atomicAdd(reinterpret_cast<double*>(&t.state[f.s0][s]), __longlong_as_double((long long)v)); break;   // func_sum.go:106, func_avg.go:444
          case TG_AGG_MIN: atomicMin(&t.state[f.s0][s], v); break;
          case TG_AGG_MAX: atomicMax(&t.state[f.s0][s], v); break;
          default: break;
        }
      }
      if (f.s1 >= 0) atomicAdd(&t.state[f.s1][s], in.state[f.s1][i]);
    }
  }
}

// re-insert every group of an old table into a bigger one (no atomics on the states: keys are unique)
__global__ void k_agg_rehash(AggTable oldt, AggTable newt, AggSpec spec, int nstates, unsigned long long* fill) {
  unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
  unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  for (; i < oldt.nslots + 2; i += stride) {
    unsigned long long s;
    if (i >= oldt.nslots) { if (oldt.rows[i] == 0) continue; s = newt.nslots + (i - oldt.nslots); }
    else {
      long long k = oldt.keys[i];
      if (k == kEmptyKey) continue;
      s = slot_of(mix64((uint64_t)k), newt.nslots);
      for (;;) {
        unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long*>(&newt.keys[s]), (unsigned long long)kEmptyKey, (unsigned long long)k);
        if (old == (unsigned long long)kEmptyKey) break;
        if (++s == newt.nslots) s = 0;
      }
    }
    newt.rows[s] = oldt.rows[i];
    for (int a = 0; a < nstates; a++) newt.state[a][s] = oldt.state[a][i];
  }
}

// number of occupied slots (distinct groups), for sizing the result columns
__global__ void k_agg_count(AggTable t, unsigned long long* count) {
  unsigned long long n_total = t.nslots + 2;
  unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
  unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  unsigned long long c = 0;
  for (; i < n_total; i += stride) c += i < t.nslots ? (t.nkw ? t.tags[(size_t)i * t.stride] != 0 : t.keys[i] != kEmptyKey) : (t.rows[(size_t)i * t.stride] != 0);
  for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(count, c);
}

struct AggOut { void* data[TG_MAX_AGG]; uint8_t* valid[TG_MAX_AGG]; };

// compact the occupied slots into the result columns (Go-map iteration order is unspecified in the
// reference too; here it is slot order within warps, warp order by the atomic cursor)
__global__ void __launch_bounds__(256)
k_agg_finalize(AggTable t, AggSpec spec, int gk_kind, AggOut out, unsigned long long* cursor) {
  unsigned long long n_total = t.nslots + 2;
  unsigned long long base = blockIdx.x * (unsigned long long)blockDim.x;
  unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  const int lane = threadIdx.x & 31;
  for (; base < n_total; base += stride) {
    unsigned long long i = base + threadIdx.x;
    bool occ = false;
    if (i < t.nslots) occ = t.nkw ? t.tags[(size_t)i * t.stride] != 0 : t.keys[i] != kEmptyKey;
    else if (i < n_total) occ = t.rows[(size_t)i * t.stride] != 0;
    unsigned b = __ballot_sync(0xffffffffu, occ);
    // one cursor atomic per CTA iteration (256 slots), not per warp: a 29 M-slot table (Q3) would otherwise put 0.9 M atomics on
    // one address
    __shared__ uint32_t s_wcnt[8];
    __shared__ unsigned long long s_cbase;
    const int warp = threadIdx.x >> 5;
    if (lane == 0) s_wcnt[warp] = __popc(b);
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t tot = 0;
      for (int w = 0; w < 8; w++) tot += s_wcnt[w];
      s_cbase = tot ? atomicAdd(cursor, (unsigned long long)tot) : 0ull;
    }
    __syncthreads();
    unsigned long long wbase = s_cbase;
    for (int w = 0; w < warp; w++) wbase += s_wcnt[w];
    __syncthreads();   // s_wcnt / s_cbase are rewritten by the next iteration
    if (!occ) continue;
    unsigned long long o = wbase + __popc(b & ((1u << lane) - 1));
    unsigned long long rows = t.rows[(size_t)i * t.stride];
    for (int k = 0; k < spec.n; k++) {
      const AggFuncDev& f = spec.f[k];
      unsigned long long nn = f.s1 >= 0 ? t.state[f.s1][(size_t)i * t.stride] : rows;   // non-NULL inputs seen
      bool valid = true;
      unsigned long long v = 0;
      switch (f.name) {
        case TG_AGG_COUNT: v = (f.arg_col < 0 || f.s0 < 0) ? rows : t.state[f.s0][(size_t)i * t.stride]; break;
        case TG_AGG_SUM: valid = nn != 0; v = t.state[f.s0][(size_t)i * t.stride]; break;   // NULL when no non-NULL input (func_sum.go:80)
        case TG_AGG_AVG:
          valid = nn != 0;
          if (valid) v = (unsigned long long)__double_as_longlong(__longlong_as_double((long long)t.state[f.s0][(size_t)i * t.stride]) / (double)nn);   // func_avg.go:332
          break;
        case TG_AGG_MIN: case TG_AGG_MAX: {
          valid = nn != 0;
          unsigned long long u = t.state[f.s0][(size_t)i * t.stride];
          if (f.is_real) v = (unsigned long long)__double_as_longlong(ordered_to_f64(u));
          else if (f.is_unsigned) v = u;
          else v = u ^ 0x8000000000000000ull;
          break;
        }
        default:   // FIRSTROW(group column): the group key itself (firstRow4Int func_first_row.go:140)
          if (t.nkw) {   // f.arg_col2 = index of the column among the GROUP BY items | word with the NULL bits << 8 (0 = none)
            const int g = f.arg_col2 & 0xff, nullword = (f.arg_col2 >> 8) & 0xff;
            if (nullword && ((unsigned long long)t.keyw[nullword][(size_t)i * t.stride] >> g) & 1ull) valid = false;
            else v = (unsigned long long)t.keyw[g][(size_t)i * t.stride];
          }
          else if (i == t.nslots) valid = false;                       // NULL group
          else if (i == t.nslots + 1) v = (unsigned long long)kEmptyKey;
          else v = (unsigned long long)t.keys[i];
          (void)gk_kind;
          break;
      }
      reinterpret_cast<unsigned long long*>(out.data[k])[o] = valid ? v : 0ull;
      if (out.valid[k]) out.valid[k][o] = valid ? 1 : 0;
    }
  }
}

__global__ void k_pack_bitmap_agg(const uint8_t* __restrict__ valid, int64_t n, uint8_t* __restrict__ bitmap) {
  int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t nbytes = (n + 7) / 8;
  for (; b < nbytes; b += stride) {
    uint8_t v = 0;
    for (int j = 0; j < 8; j++) { int64_t r = b * 8 + j; if (r < n && valid[r]) v |= (uint8_t)(1u << j); }
    bitmap[b] = v;
  }
}


// ---- several GROUP BY columns: tag-claimed slots, global table only -------------------------------------------------
struct KeyWords { long long w[TG_MAX_GROUP_COLS + 1]; };
__device__ __forceinline__ unsigned long long hash_words(const KeyWords& k, int nkw) {
  unsigned long long h = hash64((unsigned long long)k.w[0]);
  for (int j = 1; j < nkw; j++) h = hash64(h ^ ((unsigned long long)k.w[j] * 0xD6E8FEB86659FD93ull + (unsigned long long)j));
  return h;
}
__device__ __forceinline__ void load_key_words(const GroupKeys& gk, int64_t i, KeyWords& k) {
  unsigned long long nullbits = 0;
  for (int j = 0; j < gk.n; j++) {
    long long v = 0;
    if (gk.nulls[j] && !bit_not_null(gk.nulls[j], i)) nullbits |= 1ull << j;
    else {
      v = __ldcs(reinterpret_cast<const long long*>(gk.data[j]) + i);
      if (gk.kind[j] == GK_F64) { double d = __longlong_as_double(v); if (d == 0) d = 0; v = __double_as_longlong(d); }
    }
    k.w[j] = v;
  }
  if (gk.nkw > gk.n) k.w[gk.n] = (long long)nullbits;
}
// find-or-insert; returns the slot or ~0 when the probe sequence is longer than max_probe (overfull: defer)
__device__ __forceinline__ unsigned long long mk_find_or_insert(const AggTable& t, const KeyWords& k, unsigned long long h, uint32_t max_probe) {
  const unsigned long long ready = h | 3ull, busy = (h & ~3ull) | 1ull;
  uint32_t s = slot32(h, (uint32_t)t.nslots), steps = 0;
  for (;;) {
    // tag and the first three key words sit in the record's first 32 bytes: ONE L2-coherent 256-bit load (records are 32-byte aligned)
    unsigned long long cur, k0, k1, k2;
    asm volatile("ld.global.cg.v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(cur), "=l"(k0), "=l"(k1), "=l"(k2) : "l"(&t.tags[(size_t)s * t.stride]) : "memory");
    if (cur == 0) {
      cur = atomicCAS(&t.tags[(size_t)s * t.stride], 0ull, busy);
      if (cur == 0) {
        for (int j = 0; j < t.nkw; j++) t.keyw[j][(size_t)s * t.stride] = k.w[j];
        __threadfence();
        *reinterpret_cast<volatile unsigned long long*>(&t.tags[(size_t)s * t.stride]) = ready;   // publish
        return s;
      }
    }
    if ((cur | 2ull) == ready) {
      bool eq = cur == ready && (unsigned long long)k.w[0] == k0 && (t.nkw < 2 || (unsigned long long)k.w[1] == k1) && (t.nkw < 3 || (unsigned long long)k.w[2] == k2);
      if (eq && t.nkw > 3) eq = *reinterpret_cast<volatile long long*>(&t.keyw[3][(size_t)s * t.stride]) == k.w[3];
      if (!eq) {   // still being written, or the vector load raced with the writer, or a different key with the same hash: settle it with ordered loads
        while (cur != ready) cur = *reinterpret_cast<volatile unsigned long long*>(&t.tags[(size_t)s * t.stride]);
        eq = true;
        for (int j = 0; j < t.nkw; j++) eq &= *reinterpret_cast<volatile long long*>(&t.keyw[j][(size_t)s * t.stride]) == k.w[j];
      }
      if (eq) return s;
    }
    if (++steps > max_probe) return ~0ull;
    if (++s == (uint32_t)t.nslots) s = 0;
  }
}

__global__ void __launch_bounds__(256)
k_agg_update_mk(GroupKeys gk, DevCols cols, int64_t n, AggTable t, AggSpec spec, uint32_t max_probe,
                uint32_t* deferred, const uint32_t* only, unsigned long long* n_deferred) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  unsigned long long my_deferred = 0;
  for (; i < n; i += stride) {
    if (only && !((only[i >> 5] >> (i & 31)) & 1u)) continue;
    KeyWords k;
    load_key_words(gk, i, k);
    const unsigned long long s = mk_find_or_insert(t, k, hash_words(k, t.nkw), max_probe);
    if (s == ~0ull) { atomicOr(&deferred[i >> 5], 1u << (i & 31)); my_deferred++; continue; }
    agg_apply(t, spec, cols, i, s);
  }
  for (int o = 16; o; o >>= 1) my_deferred += __shfl_xor_sync(0xffffffffu, my_deferred, o);
  if ((threadIdx.x & 31) == 0 && my_deferred) atomicAdd(n_deferred, my_deferred);
}

// re-insert every group of an old multi-key table into a bigger one (keys are distinct: claim with the published tag)
__global__ void k_agg_rehash_mk(AggTable oldt, AggTable newt, int nstates) {
  unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  for (; i < oldt.nslots; i += stride) {
    const unsigned long long tag = oldt.tags[(size_t)i * oldt.stride];
    if (tag == 0) continue;
    uint32_t s = slot32(tag, (uint32_t)newt.nslots);
    for (;;) {
      if (atomicCAS(&newt.tags[(size_t)s * newt.stride], 0ull, tag) == 0ull) break;
      if (++s == (uint32_t)newt.nslots) s = 0;
    }
    for (int j = 0; j < oldt.nkw; j++) newt.keyw[j][(size_t)s * newt.stride] = oldt.keyw[j][(size_t)i * oldt.stride];
    newt.rows[(size_t)s * newt.stride] = oldt.rows[(size_t)i * oldt.stride];
    for (int a = 0; a < nstates; a++) newt.state[a][(size_t)s * newt.stride] = oldt.state[a][(size_t)i * oldt.stride];
  }
}

}  // namespace tg
#include "agg_update.cuh"
namespace tg {

}  // namespace tg

using namespace tg;

struct AggImpl;

// shell + implementation, like tg_join (join.cu): close frees the implementation, the shell stays readable
struct tg_agg {
  std::mutex mu;
  std::atomic<bool> closed{false};
  AggImpl* impl = nullptr;
};

struct AggImpl {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  int nsm = 148;

  int ncols = 0;
  std::vector<int> types, elem;
  std::vector<uint32_t> flags;
  std::vector<char> needed;
  int group_col = -1;          // -1: no GROUP BY (several GROUP BY columns: the first one)
  int gk_kind = GK_NONE;
  std::vector<int> group_cols, group_kinds;   // all GROUP BY columns
  int nkw = 0;                 // > 0: multi-key table (key words per slot)
  AggSpec spec{};
  int nstates = 0;
  std::vector<char> out_nullable;

  // table
  DevBuf tbl_mem;
  AggTable tbl{};
  unsigned long long nslots = 0;
  DevBuf scalars;              // [0] fill [1] n_deferred [2] out cursor
  DevBuf deferred, partials_mem;
  int64_t expected_groups = 0;
  int local_mode = -1;            // -1 undecided, 0 global atomics only, 1 CTA-local partial aggregation first

  // staging
  ColumnStage stage;
  std::vector<std::unique_ptr<DevBuf>> dcols, dnulls;

  // result
  bool finished = false;
  std::vector<std::unique_ptr<DevBuf>> out_cols, out_valid, out_bitmaps;
  int64_t out_rows = 0, consumed = 0;
  tg_agg_stats stats{};
};

namespace tg {

static int agrid(const AggImpl* a, int64_t n, int block = 256, int per_sm = 8) {
  int64_t need = (n + block - 1) / block, cap = (int64_t)a->nsm * per_sm;
  if (need < 1) need = 1;
  return (int)(need < cap ? need : cap);
}

static int agg_setup(AggImpl* a, const tg_agg_desc* d) {
  if (!d) return fail(TG_ERR_INVALID, "desc is NULL");
  if (d->n_cols <= 0 || d->n_cols > TG_MAX_COLS) return fail(TG_ERR_UNSUPPORTED, "child schema must have 1..16 columns");
  a->ncols = d->n_cols;
  a->types.assign(d->col_types, d->col_types + d->n_cols);
  a->flags.resize(d->n_cols);
  for (int i = 0; i < d->n_cols; i++) a->flags[i] = d->col_flags ? d->col_flags[i] : 0;
  a->elem.resize(d->n_cols);
  for (int i = 0; i < d->n_cols; i++) a->elem[i] = fixed_len(a->types[i]);
  a->needed.assign(d->n_cols, 0);
  if (d->n_group_by > TG_MAX_GROUP_COLS) return fail(TG_ERR_UNSUPPORTED, "GPU hash aggregation handles up to 4 GROUP BY columns");
  a->group_col = -1; a->gk_kind = GK_NONE; a->nkw = 0;
  a->group_cols.clear(); a->group_kinds.clear();
  bool any_nullable = false;
  for (int q = 0; q < d->n_group_by; q++) {
    int g = d->group_by_cols[q];
    if (g < 0 || g >= a->ncols) return fail(TG_ERR_INVALID, "group-by column out of range");
    int kind;
    if (is_int_family(a->types[g])) kind = GK_I64;
    else if (a->types[g] == TG_TYPE_DOUBLE) kind = GK_F64;
    else return fail(TG_ERR_UNSUPPORTED, "GROUP BY column type is not offloaded (int family / double only)");
    if (a->elem[g] != 8) return fail(TG_ERR_UNSUPPORTED, "GROUP BY columns must be 8-byte columns");
    if (q == 0) { a->group_col = g; a->gk_kind = kind; }
    a->group_cols.push_back(g); a->group_kinds.push_back(kind);
    any_nullable |= !(a->flags[g] & TG_FLAG_NOT_NULL);
    a->needed[g] = 1;
  }
  if (d->n_group_by > 1) a->nkw = d->n_group_by + (any_nullable ? 1 : 0);
  if (d->n_funcs <= 0 || d->n_funcs > TG_MAX_AGG) return fail(TG_ERR_UNSUPPORTED, "1..12 aggregate functions are offloaded");
  a->spec.n = d->n_funcs;
  a->nstates = 0;
  a->out_nullable.assign(d->n_funcs, 0);
  for (int k = 0; k < d->n_funcs; k++) {
    const tg_agg_func& f = d->funcs[k];
    AggFuncDev& o = a->spec.f[k];
    o = AggFuncDev{f.name, f.arg_col, 0, 0, -1, -1, 0, f.arg_col2, f.arg_expr, 0, f.arg_const};
    if (f.arg_expr != TG_ARGEXPR_COL) {
      if (f.arg_expr != TG_ARGEXPR_MUL && f.arg_expr != TG_ARGEXPR_MUL_CSUB) return fail(TG_ERR_INVALID, "unknown aggregate argument expression");
      if ((f.name != TG_AGG_SUM && f.name != TG_AGG_AVG) || f.mode != TG_AGGMODE_COMPLETE)
        return fail(TG_ERR_UNSUPPORTED, "argument expressions are fused for SUM / AVG in Complete mode only");
      if (f.arg_col < 0 || f.arg_col2 < 0 || f.arg_col2 >= d->n_cols || a->types[f.arg_col] != TG_TYPE_DOUBLE || a->types[f.arg_col2] != TG_TYPE_DOUBLE)
        return fail(TG_ERR_UNSUPPORTED, "argument expressions take two DOUBLE columns");
      a->needed[f.arg_col2] = 1;
    }
    if (f.mode != TG_AGGMODE_COMPLETE && f.mode != TG_AGGMODE_FINAL) return fail(TG_ERR_UNSUPPORTED, "only Complete and Final aggregate modes are offloaded");
    o.final_mode = f.mode == TG_AGGMODE_FINAL;
    if (f.arg_col >= a->ncols || f.arg_col2 >= a->ncols) return fail(TG_ERR_INVALID, "aggregate argument column out of range");
    bool arg_nullable = f.arg_col >= 0 && !(a->flags[f.arg_col] & TG_FLAG_NOT_NULL);
    if (f.arg_expr != TG_ARGEXPR_COL && f.arg_col2 >= 0 && f.arg_col2 < d->n_cols && !(a->flags[f.arg_col2] & TG_FLAG_NOT_NULL)) arg_nullable = true;
    if (f.arg_col >= 0) { if (a->elem[f.arg_col] != 8) return fail(TG_ERR_UNSUPPORTED, "aggregate arguments must be 8-byte columns"); a->needed[f.arg_col] = 1; }
    int atype = f.arg_col >= 0 ? a->types[f.arg_col] : TG_TYPE_LONGLONG;
    o.is_real = atype == TG_TYPE_DOUBLE;
    o.is_unsigned = f.arg_col >= 0 && (a->flags[f.arg_col] & TG_FLAG_UNSIGNED) != 0;
    switch (f.name) {
      case TG_AGG_COUNT:
        if (o.final_mode) { if (f.arg_col < 0) return fail(TG_ERR_INVALID, "final COUNT needs the partial count column"); o.s0 = a->nstates++; }
        else if (f.arg_col >= 0 && arg_nullable) o.s0 = a->nstates++;   // NOT NULL COUNT(x) == COUNT(*) == rows[]
        break;
      case TG_AGG_SUM:
        // SUM(int) yields DECIMAL in TiDB (aggregation/base_func.go:223-245): not offloaded
        if (f.arg_col < 0 || atype != TG_TYPE_DOUBLE) return fail(TG_ERR_UNSUPPORTED, "SUM is offloaded for DOUBLE arguments only (SUM(int) is DECIMAL)");
        o.s0 = a->nstates++;
        if (arg_nullable) o.s1 = a->nstates++;
        a->out_nullable[k] = 1;
        break;
      case TG_AGG_AVG:
        if (o.final_mode) {
          if (f.arg_col < 0 || f.arg_col2 < 0 || a->types[f.arg_col2] != TG_TYPE_DOUBLE || !is_int_family(a->types[f.arg_col]))
            return fail(TG_ERR_UNSUPPORTED, "final AVG takes (count BIGINT, sum DOUBLE)");
          a->needed[f.arg_col2] = 1;
          o.s0 = a->nstates++; o.s1 = a->nstates++;
        } else {
          if (f.arg_col < 0 || atype != TG_TYPE_DOUBLE) return fail(TG_ERR_UNSUPPORTED, "AVG is offloaded for DOUBLE arguments only");
          o.s0 = a->nstates++;
          if (arg_nullable) o.s1 = a->nstates++;
        }
        a->out_nullable[k] = 1;
        break;
      case TG_AGG_MIN: case TG_AGG_MAX:
        if (f.arg_col < 0 || !(is_int_family(atype) || atype == TG_TYPE_DOUBLE)) return fail(TG_ERR_UNSUPPORTED, "MIN/MAX are offloaded for int family / DOUBLE");
        o.s0 = a->nstates++;
        if (arg_nullable) o.s1 = a->nstates++;
        a->out_nullable[k] = 1;
        break;
      case TG_AGG_FIRSTROW: {
        int gi = -1;
        for (size_t q = 0; q < a->group_cols.size(); q++) if (a->group_cols[q] == f.arg_col) gi = (int)q;
        if (f.arg_col < 0 || gi < 0) return fail(TG_ERR_UNSUPPORTED, "FIRSTROW is offloaded only for GROUP BY columns (deterministic)");
        a->out_nullable[k] = !(a->flags[f.arg_col] & TG_FLAG_NOT_NULL);
        o.arg_col2 = gi | ((a->nkw > (int)a->group_cols.size() ? (int)a->group_cols.size() : 0) << 8);
        break;
      }
      default: return fail(TG_ERR_UNSUPPORTED, "aggregate function is not offloaded");
    }
  }
  a->device = d->device;
  a->expected_groups = d->expected_groups;
  return TG_OK;
}

static int table_record_words(const AggImpl* a) { return a->nkw ? ((1 + a->nkw + 1 + a->nstates + 3) / 4) * 4 : (2 + a->nstates); }
static void layout_table(AggImpl* a, uint8_t* mem, unsigned long long nslots, AggTable& t) {
  size_t n = (size_t)nslots + 2;
  t.nslots = nslots;
  t.nkw = a->nkw;
  if (a->nkw) {   // array of records: [tag | nkw key words | rows | states], padded to a multiple of 32 bytes
    unsigned long long* w = reinterpret_cast<unsigned long long*>(mem);
    t.stride = (uint32_t)table_record_words(a);
    t.tags = w; t.keys = reinterpret_cast<long long*>(w);
    for (int j = 0; j < a->nkw; j++) t.keyw[j] = reinterpret_cast<long long*>(w + 1 + j);
    t.rows = w + 1 + a->nkw;
    for (int s = 0; s < a->nstates; s++) t.state[s] = w + 2 + a->nkw + s;
    return;
  }
  t.stride = 1;
  t.keys = reinterpret_cast<long long*>(mem);
  t.tags = reinterpret_cast<unsigned long long*>(mem);
  t.rows = reinterpret_cast<unsigned long long*>(mem + n * 8);
  for (int s = 0; s < a->nstates; s++) t.state[s] = reinterpret_cast<unsigned long long*>(mem + n * 8 * (2 + s));
}

static int alloc_table(AggImpl* a, unsigned long long nslots, DevBuf& mem, AggTable& t) {
  size_t n = (size_t)nslots + 2;
  TG_TRY(mem.ensure(a->device, n * 8 * (size_t)table_record_words(a) + 64));
  layout_table(a, mem.as<uint8_t>(), nslots, t);
  k_agg_init<<<agrid(a, (int64_t)n), 256, 0, a->stream>>>(t, a->spec, n);
  a->stats.kernel_launches++;
  return TG_OK;
}

static int grow_table(AggImpl* a, unsigned long long want_slots) {
  std::unique_ptr<DevBuf> nm(new DevBuf());
  AggTable nt{};
  TG_TRY(alloc_table(a, want_slots, *nm, nt));
  unsigned long long* sc = a->scalars.as<unsigned long long>();
  TG_CUDA(cudaMemsetAsync(sc, 0, 8, a->stream));
  if (a->nkw) k_agg_rehash_mk<<<agrid(a, (int64_t)a->tbl.nslots), 256, 0, a->stream>>>(a->tbl, nt, a->nstates);
  else k_agg_rehash<<<agrid(a, (int64_t)a->tbl.nslots + 2), 256, 0, a->stream>>>(a->tbl, nt, a->spec, a->nstates, sc);
  a->stats.kernel_launches++;
  TG_CUDA(cudaStreamSynchronize(a->stream));
  std::swap(a->tbl_mem.p, nm->p); std::swap(a->tbl_mem.cap, nm->cap); std::swap(a->tbl_mem.device, nm->device);
  a->tbl = nt;
  a->nslots = want_slots;
  return TG_OK;
}

__global__ void k_mark_range(uint32_t* bits, int64_t lo, int64_t hi) {
  int64_t i = lo + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < hi; i += stride) atomicOr(&bits[i >> 5], 1u << (i & 31));
}
static int mark_range_deferred(AggImpl* a, int64_t lo, int64_t hi) {
  // whole 32-bit words with memset, ragged edges with a tiny kernel
  int64_t wlo = (lo + 31) / 32, whi = hi / 32;
  uint32_t* bits = a->deferred.as<uint32_t>();
  if (whi > wlo) TG_CUDA(cudaMemsetAsync(bits + wlo, 0xff, (size_t)(whi - wlo) * 4, a->stream));
  int64_t e1 = std::min<int64_t>(hi, wlo * 32);
  if (lo < e1) { k_mark_range<<<1, 64, 0, a->stream>>>(bits, lo, e1); a->stats.kernel_launches++; }
  int64_t s2 = std::max<int64_t>(std::max<int64_t>(lo, e1), whi * 32);
  if (s2 < hi) { k_mark_range<<<1, 64, 0, a->stream>>>(bits, s2, hi); a->stats.kernel_launches++; }
  return TG_OK;
}

// fold `m` partial-result tuples into the global table, growing it until every tuple found a slot
static int grow_table(AggImpl* a, unsigned long long want_slots);
static int merge_partials(AggImpl* a, const AggPartials& pp, unsigned long long m, unsigned long long* sc) {
  if (m == 0) return TG_OK;
  DevBuf mdef, mprev;
  size_t dwords = (size_t)((m + 31) / 32);
  TG_TRY(mdef.ensure(a->device, dwords * 4 + 16));
  TG_CUDA(cudaMemsetAsync(mdef.p, 0, dwords * 4, a->stream));
  TG_CUDA(cudaMemsetAsync(sc + 4, 0, 8, a->stream));
  const uint32_t* only = nullptr;
  for (int round = 0; round < 40; round++) {
    unsigned long long max_fill = 48;   // probe-length limit (see k_agg_update)
    k_agg_merge<<<agrid(a, (int64_t)m), 256, 0, a->stream>>>(pp, (int64_t)m, a->tbl, a->spec, max_fill, sc, mdef.as<uint32_t>(), only, sc + 4);
    a->stats.kernel_launches++;
    unsigned long long nd = 0;
    TG_CUDA(cudaMemcpyAsync(&nd, sc + 4, 8, cudaMemcpyDeviceToHost, a->stream));
    TG_CUDA(cudaStreamSynchronize(a->stream));
    if (nd == 0) break;
    unsigned long long want = std::max<unsigned long long>(a->nslots * 4, (unsigned long long)((a->nslots * 0.6 + (double)nd) * 2));
    TG_TRY(grow_table(a, want));
    TG_TRY(mprev.ensure(a->device, dwords * 4 + 16));
    TG_CUDA(cudaMemcpyAsync(mprev.p, mdef.p, dwords * 4, cudaMemcpyDeviceToDevice, a->stream));
    TG_CUDA(cudaMemsetAsync(mdef.p, 0, dwords * 4, a->stream));
    TG_CUDA(cudaMemsetAsync(sc + 4, 0, 8, a->stream));
    only = mprev.as<uint32_t>();
    if (round == 39) return fail(TG_ERR_CUDA, "internal: aggregation merge failed to converge");
  }
  return TG_OK;
}

static void layout_partials(uint8_t* base, size_t cap, int nstates, unsigned long long* count, AggPartials& pp) {
  pp.keys = reinterpret_cast<long long*>(base); base += cap * 8;
  pp.rows = reinterpret_cast<unsigned long long*>(base); base += cap * 8;
  for (int s = 0; s < nstates; s++) { pp.state[s] = reinterpret_cast<unsigned long long*>(base); base += cap * 8; }
  pp.kind = base;
  pp.count = count;
}

// several GROUP BY columns: global tag-claimed table only (k_agg_update_mk), same grow-and-retry protocol
static int update_grouped_mk(AggImpl* a, const DevCols& cols, int64_t n, unsigned long long* sc) {
  size_t dwords = (size_t)((n + 31) / 32);
  TG_TRY(a->deferred.ensure(a->device, dwords * 4 + 16));
  TG_CUDA(cudaMemsetAsync(a->deferred.p, 0, dwords * 4, a->stream));
  GroupKeys gk{};
  gk.n = (int)a->group_cols.size(); gk.nkw = a->nkw;
  for (int q = 0; q < gk.n; q++) { gk.data[q] = cols.data[a->group_cols[q]]; gk.nulls[q] = cols.nulls[a->group_cols[q]]; gk.kind[q] = a->group_kinds[q]; }
  DevBuf prev_deferred;
  const uint32_t* only = nullptr;
  for (int round = 0; round < 40; round++) {
    TG_CUDA(cudaMemsetAsync(sc + 1, 0, 8, a->stream));
    k_agg_update_mk<<<agrid(a, n), 256, 0, a->stream>>>(gk, cols, n, a->tbl, a->spec, 48u, a->deferred.as<uint32_t>(), only, sc + 1);
    a->stats.kernel_launches++;
    unsigned long long nd = 0;
    TG_CUDA(cudaMemcpyAsync(&nd, sc + 1, 8, cudaMemcpyDeviceToHost, a->stream));
    TG_CUDA(cudaStreamSynchronize(a->stream));
    if (nd == 0) break;
    unsigned long long want = std::max<unsigned long long>(a->nslots * 4, (unsigned long long)((a->nslots * 0.6 + (double)nd) * 2));
    TG_TRY(grow_table(a, want));
    TG_TRY(prev_deferred.ensure(a->device, dwords * 4 + 16));
    TG_CUDA(cudaMemcpyAsync(prev_deferred.p, a->deferred.p, dwords * 4, cudaMemcpyDeviceToDevice, a->stream));
    TG_CUDA(cudaMemsetAsync(a->deferred.p, 0, dwords * 4, a->stream));
    only = prev_deferred.as<uint32_t>();
    if (round == 39) return fail(TG_ERR_CUDA, "internal: aggregation table failed to converge");
  }
  return TG_OK;
}

// Round-2 update path (agg_update.cuh): one two-level kernel per round; rows / local groups that found no slot are re-run
// after the table has grown.
static int update_grouped_v2(AggImpl* a, const GroupKey& gk, const DevCols& cols, int64_t n, unsigned long long* sc) {
  size_t dwords = (size_t)((n + 31) / 32);
  TG_TRY(a->deferred.ensure(a->device, dwords * 4 + 16));
  TG_CUDA(cudaMemsetAsync(a->deferred.p, 0, dwords * 4, a->stream));
  // CTA-local level: on for small / unknown cardinalities (a CTA turns it off by itself when its hit rate is low)
  static int env_local = -1, env_slots = 0;
  if (env_local < 0) { const char* e = getenv("TG_AGG_LOCAL"); env_local = e ? atoi(e) : 1; const char* s2 = getenv("TG_AGG_LOCAL_SLOTS"); env_slots = s2 ? atoi(s2) : 0; }
  bool local = env_local != 0 && a->nstates <= AGG_LOCAL_MAX_STATES && (a->expected_groups == 0 || a->expected_groups <= 4096);
  if (env_local == 2) local = a->nstates <= AGG_LOCAL_MAX_STATES;
  int local_slots = (env_slots == 512 || env_slots == 1024 || env_slots == 2048 || env_slots == 4096) ? env_slots : 2048;
  size_t smem = (size_t)(local_slots + 2) * 8 * (2 + a->nstates);
  while (local && smem > (100u << 10) && local_slots > 512) { local_slots /= 2; smem = (size_t)(local_slots + 2) * 8 * (2 + a->nstates); }
  int per_sm = local ? (int)std::max<size_t>(1, std::min<size_t>(4, (200u << 10) / smem)) : 8;
  int grid = (int)std::min<int64_t>((n + AGG2_TILE - 1) / AGG2_TILE, (int64_t)a->nsm * per_sm);
  if (grid < 1) grid = 1;
  Agg2Params p{};
  p.gk = gk; p.n = n; p.max_probe = 48; p.nstates = a->nstates; p.local_slots = local ? local_slots : 0;
  p.deferred = a->deferred.as<uint32_t>(); p.only = nullptr; p.n_deferred = sc + 1; p.local_rows = sc + 6;
  if (local) {
    p.spill_cap = (unsigned long long)grid * (size_t)(local_slots + 2);
    size_t per = 8 + 8 + 8 * (size_t)a->nstates + 1;
    TG_TRY(a->partials_mem.ensure(a->device, (size_t)p.spill_cap * per + 256));
    layout_partials(a->partials_mem.as<uint8_t>(), (size_t)p.spill_cap, a->nstates, sc + 5, p.spill);
    TG_CUDA(cudaFuncSetAttribute(k_agg_update2<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  DevBuf prev_deferred;
  for (int round = 0; round < 40; round++) {
    TG_CUDA(cudaMemsetAsync(sc + 1, 0, 8, a->stream));
    TG_CUDA(cudaMemsetAsync(sc + 5, 0, 8, a->stream));
    if (local && round == 0) k_agg_update2<true><<<grid, AGG2_BLOCK, smem, a->stream>>>(p, cols, a->tbl, a->spec);
    else k_agg_update2<false><<<grid, AGG2_BLOCK, 0, a->stream>>>(p, cols, a->tbl, a->spec);
    a->stats.kernel_launches++;
    unsigned long long back[8] = {0};
    TG_CUDA(cudaMemcpyAsync(back, sc, 64, cudaMemcpyDeviceToHost, a->stream));
    TG_CUDA(cudaStreamSynchronize(a->stream));
    const unsigned long long nd = back[1], spilled = (local && round == 0) ? back[5] : 0;
    if (nd == 0 && spilled == 0) break;
    if (spilled > p.spill_cap) return fail(TG_ERR_CUDA, "internal: aggregation spill buffer overflow");
    // grow x4 (at least enough for every deferred row / spilled group to be a new group), then re-run just those
    unsigned long long want = std::max<unsigned long long>(a->nslots * 4, (unsigned long long)((a->nslots * 0.6 + (double)(nd + spilled)) * 2));
    TG_TRY(grow_table(a, want));
    p.max_probe = 48;
    if (spilled) TG_TRY(merge_partials(a, p.spill, spilled, sc));
    if (nd == 0) break;
    TG_TRY(prev_deferred.ensure(a->device, dwords * 4 + 16));
    TG_CUDA(cudaMemcpyAsync(prev_deferred.p, a->deferred.p, dwords * 4, cudaMemcpyDeviceToDevice, a->stream));
    TG_CUDA(cudaMemsetAsync(a->deferred.p, 0, dwords * 4, a->stream));
    p.only = prev_deferred.as<uint32_t>();
    if (round == 39) return fail(TG_ERR_CUDA, "internal: aggregation table failed to converge");
  }
  return TG_OK;
}

// rows [lo, hi): CTA-local partial aggregation, then merge of the partial results into the global table
static int local_partial_pass(AggImpl* a, const GroupKey& gk, const DevCols& cols, int64_t lo, int64_t hi, unsigned long long* sc) {
  int local_slots = 1024;   // measured best on B200 (tools/bench_ops.py): bigger tables lose more to occupancy than they gain
  if (const char* e = getenv("TG_AGG_LOCAL_SLOTS")) { int v = atoi(e); if (v == 512 || v == 1024 || v == 2048 || v == 4096) local_slots = v; }
  size_t smem_per_cta = (size_t)(local_slots + 2) * 8 * (2 + a->nstates);
  int per_sm = (int)std::max<size_t>(1, std::min<size_t>(4, (200u << 10) / smem_per_cta));
  int grid = agrid(a, hi - lo, 256, per_sm);
  size_t cap = (size_t)grid * (local_slots / 2 + 2);
  size_t per = 8 /*keys*/ + 8 /*rows*/ + 8 * (size_t)a->nstates + 1 /*kind*/;
  TG_TRY(a->partials_mem.ensure(a->device, cap * per + 256));
  AggPartials pp{};
  uint8_t* base = a->partials_mem.as<uint8_t>();
  pp.keys = reinterpret_cast<long long*>(base); base += cap * 8;
  pp.rows = reinterpret_cast<unsigned long long*>(base); base += cap * 8;
  for (int s = 0; s < a->nstates; s++) { pp.state[s] = reinterpret_cast<unsigned long long*>(base); base += cap * 8; }
  pp.kind = base;
  pp.count = sc + 3;
  TG_CUDA(cudaMemsetAsync(sc + 3, 0, 8, a->stream));
  size_t smem = (size_t)(local_slots + 2) * 8 * (2 + a->nstates);
  TG_CUDA(cudaFuncSetAttribute(k_agg_update_local, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_agg_update_local<<<grid, 256, smem, a->stream>>>(gk, cols, lo, hi, a->spec, a->nstates, local_slots, pp, a->deferred.as<uint32_t>(), sc + 1);
  a->stats.kernel_launches++;
  unsigned long long m = 0;
  TG_CUDA(cudaMemcpyAsync(&m, sc + 3, 8, cudaMemcpyDeviceToHost, a->stream));
  TG_CUDA(cudaStreamSynchronize(a->stream));
  if (m == 0) return TG_OK;
  // merge with its own grow-and-retry loop (tuples, not rows)
  DevBuf mdef, mprev;
  size_t dwords = (size_t)((m + 31) / 32);
  TG_TRY(mdef.ensure(a->device, dwords * 4 + 16));
  TG_CUDA(cudaMemsetAsync(mdef.p, 0, dwords * 4, a->stream));
  TG_CUDA(cudaMemsetAsync(sc + 4, 0, 8, a->stream));
  const uint32_t* only = nullptr;
  for (int round = 0; round < 40; round++) {
    unsigned long long max_fill = 48;   // probe-length limit (see k_agg_update)
    k_agg_merge<<<agrid(a, (int64_t)m), 256, 0, a->stream>>>(pp, (int64_t)m, a->tbl, a->spec, max_fill, sc, mdef.as<uint32_t>(), only, sc + 4);
    a->stats.kernel_launches++;
    unsigned long long nd = 0;
    TG_CUDA(cudaMemcpyAsync(&nd, sc + 4, 8, cudaMemcpyDeviceToHost, a->stream));
    TG_CUDA(cudaStreamSynchronize(a->stream));
    if (nd == 0) break;
    unsigned long long want = std::max<unsigned long long>(a->nslots * 4, (unsigned long long)((a->nslots * 0.6 + (double)nd) * 2));
    TG_TRY(grow_table(a, want));
    TG_TRY(mprev.ensure(a->device, dwords * 4 + 16));
    TG_CUDA(cudaMemcpyAsync(mprev.p, mdef.p, dwords * 4, cudaMemcpyDeviceToDevice, a->stream));
    TG_CUDA(cudaMemsetAsync(mdef.p, 0, dwords * 4, a->stream));
    TG_CUDA(cudaMemsetAsync(sc + 4, 0, 8, a->stream));
    only = mprev.as<uint32_t>();
    if (round == 39) return fail(TG_ERR_CUDA, "internal: aggregation merge failed to converge");
  }
  return TG_OK;
}

// aggregate n device-resident rows
static int update_device_impl(AggImpl* a, const DevCols& cols, int64_t n) {
  if (n == 0) return TG_OK;
  a->stats.input_rows += n;
  TG_TRY(a->scalars.ensure(a->device, 64));
  unsigned long long* sc = a->scalars.as<unsigned long long>();
  a->spec.err = sc + 7;    // raised by a fused argument expression that left the DOUBLE range (types.ErrOverflow)
  if (a->nslots == 0) {
    unsigned long long want = 1024;
    if (a->group_col >= 0) {
      if (a->expected_groups > 0) want = std::max<unsigned long long>(1024, (unsigned long long)a->expected_groups * 2);
      else want = std::max<unsigned long long>(1024, (unsigned long long)std::min<int64_t>(n, 1ll << 22) * 2);
    }
    TG_CUDA(cudaMemsetAsync(sc, 0, 64, a->stream));
    TG_TRY(alloc_table(a, want, a->tbl_mem, a->tbl));
    a->nslots = want;
  }
  TG_CUDA(cudaEventRecord(a->ev0, a->stream));
  if (a->group_col < 0) {
    k_agg_update_nogroup<<<agrid(a, n, 256, 4), 256, 0, a->stream>>>(cols, n, a->tbl, a->spec);
    a->stats.kernel_launches++;
  } else {
    if (a->nkw) {
      TG_TRY(update_grouped_mk(a, cols, n, sc));
      TG_CUDA(cudaEventRecord(a->ev1, a->stream));
      TG_CUDA(cudaStreamSynchronize(a->stream));
      TG_CUDA(cudaGetLastError());
      float ms3 = 0; cudaEventElapsedTime(&ms3, a->ev0, a->ev1); a->stats.update_ms += ms3;
      return TG_OK;
    }
    GroupKey gk{cols.data[a->group_col], cols.nulls[a->group_col], a->gk_kind, 0};
    static int v1 = -1;
    if (v1 < 0) { const char* e = getenv("TG_AGG_V1"); v1 = e ? atoi(e) : 0; }
    if (!v1) {
      TG_TRY(update_grouped_v2(a, gk, cols, n, sc));
      TG_CUDA(cudaEventRecord(a->ev1, a->stream));
      TG_CUDA(cudaStreamSynchronize(a->stream));
      TG_CUDA(cudaGetLastError());
      float ms2 = 0; cudaEventElapsedTime(&ms2, a->ev0, a->ev1); a->stats.update_ms += ms2;
      return TG_OK;
    }
    size_t dwords = (size_t)((n + 31) / 32);
    TG_TRY(a->deferred.ensure(a->device, dwords * 4 + 16));
    TG_CUDA(cudaMemsetAsync(a->deferred.p, 0, dwords * 4, a->stream));
    TG_CUDA(cudaMemsetAsync(sc + 1, 0, 8, a->stream));
    bool have_deferred = false;
    // ---- phase 1 (low cardinality): CTA-local partial aggregation, decided on a 1M-row sample when there is no hint ----
    bool try_local = a->nstates <= AGG_LOCAL_MAX_STATES && a->local_mode != 0 &&
                     (a->local_mode == 1 || a->expected_groups == 0 || a->expected_groups <= 2 * AGG_LOCAL_SLOTS_MAX);
    if (try_local) {
      int64_t done = 0;
      while (done < n) {
        int64_t hi = (a->local_mode == 1) ? n : std::min<int64_t>(n, done + (1ll << 20));
        TG_TRY(local_partial_pass(a, gk, cols, done, hi, sc));
        unsigned long long nd = 0;
        TG_CUDA(cudaMemcpyAsync(&nd, sc + 1, 8, cudaMemcpyDeviceToHost, a->stream));
        TG_CUDA(cudaStreamSynchronize(a->stream));
        int64_t span = hi - done;
        done = hi;
        if (nd) have_deferred = true;
        // Keep the CTA-local phase while it absorbs a useful share of the rows.  Measured (profiles/r1_agg_notes.md): shared-memory
        // atomics (LSU) and L2 atomics are different engines; 1000 groups with half of the rows aggregated in shared memory and
        // half deferred to the L2 path take 2.7 ms, all-L2 5.0 ms, all-shared 9 ms.
        if (a->local_mode < 0) a->local_mode = (nd * 10 <= (unsigned long long)span * 7) ? 1 : 0;
        if (a->local_mode == 0) break;
      }
      if (done < n) {   // the rest of the batch goes through the global kernel: mark it "deferred"
        TG_TRY(mark_range_deferred(a, done, n));
        have_deferred = true;
      }
      TG_CUDA(cudaMemsetAsync(sc + 1, 0, 8, a->stream));
    }
    // ---- phase 2: global atomics on every row (or only the deferred ones), growing the table on demand ----
    if (!try_local || have_deferred) {
      DevBuf prev_deferred;
      const uint32_t* only = nullptr;
      if (try_local) {
        TG_TRY(prev_deferred.ensure(a->device, dwords * 4 + 16));
        TG_CUDA(cudaMemcpyAsync(prev_deferred.p, a->deferred.p, dwords * 4, cudaMemcpyDeviceToDevice, a->stream));
        TG_CUDA(cudaMemsetAsync(a->deferred.p, 0, dwords * 4, a->stream));
        only = prev_deferred.as<uint32_t>();
      }
      for (int round = 0; round < 40; round++) {
        unsigned long long max_fill = 48;   // probe-length limit (see k_agg_update)
        k_agg_update<<<agrid(a, n), 256, 0, a->stream>>>(gk, cols, n, a->tbl, a->spec, max_fill, sc, a->deferred.as<uint32_t>(), only, sc + 1);
        a->stats.kernel_launches++;
        unsigned long long nd = 0;
        TG_CUDA(cudaMemcpyAsync(&nd, sc + 1, 8, cudaMemcpyDeviceToHost, a->stream));
        TG_CUDA(cudaStreamSynchronize(a->stream));
        if (nd == 0) break;
        // grow x4 (at least enough for every deferred row to be a new group), re-run only the deferred rows
        unsigned long long want = std::max<unsigned long long>(a->nslots * 4, (unsigned long long)((a->nslots * 0.6 + (double)nd) * 2));
        TG_TRY(grow_table(a, want));
        TG_TRY(prev_deferred.ensure(a->device, dwords * 4 + 16));
        TG_CUDA(cudaMemcpyAsync(prev_deferred.p, a->deferred.p, dwords * 4, cudaMemcpyDeviceToDevice, a->stream));
        TG_CUDA(cudaMemsetAsync(a->deferred.p, 0, dwords * 4, a->stream));
        TG_CUDA(cudaMemsetAsync(sc + 1, 0, 8, a->stream));
        only = prev_deferred.as<uint32_t>();
        if (round == 39) return fail(TG_ERR_CUDA, "internal: aggregation table failed to converge");
      }
    }
  }
  TG_CUDA(cudaEventRecord(a->ev1, a->stream));
  TG_CUDA(cudaStreamSynchronize(a->stream));
  TG_CUDA(cudaGetLastError());
  float ms = 0; cudaEventElapsedTime(&ms, a->ev0, a->ev1); a->stats.update_ms += ms;
  return TG_OK;
}

// aggregate n device-resident rows; a fused argument expression that overflowed fails the call (types.ErrOverflow)
static int update_device(AggImpl* a, const DevCols& cols, int64_t n) {
  TG_TRY(update_device_impl(a, cols, n));
  bool has_expr = false;
  for (int k = 0; k < a->spec.n; k++) has_expr |= a->spec.f[k].arg_expr != TG_ARGEXPR_COL;
  if (!has_expr || n == 0) return TG_OK;
  unsigned long long e = 0;
  TG_CUDA(cudaMemcpyAsync(&e, a->scalars.as<unsigned long long>() + 7, 8, cudaMemcpyDeviceToHost, a->stream));
  TG_CUDA(cudaStreamSynchronize(a->stream));
  if (e) return fail(TG_ERR_OVERFLOW, "ErrOverflow: DOUBLE value is out of range in an aggregate argument expression");
  return TG_OK;
}

static int avalidate(const AggImpl* a, const tg_chunk* chk) {
  if (!chk || chk->ncols != a->ncols) return fail(TG_ERR_INVALID, "chunk column count does not match the child schema");
  int64_t phys = chk->cols[0].length;
  for (int c = 0; c < a->ncols; c++) {
    if (!a->needed[c]) continue;
    if (chk->cols[c].elem_len != a->elem[c]) return fail(TG_ERR_INVALID, "chunk column elem_len does not match the schema type");
    if (chk->cols[c].length != phys) return fail(TG_ERR_INVALID, "chunk columns have different lengths");
  }
  return TG_OK;
}

static int aflush(AggImpl* a) {
  ColumnStage& st = a->stage;
  if (st.rows == 0) return TG_OK;
  DevCols v{};
  for (int c = 0; c < a->ncols; c++) {
    v.elem_len[c] = a->elem[c];
    if (!a->needed[c]) continue;
    size_t bytes = (size_t)st.rows * 8;
    TG_TRY(a->dcols[c]->ensure(a->device, bytes + 16));
    TG_CUDA(cudaMemcpyAsync(a->dcols[c]->p, st.data[c]->p, bytes, cudaMemcpyHostToDevice, a->stream));
    a->stats.h2d_bytes += bytes;
    v.data[c] = a->dcols[c]->p;
    if (st.has_nulls[c]) {
      size_t nb = (size_t)((st.rows + 7) / 8);
      TG_TRY(a->dnulls[c]->ensure(a->device, nb + 16));
      TG_CUDA(cudaMemcpyAsync(a->dnulls[c]->p, st.nulls[c]->p, nb, cudaMemcpyHostToDevice, a->stream));
      a->stats.h2d_bytes += nb;
      v.nulls[c] = a->dnulls[c]->as<uint8_t>();
    }
  }
  int64_t n = st.rows;
  int rc = update_device(a, v, n);
  st.rows = 0;
  std::fill(st.has_nulls.begin(), st.has_nulls.end(), 0);
  return rc;
}

static int afinalize(AggImpl* a) {
  TG_TRY(a->scalars.ensure(a->device, 64));
  unsigned long long* sc = a->scalars.as<unsigned long long>();
  int nf = a->spec.n;
  a->out_cols.clear(); a->out_valid.clear(); a->out_bitmaps.clear();
  for (int k = 0; k < nf; k++) { a->out_cols.emplace_back(new DevBuf()); a->out_valid.emplace_back(new DevBuf()); a->out_bitmaps.emplace_back(new DevBuf()); }
  // agg_hash_executor.go:654: empty input and no GROUP BY → one row of default values (COUNT 0, rest NULL)
  bool default_row = a->stats.input_rows == 0 && a->group_col < 0;
  if (a->nslots == 0) {
    if (!default_row) { a->out_rows = 0; return TG_OK; }
    TG_CUDA(cudaMemsetAsync(sc, 0, 64, a->stream));
    TG_TRY(alloc_table(a, 1024, a->tbl_mem, a->tbl));
    a->nslots = 1024;
  }
  unsigned long long fill = 0;
  TG_CUDA(cudaMemsetAsync(sc, 0, 8, a->stream));
  k_agg_count<<<agrid(a, (int64_t)a->nslots + 2), 256, 0, a->stream>>>(a->tbl, sc);
  a->stats.kernel_launches++;
  TG_CUDA(cudaMemcpyAsync(&fill, sc, 8, cudaMemcpyDeviceToHost, a->stream));
  TG_CUDA(cudaStreamSynchronize(a->stream));
  int64_t cap = (int64_t)fill + 2 + 1;
  AggOut ao{};
  for (int k = 0; k < nf; k++) {
    TG_TRY(a->out_cols[k]->ensure(a->device, (size_t)cap * 8 + 16));
    ao.data[k] = a->out_cols[k]->p;
    ao.valid[k] = nullptr;
    if (a->out_nullable[k] || default_row) { TG_TRY(a->out_valid[k]->ensure(a->device, (size_t)cap + 16)); ao.valid[k] = a->out_valid[k]->as<uint8_t>(); }
  }
  TG_CUDA(cudaEventRecord(a->ev0, a->stream));
  TG_CUDA(cudaMemsetAsync(sc + 2, 0, 8, a->stream));
  k_agg_finalize<<<agrid(a, (int64_t)a->nslots + 2), 256, 0, a->stream>>>(a->tbl, a->spec, a->gk_kind, ao, sc + 2);
  a->stats.kernel_launches++;
  unsigned long long nrows = 0;
  TG_CUDA(cudaMemcpyAsync(&nrows, sc + 2, 8, cudaMemcpyDeviceToHost, a->stream));
  TG_CUDA(cudaStreamSynchronize(a->stream));
  if (default_row && nrows == 0) {
    // write the default row on the host side: COUNT → 0, everything else NULL
    for (int k = 0; k < nf; k++) {
      unsigned long long zero = 0; uint8_t v = a->spec.f[k].name == TG_AGG_COUNT ? 1 : 0;
      TG_CUDA(cudaMemcpyAsync(a->out_cols[k]->p, &zero, 8, cudaMemcpyHostToDevice, a->stream));
      TG_CUDA(cudaMemcpyAsync(a->out_valid[k]->p, &v, 1, cudaMemcpyHostToDevice, a->stream));
      TG_CUDA(cudaStreamSynchronize(a->stream));
    }
    nrows = 1;
  }
  a->out_rows = (int64_t)nrows;
  a->stats.groups = a->out_rows;
  a->stats.table_slots = (int64_t)a->nslots;
  for (int k = 0; k < nf; k++) {
    if (!ao.valid[k]) continue;
    TG_TRY(a->out_bitmaps[k]->ensure(a->device, (size_t)((a->out_rows + 7) / 8) + 16));
    if (a->out_rows) { k_pack_bitmap_agg<<<agrid(a, (a->out_rows + 7) / 8), 256, 0, a->stream>>>(ao.valid[k], a->out_rows, a->out_bitmaps[k]->as<uint8_t>()); a->stats.kernel_launches++; }
  }
  TG_CUDA(cudaEventRecord(a->ev1, a->stream));
  TG_CUDA(cudaStreamSynchronize(a->stream));
  TG_CUDA(cudaGetLastError());
  float ms = 0; cudaEventElapsedTime(&ms, a->ev0, a->ev1); a->stats.finalize_ms += ms;
  return TG_OK;
}

}  // namespace tg

#define TGA_LOCK(h)                                                            \
  if (!(h)) return tg::fail(TG_ERR_INVALID, "handle is NULL");                 \
  if ((h)->closed.load()) return tg::fail(TG_ERR_CANCELLED, "handle is closed"); \
  std::lock_guard<std::mutex> lock__((h)->mu);                                 \
  if ((h)->closed.load() || !(h)->impl) return tg::fail(TG_ERR_CANCELLED, "handle is closed"); \
  AggImpl* a = (h)->impl;                                                      \
  tg::DeviceGuard guard__(a->device);                                          \
  if (!guard__.ok) return tg::fail(TG_ERR_CUDA, "cudaSetDevice failed (no usable CUDA device)")

extern "C" {

int tg_agg_supported(const tg_agg_desc* desc) { AggImpl tmp; return agg_setup(&tmp, desc); }

int tg_agg_open(const tg_agg_desc* desc, tg_agg** out) {
  if (!out) return fail(TG_ERR_INVALID, "out is NULL");
  *out = nullptr;
  std::unique_ptr<tg_agg> shell(new tg_agg());
  std::unique_ptr<AggImpl> a(new AggImpl());
  TG_TRY(agg_setup(a.get(), desc));
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(TG_ERR_CUDA, "no CUDA device: the GPU hash aggregation has no CPU fallback"); }
  if (a->device < 0 || a->device >= ndev) return fail(TG_ERR_INVALID, "device ordinal out of range");
  DeviceGuard g(a->device);
  if (!g.ok) return fail(TG_ERR_CUDA, "cudaSetDevice failed");
  if (desc->stream) { a->stream = (cudaStream_t)desc->stream; a->own_stream = false; }
  else { TG_CUDA(cudaStreamCreateWithFlags(&a->stream, cudaStreamNonBlocking)); a->own_stream = true; }
  TG_CUDA(cudaEventCreate(&a->ev0));
  TG_CUDA(cudaEventCreate(&a->ev1));
  a->nsm = device_sm_count(a->device);
  a->stage.init(a->ncols);
  for (int c = 0; c < a->ncols; c++) { a->dcols.emplace_back(new DevBuf()); a->dnulls.emplace_back(new DevBuf()); }
  shell->impl = a.release();
  *out = shell.release();
  return TG_OK;
}

int tg_agg_push(tg_agg* h, const tg_chunk* chk) {
  TGA_LOCK(h);
  if (a->finished) return fail(TG_ERR_STATE, "push after finish");
  TG_TRY(avalidate(a, chk));
  TG_TRY(stage_append(a->stage, chk, a->needed));
  if (a->stage.rows >= (4ll << 20)) TG_TRY(aflush(a));
  return TG_OK;
}

int tg_agg_push_dev(tg_agg* h, const tg_chunk* chk) {
  TGA_LOCK(h);
  if (a->finished) return fail(TG_ERR_STATE, "push after finish");
  TG_TRY(avalidate(a, chk));
  if (chk->sel) return fail(TG_ERR_UNSUPPORTED, "device-resident chunks must not carry a sel vector");
  TG_TRY(aflush(a));
  DevCols v{};
  for (int c = 0; c < a->ncols; c++) {
    v.elem_len[c] = a->elem[c];
    if (!a->needed[c]) continue;
    v.data[c] = chk->cols[c].data; v.nulls[c] = chk->cols[c].null_bitmap;
  }
  return update_device(a, v, chk->cols[0].length);
}

int tg_agg_finish(tg_agg* h) {
  TGA_LOCK(h);
  if (a->finished) return TG_OK;
  TG_TRY(aflush(a));
  TG_TRY(afinalize(a));
  a->finished = true;
  return TG_OK;
}

int tg_agg_next(tg_agg* h, tg_mut_chunk* out, int64_t max_rows, int64_t* nrows) {
  TGA_LOCK(h);
  if (!out || !nrows) return fail(TG_ERR_INVALID, "out / nrows is NULL");
  *nrows = 0;
  if (!a->finished) return fail(TG_ERR_STATE, "next before finish (hash aggregation is a pipeline breaker)");
  if (out->ncols != a->spec.n) return fail(TG_ERR_INVALID, "output chunk column count does not match the aggregate list");
  int64_t lo = a->consumed;
  int64_t want = std::min<int64_t>(std::min<int64_t>(max_rows, out->capacity_rows), a->out_rows - lo);
  if (want <= 0) return TG_OK;
  std::vector<const void*> cols(a->spec.n);
  std::vector<const uint8_t*> bitmaps(a->spec.n);
  for (int k = 0; k < a->spec.n; k++) { cols[k] = a->out_cols[k]->p; bitmaps[k] = a->out_bitmaps[k]->as<uint8_t>(); }
  TG_TRY(copy_out_rows(a->stream, a->spec.n, cols.data(), bitmaps.data(), lo, want, out, &a->stats.d2h_bytes));
  a->consumed += want;
  *nrows = want;
  return TG_OK;
}

int tg_agg_result_dev(tg_agg* h, int64_t* out_rows, void** out_cols, void** out_nulls) {
  TGA_LOCK(h);
  if (!a->finished) return fail(TG_ERR_STATE, "result before finish");
  if (out_rows) *out_rows = a->out_rows;
  for (int k = 0; k < a->spec.n; k++) {
    if (out_cols) out_cols[k] = a->out_cols[k]->p;
    if (out_nulls) out_nulls[k] = a->out_bitmaps[k]->p;
  }
  return TG_OK;
}

int tg_agg_get_stats(tg_agg* h, tg_agg_stats* out) {
  TGA_LOCK(h);
  if (!out) return fail(TG_ERR_INVALID, "out is NULL");
  *out = a->stats;
  return TG_OK;
}

int tg_agg_close(tg_agg* h) {
  if (!h) return TG_OK;
  bool was = h->closed.exchange(true);
  if (was) return TG_OK;
  {
    std::lock_guard<std::mutex> lock(h->mu);   // waits for an in-flight call; later calls see `closed`
    AggImpl* a = h->impl;
    h->impl = nullptr;
    if (a) {
      DeviceGuard g(a->device);
      if (a->stream) cudaStreamSynchronize(a->stream);
      if (a->ev0) cudaEventDestroy(a->ev0);
      if (a->ev1) cudaEventDestroy(a->ev1);
      if (a->own_stream && a->stream) cudaStreamDestroy(a->stream);
      cudaGetLastError();
      delete a;
    }
  }
  bury_handle(h);
  return TG_OK;
}

}  // extern "C"
