/*
 * tidbgpu.h — C ABI of libtidbgpu.so: the B200 (sm_100a) operator hot path of TiDB's
 * chunk-based vectorized executor (hash join build/probe, hash aggregation, VecEval*
 * filter/projection kernels, key-hash repartition for multi-GPU).
 *
 * This is the drop-in boundary a cgo shim binds (see INTEGRATION.md).  TiDB has no FFI for
 * this path today; the interface it sits behind is the Go interface
 *     exec.Executor { Open(ctx) / Next(ctx, *chunk.Chunk) / Close() }
 *     (reference: pkg/executor/internal/exec/executor.go:51-77)
 * and the data that crosses it is chunk.Chunk / chunk.Column
 *     (reference: pkg/util/chunk/chunk.go:35-54, pkg/util/chunk/column.go:74-82).
 * Every entry point below names the reference function it replaces.
 *
 * Conventions
 *   - plain C, no C++ types; every call returns int: 0 = TG_OK, >0 = tg_status code.
 *     tg_last_error() returns a thread-local human readable message for the last failure.
 *   - input buffers are BORROWED for the duration of the call only (cgo pointer rule);
 *     output buffers are caller-owned and caller-sized.
 *   - the library never falls back to a CPU implementation: if no CUDA device is usable every
 *     compute entry point fails with TG_ERR_CUDA.
 *   - calls on one handle are serialised internally; tg_*_close may race with an in-flight
 *     tg_*_next (executor.go:65 "Close may be called with Next at the same time"): the
 *     in-flight call returns TG_ERR_CANCELLED.
 */
#ifndef TIDBGPU_H
#define TIDBGPU_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TIDBGPU_ABI_VERSION 1

/* ---------------------------------------------------------------------------------------------
 * status codes
 * ------------------------------------------------------------------------------------------- */
typedef enum tg_status {
  TG_OK = 0,
  TG_ERR_INVALID = 1,      /* bad argument / descriptor */
  TG_ERR_UNSUPPORTED = 2,  /* valid plan, but not offloadable: the Go shim keeps the CPU executor
                              (same spirit as join.IsHashJoinV2Supported / CanUseHashJoinV2,
                              pkg/executor/builder.go:1934) */
  TG_ERR_CUDA = 3,         /* CUDA runtime failure or no device */
  TG_ERR_OOM = 4,          /* device or pinned-host allocation failed */
  TG_ERR_STATE = 5,        /* call out of order (e.g. probe before build_finish) */
  TG_ERR_CANCELLED = 6,    /* handle closed / killed while the call was running */
  TG_ERR_OVERFLOW = 7,     /* types.ErrOverflow raised by an arithmetic VecEval kernel
                              (pkg/expression/builtin_arithmetic_vec.go:513-519, :957) */
  TG_ERR_CAPACITY = 8      /* caller-provided output buffer too small */
} tg_status;

const char* tg_last_error(void);
int tg_abi_version(void);
/* number of visible CUDA devices (0 if none, never an error) */
int tg_device_count(void);
/* name / SM count / HBM bytes of a device */
int tg_device_info(int device, char* name, size_t name_cap, int* sm_count, int64_t* hbm_bytes);

/* ---------------------------------------------------------------------------------------------
 * enumerations reused verbatim from the reference so the Go shim is a plain copy
 * ------------------------------------------------------------------------------------------- */
/* pkg/parser/mysql/type.go:17-48 */
enum {
  TG_TYPE_TINY = 1, TG_TYPE_SHORT = 2, TG_TYPE_LONG = 3, TG_TYPE_FLOAT = 4, TG_TYPE_DOUBLE = 5,
  TG_TYPE_TIMESTAMP = 7, TG_TYPE_LONGLONG = 8, TG_TYPE_INT24 = 9, TG_TYPE_DATE = 10,
  TG_TYPE_DURATION = 11, TG_TYPE_DATETIME = 12, TG_TYPE_YEAR = 13, TG_TYPE_NEWDECIMAL = 0xf6,
  TG_TYPE_VARSTRING = 0xfd
};
/* pkg/parser/mysql/type.go:54-77 */
enum { TG_FLAG_NOT_NULL = 1u << 0, TG_FLAG_UNSIGNED = 1u << 5 };
/* pkg/planner/core/base/plan_base.go:310-322 (JoinType) */
enum {
  TG_JOIN_INNER = 0, TG_JOIN_LEFT_OUTER = 1, TG_JOIN_RIGHT_OUTER = 2, TG_JOIN_SEMI = 3,
  TG_JOIN_ANTI_SEMI = 4, TG_JOIN_LEFT_OUTER_SEMI = 5, TG_JOIN_ANTI_LEFT_OUTER_SEMI = 6
};
/* aggregate function names (pkg/parser/ast/functions.go AggFuncCount.. ) */
enum { TG_AGG_COUNT = 0, TG_AGG_SUM = 1, TG_AGG_AVG = 2, TG_AGG_MIN = 3, TG_AGG_MAX = 4,
       TG_AGG_FIRSTROW = 5 };
/* pkg/expression/aggregation/descriptor.go:155-165 (AggFunctionMode) */
enum { TG_AGGMODE_COMPLETE = 0, TG_AGGMODE_FINAL = 1, TG_AGGMODE_PARTIAL1 = 2,
       TG_AGGMODE_PARTIAL2 = 3, TG_AGGMODE_DEDUP = 4 };

/* fixed element length of a MySQL type inside a chunk column, -1 = var-len
 * (pkg/util/chunk/codec.go:165-179 getFixedLen) */
int tg_fixed_len(int mysql_type);

/* ---------------------------------------------------------------------------------------------
 * chunk.Column / chunk.Chunk views            (pkg/util/chunk/column.go:74-82, chunk.go:35-54)
 * ------------------------------------------------------------------------------------------- */
typedef struct tg_column {
  int64_t length;             /* Column.length: physical rows                                   */
  const uint8_t* null_bitmap; /* Column.nullBitmap: LSB-first, bit 1 = NOT NULL, ceil(length/8)
                                 bytes; NULL pointer = no NULLs in this column                  */
  const int64_t* offsets;     /* Column.offsets (length+1) for var-len columns, else NULL       */
  const uint8_t* data;        /* Column.data: length*elem_len little-endian bytes (fixed)       */
  int32_t elem_len;           /* 8, 4, 40, or -1 (var-len)                                      */
  int32_t reserved;
} tg_column;

typedef struct tg_chunk {
  int32_t ncols;
  int32_t reserved;
  const tg_column* cols;
  const int64_t* sel;         /* Chunk.sel: logical row i -> physical row sel[i]; NULL = identity
                                 (chunk.go:38, :394-407).  Go `int` is 64-bit on every TiDB target */
  int64_t nsel;               /* logical rows when sel != NULL (Chunk.NumRows, chunk.go:384)    */
} tg_chunk;

/* caller-owned output column: the Go side passes Column.data / Column.nullBitmap capacity */
typedef struct tg_mut_column {
  uint8_t* null_bitmap;       /* capacity ceil(capacity_rows/8) bytes, may be NULL if the caller
                                 knows the column is NOT NULL (then a NULL produced is an error) */
  uint8_t* data;              /* capacity capacity_rows*elem_len bytes                           */
  int32_t elem_len;
  int32_t reserved;
} tg_mut_column;

typedef struct tg_mut_chunk {
  int32_t ncols;
  int32_t reserved;
  tg_mut_column* cols;
  int64_t capacity_rows;
} tg_mut_chunk;

/* ---------------------------------------------------------------------------------------------
 * Chunk wire format (host code): chunk.Codec, pkg/util/chunk/codec.go — Encode :41, DecodeToChunk :93,
 * decodeColumn :101, setAllNotNull :145.  Per column: u32 length | u32 nullCount | [bitmap if nullCount > 0] |
 * [offsets (length+1) x i64 if var-len] | data.  Coprocessor / TiFlash responses use it, so a cgo shim can hand the
 * response buffer over as is (SURVEY §8 f.2).
 * ------------------------------------------------------------------------------------------- */
int tg_chunk_wire_size(const tg_chunk* chk, size_t* bytes);
int tg_chunk_encode(const tg_chunk* chk, uint8_t* buf, size_t cap, size_t* written);
/* zero copy: cols_out[i] alias buf, like the Go decoder's Columns alias the gRPC message; null_bitmap == NULL where the
 * wire carried no NULLs.  `consumed` = bytes of buf that belonged to these ncols columns.                          */
int tg_chunk_decode(const uint8_t* buf, size_t len, int32_t ncols, const int32_t* mysql_types, tg_column* cols_out,
                    size_t* consumed);
/* decode the fixed-width columns straight into caller-owned (e.g. tg_host_alloc'ed, pinned) buffers; columns whose
 * out->cols[i].data is NULL are skipped                                                                           */
int tg_chunk_decode_into(const uint8_t* buf, size_t len, int32_t ncols, const int32_t* mysql_types, tg_mut_chunk* out,
                         int64_t* rows, size_t* consumed);

/* ---------------------------------------------------------------------------------------------
 * pinned host memory for a chunk.ColumnAllocator (pkg/util/chunk/column.go:85) backed by
 * cudaHostAlloc, precedent: pkg/lightning/manual/manual.go (C.calloc behind Go slices).
 * Buffers from here make H2D/D2H copies true DMA; any other host pointer is accepted too.
 * ------------------------------------------------------------------------------------------- */
int tg_host_alloc(size_t bytes, void** out);
int tg_host_free(void* p);

/* raw device memory + copies, for device-resident ("synthetic columnar") runs and tests */
int tg_dev_alloc(int device, size_t bytes, void** out);
int tg_dev_free(int device, void* p);
int tg_memcpy_h2d(int device, void* dst_dev, const void* src_host, size_t bytes);
int tg_memcpy_d2h(int device, void* dst_host, const void* src_dev, size_t bytes);
/* Asynchronous device-to-device copy on `stream` (cudaMemcpyAsync, copy engine): `dst` may be memory of a peer GPU mapped
 * with tg_ipc_open — the DMA then crosses NVLink without occupying SMs (SegmentExchange's transfer step).          */
int tg_memcpy_d2d_async(int device, void* dst_dev, const void* src_dev, size_t bytes, void* stream);
int tg_device_synchronize(int device);

/* ---------------------------------------------------------------------------------------------
 * Hash join                      replaces join.HashJoinV2Exec (pkg/executor/join/hash_join_v2.go:608)
 * ------------------------------------------------------------------------------------------- */
typedef struct tg_join tg_join;

/* scalar filter program: CNF of (column OP constant) / (column OP column) items on 8-byte columns;
 * replaces expression.VectorizedFilter (pkg/expression/chunk_executor.go:413) for
 * BuildFilter / ProbeFilter / OtherCondition (pkg/executor/builder.go:1771-1931). */
enum { TG_CMP_LT = 0, TG_CMP_LE = 1, TG_CMP_GT = 2, TG_CMP_GE = 3, TG_CMP_EQ = 4, TG_CMP_NE = 5 };
typedef struct tg_filter_item {
  int32_t op;          /* TG_CMP_*                                                      */
  int32_t lhs_col;     /* column index in the chunk the filter is evaluated on           */
  int32_t rhs_col;     /* -1 = compare with constant                                     */
  int32_t is_real;     /* 0: int64 compare (signed unless lhs_unsigned), 1: float64      */
  int32_t lhs_unsigned;
  int32_t rhs_unsigned; /* signedness of the right column / constant (types.CompareInt takes both flags) */
  int64_t const_i64;   /* constant when rhs_col < 0 and !is_real                         */
  double const_f64;    /* constant when rhs_col < 0 and is_real                          */
} tg_filter_item;

/* One CNF item of HashJoinV2Exec.OtherCondition (inner_join_probe.go:72-79, base_join_probe.go:758
 * buildResultAfterOtherCondition): `operand OP operand` over the JOINED row, each operand a column of the left or the
 * right child (side 0 / 1), the right operand optionally a constant (rhs_side = -1).  A candidate pair (equal keys)
 * is a match only if every item is non-NULL true (VectorizedFilter semantics).                                     */
typedef struct tg_other_item {
  int32_t op;            /* TG_CMP_*                                                      */
  int32_t is_real;       /* 0: int64 compare, 1: float64                                  */
  int32_t lhs_side, lhs_col;
  int32_t rhs_side, rhs_col;   /* rhs_side = -1: constant                                 */
  int32_t lhs_unsigned, rhs_unsigned;
  int64_t const_i64;
  double const_f64;
} tg_other_item;

typedef struct tg_join_desc {
  int32_t join_type;          /* TG_JOIN_*                                                       */
  int32_t build_is_right;     /* HashJoinV2Exec RightAsBuildSide: 1 = right child is build side  */
  /* schema of both children: MySQL type + flag per column (FieldType.tp / .flag)               */
  int32_t n_left_cols;
  int32_t n_right_cols;
  const int32_t* left_types;  const uint32_t* left_flags;
  const int32_t* right_types; const uint32_t* right_flags;
  /* equal-condition keys: column index per side (BuildKeyColIdx / ProbeKeyColIdx after
   * mapping to left/right, builder.go:1780-1830).  nkeys = 1: int family / float / double key (OneInt64 mode and the
   * 8-byte fixed keys).  nkeys = 2..4: FixedSerializedKey mode (join_table_meta.go:174-178) for 8-byte integer-family
   * columns — a row with a NULL in any key column has no key; a pair matches iff every key column is equal by value
   * (signed vs unsigned compared by value).  Join shapes that need a build-side scan or the NULL-aware match flag are
   * declined with several keys (TG_ERR_UNSUPPORTED → the planner keeps the CPU executor), like with OtherCondition.  */
  int32_t nkeys;
  int32_t reserved0;
  const int32_t* left_key_idx;
  const int32_t* right_key_idx;
  /* output = LUsed columns of left ‖ RUsed columns of right (builder.go:1868-1871).
   * NULL pointer with n = -1 means "all columns" (the reference's nil slice).                  */
  int32_t n_lused; int32_t n_rused;
  const int32_t* lused; const int32_t* rused;
  /* optional filters evaluated on the build-side / probe-side child chunk                      */
  int32_t n_build_filter; int32_t n_probe_filter;
  const tg_filter_item* build_filter;
  const tg_filter_item* probe_filter;
  int32_t device;             /* CUDA device ordinal                                             */
  int32_t reserved1;
  void* stream;               /* cudaStream_t to launch on; NULL = library-owned stream          */
  double load_factor;         /* 0 = default                                                     */
  /* OtherCondition (non-equi residual evaluated on candidate pairs); offloaded for inner, probe-side outer, semi and
   * anti-semi joins with the right child as build side (the gate declines the rest)              */
  int32_t n_other_cond; int32_t reserved2;
  const tg_other_item* other_cond;
} tg_join_desc;

/* planner gate: 0 if this descriptor can run on the GPU, TG_ERR_UNSUPPORTED otherwise        */
int tg_join_supported(const tg_join_desc* desc);

/* HashJoinV2Exec.Open (hash_join_v2.go:690)                                                  */
int tg_join_open(const tg_join_desc* desc, tg_join** out);
/* buildWorkerBase.fetchBuildSideRows + BuildWorkerV2.processOneChunk (hash_join_base.go:257,
 * hash_join_v2.go:536): one build-side child chunk. Host buffers; copied before returning.    */
int tg_join_build_push(tg_join* j, const tg_chunk* chk);
/* same, columns already resident in device memory (borrowed until tg_join_build_finish)       */
int tg_join_build_push_dev(tg_join* j, const tg_chunk* dev_chk);
/* mergeRowTablesToHashTable + buildHashTable (hash_join_v2.go:217, :1458)                     */
int tg_join_build_finish(tg_join* j);
/* ProbeWorkerV2.processOneProbeChunk → JoinProbe.SetChunkForProbe + Probe
 * (hash_join_v2.go:932, base_join_probe.go:179, inner_join_probe.go:27): one probe-side child
 * chunk from host memory.  The library batches internally; joined rows become available to
 * tg_join_next.                                                                               */
int tg_join_probe_push(tg_join* j, const tg_chunk* chk);
/* end of probe side: flush the batcher; for build-side-outer joins also runs
 * JoinProbe.ScanRowTable (outer_join_probe.go:117)                                            */
int tg_join_probe_finish(tg_join* j);
/* HashJoinV2Exec.Next (hash_join_v2.go:1161): fill at most min(max_rows, out->capacity_rows)
 * joined rows; *nrows == 0 means EOF (only after tg_join_probe_finish).                       */
int tg_join_next(tg_join* j, tg_mut_chunk* out, int64_t max_rows, int64_t* nrows);
/* Same, but blocks until rows are available or the probe side is finished (then 0 = EOF).  One thread may sit in
 * tg_join_next_wait while another pushes probe chunks — the reference's probe fetcher goroutine vs the consumer of
 * joinResultCh (hash_join_v2.go:840, :1176); results are copied on their own stream, so D2H overlaps the next H2D. */
int tg_join_next_wait(tg_join* j, tg_mut_chunk* out, int64_t max_rows, int64_t* nrows);
/* Start another probe pass against the SAME built table (results not yet fetched are dropped).  Mirrors re-execution
 * of the probe side under Apply with a cached build side; not available for joins that scan the build side. */
int tg_join_probe_rewind(tg_join* j);
/* HashJoinV2Exec.Close (hash_join_v2.go:647); idempotent                                     */
int tg_join_close(tg_join* j);

/* Device-resident probe (inputs and outputs stay in HBM): probe `dev_chk` against the built table,
 * write the joined columns into library-owned device buffers, return their device pointers.
 * out_cols[i] receives the device address of output column i (n_lused+n_rused entries),
 * out_nulls[i] the device null bitmap of that column or NULL.  Valid until the next probe call
 * on this handle or close.  This is the kernel-only path bench.py times as `value`.           */
int tg_join_probe_dev(tg_join* j, const tg_chunk* dev_chk, int64_t* out_rows,
                      void** out_cols, void** out_nulls);
/* Same, for a device chunk that is SEGMENTED: `nseg` segments of `seg_cap` rows each (seg_cap a multiple of
 * 1024), segment s holding seg_cnt_dev[s] valid rows at its start; dev_chk->cols[*].length = nseg*seg_cap.  This is
 * the shape a count-free exchange delivers (tg_partition_exchange_cf: one fixed-capacity region per sending GPU,
 * fill counts known only on the device), so the receiver probes without compacting and without a host round trip.
 * Only for plans the fused fast path covers (tg_join_get_stats().table_mode == 1); others: TG_ERR_UNSUPPORTED.  */
int tg_join_probe_dev_seg(tg_join* j, const tg_chunk* dev_chk, const int64_t* seg_cnt_dev, int32_t nseg,
                          int64_t seg_cap, int64_t* out_rows, void** out_cols, void** out_nulls);


/* hashJoinRuntimeStatsV2 (pkg/executor/join/hash_join_stats.go:142)                          */
typedef struct tg_join_stats {
  int64_t build_rows;         /* rows pushed on the build side                       */
  int64_t build_valid_keys;   /* rows inserted into the table (non-NULL key, passed filter) */
  int64_t table_slots;        /* slots allocated                                      */
  int64_t distinct_keys;
  int64_t max_dup;            /* largest multiplicity of one key                      */
  int64_t probe_rows;
  int64_t output_rows;
  int64_t kernel_launches;    /* CUDA kernels launched by this handle                 */
  int32_t table_mode;         /* 0 none, 1 unique-inline, 2 grouped row store         */
  int32_t reserved;
  double build_ms, probe_ms;  /* device time measured with CUDA events                */
  int64_t h2d_bytes, d2h_bytes;
} tg_join_stats;
int tg_join_get_stats(tg_join* j, tg_join_stats* out);

/* ---------------------------------------------------------------------------------------------
 * Hash aggregation            replaces aggregate.HashAggExec (pkg/executor/aggregate/agg_hash_executor.go:93)
 * ------------------------------------------------------------------------------------------- */
typedef struct tg_agg tg_agg;

typedef struct tg_agg_func {
  int32_t name;      /* TG_AGG_*                                                               */
  int32_t mode;      /* TG_AGGMODE_*                                                           */
  int32_t arg_col;   /* input column index; -1 for COUNT(*) / count(constant)                  */
  int32_t arg_type;  /* MySQL type of the argument (TG_TYPE_DOUBLE / TG_TYPE_LONGLONG ...)      */
  uint32_t arg_flag;
  int32_t arg_col2;  /* Final/Partial2 AVG: second input column (count, then sum: func_avg.go:444);
                      * arg_expr != 0: the second column of the argument expression                */
  /* The argument as a small scalar expression instead of a plain column (AggFuncDesc.Args[0] is an expression.Expression
   * evaluated per row: args[0].EvalReal, func_sum.go:90).  Fused into the update kernel — no projected column is
   * materialised.  DOUBLE columns, SUM / AVG in Complete mode.  NULL if either column is NULL; a non-finite intermediate
   * on a non-NULL row fails the call with TG_ERR_OVERFLOW (builtinArithmetic{Minus,Multiply}RealSig).
   *   TG_ARGEXPR_COL        arg_col
   *   TG_ARGEXPR_MUL        arg_col * arg_col2
   *   TG_ARGEXPR_MUL_CSUB   arg_col * (arg_const - arg_col2)      e.g. l_extendedprice * (1 - l_discount)            */
  int32_t arg_expr;
  int32_t reserved;
  double arg_const;
} tg_agg_func;
enum { TG_ARGEXPR_COL = 0, TG_ARGEXPR_MUL = 1, TG_ARGEXPR_MUL_CSUB = 2 };

typedef struct tg_agg_desc {
  int32_t n_cols;                 /* child schema                                               */
  int32_t n_group_by;
  const int32_t* col_types; const uint32_t* col_flags;
  const int32_t* group_by_cols;   /* GroupByItems as plain column refs (agg_util.go:106)        */
  int32_t n_funcs;
  int32_t device;
  const tg_agg_func* funcs;       /* AggFuncDescs (builder.go:2106-2181)                        */
  void* stream;
  int64_t expected_groups;        /* hint (planner NDV estimate); 0 = grow on demand            */
} tg_agg_desc;

int tg_agg_supported(const tg_agg_desc* desc);
/* HashAggExec.Open (agg_hash_executor.go:237) */
int tg_agg_open(const tg_agg_desc* desc, tg_agg** out);
/* fetchChildData + HashAggPartialWorker.updatePartialResult (agg_hash_executor.go:449,
 * agg_hash_partial_worker.go:256): one child chunk (host / device-resident)                    */
int tg_agg_push(tg_agg* a, const tg_chunk* chk);
int tg_agg_push_dev(tg_agg* a, const tg_chunk* dev_chk);
/* end of input: HashAggFinalWorker merge + result generation (agg_hash_final_worker.go:73,:121) */
int tg_agg_finish(tg_agg* a);
/* HashAggExec.Next (agg_hash_executor.go:441). Output schema = one column per agg func in
 * desc order (the reference emits group columns through firstrow() funcs, SURVEY §8 note 4).   */
int tg_agg_next(tg_agg* a, tg_mut_chunk* out, int64_t max_rows, int64_t* nrows);
int tg_agg_close(tg_agg* a);
/* device-resident result: number of groups + device pointers of the output columns            */
int tg_agg_result_dev(tg_agg* a, int64_t* out_rows, void** out_cols, void** out_nulls);

typedef struct tg_agg_stats {
  int64_t input_rows, groups, table_slots, kernel_launches;
  double update_ms, finalize_ms;
  int64_t h2d_bytes, d2h_bytes;
} tg_agg_stats;
int tg_agg_get_stats(tg_agg* a, tg_agg_stats* out);

/* ---------------------------------------------------------------------------------------------
 * VecEval* kernels             replace pkg/expression builtin_*_vec.go signatures
 * All operate on one column-at-a-time over host or device buffers (`on_device` flag).
 * Result null bitmap = MergeNulls of the argument bitmaps (pkg/util/chunk/column.go:906).
 * ------------------------------------------------------------------------------------------- */
enum { TG_ARITH_PLUS = 0, TG_ARITH_MINUS = 1, TG_ARITH_MUL = 2 };

/* builtinLTIntSig.vecEvalInt & friends (pkg/expression/builtin_compare_vec.go:524-561, :619):
 * result int64 0/1, NULL if either side NULL.  b == NULL -> compare with the constant.         */
int tg_vec_compare_int(int device, int on_device, int op, int a_unsigned, int b_unsigned,
                       const tg_column* a, const tg_column* b, int64_t b_const,
                       int64_t* result, uint8_t* result_nulls, void* stream);
/* builtinLTRealSig etc (builtin_compare_vec_generated.go:54, cmp.Compare NaN ordering)        */
int tg_vec_compare_real(int device, int on_device, int op,
                        const tg_column* a, const tg_column* b, double b_const,
                        int64_t* result, uint8_t* result_nulls, void* stream);
/* builtinArithmeticPlusIntSig.vecEvalInt (builtin_arithmetic_vec.go:856-908, overflow :957),
 * MinusInt (:365, overflowCheck builtin_arithmetic.go:491), MultiplyInt / MultiplyIntUnsigned
 * (:646, :1011): the four signed/unsigned combinations; overflow on a non-NULL row ->
 * TG_ERR_OVERFLOW                                                                               */
int tg_vec_arith_int(int device, int on_device, int op, int a_unsigned, int b_unsigned,
                     const tg_column* a, const tg_column* b, int64_t b_const,
                     int64_t* result, uint8_t* result_nulls, void* stream);
/* builtinArithmeticPlusRealSig.vecEvalReal (:496-523), MinusReal, MultiplyReal:
 * +-Inf/NaN on a non-NULL row -> TG_ERR_OVERFLOW                                               */
int tg_vec_arith_real(int device, int on_device, int op,
                      const tg_column* a, const tg_column* b, double b_const,
                      double* result, uint8_t* result_nulls, void* stream);
/* expression.VectorizedFilter (chunk_executor.go:413) over a CNF of tg_filter_item:
 * selected[i] (1 byte per physical row, Go []bool) = all items true and not NULL.              */
int tg_vec_filter(int device, int on_device, const tg_chunk* chk,
                  const tg_filter_item* items, int32_t n_items,
                  uint8_t* selected, int64_t* n_selected, void* stream);

/* ---------------------------------------------------------------------------------------------
 * TopN                         replaces sortexec.TopNExec (pkg/executor/sortexec/topn.go:74, :230)
 * ORDER BY items over plain columns, LIMIT offset, count.  Rows [offset, offset + count) of the child's rows in item
 * order (NULL sorts before every value, DESC reverses: chunk.GetCompareFunc) are written to `out` (child schema, host
 * buffers, capacity >= count); ties are broken arbitrarily, as by the reference's heap.  `on_device` as in the VecEval
 * calls.  8-byte int-family / double / time columns.
 * ------------------------------------------------------------------------------------------- */
typedef struct tg_sort_item { int32_t col; int32_t desc; } tg_sort_item;
int tg_topn(int device, int on_device, const tg_chunk* chk, const int32_t* col_types, const uint32_t* col_flags,
            const tg_sort_item* items, int32_t n_items, int64_t offset, int64_t count,
            tg_mut_chunk* out, int64_t* nrows, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Sort                          replaces sortexec.SortExec (pkg/executor/sortexec/sort.go:43) for ORDER BY without LIMIT
 * Every row of the child in ORDER BY order: items compared one after another with chunk.GetCompareFunc
 * (SortExec.lessRow sort.go:804; util/chunk/compare.go:30-60): NULL before every value, DESC negates; signed / unsigned
 * int family and YEAR as int64 / uint64 (unsigned flag), DURATION as int64, DOUBLE as Go cmp.Compare (NaN first, NaNs equal, -0 == +0),
 * DATE / DATETIME / TIMESTAMP as the packed CoreTime word without its 4 fsp bits.  The device sort is stable (rows that
 * tie on every item keep their input order); the reference's is not, so callers must not rely on it.
 * 1..8 items over plain columns, 1..16 columns, every column 8 bytes (int family, YEAR, DURATION, DOUBLE, time);
 * at most 2^32 - 1 rows (row ids are 32-bit).  The whole input and the result live in HBM: no spill.
 * ------------------------------------------------------------------------------------------- */
typedef struct tg_sort tg_sort;
typedef struct tg_sort_desc {
  int32_t n_cols;                 /* child schema                                               */
  int32_t n_items;
  const int32_t* col_types; const uint32_t* col_flags;
  const tg_sort_item* items;      /* ByItems as plain column refs (buildKeyColumns sort.go:789)  */
  int32_t device;
  int32_t reserved;
  void* stream;                   /* cudaStream_t; NULL = library-owned stream                   */
  int64_t expected_rows;          /* hint for buffer sizing (planner estimate); 0 = grow on demand */
} tg_sort_desc;

/* planner gate: 0 if this descriptor can run on the GPU; answers without a device               */
int tg_sort_supported(const tg_sort_desc* desc);
/* SortExec.Open (sort.go:155)                                                                   */
int tg_sort_open(const tg_sort_desc* desc, tg_sort** out);
/* SortExec.fetchChunks (sort.go:526): one child chunk from host memory, sel honoured; copied before returning */
int tg_sort_push(tg_sort* s, const tg_chunk* chk);
/* same, columns already resident in device memory (no sel; borrowed until tg_sort_finish)       */
int tg_sort_push_dev(tg_sort* s, const tg_chunk* dev_chk);
/* end of input: the sort itself (LSD radix sort of the ORDER BY items) and the gather of every column */
int tg_sort_finish(tg_sort* s);
/* SortExec.Next (sort.go:265): the next min(max_rows, out->capacity_rows) rows; *nrows == 0 means EOF */
int tg_sort_next(tg_sort* s, tg_mut_chunk* out, int64_t max_rows, int64_t* nrows);
/* device-resident result: row count + device pointers of the sorted columns and their null bitmaps (NULL: no NULLs);
 * valid until close                                                                             */
int tg_sort_result_dev(tg_sort* s, int64_t* out_rows, void** out_cols, void** out_nulls);

typedef struct tg_sort_stats {
  int64_t input_rows;
  int64_t digit_passes;           /* 8-bit digit scatter passes run                              */
  int64_t skipped_passes;         /* digit passes skipped: every row had the same digit          */
  int64_t null_passes;            /* NULL-flag passes run                                        */
  int64_t kernel_launches;
  double sort_ms, gather_ms;      /* device time measured with CUDA events                       */
  int64_t h2d_bytes, d2h_bytes;
} tg_sort_stats;
int tg_sort_get_stats(tg_sort* s, tg_sort_stats* out);
/* SortExec.Close (sort.go:109); idempotent, may race with an in-flight call                    */
int tg_sort_close(tg_sort* s);
/* The order-preserving 64-bit key the sort gives one non-NULL value of a column (host evaluation of the device
 * normalizer; tests and planners): keys compare as uint64 exactly as the values compare under ORDER BY.      */
int tg_sort_key_host(int32_t mysql_type, uint32_t flag, int32_t desc, uint64_t raw, uint64_t* key);

/* ---------------------------------------------------------------------------------------------
 * Key-hash repartition for the multi-GPU exchange (the B200 analogue of the MPP
 * ExchangeSender HashPartition, pkg/planner/core/operator/physicalop/physical_exchange_sender.go:115;
 * in-process analogue: partitionHashSplitter.split, pkg/executor/shuffle.go:450).
 * Device-resident: scatter `ncols` 8-byte columns of `rows` rows into `nparts` contiguous
 * regions by hash(key) (bits disjoint from the local table slot bits).  part_offsets receives
 * nparts+1 row offsets (device int64).  dst columns have capacity `rows`.
 * ------------------------------------------------------------------------------------------- */
int tg_partition_by_key(int device, const int64_t* key_dev, const uint8_t* key_nulls_dev,
                        int64_t rows, int32_t nparts, int32_t ncols,
                        const void* const* src_cols_dev, void* const* dst_cols_dev,
                        int64_t* part_offsets_dev, void* stream);
/* Same partition function evaluated on the host for one key (tests / planner)                 */
int32_t tg_partition_of_key(int64_t key, int32_t nparts);

/* Fused partition + NVLink exchange: like tg_partition_by_key but region p is written straight
 * into peer p's receive buffer (peer pointers mapped with tg_ipc_open) — the repartition step and
 * its all-to-all in one kernel.  recv_cols_peer[p*ncols + c] = device address (on peer p, mapped
 * here) of column c's receive buffer; recv_base[p] = first row this rank may write on peer p.   */
int tg_partition_exchange(int device, const int64_t* key_dev, int64_t rows, int32_t nparts,
                          int32_t ncols, const void* const* src_cols_dev,
                          void* const* recv_cols_peer, const int64_t* part_counts_dev,
                          const int64_t* recv_base_dev, void* stream);
/* Count-free variant (no histogram pass, no host round trip): every destination p owns, inside each receiver's
 * buffers, the fixed-capacity region [region_base, region_base + region_cap) reserved for THIS sender; rows are
 * appended there in arrival order and sent_rows_dev[p] (device, zeroed by the call) ends up holding how many rows went
 * to p.  A destination that would overflow raises *overflow_dev (device u64, sticky: the caller zeroes it once) and drops the excess —
 * the caller re-runs that step through tg_partition_count + tg_partition_exchange.  Returns after ENQUEUEING on `stream`.
 * The MPP analogue is still ExchangeSender/HashPartition (physical_exchange_sender.go:115); the reference sizes
 * its per-partition chunks dynamically on the host (shuffle.go:450), which a single GPU kernel cannot.            */
int tg_partition_exchange_cf(int device, const int64_t* key_dev, int64_t rows, int32_t nparts, int32_t ncols,
                             const void* const* src_cols_dev, void* const* recv_cols_peer, int64_t region_base,
                             int64_t region_cap, int64_t* sent_rows_dev, uint64_t* overflow_dev, void* stream);

/* tg_partition_exchange_cf with a cap on the scatter kernel's CTAs per SM (0 = as many as fit).  When the exchange
 * is NVLink-bound a few CTAs per SM already saturate the links, and the probe kernel of the previous step — running
 * next to it on another stream — keeps the SMs' L1 (the bulk-store scatter holds 49 KB of shared memory per CTA).   */
int tg_partition_exchange_cf_ex(int device, const int64_t* key_dev, int64_t rows, int32_t nparts, int32_t ncols,
                                const void* const* src_cols_dev, void* const* recv_cols_peer, int64_t region_base,
                                int64_t region_cap, int64_t* sent_rows_dev, uint64_t* overflow_dev, int32_t ctas_per_sm,
                                void* stream);

/* tg_partition_exchange_cf_ex whose destinations cannot lose rows to skew: a row that does not fit its destination's region
 * is appended to a LOCAL spill area instead (column c at spill_cols_dev[c], at most spill_cap rows in total, filled through
 * *spill_cursor_dev — device u64, zeroed by the caller, it keeps counting across calls).  After the pipeline the caller reads
 * the cursor once and moves the spilled rows with the counted exchange (tg_partition_count + tg_partition_exchange).
 * *overflow_dev is raised only when the spill area itself is full.  The reference's exchange has unbounded per-partition
 * queues (executor/shuffle.go:450) — skew makes it slower, never wrong; this is the fixed-capacity equivalent.           */
int tg_partition_exchange_cf_spill(int device, const int64_t* key_dev, int64_t rows, int32_t nparts, int32_t ncols,
                                   const void* const* src_cols_dev, void* const* recv_cols_peer, int64_t region_base,
                                   int64_t region_cap, int64_t* sent_rows_dev, uint64_t* overflow_dev,
                                   void* const* spill_cols_dev, int64_t spill_cap, uint64_t* spill_cursor_dev,
                                   int32_t ctas_per_sm, void* stream);

/* Transfer stage of the count-free exchange on the SMs instead of the copy engines: region r = the first
 * min(counts_dev[count_index[r]], cap_rows) rows (8 bytes each) of src_dev[r] -> dst_peer[r] (a peer address mapped with
 * tg_ipc_open).  128-bit loads / stores, no shared memory, <= 32 registers: the kernel fits NEXT TO the persistent probe
 * kernel on every SM and copies only the filled part of each region (the copy engines move whole regions: the host
 * never learns the fill).  ctas = 0: one 128-thread CTA per SM.                                                        */
#define TG_COPY_MAX_REGIONS 64
int tg_peer_copy_regions(int device, int32_t n_regions, const void* const* src_dev, void* const* dst_peer,
                         const int32_t* count_index, const int64_t* counts_dev, int64_t cap_rows, int32_t ctas, void* stream);

/* Cross-GPU mailboxes — the synchronisation of the count-free exchange without NCCL and without the host: one 8-byte
 * word per (sender) in a device buffer of the RECEIVER that every sender has mapped with tg_ipc_open.
 *   tg_mail_signal: after everything already enqueued on `stream` (the scatter kernel whose peer stores it publishes),
 *                   store  epoch << 40 | values_dev[p]  into targets->slot[p] for every p (values_dev NULL: 0).
 *   tg_mail_wait  : block `stream` (a spinning 32-thread kernel, the host never waits) until every one of the n words at
 *                   mail_dev carries an epoch >= `epoch`; the low 40 bits go to values_out_dev[p] (e.g. the fill count of
 *                   sender p's region = tg_join_probe_dev_seg's seg_cnt_dev).  A sender that stays silent for
 *                   `timeout_ms` (0 = 10 s) raises *error_flag_dev = 1 + p and the wait ends: the GPU is never hung.
 * The MPP analogue: the ExchangeReceiver waiting for every sender's stream end (the reference does it over gRPC).   */
#define TG_MAIL_MAX_PEERS 16
typedef struct tg_mail_targets { int32_t n, pad; uint64_t* slot[TG_MAIL_MAX_PEERS]; } tg_mail_targets;
int tg_mail_signal(int device, const tg_mail_targets* targets, const int64_t* values_dev, int64_t epoch, void* stream);
int tg_mail_wait(int device, const uint64_t* mail_dev, int32_t n, int64_t epoch, int64_t* values_out_dev,
                 uint64_t* error_flag_dev, int64_t timeout_ms, void* stream);

/* count rows per destination (first half of the exchange: counts are all-gathered by the host) */
int tg_partition_count(int device, const int64_t* key_dev, int64_t rows, int32_t nparts,
                       int64_t* part_counts_dev, void* stream);
/* cudaIpc handle plumbing for one-process-per-GPU peer access (64-byte opaque handle)           */
int tg_ipc_export(int device, void* dev_ptr, uint8_t handle_out[64]);
int tg_ipc_open(int device, const uint8_t handle[64], void** out_ptr);
int tg_ipc_close(int device, void* mapped_ptr);

#ifdef __cplusplus
}
#endif
#endif /* TIDBGPU_H */
