// common.cuh — shared host/device helpers of libtidbgpu.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include <mutex>
#include <atomic>
#include <memory>
#include "../../include/tidbgpu.h"

namespace tg {

// ---- error plumbing ---------------------------------------------------------------------------
void set_error(const std::string& msg);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define TG_CUDA(call)                                                         \
  do {                                                                        \
    cudaError_t e__ = (call);                                                 \
    if (e__ != cudaSuccess) return tg::cuda_fail(e__, #call, __FILE__, __LINE__); \
  } while (0)

#define TG_TRY(call)                  \
  do {                                \
    int rc__ = (call);                \
    if (rc__ != TG_OK) return rc__;   \
  } while (0)

inline int fail(int code, const std::string& msg) { set_error(msg); return code; }

// pkg/util/chunk/codec.go:165-179 getFixedLen
inline int fixed_len(int tp) {
  switch (tp) {
    case TG_TYPE_FLOAT: return 4;
    case TG_TYPE_TINY: case TG_TYPE_SHORT: case TG_TYPE_INT24: case TG_TYPE_LONG: case TG_TYPE_LONGLONG:
    case TG_TYPE_DOUBLE: case TG_TYPE_YEAR: case TG_TYPE_DURATION:
    case TG_TYPE_DATE: case TG_TYPE_DATETIME: case TG_TYPE_TIMESTAMP: return 8;
    case TG_TYPE_NEWDECIMAL: return 40;
    default: return -1;
  }
}
inline bool is_int_family(int tp) {
  return tp == TG_TYPE_TINY || tp == TG_TYPE_SHORT || tp == TG_TYPE_INT24 || tp == TG_TYPE_LONG ||
         tp == TG_TYPE_LONGLONG || tp == TG_TYPE_YEAR || tp == TG_TYPE_DURATION;
}

// ---- device buffer (grow-only) ------------------------------------------------------------------
// Stream-ordered pool allocation (cudaMallocAsync on a per-device service stream, pool never trimmed): a handle's
// setup otherwise spends milliseconds in cudaMalloc / cudaFree, which also synchronise the whole device
// (profiles/r1_agg_update_global.md: 1.8 ms kernel inside a 5.2 ms one-shot aggregation).
cudaStream_t service_stream(int device);
inline cudaError_t pool_alloc(int dev, void** p, size_t bytes) {
  cudaStream_t st = service_stream(dev);
  cudaError_t e = cudaMallocAsync(p, bytes, st);
  if (e != cudaSuccess) return e;
  return cudaStreamSynchronize(st);
}
inline void pool_free(int dev, void* p) {
  // Frees are rare (growth, handle close).  Like cudaFree, wait for everything in flight first: kernels on the
  // handle's streams may still be using the buffer, and the pool may hand it out again immediately.
  if (cudaDeviceSynchronize() != cudaSuccess) cudaGetLastError();
  cudaStream_t st = service_stream(dev);
  if (cudaFreeAsync(p, st) != cudaSuccess) cudaGetLastError();
}
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  int device = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  // the caller guarantees that no kernel still uses the buffer (every handle synchronises its stream before freeing)
  void release() {
    if (p) { int prev = -1; cudaGetDevice(&prev); cudaSetDevice(device); pool_free(device, p); if (prev >= 0) cudaSetDevice(prev); p = nullptr; cap = 0; }
  }
  // contents are NOT preserved on growth
  int ensure(int dev, size_t bytes) {
    if (bytes <= cap && p) return TG_OK;
    release();
    device = dev;
    size_t want = bytes < 256 ? 256 : bytes;
    cudaError_t e = pool_alloc(dev, &p, want);
    if (e != cudaSuccess) { p = nullptr; cudaGetLastError(); return fail(TG_ERR_OOM, "device allocation failed: " + std::string(cudaGetErrorString(e))); }
    cap = want;
    return TG_OK;
  }
  // contents preserved (device-to-device copy on the given stream, then sync)
  int ensure_preserve(int dev, size_t bytes, size_t used, cudaStream_t st) {
    if (bytes <= cap && p) return TG_OK;
    size_t want = bytes < 2 * cap ? 2 * cap : bytes;
    if (want < 256) want = 256;
    void* np = nullptr;
    cudaError_t e = pool_alloc(dev, &np, want);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(TG_ERR_OOM, "device allocation failed: " + std::string(cudaGetErrorString(e))); }
    if (p && used) {
      TG_CUDA(cudaMemcpyAsync(np, p, used, cudaMemcpyDeviceToDevice, st));
      TG_CUDA(cudaStreamSynchronize(st));
    }
    if (p) pool_free(dev, p);
    p = np; cap = want; device = dev;
    return TG_OK;
  }
  template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

// pinned host buffer (grow, preserving contents)
struct PinBuf {
  uint8_t* p = nullptr;
  size_t cap = 0, used = 0;
  PinBuf() = default;
  PinBuf(const PinBuf&) = delete;
  PinBuf& operator=(const PinBuf&) = delete;
  ~PinBuf() { if (p) cudaFreeHost(p); }
  int reserve(size_t bytes) {
    if (bytes <= cap) return TG_OK;
    size_t want = bytes < 2 * cap ? 2 * cap : bytes;
    if (want < 4096) want = 4096;
    uint8_t* np = nullptr;
    cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(&np), want, cudaHostAllocDefault);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(TG_ERR_OOM, "cudaHostAlloc failed: " + std::string(cudaGetErrorString(e))); }
    if (p && used) std::memcpy(np, p, used);
    if (p) cudaFreeHost(p);
    p = np; cap = want;
    return TG_OK;
  }
};

// ---- handle graveyard ------------------------------------------------------------------------------
// Closed handle shells (tg_join / tg_agg: two mutexes, a flag and a null impl pointer) stay readable for callers that
// raced with close; only the oldest is freed once more than kGraveyardDepth have accumulated, so memory stays bounded.
constexpr size_t kGraveyardDepth = 4096;
template <typename H>
inline void bury_handle(H* h) {
  static std::mutex mu;
  static std::vector<H*> ring(kGraveyardDepth, nullptr);
  static size_t pos = 0;
  H* old = nullptr;
  { std::lock_guard<std::mutex> lk(mu); old = ring[pos]; ring[pos] = h; pos = (pos + 1) % kGraveyardDepth; }
  delete old;
}

// ---- hashing --------------------------------------------------------------------------------------
// The reference hashes the serialised key with FNV-1 64 (join/row_table_builder.go:103).  The hash only selects a
// bucket / partition, never a result, so the GPU is free to use something cheaper.  These kernels turned out to be
// instruction-bound (profiles/r1_partitioned_*): murmur's 64-bit finaliser plus a 64-bit multiply-high cost ~40 SASS
// instructions per row.  hash64 is one xor-fold and ONE 64-bit multiply (Fibonacci hashing, ~5 instructions); every
// range reduction is a 32-bit multiply-high:
//   slot   = mulhi32(hi32(h), nslots)      table slot, monotone in hi32(h)   (tables are limited to < 2^32 slots)
//   lpart  = mulhi32(hi32(h), P)           L2 partition = same top bits, so partition p owns a contiguous slot range
//   gpart  = mulhi32(remix(lo32,hi32), N)  destination GPU, from bits the slot does not use (the reference splits
//                                          top bits / low bits the same way: hash_join_v2.go:306 vs hash_table_v2.go:46)
__host__ __device__ __forceinline__ uint64_t hash64(uint64_t k) {
  k ^= k >> 32;
  return k * 0x9E3779B97F4A7C15ULL;
}
__host__ __device__ __forceinline__ uint32_t mulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * (uint64_t)b) >> 32); }
__host__ __device__ __forceinline__ uint32_t slot32(uint64_t h, uint32_t nslots) { return mulhi32((uint32_t)(h >> 32), nslots); }
__host__ __device__ __forceinline__ uint32_t part_of(uint64_t h, uint32_t nparts) {
  uint32_t g = (uint32_t)h ^ ((uint32_t)(h >> 32) * 0x85EBCA6Bu);
  g *= 0xC2B2AE35u;
  g ^= g >> 16;
  return mulhi32(g, nparts);
}
// kept for the aggregation table (64-bit slot counts are never needed there either, but its keys are group ids that
// deserve a stronger mix: low-cardinality integer ranges)
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdULL;
  k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ULL;
  k ^= k >> 33;
  return k;
}
#ifdef __CUDACC__
__device__ __forceinline__ uint64_t slot_of(uint64_t h, uint64_t nslots) { return __umul64hi(h, nslots); }
#endif

static const int64_t kEmptyKey = INT64_MIN;   // sentinel of an unoccupied slot; the key value itself
                                              // lives in a dedicated side slot (see join.cu)

// ---- null bitmap helpers (bit 1 = NOT NULL, LSB first: pkg/util/chunk/column.go:225) ------------
__host__ __device__ __forceinline__ bool bit_not_null(const uint8_t* bm, int64_t row) {
  return (bm[row >> 3] >> (row & 7)) & 1;
}

// append nbits of src (starting at src bit 0) to dst at bit position pos (host side)
void append_bits(uint8_t* dst, int64_t pos, const uint8_t* src, int64_t nbits);

// ---- host staging of pipeline breakers (tg_agg_push / tg_sort_push) ------------------------------------------------
// Child chunks arrive as small host chunks (1024 rows) with an optional sel vector; they are appended, sel applied, into
// pinned buffers that are flushed to the device in batches of millions of rows.  Per column: 8-byte values and, once any
// chunk carried a bitmap, a null bitmap (earlier rows all NOT NULL).  Only columns with needed[c] != 0 are staged.
struct ColumnStage {
  std::vector<std::unique_ptr<PinBuf>> data, nulls;
  std::vector<char> has_nulls;
  int64_t rows = 0;
  void init(int ncols) {
    for (int c = 0; c < ncols; c++) { data.emplace_back(new PinBuf()); nulls.emplace_back(new PinBuf()); }
    has_nulls.assign(ncols, 0);
  }
};
inline int64_t logical_rows(const tg_chunk* c) { return c->sel ? c->nsel : (c->ncols > 0 ? c->cols[0].length : 0); }
int stage_append(ColumnStage& st, const tg_chunk* chk, const std::vector<char>& needed);

// Copy rows [lo, lo + want) of ncols device-resident 8-byte columns to the caller's host chunk (the Next of a pipeline
// breaker).  bitmaps[k] = packed device null bitmap of column k, or nullptr when the column has no NULLs.  Any `lo` is
// served: a bitmap slice that starts inside a byte is fetched whole and shifted on the host.  Synchronises `st`.
int copy_out_rows(cudaStream_t st, int ncols, const void* const* cols, const uint8_t* const* bitmaps, int64_t lo,
                  int64_t want, tg_mut_chunk* out, int64_t* d2h_bytes);

// device ordinal guard
struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; cudaGetLastError(); }
    if (cudaSetDevice(dev) != cudaSuccess) { ok = false; cudaGetLastError(); }
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

int device_sm_count(int device);

// scalar filter program passed to kernels by value
#define TG_MAX_COLS 16
#define TG_MAX_FILTER 8
struct DevCols {
  const void* data[TG_MAX_COLS];
  const uint8_t* nulls[TG_MAX_COLS];
  int32_t elem_len[TG_MAX_COLS];
};
struct DevFilter {
  int32_t n;
  int32_t pad;
  tg_filter_item items[TG_MAX_FILTER];
};

#ifdef __CUDACC__
__device__ __forceinline__ int cmp_int(int64_t a, bool ua, int64_t b, bool ub) {
  // types.CompareInt pkg/types/compare.go:86
  if (ua && ub) { uint64_t x = (uint64_t)a, y = (uint64_t)b; return x < y ? -1 : (x == y ? 0 : 1); }
  if (ua && !ub) { if (b < 0 || (uint64_t)a > (uint64_t)INT64_MAX) return 1; }
  else if (!ua && ub) { if (a < 0 || (uint64_t)b > (uint64_t)INT64_MAX) return -1; }
  return a < b ? -1 : (a == b ? 0 : 1);
}
__device__ __forceinline__ int cmp_real(double a, double b) {
  // Go cmp.Compare: NaN < everything, NaN == NaN
  bool an = a != a, bn = b != b;
  if (an) return bn ? 0 : -1;
  if (bn) return 1;
  return a < b ? -1 : (a > b ? 1 : 0);
}
__device__ __forceinline__ bool apply_cmp(int op, int c) {
  switch (op) {
    case TG_CMP_LT: return c < 0;
    case TG_CMP_LE: return c <= 0;
    case TG_CMP_GT: return c > 0;
    case TG_CMP_GE: return c >= 0;
    case TG_CMP_EQ: return c == 0;
    default: return c != 0;
  }
}
// VecEvalBool semantics (expression.go:409-494): selected iff every CNF item is non-NULL true
__device__ __forceinline__ bool eval_filter(const DevFilter& f, const DevCols& c, int64_t row) {
  for (int i = 0; i < f.n; i++) {
    const tg_filter_item& it = f.items[i];
    const uint8_t* ln = c.nulls[it.lhs_col];
    if (ln && !bit_not_null(ln, row)) return false;
    int r;
    if (it.rhs_col >= 0) {
      const uint8_t* rn = c.nulls[it.rhs_col];
      if (rn && !bit_not_null(rn, row)) return false;
    }
    if (it.is_real) {
      double x = reinterpret_cast<const double*>(c.data[it.lhs_col])[row];
      double y = it.rhs_col >= 0 ? reinterpret_cast<const double*>(c.data[it.rhs_col])[row] : it.const_f64;
      r = cmp_real(x, y);
    } else {
      int64_t x = reinterpret_cast<const int64_t*>(c.data[it.lhs_col])[row];
      int64_t y = it.rhs_col >= 0 ? reinterpret_cast<const int64_t*>(c.data[it.rhs_col])[row] : it.const_i64;
      r = cmp_int(x, it.lhs_unsigned != 0, y, it.rhs_unsigned != 0);
    }
    if (!apply_cmp(it.op, r)) return false;
  }
  return true;
}
#endif

}  // namespace tg
