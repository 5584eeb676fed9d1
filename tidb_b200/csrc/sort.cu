// sort.cu — tg_sort_*: SortExec (pkg/executor/sortexec/sort.go:43) for ORDER BY without LIMIT on the device.
//
// The reference sorts row pointers with SortExec.lessRow (sort.go:804): ORDER BY items one after another, each with
// chunk.GetCompareFunc (util/chunk/compare.go:30-60; NULL first, DESC negated).  Here the items become one exact,
// order-preserving u64 key each and the rows are sorted by a key-index LSD radix sort (8-bit digits), items last to first:
//   1. k_sort_key_hist : key[i] = norm(col[idx[i]]) (the gather through the current permutation is fused into the key
//                        pass; the first item reads no index) plus all eight 256-bin digit histograms in the same read
//                        (Onesweep's global histogram, Adinets & Merrill 2022).  One 8 KB D2H per item lets the host
//                        skip every digit whose histogram has a single non-empty bin.
//   2. k_sort_scatter  : one launch per remaining digit: a stable scatter of (u64 key, u32 row id) pairs with decoupled
//                        look-back across 4096-row tiles.
//   3. NULL pass       : an item whose column has a bitmap gets one more stable pass on the NOT-NULL flag after its digit
//                        passes (same two kernels, key = one bit).  NULL rows carry key 0 in the digit passes, so they
//                        keep the order of the less significant items.
//   4. k_sort_gather   : every column permuted by the final row ids, output bitmaps built by warp ballot.
// Row ids are u32: at most 2^32 - 1 rows per sort.
#include <algorithm>
#include <memory>
#include <vector>
#include "common.cuh"

namespace tg {

// key kinds (chunk.GetCompareFunc): cmpInt64 (int family, YEAR, DURATION), cmpUint64, cmpFloat64, cmpTime
enum { SK_SIGNED = 0, SK_UNSIGNED = 1, SK_REAL = 2, SK_TIME = 3, SK_NULLFLAG = 4 };

// Exact order-preserving map of a non-NULL value to u64.  Unlike TopN's rank_of (a lossy candidate filter) no two values
// that compare differently share a key and no two values that compare equal get different ones: -0.0 == +0.0, every NaN
// is one key below -inf (Go cmp.Compare), time words lose their fsp bits (types/time.go:235-251, compareTime
// core_time.go:256 compares the calendar fields and microseconds only).
__host__ __device__ __forceinline__ unsigned long long sort_key(unsigned long long raw, int kind, bool desc) {
  unsigned long long o;
  if (kind == SK_SIGNED) o = raw ^ 0x8000000000000000ull;
  else if (kind == SK_UNSIGNED) o = raw;
  else if (kind == SK_TIME) o = raw & ~0xFull;
  else {
    const bool nan = (raw & 0x7FF0000000000000ull) == 0x7FF0000000000000ull && (raw & 0x000FFFFFFFFFFFFFull);
    if (nan) o = 0ull;                                     // -inf maps to 0x000F..F; only NaN words map to 0 otherwise
    else {
      if (raw == 0x8000000000000000ull) raw = 0ull;        // -0.0 -> +0.0
      o = (raw >> 63) ? ~raw : (raw | 0x8000000000000000ull);
    }
  }
  return desc ? ~o : o;
}

static int sort_kind_of(int tp, uint32_t flag) {
  if (tp == TG_TYPE_DOUBLE) return SK_REAL;
  if (tp == TG_TYPE_DURATION) return SK_SIGNED;                            // cmpDuration: cmp.Compare(int64), compare.go:138
  if (is_int_family(tp)) return (flag & TG_FLAG_UNSIGNED) ? SK_UNSIGNED : SK_SIGNED;
  if (tp == TG_TYPE_DATE || tp == TG_TYPE_DATETIME || tp == TG_TYPE_TIMESTAMP) return SK_TIME;
  return -1;
}

constexpr int kHistThreads = 256;
constexpr int kSortThreads = 256, kSortItems = 16, kSortTile = kSortThreads * kSortItems, kSortWarps = kSortThreads / 32;
constexpr size_t kScatterSmem = (size_t)kSortTile * 8 + (size_t)kSortTile * 4 + (size_t)kSortWarps * 256 * 4;
constexpr unsigned long long kLbAggregate = 1ull << 62, kLbInclusive = 2ull << 62, kLbCount = (1ull << 62) - 1;

// key pass of one ORDER BY item (or of its NULL flag, kind == SK_NULLFLAG) + the eight digit histograms of the keys
__global__ void __launch_bounds__(kHistThreads)
k_sort_key_hist(const unsigned long long* __restrict__ col, const uint8_t* __restrict__ nulls, const uint32_t* __restrict__ idx,
                uint32_t n, int kind, int desc, unsigned long long* __restrict__ keys, uint32_t* __restrict__ hist) {
  __shared__ uint32_t s_h[8 * 256];
  for (int i = threadIdx.x; i < 8 * 256; i += kHistThreads) s_h[i] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  // every lane of a warp runs the same iterations (base is warp aligned), so the warp votes below see all 32 lanes
  for (uint64_t base = (uint64_t)blockIdx.x * kHistThreads; base < n; base += (uint64_t)gridDim.x * kHistThreads) {
    const uint64_t i = base + threadIdx.x;
    const bool valid = i < n;
    unsigned long long key = 0;
    if (valid) {
      const uint64_t r = idx ? idx[i] : i;
      const bool is_null = nulls && !bit_not_null(nulls, (int64_t)r);
      if (kind == SK_NULLFLAG) key = (unsigned long long)((is_null ? 0 : 1) ^ (desc ? 1 : 0));   // ASC: NULL first; DESC: last
      else key = is_null ? 0ull : sort_key(col[r], kind, desc != 0);
      keys[i] = key;
    }
    const unsigned vmask = __ballot_sync(0xffffffffu, valid);
    if (!vmask) continue;                                  // lane 0 is valid from here on
#pragma unroll
    for (int b = 0; b < 8; b++) {
      const uint32_t d = (uint32_t)(key >> (8 * b)) & 0xFFu;
      const uint32_t d0 = __shfl_sync(0xffffffffu, d, 0);
      // a byte that is equal across the warp (high bytes of small ints, dates, constants) is one shared-memory atomic
      if (__all_sync(0xffffffffu, !valid || d == d0)) { if (lane == 0) atomicAdd(&s_h[b * 256 + d0], (uint32_t)__popc(vmask)); }
      else if (valid) atomicAdd(&s_h[b * 256 + d], 1u);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 8 * 256; i += kHistThreads) if (s_h[i]) atomicAdd(&hist[i], s_h[i]);
}

struct DigitOffsets { uint32_t off[256]; };   // exclusive prefix of the digit's global histogram

__device__ __forceinline__ unsigned long long ld_relaxed(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_relaxed(unsigned long long* p, unsigned long long v) {
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// One stable counting-sort pass on the digit at `shift`: (keys_in, vals_in) -> (keys_out, vals_out).  vals_in == nullptr:
// the row ids are the positions (first pass of the sort).  One CTA per 4096-row tile; tile ids come from a global atomic
// counter, in the order CTAs start, so the look-back of tile t only ever waits for tiles < t, which have already started
// and publish their counts without waiting on anybody: progress does not depend on the order the hardware schedules CTAs.
// lookback: [tiles][256] status words (2-bit flag | 62-bit count), zeroed with the counter before the launch.
__global__ void __launch_bounds__(kSortThreads, 3)
k_sort_scatter(const unsigned long long* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
               unsigned long long* __restrict__ keys_out, uint32_t* __restrict__ vals_out, uint32_t n, int shift,
               DigitOffsets g, unsigned long long* __restrict__ lookback, uint32_t* __restrict__ tile_counter) {
  extern __shared__ __align__(16) unsigned char smem[];
  unsigned long long* s_keys = reinterpret_cast<unsigned long long*>(smem);
  uint32_t* s_vals = reinterpret_cast<uint32_t*>(smem + (size_t)kSortTile * 8);
  uint32_t* s_whist = reinterpret_cast<uint32_t*>(smem + (size_t)kSortTile * 12);   // [warp][digit]
  __shared__ uint32_t s_start[256], s_wsum[kSortWarps], s_tile;
  __shared__ unsigned long long s_gbase[256];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(tile_counter, 1u);
  for (int i = tid; i < kSortWarps * 256; i += kSortThreads) s_whist[i] = 0;
  __syncthreads();
  const uint32_t tile = s_tile;
  const uint64_t tbase = (uint64_t)tile * kSortTile;
  const uint64_t wbase = tbase + (uint64_t)warp * 32 * kSortItems;
  uint32_t* wh = s_whist + warp * 256;
  const unsigned lt_mask = (1u << lane) - 1u;

  // rank inside the warp: warp-striped rows (row = wbase + j*32 + lane), so j-major, lane-minor order is row order and
  // the rank of a row among the warp's rows with its digit is stable
  unsigned long long k[kSortItems];
  uint32_t rank[kSortItems];
#pragma unroll
  for (int j = 0; j < kSortItems; j++) {
    const uint64_t i = wbase + (uint64_t)j * 32 + lane;
    k[j] = i < n ? __ldcs(keys_in + i) : 0ull;
  }
#pragma unroll
  for (int j = 0; j < kSortItems; j++) {
    const uint64_t i = wbase + (uint64_t)j * 32 + lane;
    const uint32_t d = i < n ? ((uint32_t)(k[j] >> shift) & 0xFFu) : 256u;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const uint32_t below = (uint32_t)__popc(peers & lt_mask);
    const uint32_t pre = d < 256 ? wh[d] : 0u;
    rank[j] = pre + below;
    __syncwarp();
    if (d < 256 && below == 0) wh[d] = pre + (uint32_t)__popc(peers);
    __syncwarp();
  }
  __syncthreads();

  // thread b owns digit b: warp offsets inside the tile, tile count, publish, look back
  const int b = tid;
  uint32_t cnt = 0;
#pragma unroll
  for (int w = 0; w < kSortWarps; w++) { const uint32_t c = s_whist[w * 256 + b]; s_whist[w * 256 + b] = cnt; cnt += c; }
  unsigned long long* my_lb = lookback + (size_t)tile * 256 + b;
  st_relaxed(my_lb, (tile == 0 ? kLbInclusive : kLbAggregate) | cnt);
  // exclusive scan of the tile's digit counts -> where each digit starts inside the tile
  uint32_t x = cnt;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
  if (lane == 31) s_wsum[warp] = x;
  unsigned long long prefix = 0;
  if (tile > 0) {
    for (int64_t t = (int64_t)tile - 1; t >= 0;) {
      const unsigned long long v = ld_relaxed(lookback + (size_t)t * 256 + b);
      const unsigned long long flag = v & ~kLbCount;
      if (flag == 0) continue;                             // tile t has started but not published yet
      prefix += v & kLbCount;
      if (flag == kLbInclusive) break;
      t--;
    }
    st_relaxed(my_lb, kLbInclusive | (prefix + cnt));
  }
  s_gbase[b] = (unsigned long long)g.off[b] + prefix;
  __syncthreads();
  uint32_t wprefix = 0;
  for (int w = 0; w < warp; w++) wprefix += s_wsum[w];
  s_start[b] = wprefix + x - cnt;
  __syncthreads();

  // place the tile in shared memory in (digit, row) order, then write it out: rows of one digit go to consecutive
  // global addresses
#pragma unroll
  for (int j = 0; j < kSortItems; j++) {
    const uint64_t i = wbase + (uint64_t)j * 32 + lane;
    if (i < n) {
      const uint32_t d = (uint32_t)(k[j] >> shift) & 0xFFu;
      const uint32_t pos = s_start[d] + wh[d] + rank[j];
      s_keys[pos] = k[j];
      s_vals[pos] = vals_in ? __ldcs(vals_in + i) : (uint32_t)i;
    }
  }
  __syncthreads();
  const uint32_t tile_n = (uint32_t)min((uint64_t)kSortTile, (uint64_t)n - tbase);
  for (uint32_t i = tid; i < tile_n; i += kSortThreads) {
    const unsigned long long key = s_keys[i];
    const uint32_t d = (uint32_t)(key >> shift) & 0xFFu;
    const uint64_t dst = s_gbase[d] + (i - s_start[d]);
    keys_out[dst] = key;
    vals_out[dst] = s_vals[i];
  }
}

struct SortCols {
  const unsigned long long* in[TG_MAX_COLS];
  const uint8_t* in_nulls[TG_MAX_COLS];
  unsigned long long* out[TG_MAX_COLS];
  uint32_t* out_nulls[TG_MAX_COLS];       // packed bitmap, one 32-bit word per 32 rows; nullptr: the column has no NULLs
};

// out[c][i] = in[c][perm[i]] for every column; bitmaps by warp ballot, one 32-bit store per 32 rows.  Every column's
// random load is issued before the first store (a store could alias a later load), so a thread keeps ncols loads in flight.
__global__ void __launch_bounds__(256)
k_sort_gather(SortCols sc, int ncols, const uint32_t* __restrict__ perm, uint32_t n) {
  const int lane = threadIdx.x & 31;
  for (uint64_t base = (uint64_t)blockIdx.x * blockDim.x; base < n; base += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t i = base + threadIdx.x;
    const bool valid = i < n;
    const uint64_t r = valid ? (perm ? __ldcs(perm + i) : i) : 0;
    unsigned long long v[TG_MAX_COLS];
#pragma unroll
    for (int c = 0; c < TG_MAX_COLS; c++) if (c < ncols && valid) v[c] = __ldg(sc.in[c] + r);
#pragma unroll
    for (int c = 0; c < TG_MAX_COLS; c++) {
      if (c >= ncols) break;
      if (valid) __stcs(sc.out[c] + i, v[c]);
      if (sc.in_nulls[c]) {
        const unsigned m = __ballot_sync(0xffffffffu, valid && bit_not_null(sc.in_nulls[c], (int64_t)r));
        if (lane == 0 && valid) sc.out_nulls[c][i >> 5] = m;
      }
    }
  }
}

// bits [pos, pos + nbits) of dst = src bits [0, nbits) (src == nullptr: all NOT NULL); other bits of dst are kept
__global__ void __launch_bounds__(256)
k_sort_append_bits(uint8_t* __restrict__ dst, int64_t pos, const uint8_t* __restrict__ src, int64_t nbits) {
  const int64_t first = pos >> 3, last = (pos + nbits - 1) >> 3;
  for (int64_t byte = first + blockIdx.x * (int64_t)blockDim.x + threadIdx.x; byte <= last; byte += (int64_t)gridDim.x * blockDim.x) {
    uint8_t v = dst[byte];
    for (int bit = 0; bit < 8; bit++) {
      const int64_t gbit = byte * 8 + bit;
      if (gbit < pos || gbit >= pos + nbits) continue;
      const int64_t s = gbit - pos;
      const bool nn = src ? ((src[s >> 3] >> (s & 7)) & 1) : true;
      v = nn ? (uint8_t)(v | (1u << bit)) : (uint8_t)(v & ~(1u << bit));
    }
    dst[byte] = v;
  }
}

}  // namespace tg

using namespace tg;

struct SortImpl;

// shell + implementation, like tg_agg (agg.cu): close frees the implementation, the shell stays readable
struct tg_sort {
  std::mutex mu;
  std::atomic<bool> closed{false};
  SortImpl* impl = nullptr;
};

struct SortImpl {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
  int nsm = 148;

  int ncols = 0;
  std::vector<int> types, kinds;
  std::vector<tg_sort_item> items;
  int64_t expected_rows = 0;

  // input: staged host chunks are appended to owned device columns; a single device chunk is used in place (borrowed)
  ColumnStage stage;
  std::vector<char> all_cols;
  std::vector<std::unique_ptr<DevBuf>> in_data, in_nulls;
  std::vector<char> in_has_nulls;
  int64_t in_rows = 0;
  bool borrowed = false;
  std::vector<const void*> b_data;
  std::vector<const uint8_t*> b_nulls;
  int64_t b_rows = 0;
  DevBuf tmp_bits;

  // sort scratch
  DevBuf keys[2], vals[2], hist, lookback;

  // result
  bool finished = false;
  std::vector<std::unique_ptr<DevBuf>> out_cols, out_bitmaps;
  std::vector<char> out_has_nulls;
  int64_t out_rows = 0, consumed = 0;
  tg_sort_stats stats{};
};

namespace tg {

static int sort_setup(SortImpl* s, const tg_sort_desc* d) {
  if (!d) return fail(TG_ERR_INVALID, "descriptor is NULL");
  if (!d->col_types || !d->items) return fail(TG_ERR_INVALID, "col_types / items is NULL");
  if (d->n_cols < 1) return fail(TG_ERR_INVALID, "the child schema has no columns");
  if (d->n_cols > TG_MAX_COLS) return fail(TG_ERR_UNSUPPORTED, "the GPU sort handles up to 16 columns");
  if (d->n_items < 1 || d->n_items > 8) return fail(TG_ERR_UNSUPPORTED, "1..8 ORDER BY items are offloaded");
  if (d->expected_rows < 0) return fail(TG_ERR_INVALID, "expected_rows is negative");
  s->ncols = d->n_cols;
  s->types.assign(d->col_types, d->col_types + d->n_cols);
  s->kinds.resize(d->n_cols);
  for (int c = 0; c < d->n_cols; c++) {
    s->kinds[c] = sort_kind_of(s->types[c], d->col_flags ? d->col_flags[c] : 0);
    // FLOAT (4 bytes), DECIMAL (40 bytes) and var-len columns stay on the CPU, as ORDER BY items and as payload
    if (s->kinds[c] < 0) return fail(TG_ERR_UNSUPPORTED, "the GPU sort handles 8-byte int family / YEAR / DURATION / DOUBLE / DATE / DATETIME / TIMESTAMP columns only");
  }
  s->items.assign(d->items, d->items + d->n_items);
  for (const tg_sort_item& it : s->items)
    if (it.col < 0 || it.col >= d->n_cols) return fail(TG_ERR_INVALID, "ORDER BY column out of range");
  s->device = d->device;
  s->expected_rows = d->expected_rows;
  s->all_cols.assign(d->n_cols, 1);
  return TG_OK;
}

static int sgrid(const SortImpl* s, int64_t n, int block = 256, int per_sm = 8) {
  int64_t need = (n + block - 1) / block, cap = (int64_t)s->nsm * per_sm;
  if (need < 1) need = 1;
  return (int)(need < cap ? need : cap);
}

static int svalidate(const SortImpl* s, const tg_chunk* chk) {
  if (!chk || chk->ncols != s->ncols || !chk->cols) return fail(TG_ERR_INVALID, "chunk column count does not match the child schema");
  for (int c = 0; c < s->ncols; c++) {
    if (chk->cols[c].elem_len != 8) return fail(TG_ERR_INVALID, "chunk column elem_len does not match the schema type");
    if (chk->cols[c].length != chk->cols[0].length) return fail(TG_ERR_INVALID, "chunk columns have different lengths");
  }
  return TG_OK;
}

static int64_t sort_rows_pending(const SortImpl* s) { return s->in_rows + s->b_rows + s->stage.rows; }

static int check_row_limit(int64_t rows) {
  if (rows > (int64_t)UINT32_MAX) return fail(TG_ERR_UNSUPPORTED, "the GPU sort handles at most 2^32 - 1 rows (32-bit row ids)");
  return TG_OK;
}

// append n rows to the owned device input: data[c] / nulls[c] are device pointers, or pinned host pointers when `host`
static int append_input(SortImpl* s, const void* const* data, const uint8_t* const* nulls, int64_t n, bool host) {
  if (n == 0) return TG_OK;
  const int64_t rows = s->in_rows + n;
  const int64_t want = std::max(rows, s->expected_rows);
  const cudaMemcpyKind kind = host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  for (int c = 0; c < s->ncols; c++) {
    TG_TRY(s->in_data[c]->ensure_preserve(s->device, (size_t)want * 8 + 16, (size_t)s->in_rows * 8, s->stream));
    TG_CUDA(cudaMemcpyAsync(s->in_data[c]->as<uint8_t>() + (size_t)s->in_rows * 8, data[c], (size_t)n * 8, kind, s->stream));
    if (host) s->stats.h2d_bytes += n * 8;
    if (!nulls[c] && !s->in_has_nulls[c]) continue;
    TG_TRY(s->in_nulls[c]->ensure_preserve(s->device, (size_t)(want + 7) / 8 + 16, s->in_has_nulls[c] ? (size_t)(s->in_rows + 7) / 8 : 0, s->stream));
    uint8_t* bm = s->in_nulls[c]->as<uint8_t>();
    if (!s->in_has_nulls[c] && s->in_rows) {       // the first bitmap of this column: the rows before it are NOT NULL
      k_sort_append_bits<<<sgrid(s, (s->in_rows + 7) / 8 + 1), 256, 0, s->stream>>>(bm, 0, nullptr, s->in_rows);
      s->stats.kernel_launches++;
    }
    s->in_has_nulls[c] = 1;
    const uint8_t* src = nulls[c];
    if (src && host) {
      const size_t nb = (size_t)(n + 7) / 8;
      TG_TRY(s->tmp_bits.ensure(s->device, nb + 16));
      TG_CUDA(cudaMemcpyAsync(s->tmp_bits.p, src, nb, cudaMemcpyHostToDevice, s->stream));
      s->stats.h2d_bytes += nb;
      src = s->tmp_bits.as<uint8_t>();
    }
    k_sort_append_bits<<<sgrid(s, (n + 7) / 8 + 1), 256, 0, s->stream>>>(bm, s->in_rows, src, n);
    s->stats.kernel_launches++;
    if (host) TG_CUDA(cudaStreamSynchronize(s->stream));   // tmp_bits is reused by the next column
  }
  s->in_rows = rows;
  TG_CUDA(cudaStreamSynchronize(s->stream));               // the pinned staging buffers are reused after this
  TG_CUDA(cudaGetLastError());
  return TG_OK;
}

// a borrowed device chunk becomes owned as soon as a second piece of input arrives
static int materialize_borrowed(SortImpl* s) {
  if (!s->borrowed) return TG_OK;
  s->borrowed = false;
  const int64_t n = s->b_rows;
  s->b_rows = 0;
  return append_input(s, s->b_data.data(), s->b_nulls.data(), n, false);
}

static int sflush(SortImpl* s) {
  ColumnStage& st = s->stage;
  if (st.rows == 0) return TG_OK;
  TG_TRY(materialize_borrowed(s));
  std::vector<const void*> data(s->ncols);
  std::vector<const uint8_t*> nulls(s->ncols);
  for (int c = 0; c < s->ncols; c++) { data[c] = st.data[c]->p; nulls[c] = st.has_nulls[c] ? st.nulls[c]->p : nullptr; }
  const int64_t n = st.rows;
  st.rows = 0;
  std::fill(st.has_nulls.begin(), st.has_nulls.end(), 0);
  return append_input(s, data.data(), nulls.data(), n, true);
}

// D2H of one item's eight digit histograms
static int read_hist(SortImpl* s, uint32_t* h) {
  TG_CUDA(cudaMemcpyAsync(h, s->hist.p, 8 * 256 * 4, cudaMemcpyDeviceToHost, s->stream));
  TG_CUDA(cudaStreamSynchronize(s->stream));
  s->stats.d2h_bytes += 8 * 256 * 4;
  return TG_OK;
}

static int ssort(SortImpl* s, const unsigned long long* const* cols, const uint8_t* const* nulls, uint32_t n, const uint32_t** perm_out) {
  *perm_out = nullptr;
  if (n == 0) return TG_OK;
  const uint32_t tiles = (n + kSortTile - 1) / kSortTile;
  for (int q = 0; q < 2; q++) {
    TG_TRY(s->keys[q].ensure(s->device, (size_t)n * 8 + 16));
    TG_TRY(s->vals[q].ensure(s->device, (size_t)n * 4 + 16));
  }
  TG_TRY(s->hist.ensure(s->device, 8 * 256 * 4));
  TG_TRY(s->lookback.ensure(s->device, (size_t)tiles * 256 * 8 + 64));
  static bool smem_set[64] = {};
  if (!smem_set[s->device & 63]) {
    TG_CUDA(cudaFuncSetAttribute(k_sort_scatter, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kScatterSmem));
    smem_set[s->device & 63] = true;
  }
  unsigned long long* lb = s->lookback.as<unsigned long long>();
  uint32_t* counter = reinterpret_cast<uint32_t*>(lb + (size_t)tiles * 256);
  int cur = 0;                       // keys[cur] / vals[cur] hold the current order
  const uint32_t* perm = nullptr;    // nullptr: identity (nothing moved yet)
  std::vector<uint32_t> h(8 * 256);
  auto scatter = [&](int shift, const uint32_t* bins) -> int {
    DigitOffsets g;
    uint32_t run = 0;
    for (int b = 0; b < 256; b++) { g.off[b] = run; run += bins[b]; }
    TG_CUDA(cudaMemsetAsync(lb, 0, (size_t)tiles * 256 * 8 + 64, s->stream));
    k_sort_scatter<<<tiles, kSortThreads, kScatterSmem, s->stream>>>(s->keys[cur].as<unsigned long long>(), perm,
        s->keys[cur ^ 1].as<unsigned long long>(), s->vals[cur ^ 1].as<uint32_t>(), n, shift, g, lb, counter);
    s->stats.kernel_launches++;
    cur ^= 1;
    perm = s->vals[cur].as<uint32_t>();
    return TG_OK;
  };
  auto nonempty = [](const uint32_t* bins) { int k = 0; for (int b = 0; b < 256; b++) k += bins[b] != 0; return k; };
  for (int q = (int)s->items.size() - 1; q >= 0; q--) {
    const int c = s->items[q].col;
    const int desc = s->items[q].desc != 0;
    TG_CUDA(cudaMemsetAsync(s->hist.p, 0, 8 * 256 * 4, s->stream));
    k_sort_key_hist<<<sgrid(s, n, kHistThreads, 8), kHistThreads, 0, s->stream>>>(cols[c], nulls[c], perm, n, s->kinds[c], desc,
                                                                                    s->keys[cur].as<unsigned long long>(), s->hist.as<uint32_t>());
    s->stats.kernel_launches++;
    TG_TRY(read_hist(s, h.data()));
    for (int b = 0; b < 8; b++) {
      if (nonempty(&h[b * 256]) <= 1) { s->stats.skipped_passes++; continue; }
      TG_TRY(scatter(8 * b, &h[b * 256]));
      s->stats.digit_passes++;
    }
    if (!nulls[c]) continue;
    TG_CUDA(cudaMemsetAsync(s->hist.p, 0, 8 * 256 * 4, s->stream));
    k_sort_key_hist<<<sgrid(s, n, kHistThreads, 8), kHistThreads, 0, s->stream>>>(cols[c], nulls[c], perm, n, SK_NULLFLAG, desc,
                                                                                    s->keys[cur].as<unsigned long long>(), s->hist.as<uint32_t>());
    s->stats.kernel_launches++;
    TG_TRY(read_hist(s, h.data()));
    if (nonempty(&h[0]) > 1) { TG_TRY(scatter(0, &h[0])); s->stats.null_passes++; }
  }
  *perm_out = perm;
  return TG_OK;
}

static int sfinish(SortImpl* s) {
  TG_TRY(sflush(s));
  const int64_t n64 = sort_rows_pending(s);
  TG_TRY(check_row_limit(n64));
  const uint32_t n = (uint32_t)n64;
  std::vector<const unsigned long long*> cols(s->ncols);
  std::vector<const uint8_t*> nulls(s->ncols);
  for (int c = 0; c < s->ncols; c++) {
    cols[c] = reinterpret_cast<const unsigned long long*>(s->borrowed ? s->b_data[c] : s->in_data[c]->p);
    nulls[c] = s->borrowed ? s->b_nulls[c] : (s->in_has_nulls[c] ? s->in_nulls[c]->as<uint8_t>() : nullptr);
  }
  s->stats.input_rows = n64;
  TG_CUDA(cudaEventRecord(s->ev0, s->stream));
  const uint32_t* perm = nullptr;
  TG_TRY(ssort(s, cols.data(), nulls.data(), n, &perm));
  TG_CUDA(cudaEventRecord(s->ev1, s->stream));
  SortCols sc{};
  s->out_has_nulls.assign(s->ncols, 0);
  for (int c = 0; c < s->ncols; c++) {
    TG_TRY(s->out_cols[c]->ensure(s->device, (size_t)n * 8 + 16));
    sc.in[c] = cols[c];
    sc.in_nulls[c] = nulls[c];
    sc.out[c] = s->out_cols[c]->as<unsigned long long>();
    if (nulls[c]) {
      TG_TRY(s->out_bitmaps[c]->ensure(s->device, ((size_t)n + 31) / 32 * 4 + 16));
      sc.out_nulls[c] = s->out_bitmaps[c]->as<uint32_t>();
      s->out_has_nulls[c] = 1;
    }
  }
  if (n) { k_sort_gather<<<sgrid(s, n), 256, 0, s->stream>>>(sc, s->ncols, perm, n); s->stats.kernel_launches++; }
  TG_CUDA(cudaEventRecord(s->ev2, s->stream));
  TG_CUDA(cudaStreamSynchronize(s->stream));
  TG_CUDA(cudaGetLastError());
  float ms = 0;
  cudaEventElapsedTime(&ms, s->ev0, s->ev1); s->stats.sort_ms += ms;
  cudaEventElapsedTime(&ms, s->ev1, s->ev2); s->stats.gather_ms += ms;
  s->out_rows = n64;
  s->consumed = 0;
  // the scratch is not needed any more; a borrowed input is not touched after finish
  for (int q = 0; q < 2; q++) { s->keys[q].release(); s->vals[q].release(); }
  s->lookback.release();
  s->borrowed = false;
  return TG_OK;
}

}  // namespace tg

#define TGS_LOCK(h)                                                            \
  if (!(h)) return tg::fail(TG_ERR_INVALID, "handle is NULL");                 \
  if ((h)->closed.load()) return tg::fail(TG_ERR_CANCELLED, "handle is closed"); \
  std::lock_guard<std::mutex> lock__((h)->mu);                                 \
  if ((h)->closed.load() || !(h)->impl) return tg::fail(TG_ERR_CANCELLED, "handle is closed"); \
  SortImpl* s = (h)->impl;                                                     \
  tg::DeviceGuard guard__(s->device);                                          \
  if (!guard__.ok) return tg::fail(TG_ERR_CUDA, "cudaSetDevice failed (no usable CUDA device)")

extern "C" {

int tg_sort_supported(const tg_sort_desc* desc) { SortImpl tmp; return sort_setup(&tmp, desc); }

int tg_sort_open(const tg_sort_desc* desc, tg_sort** out) {
  if (!out) return fail(TG_ERR_INVALID, "out is NULL");
  *out = nullptr;
  std::unique_ptr<tg_sort> shell(new tg_sort());
  std::unique_ptr<SortImpl> s(new SortImpl());
  TG_TRY(sort_setup(s.get(), desc));
  TG_TRY(check_row_limit(s->expected_rows));
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return fail(TG_ERR_CUDA, "no CUDA device: the GPU sort has no CPU fallback"); }
  if (s->device < 0 || s->device >= ndev) return fail(TG_ERR_INVALID, "device ordinal out of range");
  DeviceGuard g(s->device);
  if (!g.ok) return fail(TG_ERR_CUDA, "cudaSetDevice failed");
  if (desc->stream) { s->stream = (cudaStream_t)desc->stream; s->own_stream = false; }
  else { TG_CUDA(cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking)); s->own_stream = true; }
  TG_CUDA(cudaEventCreate(&s->ev0));
  TG_CUDA(cudaEventCreate(&s->ev1));
  TG_CUDA(cudaEventCreate(&s->ev2));
  s->nsm = device_sm_count(s->device);
  s->stage.init(s->ncols);
  for (int c = 0; c < s->ncols; c++) {
    s->in_data.emplace_back(new DevBuf()); s->in_nulls.emplace_back(new DevBuf());
    s->out_cols.emplace_back(new DevBuf()); s->out_bitmaps.emplace_back(new DevBuf());
  }
  s->in_has_nulls.assign(s->ncols, 0);
  shell->impl = s.release();
  *out = shell.release();
  return TG_OK;
}

int tg_sort_push(tg_sort* h, const tg_chunk* chk) {
  TGS_LOCK(h);
  if (s->finished) return fail(TG_ERR_STATE, "push after finish");
  TG_TRY(svalidate(s, chk));
  TG_TRY(check_row_limit(sort_rows_pending(s) + logical_rows(chk)));
  TG_TRY(stage_append(s->stage, chk, s->all_cols));
  if (s->stage.rows >= (4ll << 20)) TG_TRY(sflush(s));
  return TG_OK;
}

int tg_sort_push_dev(tg_sort* h, const tg_chunk* chk) {
  TGS_LOCK(h);
  if (s->finished) return fail(TG_ERR_STATE, "push after finish");
  TG_TRY(svalidate(s, chk));
  if (chk->sel) return fail(TG_ERR_UNSUPPORTED, "device-resident chunks must not carry a sel vector");
  const int64_t n = chk->cols[0].length;
  if (n == 0) return TG_OK;
  TG_TRY(check_row_limit(sort_rows_pending(s) + n));
  std::vector<const void*> data(s->ncols);
  std::vector<const uint8_t*> nulls(s->ncols);
  for (int c = 0; c < s->ncols; c++) { data[c] = chk->cols[c].data; nulls[c] = chk->cols[c].null_bitmap; }
  if (sort_rows_pending(s) == 0) {   // the only input so far: sort it in place, no copy
    s->borrowed = true; s->b_data = data; s->b_nulls = nulls; s->b_rows = n;
    return TG_OK;
  }
  TG_TRY(sflush(s));
  TG_TRY(materialize_borrowed(s));
  return append_input(s, data.data(), nulls.data(), n, false);
}

int tg_sort_finish(tg_sort* h) {
  TGS_LOCK(h);
  if (s->finished) return TG_OK;
  TG_TRY(sfinish(s));
  s->finished = true;
  return TG_OK;
}

int tg_sort_next(tg_sort* h, tg_mut_chunk* out, int64_t max_rows, int64_t* nrows) {
  TGS_LOCK(h);
  if (!out || !nrows) return fail(TG_ERR_INVALID, "out / nrows is NULL");
  *nrows = 0;
  if (!s->finished) return fail(TG_ERR_STATE, "next before finish (sort is a pipeline breaker)");
  if (out->ncols != s->ncols) return fail(TG_ERR_INVALID, "output chunk has the child's schema");
  for (int c = 0; c < s->ncols; c++) if (out->cols[c].elem_len != 8) return fail(TG_ERR_INVALID, "output column elem_len mismatch");
  const int64_t lo = s->consumed;
  const int64_t want = std::min<int64_t>(std::min<int64_t>(max_rows, out->capacity_rows), s->out_rows - lo);
  if (want <= 0) return TG_OK;
  std::vector<const void*> cols(s->ncols);
  std::vector<const uint8_t*> bitmaps(s->ncols);
  for (int c = 0; c < s->ncols; c++) { cols[c] = s->out_cols[c]->p; bitmaps[c] = s->out_has_nulls[c] ? s->out_bitmaps[c]->as<uint8_t>() : nullptr; }
  TG_TRY(copy_out_rows(s->stream, s->ncols, cols.data(), bitmaps.data(), lo, want, out, &s->stats.d2h_bytes));
  s->consumed += want;
  *nrows = want;
  return TG_OK;
}

int tg_sort_result_dev(tg_sort* h, int64_t* out_rows, void** out_cols, void** out_nulls) {
  TGS_LOCK(h);
  if (!s->finished) return fail(TG_ERR_STATE, "result before finish");
  if (out_rows) *out_rows = s->out_rows;
  for (int c = 0; c < s->ncols; c++) {
    if (out_cols) out_cols[c] = s->out_cols[c]->p;
    if (out_nulls) out_nulls[c] = s->out_has_nulls[c] ? s->out_bitmaps[c]->p : nullptr;
  }
  return TG_OK;
}

int tg_sort_get_stats(tg_sort* h, tg_sort_stats* out) {
  TGS_LOCK(h);
  if (!out) return fail(TG_ERR_INVALID, "out is NULL");
  *out = s->stats;
  return TG_OK;
}

int tg_sort_close(tg_sort* h) {
  if (!h) return TG_OK;
  bool was = h->closed.exchange(true);
  if (was) return TG_OK;
  {
    std::lock_guard<std::mutex> lock(h->mu);   // waits for an in-flight call; later calls see `closed`
    SortImpl* s = h->impl;
    h->impl = nullptr;
    if (s) {
      DeviceGuard g(s->device);
      if (s->stream) cudaStreamSynchronize(s->stream);
      if (s->ev0) cudaEventDestroy(s->ev0);
      if (s->ev1) cudaEventDestroy(s->ev1);
      if (s->ev2) cudaEventDestroy(s->ev2);
      if (s->own_stream && s->stream) cudaStreamDestroy(s->stream);
      cudaGetLastError();
      delete s;
    }
  }
  bury_handle(h);
  return TG_OK;
}

int tg_sort_key_host(int32_t mysql_type, uint32_t flag, int32_t desc, uint64_t raw, uint64_t* key) {
  if (!key) return fail(TG_ERR_INVALID, "key is NULL");
  const int kind = sort_kind_of(mysql_type, flag);
  if (kind < 0) return fail(TG_ERR_UNSUPPORTED, "type is not a GPU sort key");
  *key = sort_key(raw, kind, desc != 0);
  return TG_OK;
}

}  // extern "C"
