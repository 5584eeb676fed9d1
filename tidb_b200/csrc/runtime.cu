// runtime.cu — device/host memory plumbing of the C-ABI (include/tidbgpu.h), no kernels.
#include "common.cuh"

namespace tg {

static thread_local std::string g_last_error;

void set_error(const std::string& msg) { g_last_error = msg; }

int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
  char buf[512];
  snprintf(buf, sizeof(buf), "CUDA error %d (%s) at %s:%d: %s", (int)e, cudaGetErrorString(e), file, line, what);
  g_last_error = buf;
  cudaGetLastError();   // clear the sticky non-fatal error state
  return e == cudaErrorMemoryAllocation ? TG_ERR_OOM : TG_ERR_CUDA;
}

void append_bits(uint8_t* dst, int64_t pos, const uint8_t* src, int64_t nbits) {
  if (nbits <= 0) return;
  int shift = (int)(pos & 7);
  int64_t d = pos >> 3;
  if (shift == 0) {
    std::memcpy(dst + d, src, (size_t)((nbits + 7) / 8));
    if (nbits & 7) dst[d + (nbits >> 3)] &= (uint8_t)((1u << (nbits & 7)) - 1);
    return;
  }
  // keep the low `shift` bits already in dst[d]
  int64_t nbytes = (nbits + 7) / 8;
  uint8_t carry = (uint8_t)(dst[d] & ((1u << shift) - 1));
  for (int64_t i = 0; i < nbytes; i++) {
    uint8_t s = src[i];
    if (i == nbytes - 1 && (nbits & 7)) s &= (uint8_t)((1u << (nbits & 7)) - 1);
    dst[d + i] = (uint8_t)(carry | (uint8_t)(s << shift));
    carry = (uint8_t)(s >> (8 - shift));
  }
  // spill of the last byte, only if bits remain beyond the bytes written above
  if (((pos + nbits + 7) >> 3) > d + nbytes) dst[d + nbytes] = carry;
}

int stage_append(ColumnStage& st, const tg_chunk* chk, const std::vector<char>& needed) {
  int64_t n = logical_rows(chk);
  if (n == 0) return TG_OK;
  for (size_t c = 0; c < needed.size(); c++) {
    if (!needed[c]) continue;
    const tg_column& col = chk->cols[c];
    PinBuf& d = *st.data[c];
    TG_TRY(d.reserve((size_t)(st.rows + n) * 8));
    uint64_t* dst = reinterpret_cast<uint64_t*>(d.p) + st.rows;
    const uint64_t* src = reinterpret_cast<const uint64_t*>(col.data);
    if (!chk->sel) std::memcpy(dst, src, (size_t)n * 8);
    else for (int64_t i = 0; i < n; i++) dst[i] = src[chk->sel[i]];
    d.used = (size_t)(st.rows + n) * 8;
    bool bring = col.null_bitmap != nullptr;
    if (bring || st.has_nulls[c]) {
      PinBuf& nb = *st.nulls[c];
      size_t need = (size_t)((st.rows + n + 7) / 8) + 1;
      TG_TRY(nb.reserve(need));
      if (!st.has_nulls[c]) { std::memset(nb.p, 0xff, (size_t)((st.rows + 7) / 8) + 1); st.has_nulls[c] = 1; }
      if (bring && !chk->sel) append_bits(nb.p, st.rows, col.null_bitmap, n);
      else for (int64_t i = 0; i < n; i++) {
        bool nn = bring ? bit_not_null(col.null_bitmap, chk->sel ? chk->sel[i] : i) : true;
        int64_t r = st.rows + i;
        if (nn) nb.p[r >> 3] |= (uint8_t)(1u << (r & 7)); else nb.p[r >> 3] &= (uint8_t)~(1u << (r & 7));
      }
      nb.used = need;
    }
  }
  st.rows += n;
  return TG_OK;
}

int copy_out_rows(cudaStream_t st, int ncols, const void* const* cols, const uint8_t* const* bitmaps, int64_t lo,
                  int64_t want, tg_mut_chunk* out, int64_t* d2h_bytes) {
  const int shift = (int)(lo & 7);
  std::vector<std::vector<uint8_t>> shifted;
  for (int k = 0; k < ncols; k++) {
    TG_CUDA(cudaMemcpyAsync(out->cols[k].data, reinterpret_cast<const uint8_t*>(cols[k]) + (size_t)lo * 8, (size_t)want * 8, cudaMemcpyDeviceToHost, st));
    *d2h_bytes += want * 8;
    size_t nb = (size_t)((want + 7) / 8);
    if (bitmaps[k]) {
      if (!out->cols[k].null_bitmap) return fail(TG_ERR_INVALID, "output column can be NULL but the caller passed no null bitmap");
      if (shift == 0) TG_CUDA(cudaMemcpyAsync(out->cols[k].null_bitmap, bitmaps[k] + lo / 8, nb, cudaMemcpyDeviceToHost, st));
      else {
        shifted.emplace_back((size_t)((shift + want + 7) / 8) + 1, (uint8_t)0);
        TG_CUDA(cudaMemcpyAsync(shifted.back().data(), bitmaps[k] + lo / 8, shifted.back().size() - 1, cudaMemcpyDeviceToHost, st));
      }
    } else if (out->cols[k].null_bitmap) {
      std::memset(out->cols[k].null_bitmap, 0xff, nb);
      if (want & 7) out->cols[k].null_bitmap[nb - 1] = (uint8_t)((1u << (want & 7)) - 1);
    }
  }
  TG_CUDA(cudaStreamSynchronize(st));
  if (shift) {
    size_t q = 0;
    for (int k = 0; k < ncols; k++) {
      if (!bitmaps[k]) continue;
      const std::vector<uint8_t>& src = shifted[q++];
      size_t nb = (size_t)((want + 7) / 8);
      for (size_t b = 0; b < nb; b++) out->cols[k].null_bitmap[b] = (uint8_t)((src[b] >> shift) | (src[b + 1] << (8 - shift)));
    }
  }
  if (want & 7) for (int k = 0; k < ncols; k++) if (bitmaps[k]) out->cols[k].null_bitmap[want >> 3] &= (uint8_t)((1u << (want & 7)) - 1);
  return TG_OK;
}

cudaStream_t service_stream(int device) {
  static std::mutex mu;
  static cudaStream_t streams[64];
  std::lock_guard<std::mutex> lk(mu);
  int d = device & 63;
  if (!streams[d]) {
    int prev = -1; cudaGetDevice(&prev); cudaSetDevice(device);
    if (cudaStreamCreateWithFlags(&streams[d], cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); streams[d] = nullptr; }
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
      unsigned long long keep = ~0ull;   // never give memory back to the driver between operators
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaGetLastError();
    if (prev >= 0) cudaSetDevice(prev);
  }
  return streams[d];
}

int device_sm_count(int device) {
  static int cache[64];
  if (device >= 0 && device < 64 && cache[device] > 0) return cache[device];
  int n = 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device) != cudaSuccess) { cudaGetLastError(); n = 148; }
  if (device >= 0 && device < 64) cache[device] = n;
  return n;
}

}  // namespace tg

using namespace tg;

extern "C" {

const char* tg_last_error(void) { return tg::g_last_error.c_str(); }
int tg_abi_version(void) { return TIDBGPU_ABI_VERSION; }

int tg_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int tg_device_info(int device, char* name, size_t name_cap, int* sm_count, int64_t* hbm_bytes) {
  cudaDeviceProp p;
  TG_CUDA(cudaGetDeviceProperties(&p, device));
  if (name && name_cap) { strncpy(name, p.name, name_cap - 1); name[name_cap - 1] = 0; }
  if (sm_count) *sm_count = p.multiProcessorCount;
  if (hbm_bytes) *hbm_bytes = (int64_t)p.totalGlobalMem;
  return TG_OK;
}

int tg_fixed_len(int mysql_type) { return tg::fixed_len(mysql_type); }

int tg_host_alloc(size_t bytes, void** out) {
  if (!out) return fail(TG_ERR_INVALID, "tg_host_alloc: out is NULL");
  *out = nullptr;
  cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(e == cudaErrorMemoryAllocation ? TG_ERR_OOM : TG_ERR_CUDA, std::string("cudaHostAlloc: ") + cudaGetErrorString(e)); }
  return TG_OK;
}
int tg_host_free(void* p) {
  if (!p) return TG_OK;
  TG_CUDA(cudaFreeHost(p));
  return TG_OK;
}
int tg_dev_alloc(int device, size_t bytes, void** out) {
  if (!out) return fail(TG_ERR_INVALID, "tg_dev_alloc: out is NULL");
  DeviceGuard g(device);
  if (!g.ok) return fail(TG_ERR_CUDA, "cudaSetDevice failed (no usable CUDA device)");
  *out = nullptr;
  cudaError_t e = cudaMalloc(out, bytes ? bytes : 1);
  if (e != cudaSuccess) { cudaGetLastError(); return fail(e == cudaErrorMemoryAllocation ? TG_ERR_OOM : TG_ERR_CUDA, std::string("cudaMalloc: ") + cudaGetErrorString(e)); }
  return TG_OK;
}
int tg_dev_free(int device, void* p) {
  if (!p) return TG_OK;
  DeviceGuard g(device);
  TG_CUDA(cudaFree(p));
  return TG_OK;
}
int tg_memcpy_h2d(int device, void* dst, const void* src, size_t bytes) {
  DeviceGuard g(device);
  if (!g.ok) return fail(TG_ERR_CUDA, "cudaSetDevice failed (no usable CUDA device)");
  TG_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
  return TG_OK;
}
int tg_memcpy_d2h(int device, void* dst, const void* src, size_t bytes) {
  DeviceGuard g(device);
  if (!g.ok) return fail(TG_ERR_CUDA, "cudaSetDevice failed (no usable CUDA device)");
  TG_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
  return TG_OK;
}
int tg_memcpy_d2d_async(int device, void* dst, const void* src, size_t bytes, void* stream) {
  DeviceGuard g(device);
  if (!g.ok) return fail(TG_ERR_CUDA, "cudaSetDevice failed (no usable CUDA device)");
  TG_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, (cudaStream_t)stream));
  return TG_OK;
}
int tg_device_synchronize(int device) {
  DeviceGuard g(device);
  if (!g.ok) return fail(TG_ERR_CUDA, "cudaSetDevice failed (no usable CUDA device)");
  TG_CUDA(cudaDeviceSynchronize());
  return TG_OK;
}

int tg_ipc_export(int device, void* dev_ptr, uint8_t handle_out[64]) {
  DeviceGuard g(device);
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  cudaIpcMemHandle_t h;
  TG_CUDA(cudaIpcGetMemHandle(&h, dev_ptr));
  std::memcpy(handle_out, &h, 64);
  return TG_OK;
}
int tg_ipc_open(int device, const uint8_t handle[64], void** out_ptr) {
  DeviceGuard g(device);
  cudaIpcMemHandle_t h;
  std::memcpy(&h, handle, 64);
  TG_CUDA(cudaIpcOpenMemHandle(out_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return TG_OK;
}
int tg_ipc_close(int device, void* mapped_ptr) {
  DeviceGuard g(device);
  TG_CUDA(cudaIpcCloseMemHandle(mapped_ptr));
  return TG_OK;
}

}  // extern "C"
