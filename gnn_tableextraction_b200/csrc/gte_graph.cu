// Sparse-format construction for batched page graphs (int32 ids, bit-exact
// against a stable sort of the COO) + small graph utilities.
//
// Replaces the per-batch lazy COO->CSC / COO->CSR build that DGL performs under
// `g.update_all(...)` (/root/reference/src/components/graphs/models.py:53-54)
// and under autograd's reverse-graph SpMM, and `g.in_degrees()` (models.py:75).
#include "gte_common.cuh"

#include <atomic>
#include <mutex>
#include <vector>

namespace gte {

static thread_local char g_err[512] = "";
char* err_buf() { return g_err; }

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

static std::atomic<long long> g_launches{0};
void note_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
long long launches() { return g_launches.load(std::memory_order_relaxed); }

int ensure_dynamic_smem(const void* func, size_t bytes, const char* name) {
  if (bytes <= 48 * 1024) return GTE_OK;
  struct Entry { int dev; const void* func; size_t bytes; };
  static std::mutex mu;
  static std::vector<Entry> seen;
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
  std::lock_guard<std::mutex> lock(mu);
  for (Entry& e : seen)
    if (e.dev == dev && e.func == func) {
      if (e.bytes >= bytes) return GTE_OK;
      cudaError_t err = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
      if (err != cudaSuccess) return fail(GTE_ERR_CUDA, "%s(smem attr): %s", name, cudaGetErrorString(err));
      e.bytes = bytes;
      return GTE_OK;
    }
  cudaError_t err = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (err != cudaSuccess) return fail(GTE_ERR_CUDA, "%s(smem attr): %s", name, cudaGetErrorString(err));
  seen.push_back(Entry{dev, func, bytes});
  return GTE_OK;
}

// process-wide switches (gte_set_tuning); defaults = the product path
static std::atomic<int> g_tuning[GTE_TUNE_COUNT] = {{1}};
int tuning(int key) { return (key >= 0 && key < GTE_TUNE_COUNT) ? g_tuning[key].load(std::memory_order_relaxed) : 0; }

int sm_count() {
  static int cached[64];
  static std::once_flag once;
  std::call_once(once, [] {
    for (int i = 0; i < 64; ++i) cached[i] = 0;
  });
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

// ------------------------------------------------------------- kernels ----
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

// `bad` is only ever raised here (the caller clears it), so one flag can collect several builds.
__global__ void k_count_keys(const int32_t* __restrict__ key, const int32_t* __restrict__ other, int64_t e, int32_t n,
                             int32_t n_other, int32_t* __restrict__ cnt, int* __restrict__ bad) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < e; i += stride) {
    int32_t k = key[i];
    const int32_t o = other[i];
    if (o < 0 || o >= n_other) *bad = 1;  // a gather index outside the feature matrix (clamped when stored)
    if (k < 0 || k >= n) {
      *bad = 1;
      continue;
    }
    atomicAdd(&cnt[k], 1);
  }
}

// tile sums of cnt[0..m)
__global__ void k_scan_tile_sums(const int32_t* __restrict__ cnt, int64_t m, int32_t* __restrict__ tile_sums) {
  __shared__ int32_t red[SCAN_THREADS / 32];
  int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  int32_t s = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) {
    int64_t j = base + i;
    if (j < m) s += cnt[j];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    int32_t t = 0;
    for (int w = 0; w < SCAN_THREADS / 32; ++w) t += red[w];
    tile_sums[blockIdx.x] = t;
  }
}

// exclusive scan of tile_sums in place (single block)
__global__ void k_scan_tile_offsets(int32_t* __restrict__ tile_sums, int32_t num_tiles) {
  __shared__ int32_t warp_tot[32];
  __shared__ int32_t carry_s;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  for (int32_t base = 0; base < num_tiles; base += blockDim.x) {
    int32_t i = base + threadIdx.x;
    int32_t v = (i < num_tiles) ? tile_sums[i] : 0;
    int32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if ((threadIdx.x & 31) >= o) incl += t;
    }
    if ((threadIdx.x & 31) == 31) warp_tot[threadIdx.x >> 5] = incl;
    __syncthreads();
    if (threadIdx.x < 32) {
      int32_t nw = blockDim.x >> 5;
      int32_t wv = (threadIdx.x < nw) ? warp_tot[threadIdx.x] : 0;
      int32_t wi = wv;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int32_t t = __shfl_up_sync(0xffffffffu, wi, o);
        if (threadIdx.x >= o) wi += t;
      }
      warp_tot[threadIdx.x] = wi - wv;  // exclusive warp offsets
    }
    __syncthreads();
    int32_t carry = carry_s;
    int32_t excl = carry + warp_tot[threadIdx.x >> 5] + incl - v;
    if (i < num_tiles) tile_sums[i] = excl;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry_s = excl + v;
    __syncthreads();
  }
}

// indptr[j] = exclusive scan of cnt; cursor (aliasing cnt) is reset to the same
__global__ void k_scan_apply(int32_t* __restrict__ cnt_cursor, int64_t m, const int32_t* __restrict__ tile_offs,
                             int32_t* __restrict__ indptr) {
  __shared__ int32_t warp_tot[SCAN_THREADS / 32];
  int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_ITEMS;
  int32_t v[SCAN_ITEMS];
  int32_t s = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) {
    int64_t j = base + i;
    v[i] = (j < m) ? cnt_cursor[j] : 0;
    s += v[i];
  }
  int32_t incl = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int32_t t = __shfl_up_sync(0xffffffffu, incl, o);
    if ((threadIdx.x & 31) >= o) incl += t;
  }
  if ((threadIdx.x & 31) == 31) warp_tot[threadIdx.x >> 5] = incl;
  __syncthreads();
  int32_t woff = 0;
  for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) woff += warp_tot[w];
  int32_t run = tile_offs[blockIdx.x] + woff + incl - s;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) {
    int64_t j = base + i;
    if (j < m) {
      indptr[j] = run;
      cnt_cursor[j] = run;
    }
    run += v[i];
  }
}

__global__ void k_fill_rows(const int32_t* __restrict__ key, const int32_t* __restrict__ other, int64_t e,
                            int32_t n, int32_t n_other, int32_t* __restrict__ cursor, int32_t* __restrict__ tmp_idx,
                            int32_t* __restrict__ tmp_eid) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < e; i += stride) {
    int32_t k = key[i];
    if (k < 0 || k >= n) continue;  // flagged by k_count_keys
    int32_t pos = atomicAdd(&cursor[k], 1);
    int32_t o = other[i];
    if (o < 0 || o >= n_other) o = 0;  // flagged by k_count_keys; stored in range so that no later gather leaves the matrix
    tmp_idx[pos] = o;
    tmp_eid[pos] = (int32_t)i;
  }
}

// Order every row by original edge position (eid unique => result independent of
// the arrival order of the atomics above => equals the stable sort).  A group of
// LPR lanes owns one row; element i's final slot is the number of row elements
// with a smaller eid.
template <int LPR>
__global__ void k_rank_rows(const int32_t* __restrict__ indptr, int32_t n, const int32_t* __restrict__ tmp_idx,
                            const int32_t* __restrict__ tmp_eid, int32_t* __restrict__ indices,
                            int32_t* __restrict__ eid) {
  int64_t gthread = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t row = gthread / LPR;
  int lane = (int)(gthread % LPR);
  if (row >= n) return;
  int32_t beg = indptr[row], end = indptr[row + 1];
  for (int32_t i = beg + lane; i < end; i += LPR) {
    int32_t my = tmp_eid[i];
    int32_t rank = 0;
    for (int32_t j = beg; j < end; ++j) rank += (tmp_eid[j] < my) ? 1 : 0;
    indices[beg + rank] = tmp_idx[i];
    eid[beg + rank] = my;
  }
}

__global__ void k_batch_concat(const int32_t* __restrict__ pool_indptr, const int32_t* __restrict__ pool_indices,
                               const int32_t* __restrict__ pool_eid, const float* __restrict__ pool_w,
                               const int64_t* __restrict__ pool_node_off, const int64_t* __restrict__ pool_edge_off,
                               const int32_t* __restrict__ page_ids, const int64_t* __restrict__ batch_node_off,
                               const int64_t* __restrict__ batch_edge_off, int32_t num_pages,
                               int32_t* __restrict__ indptr, int32_t* __restrict__ indices, int32_t* __restrict__ eid,
                               float* __restrict__ w_out) {
  int p = blockIdx.x;
  int32_t pid = page_ids[p];
  int64_t pn0 = pool_node_off[pid], pe0 = pool_edge_off[pid];
  int32_t ni = (int32_t)(pool_node_off[pid + 1] - pn0);
  int32_t ei = (int32_t)(pool_edge_off[pid + 1] - pe0);
  int64_t bn0 = batch_node_off[p], be0 = batch_edge_off[p];
  const int32_t* ip = pool_indptr + pn0 + pid;  // n_i + 1 entries per page
  int32_t lim = ni + ((p == num_pages - 1) ? 1 : 0);
  for (int32_t i = threadIdx.x; i < lim; i += blockDim.x) indptr[bn0 + i] = ip[i] + (int32_t)be0;
  for (int32_t j = threadIdx.x; j < ei; j += blockDim.x) {
    indices[be0 + j] = pool_indices[pe0 + j] + (int32_t)bn0;
    if (eid) eid[be0 + j] = pool_eid[pe0 + j] + (int32_t)be0;
    if (w_out) w_out[be0 + j] = pool_w[pe0 + j];
  }
}

__global__ void k_gather_f32(const float* __restrict__ in, const int32_t* __restrict__ idx, float* __restrict__ out,
                             int64_t count) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (; i < count; i += stride) out[i] = __ldg(in + idx[i]);
}

__global__ void k_degree_norm(const int32_t* __restrict__ indptr, int32_t n, int mode, float* __restrict__ norm) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int32_t deg = indptr[i + 1] - indptr[i];
  float v;
  if (mode == GTE_NORM_INV_DEG_ZERO)
    v = deg > 0 ? 1.0f / (float)deg : 0.0f;  // 1./deg ; inf -> 0  (models.py:75-76)
  else
    v = 1.0f / (float)(deg > 1 ? deg : 1);
  norm[i] = v;
}

struct CsxWs {
  size_t cnt_off, tiles_off, tmp_idx_off, tmp_eid_off, bad_off, total;
  int32_t num_tiles;
};

static CsxWs csx_ws_layout(int32_t n, int64_t e) {
  auto up = [](size_t v) { return (v + 255) & ~size_t(255); };
  CsxWs w;
  int64_t m = (int64_t)n + 1;
  w.num_tiles = (int32_t)ceil_div64(m, SCAN_TILE);
  size_t o = 0;
  w.cnt_off = o;
  o = up(o + (size_t)m * 4);
  w.tiles_off = o;
  o = up(o + (size_t)w.num_tiles * 4);
  w.tmp_idx_off = o;
  o = up(o + (size_t)e * 4);
  w.tmp_eid_off = o;
  o = up(o + (size_t)e * 4);
  w.bad_off = o;
  o = up(o + 4);
  w.total = o;
  return w;
}

static int grid_for(int64_t work, int threads) {
  int64_t b = ceil_div64(work, threads);
  int64_t cap = (int64_t)sm_count() * 16;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

}  // namespace gte

using namespace gte;

extern "C" {

int gte_abi_version(void) { return GTE_ABI_VERSION; }

int64_t gte_launch_count(void) { return (int64_t)launches(); }

const char* gte_last_error_string(void) { return err_buf(); }

int gte_set_tuning(int key, int value) {
  GTE_CHECK_ARG(key >= 0 && key < GTE_TUNE_COUNT, "gte_set_tuning: unknown key %d", key);
  g_tuning[key].store(value, std::memory_order_relaxed);
  return GTE_OK;
}

int gte_get_tuning(int key) { return tuning(key); }

int gte_device_info(int* sm_count_host, int* cc_major_host, int* cc_minor_host) {
  int dev = 0;
  GTE_CHECK_CUDA(cudaGetDevice(&dev), "gte_device_info");
  int sms = 0, maj = 0, min = 0;
  GTE_CHECK_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev), "gte_device_info");
  GTE_CHECK_CUDA(cudaDeviceGetAttribute(&maj, cudaDevAttrComputeCapabilityMajor, dev), "gte_device_info");
  GTE_CHECK_CUDA(cudaDeviceGetAttribute(&min, cudaDevAttrComputeCapabilityMinor, dev), "gte_device_info");
  if (sm_count_host) *sm_count_host = sms;
  if (cc_major_host) *cc_major_host = maj;
  if (cc_minor_host) *cc_minor_host = min;
  return GTE_OK;
}

size_t gte_csx_from_coo_workspace_bytes(int32_t n, int64_t e) {
  if (n < 0 || e < 0) return 0;
  return csx_ws_layout(n, e).total;
}

int gte_csx_from_coo(const int32_t* key, const int32_t* other, int32_t n, int64_t e, int32_t* indptr,
                     int32_t* indices, int32_t* eid, void* ws, size_t ws_bytes, gte_stream_t stream) {
  return gte_csx_from_coo_checked(key, other, n, n, e, indptr, indices, eid, nullptr, ws, ws_bytes, stream);
}

int gte_csx_from_coo_checked(const int32_t* key, const int32_t* other, int32_t n, int32_t n_other, int64_t e,
                             int32_t* indptr, int32_t* indices, int32_t* eid, int32_t* bad_ids, void* ws,
                             size_t ws_bytes, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0 && n_other >= 0 && e >= 0, "gte_csx_from_coo: negative size (n=%d, e=%lld)", n, (long long)e);
  GTE_CHECK_ARG(e < (int64_t)INT32_MAX, "gte_csx_from_coo: e=%lld exceeds int32 edge ids", (long long)e);
  GTE_CHECK_ARG(indptr != nullptr, "gte_csx_from_coo: indptr is null");
  GTE_CHECK_ARG(e == 0 || (key && other && indices && eid), "gte_csx_from_coo: null edge array");
  CsxWs L = csx_ws_layout(n, e);
  if (ws == nullptr || ws_bytes < L.total)
    return fail(GTE_ERR_WORKSPACE, "gte_csx_from_coo: workspace %zu < required %zu", ws_bytes, L.total);
  cudaStream_t st = as_stream(stream);
  char* base = static_cast<char*>(ws);
  int32_t* cnt = reinterpret_cast<int32_t*>(base + L.cnt_off);
  int32_t* tiles = reinterpret_cast<int32_t*>(base + L.tiles_off);
  int32_t* tmp_idx = reinterpret_cast<int32_t*>(base + L.tmp_idx_off);
  int32_t* tmp_eid = reinterpret_cast<int32_t*>(base + L.tmp_eid_off);
  int* bad = bad_ids ? bad_ids : reinterpret_cast<int*>(base + L.bad_off);
  int64_t m = (int64_t)n + 1;
  GTE_CHECK_CUDA(cudaMemsetAsync(cnt, 0, (size_t)m * 4, st), "gte_csx_from_coo(memset)");
  if (!bad_ids) GTE_CHECK_CUDA(cudaMemsetAsync(bad, 0, 4, st), "gte_csx_from_coo(memset)");
  if (e > 0) {
    k_count_keys<<<grid_for(e, 256), 256, 0, st>>>(key, other, e, n, n_other, cnt, bad);
    GTE_CHECK_LAUNCH("k_count_keys");
  }
  k_scan_tile_sums<<<L.num_tiles, SCAN_THREADS, 0, st>>>(cnt, m, tiles);
  GTE_CHECK_LAUNCH("k_scan_tile_sums");
  k_scan_tile_offsets<<<1, 1024, 0, st>>>(tiles, L.num_tiles);
  GTE_CHECK_LAUNCH("k_scan_tile_offsets");
  k_scan_apply<<<L.num_tiles, SCAN_THREADS, 0, st>>>(cnt, m, tiles, indptr);
  GTE_CHECK_LAUNCH("k_scan_apply");
  if (e > 0) {
    k_fill_rows<<<grid_for(e, 256), 256, 0, st>>>(key, other, e, n, n_other, cnt, tmp_idx, tmp_eid);
    GTE_CHECK_LAUNCH("k_fill_rows");
    constexpr int LPR = 8;
    int64_t threads = (int64_t)n * LPR;
    k_rank_rows<LPR><<<(unsigned)ceil_div64(threads, 256), 256, 0, st>>>(indptr, n, tmp_idx, tmp_eid, indices, eid);
    GTE_CHECK_LAUNCH("k_rank_rows");
  }
  return GTE_OK;
}

int gte_batch_concat_csx(const int32_t* pool_indptr, const int32_t* pool_indices, const int32_t* pool_eid,
                         const float* pool_w, const int64_t* pool_node_off, const int64_t* pool_edge_off,
                         const int32_t* page_ids, const int64_t* batch_node_off, const int64_t* batch_edge_off,
                         int32_t num_pages, int32_t* indptr, int32_t* indices, int32_t* eid, float* w_out,
                         gte_stream_t stream) {
  GTE_CHECK_ARG(num_pages >= 0, "gte_batch_concat_csx: num_pages < 0");
  if (num_pages == 0) return GTE_OK;
  GTE_CHECK_ARG(pool_indptr && pool_indices && pool_node_off && pool_edge_off && page_ids && batch_node_off &&
                    batch_edge_off && indptr && indices,
                "gte_batch_concat_csx: null argument");
  GTE_CHECK_ARG((eid == nullptr) || (pool_eid != nullptr), "gte_batch_concat_csx: eid requested without pool_eid");
  GTE_CHECK_ARG((w_out == nullptr) || (pool_w != nullptr), "gte_batch_concat_csx: w_out requested without pool_w");
  k_batch_concat<<<num_pages, 256, 0, as_stream(stream)>>>(pool_indptr, pool_indices, pool_eid, pool_w,
                                                          pool_node_off, pool_edge_off, page_ids, batch_node_off,
                                                          batch_edge_off, num_pages, indptr, indices, eid, w_out);
  GTE_CHECK_LAUNCH("k_batch_concat");
  return GTE_OK;
}

int gte_gather_f32(const float* in, const int32_t* idx, float* out, int64_t count, gte_stream_t stream) {
  GTE_CHECK_ARG(count >= 0, "gte_gather_f32: negative count");
  if (count == 0) return GTE_OK;
  GTE_CHECK_ARG(in && idx && out, "gte_gather_f32: null argument");
  k_gather_f32<<<grid_for(count, 256), 256, 0, as_stream(stream)>>>(in, idx, out, count);
  GTE_CHECK_LAUNCH("k_gather_f32");
  return GTE_OK;
}

int gte_degree_norm(const int32_t* indptr, int32_t n, int mode, float* norm, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0, "gte_degree_norm: negative n");
  GTE_CHECK_ARG(mode == GTE_NORM_INV_DEG_ZERO || mode == GTE_NORM_INV_DEG_CLAMP, "gte_degree_norm: bad mode %d", mode);
  if (n == 0) return GTE_OK;
  GTE_CHECK_ARG(indptr && norm, "gte_degree_norm: null argument");
  k_degree_norm<<<(unsigned)ceil_div64(n, 256), 256, 0, as_stream(stream)>>>(indptr, n, mode, norm);
  GTE_CHECK_LAUNCH("k_degree_norm");
  return GTE_OK;
}

}  // extern "C"
