// Gather + segment-reduce SpMM over compressed rows: the neighbour aggregation
// of the GraphSAGE layers, forward (CSC) and backward (transposed CSR).
//
// Replaces `g.update_all(fn.u_mul_e('h','feat','m'), fn.sum('m','h'))` and the
// `ah * norm` of `concat` (/root/reference/src/components/graphs/models.py:53-54,
// 69-71), `fn.mean` (models.py:149), and autograd's reverse-graph SpMM.
//
// Kernel `k_spmm_rows`: a group of G lanes owns one output row (G = 4..32 by
// feature width, so narrow rows pack 8 per warp); the group's lanes fetch up to
// G (index, weight) pairs with one coalesced load and broadcast them by
// shuffle; each lane accumulates C 128-bit column chunks in registers in edge
// order (deterministic, no atomics); the edge weight, the optional source-side
// scale (backward: norm[dst]), the degree normalisation and the optional addend
// (backward: the self-path gradient) are fused.
//
// Roofline: HBM.  Algorithmic bytes per launch = 8*N*F + 8*E + 4*N  (read x,
// write y, indptr, indices, weights; SURVEY.md section 8d); the gathered rows
// (4*E*F bytes) are served by L1/L2 because a page's sources are page-local.
#include "gte_common.cuh"
#include "gte_umma_ptx.cuh"

namespace gte {

template <int VEC>
struct Acc;
template <>
struct Acc<4> {
  float4 v;
  __device__ __forceinline__ void zero() { v = make_float4(0.f, 0.f, 0.f, 0.f); }
  __device__ __forceinline__ void fma(float w, const float4& x) {
    v.x = fmaf(w, x.x, v.x);
    v.y = fmaf(w, x.y, v.y);
    v.z = fmaf(w, x.z, v.z);
    v.w = fmaf(w, x.w, v.w);
  }
};
template <>
struct Acc<1> {
  float v;
  __device__ __forceinline__ void zero() { v = 0.f; }
  __device__ __forceinline__ void fma(float w, float x) { v = fmaf(w, x, v); }
};

template <int VEC>
struct VecT;
template <>
struct VecT<4> {
  using type = float4;
  static __device__ __forceinline__ float4 load(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
  static __device__ __forceinline__ float4 zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
};
template <>
struct VecT<1> {
  using type = float;
  static __device__ __forceinline__ float load(const float* p) { return __ldg(p); }
  static __device__ __forceinline__ float zero() { return 0.f; }
};

constexpr int SPMM_THREADS = 256;
constexpr int EDGE_UNROLL = 4;

template <int VEC, int G, int C>
__global__ void __launch_bounds__(SPMM_THREADS)
    k_spmm_rows(const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices, const float* __restrict__ w,
                const float* __restrict__ pre_scale, const float* __restrict__ row_norm, int mode,
                const float* __restrict__ x, int64_t ldx, const float* __restrict__ addend, int64_t ldadd,
                float* __restrict__ y, int64_t ldy, int32_t n_rows, int32_t f) {
  using V = typename VecT<VEC>::type;
  constexpr int ROWS_PER_BLOCK = SPMM_THREADS / G;
  const int lane = threadIdx.x % G;
  const int grp = threadIdx.x / G;
  const int64_t row = (int64_t)blockIdx.x * ROWS_PER_BLOCK + grp;
  const int col_base = blockIdx.y * (G * C * VEC);
  const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << ((threadIdx.x & 31) / G * G));
  if (row >= n_rows) return;  // whole group leaves together; shuffles below use the group mask

  const int32_t beg = indptr[row], end = indptr[row + 1];
  Acc<VEC> acc[C];
  int col[C];
  bool on[C];
#pragma unroll
  for (int c = 0; c < C; ++c) {
    acc[c].zero();
    col[c] = col_base + (lane + c * G) * VEC;
    on[c] = col[c] < f;
  }

  for (int32_t base = beg; base < end; base += G) {
    const int32_t mine = base + lane;
    int32_t idx = 0;
    float wv = 0.f;
    if (mine < end) {
      idx = __ldg(indices + mine);
      wv = w ? __ldg(w + mine) : 1.0f;
      if (pre_scale) wv *= __ldg(pre_scale + idx);
    }
    const int cnt = min(G, end - base);
    int t = 0;
    for (; t + EDGE_UNROLL <= cnt; t += EDGE_UNROLL) {
      V xv[EDGE_UNROLL][C];
      float wt[EDGE_UNROLL];
#pragma unroll
      for (int u = 0; u < EDGE_UNROLL; ++u) {
        const int32_t src = __shfl_sync(gmask, idx, t + u, G);
        wt[u] = __shfl_sync(gmask, wv, t + u, G);
        const float* xr = x + (int64_t)src * ldx;
#pragma unroll
        for (int c = 0; c < C; ++c) xv[u][c] = on[c] ? VecT<VEC>::load(xr + col[c]) : VecT<VEC>::zero();
      }
#pragma unroll
      for (int u = 0; u < EDGE_UNROLL; ++u)
#pragma unroll
        for (int c = 0; c < C; ++c) acc[c].fma(wt[u], xv[u][c]);
    }
    for (; t < cnt; ++t) {
      const int32_t src = __shfl_sync(gmask, idx, t, G);
      const float wt = __shfl_sync(gmask, wv, t, G);
      const float* xr = x + (int64_t)src * ldx;
#pragma unroll
      for (int c = 0; c < C; ++c)
        if (on[c]) acc[c].fma(wt, VecT<VEC>::load(xr + col[c]));
    }
  }

  float post = 1.0f;
  bool divide = false;
  if (mode == GTE_AGG_SUM_NORM) {
    post = __ldg(row_norm + row);
  } else if (mode == GTE_AGG_MEAN) {
    const int32_t deg = end - beg;
    post = (float)(deg > 1 ? deg : 1);
    divide = true;
  }
  float* yr = y + row * ldy;
  const float* ar = addend ? addend + row * ldadd : nullptr;
#pragma unroll
  for (int c = 0; c < C; ++c) {
    if (!on[c]) continue;
    if constexpr (VEC == 4) {
      float4 r = acc[c].v;
      if (divide) {
        r.x /= post; r.y /= post; r.z /= post; r.w /= post;
      } else {
        r.x *= post; r.y *= post; r.z *= post; r.w *= post;
      }
      if (ar) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(ar + col[c]));
        r.x += a.x; r.y += a.y; r.z += a.z; r.w += a.w;
      }
      *reinterpret_cast<float4*>(yr + col[c]) = r;
    } else {
      float r = divide ? acc[c].v / post : acc[c].v * post;
      if (ar) r += __ldg(ar + col[c]);
      yr[col[c]] = r;
    }
  }
}

template <int VEC, int G, int C>
static int launch_spmm(const int32_t* indptr, const int32_t* indices, const float* w, const float* pre_scale,
                       const float* row_norm, int mode, const float* x, int64_t ldx, const float* addend,
                       int64_t ldadd, float* y, int64_t ldy, int32_t n_rows, int32_t f, cudaStream_t st) {
  constexpr int ROWS_PER_BLOCK = SPMM_THREADS / G;
  const int cols_per_block = G * C * VEC;
  dim3 grid((unsigned)ceil_div64(n_rows, ROWS_PER_BLOCK), (unsigned)ceil_div64(f, cols_per_block));
  k_spmm_rows<VEC, G, C><<<grid, SPMM_THREADS, 0, st>>>(indptr, indices, w, pre_scale, row_norm, mode, x, ldx, addend,
                                                       ldadd, y, ldy, n_rows, f);
  GTE_CHECK_LAUNCH("k_spmm_rows");
  return GTE_OK;
}

// ----------------------------------------------------------------------------------------------
// Block-diagonal (page-batched) variant: one CTA per (page, column slice).  A batch of page graphs has
// no edge between pages, so every source row a page's rows can touch lies in that page's own node
// range.  The CTA stages, once and coalesced, everything the page needs in shared memory:
//   x[page rows, slice] (cp.async), the page's row pointers, its column indices (made page-local) and
//   its edge weights (with the source-side scale folded in),
// after which the whole aggregation of the page runs out of shared memory: no dependent global
// load is left in the per-row loop, and the L2->SM gather traffic (4*E*F bytes, ~10x the compulsory
// bytes at degree 10) disappears -- the kernel streams x in / y out at HBM rate.  Indices outside
// the page window (not block diagonal) fall back to a global load, so the result is always correct.
constexpr int PAGED_THREADS = 512;

template <int G>
__global__ void __launch_bounds__(PAGED_THREADS)
    k_spmm_paged(const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices, const float* __restrict__ w,
                 const float* __restrict__ pre_scale, const float* __restrict__ row_norm, int mode,
                 const float* __restrict__ x, int64_t ldx, const float* __restrict__ addend, int64_t ldadd,
                 float* __restrict__ y, int64_t ldy, const int32_t* __restrict__ page_off, int32_t f,
                 int32_t np_cap, int32_t ne_cap) {
  extern __shared__ __align__(16) float smem_f[];
  constexpr int CS = G * 4;
  constexpr int ROWS_PER_ITER = PAGED_THREADS / G;
  float* sx = smem_f;                                                     // [np_cap][CS]
  uint32_t* s_off = reinterpret_cast<uint32_t*>(sx + (size_t)np_cap * CS);  // [ne_cap] byte offset of the source row in sx
  float* s_w = reinterpret_cast<float*>(s_off + ne_cap);                  // [ne_cap] edge weight (* source-side scale)
  int32_t* s_ptr = reinterpret_cast<int32_t*>(s_w + ne_cap);              // [np_cap + 1] page-local row pointers
  int32_t* s_flag = s_ptr + np_cap + 1;                                   // some edge needs the global slow path
  // the slices of one page are adjacent in launch order (blockIdx.x fastest) so that cache lines shared
  // by neighbouring slices are fetched from DRAM once
  const int page = blockIdx.y;
  const int c0 = blockIdx.x * CS;
  const int32_t n0 = page_off[page], n1 = page_off[page + 1];
  const int32_t np = n1 - n0;
  const int32_t e0 = indptr[n0];
  const int32_t ne = indptr[n1] - e0;
  const bool staged_edges = ne <= ne_cap;  // always true when the caller's max_page_edges is right
  if (threadIdx.x == 0) *s_flag = staged_edges ? 0 : 1;
  for (int i = threadIdx.x; i < np * G; i += PAGED_THREADS) {
    const int r = i / G, ch = i % G;
    const int col = c0 + ch * 4;
    float* dst = sx + (size_t)r * CS + ch * 4;
    if (col < f) {  // 16-byte chunks; chunks entirely beyond f are zero-filled
      const float* src = x + (int64_t)(n0 + r) * ldx + col;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src)
                   : "memory");
    } else {
      *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  for (int i = threadIdx.x; i <= np; i += PAGED_THREADS) s_ptr[i] = indptr[n0 + i] - e0;
  __syncthreads();  // s_flag initialised before anyone raises it
  if (staged_edges) {
    for (int i = threadIdx.x; i < ne; i += PAGED_THREADS) {
      const int32_t c = __ldg(indices + e0 + i);
      float wv = w ? __ldg(w + e0 + i) : 1.0f;
      if (pre_scale) wv *= __ldg(pre_scale + c);
      const int32_t sl = c - n0;
      const bool inside = sl >= 0 && sl < np;
      s_off[i] = inside ? (uint32_t)sl * (CS * 4) : 0u;
      s_w[i] = inside ? wv : 0.f;  // outside edges contribute through the slow path below
      if (!inside) *s_flag = 1;
    }
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();

  const int lane = threadIdx.x % G;
  const int grp = threadIdx.x / G;
  const int col = c0 + lane * 4;
  const bool on = col < f;
  const bool slow = *s_flag != 0;
  const char* xb = reinterpret_cast<const char*>(sx) + lane * 16;
  for (int32_t rl = grp; rl < np; rl += ROWS_PER_ITER) {
    const int64_t row = n0 + rl;
    const int32_t beg = s_ptr[rl], end = s_ptr[rl + 1];
    // issue the row-end operands early so their latency overlaps the neighbour loop
    float4 av = make_float4(0.f, 0.f, 0.f, 0.f);
    if (addend && on) av = __ldg(reinterpret_cast<const float4*>(addend + row * ldadd + col));
    const float nrm = (mode == GTE_AGG_SUM_NORM) ? __ldg(row_norm + row) : 1.0f;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    if (staged_edges) {
      int32_t j = beg;
      for (; j + 4 <= end; j += 4) {  // edge order preserved: deterministic, same sums as the generic kernel
        const uint32_t o0 = s_off[j], o1 = s_off[j + 1], o2 = s_off[j + 2], o3 = s_off[j + 3];
        const float w0 = s_w[j], w1 = s_w[j + 1], w2 = s_w[j + 2], w3 = s_w[j + 3];
        const float4 x0 = *reinterpret_cast<const float4*>(xb + o0);
        const float4 x1 = *reinterpret_cast<const float4*>(xb + o1);
        const float4 x2 = *reinterpret_cast<const float4*>(xb + o2);
        const float4 x3 = *reinterpret_cast<const float4*>(xb + o3);
        acc.x = fmaf(w0, x0.x, acc.x); acc.y = fmaf(w0, x0.y, acc.y); acc.z = fmaf(w0, x0.z, acc.z); acc.w = fmaf(w0, x0.w, acc.w);
        acc.x = fmaf(w1, x1.x, acc.x); acc.y = fmaf(w1, x1.y, acc.y); acc.z = fmaf(w1, x1.z, acc.z); acc.w = fmaf(w1, x1.w, acc.w);
        acc.x = fmaf(w2, x2.x, acc.x); acc.y = fmaf(w2, x2.y, acc.y); acc.z = fmaf(w2, x2.z, acc.z); acc.w = fmaf(w2, x2.w, acc.w);
        acc.x = fmaf(w3, x3.x, acc.x); acc.y = fmaf(w3, x3.y, acc.y); acc.z = fmaf(w3, x3.z, acc.z); acc.w = fmaf(w3, x3.w, acc.w);
      }
      for (; j < end; ++j) {
        const float wt = s_w[j];
        const float4 xv = *reinterpret_cast<const float4*>(xb + s_off[j]);
        acc.x = fmaf(wt, xv.x, acc.x); acc.y = fmaf(wt, xv.y, acc.y); acc.z = fmaf(wt, xv.z, acc.z); acc.w = fmaf(wt, xv.w, acc.w);
      }
    }
    if (slow && on) {  // rare: the page table does not describe a block-diagonal graph (or edge capacity too small)
      for (int32_t j = beg; j < end; ++j) {
        const int32_t c = __ldg(indices + e0 + j);
        const int32_t sl = c - n0;
        if (staged_edges && sl >= 0 && sl < np) continue;  // already accumulated from shared memory
        float wt = w ? __ldg(w + e0 + j) : 1.0f;
        if (pre_scale) wt *= __ldg(pre_scale + c);
        const float4 xv = __ldg(reinterpret_cast<const float4*>(x + (int64_t)c * ldx + col));
        acc.x = fmaf(wt, xv.x, acc.x); acc.y = fmaf(wt, xv.y, acc.y); acc.z = fmaf(wt, xv.z, acc.z); acc.w = fmaf(wt, xv.w, acc.w);
      }
    }
    if (!on) continue;
    if (mode == GTE_AGG_MEAN) {
      const int32_t deg = end - beg;
      const float d = (float)(deg > 1 ? deg : 1);
      acc.x /= d; acc.y /= d; acc.z /= d; acc.w /= d;
    } else if (mode == GTE_AGG_SUM_NORM) {
      acc.x *= nrm; acc.y *= nrm; acc.z *= nrm; acc.w *= nrm;
    }
    if (addend) {
      acc.x += av.x; acc.y += av.y; acc.z += av.z; acc.w += av.w;
    }
    *reinterpret_cast<float4*>(y + row * ldy + col) = acc;
  }
}

static size_t paged_smem_bytes(int G, int32_t np_cap, int32_t ne_cap) {
  return (size_t)np_cap * G * 16 + (size_t)ne_cap * 8 + ((size_t)np_cap + 2) * 4 + 16;
}

template <int G>
static int launch_spmm_paged(const int32_t* indptr, const int32_t* indices, const float* w, const float* pre_scale,
                             const float* row_norm, int mode, const float* x, int64_t ldx, const float* addend,
                             int64_t ldadd, float* y, int64_t ldy, const int32_t* page_off, int32_t num_pages,
                             int32_t np_cap, int32_t ne_cap, int32_t f, cudaStream_t st) {
  constexpr int CS = G * 4;
  const size_t smem = paged_smem_bytes(G, np_cap, ne_cap);
  if (int rc = ensure_dynamic_smem(reinterpret_cast<const void*>(&k_spmm_paged<G>), smem, "k_spmm_paged")) return rc;
  dim3 grid((unsigned)ceil_div64(f, CS), (unsigned)num_pages);
  k_spmm_paged<G><<<grid, PAGED_THREADS, smem, st>>>(indptr, indices, w, pre_scale, row_norm, mode, x, ldx, addend, ldadd, y,
                                                    ldy, page_off, f, np_cap, ne_cap);
  GTE_CHECK_LAUNCH("k_spmm_paged");
  return GTE_OK;
}


// ----------------------------------------------------------------------------------------------
// Packed + persistent + double-buffered page kernel (the headline conv-layer kernel).
//
// What bounds k_spmm_paged above at F = 218, degree 10 (ncu, profiles/): no single pipe -- the
// shared-memory pipe is ~45 % busy, the issue slots ~40 %, DRAM ~25 %: every CTA waits for its own
// staging before it computes, about half of the instructions issue and address that staging, every
// row waits a global-memory round trip for its normaliser / addend, and two 32-bit metadata words
// are re-read per (edge, row group).  This variant
//   * reads the edges pre-packed as 8-byte (page-local source row, weight * source scale) pairs
//     (k_paged_pack_edges, once per graph and direction instead of once per CTA and slice),
//   * runs one persistent CTA per SM over a contiguous range of (page, column slice) items with two
//     shared-memory stages filled by the TMA unit (x slice: 2-D tensor boxes; packed edges: one bulk
//     copy; row pointers / normalisers: 4-byte cp.async tracked by the stage's mbarrier, so the producer
//     never waits for them) while the previous item is reduced,
//   * gives each lane V 128-bit column chunks of TWO rows at a time (G lanes per row) with the next
//     group's metadata loaded ahead, so 8 independent 128-bit shared loads are in flight per lane,
//   * prefetches the addend rows of the next item into L2 when it stages that item.
// Sums run in row order exactly like the kernels above (deterministic, same rounding).
// 15 consumer warps + 1 producer warp = 16 warps = 4 per SM sub-partition, so each thread may use 128 registers
// (17 warps put 5 on one sub-partition and cap everybody at 96: the compiler then splits the gather batches)
constexpr int PK_CONSUMERS = 480;
constexpr int PK_THREADS = PK_CONSUMERS + 32;   // + 1 producer warp
constexpr int PK_BOX_BIG = 64;    // rows per large TMA box
constexpr int PK_BOX_SMALL = 8;   // rows per small TMA box (page tail): at most 7 rows over-read per page
constexpr uint32_t PK_OUTSIDE = 0xFFFFFFFFu;  // packed source row of an edge that leaves its page

__global__ void __launch_bounds__(256)
    k_paged_pack_edges(const int32_t* __restrict__ indptr, const int32_t* __restrict__ indices,
                       const int32_t* __restrict__ eid, const float* __restrict__ w, const float* __restrict__ pre_scale,
                       const int32_t* __restrict__ page_off, uint2* __restrict__ packed, int32_t* __restrict__ page_flag) {
  const int page = blockIdx.x;
  const int32_t n0 = page_off[page], n1 = page_off[page + 1];
  const int32_t np = n1 - n0;
  const int32_t e0 = indptr[n0], e1 = indptr[n1];
  int outside = 0;
  for (int32_t e = e0 + threadIdx.x; e < e1; e += blockDim.x) {
    const int32_t c = __ldg(indices + e);
    float wv = w ? __ldg(w + (eid ? __ldg(eid + e) : e)) : 1.0f;
    if (pre_scale) wv *= __ldg(pre_scale + c);
    const int32_t sl = c - n0;
    const bool inside = sl >= 0 && sl < np;
    packed[e] = inside ? make_uint2((uint32_t)sl, __float_as_uint(wv)) : make_uint2(PK_OUTSIDE, 0u);
    outside |= inside ? 0 : 1;
  }
  outside = __syncthreads_or(outside);
  if (threadIdx.x == 0) page_flag[page] = outside;
}

__device__ __forceinline__ void fma4(float4& acc, float w, const float4& x) {
  acc.x = fmaf(w, x.x, acc.x);
  acc.y = fmaf(w, x.y, acc.y);
  acc.z = fmaf(w, x.z, acc.z);
  acc.w = fmaf(w, x.w, acc.w);
}
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
               "r"(bytes), "r"(bar)
               : "memory");
}

// 4-byte asynchronous copy global -> shared (no register round trip: every copy of a lane is in flight at once)
__device__ __forceinline__ void cp_async_4(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
// the mbarrier's current phase also waits for every cp.async this thread issued so far (pending count +1, then an
// arrive when they have landed: the expected arrival count is unchanged)
__device__ __forceinline__ void cp_async_mbar_arrive(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.shared.b64 [%0];" ::"r"(bar) : "memory");
}

struct PkStageLayout {
  uint32_t x_bytes, pk_bytes, ptr_bytes, nrm_bytes, info_bytes;
  // stages start on 128-byte boundaries (TMA destination alignment)
  __host__ __device__ uint32_t stage_bytes() const {
    return (x_bytes + pk_bytes + ptr_bytes + nrm_bytes + info_bytes + 127u) & ~127u;
  }
};
__host__ __device__ inline PkStageLayout pk_layout(int cs, int32_t np_cap, int32_t ne_cap) {
  PkStageLayout l;
  // staged rows (whole TMA boxes) + one all-zero row that padding / outside edges gather from
  l.x_bytes = ((((uint32_t)np_cap + PK_BOX_SMALL - 1) / PK_BOX_SMALL * PK_BOX_SMALL) + 1) * cs * 4;
  l.pk_bytes = (((uint32_t)ne_cap + 2) * 8 + 15u) & ~15u;  // +2: the bulk copy starts and ends on even edges
  l.ptr_bytes = (((uint32_t)np_cap + 1) * 4 + 15u) & ~15u;
  l.nrm_bytes = ((uint32_t)np_cap * 4 + 15u) & ~15u;
  l.info_bytes = 32;  // PkItem of the staged item, written by the producer warp
  return l;
}

struct PkItem {
  int32_t n0, np, e0, ne, c0, flag, staged, pad;
};

struct PkMaps {
  CUtensorMap big, small;  // x as [rows, f] fp32, boxes CS x 64 rows / CS x 8 rows, no swizzle
};

struct PkRowArgs {
  const uint8_t* xb;     // staged x slice [rows][CS] (+ one all-zero row at index zrow), already offset by lane * 16
  const uint2* spk;      // staged packed edges of the page
  const uint2* gpk;      // the same entries in global memory (MG variant: metadata through L1 instead of a stage)
  const int32_t* sptr;   // staged row pointers
  const float* snrm;     // staged row normalisers
  uint32_t zrow;
  bool slow;
  PkItem it;
  const int32_t *indptr, *indices, *eid;
  const float *w, *pre_scale, *row_norm;
  int mode;
  const float* x;
  int64_t ldx;
  const float* addend;
  int64_t ldadd;
  float* y;
  int64_t ldy;
  int32_t f;
};

// One pass of a row group over R (1 or 2) rows of a staged item: G lanes per row, each lane VV (<= V) 128-bit
// column chunks, U = 2 edges per step.  Every gather is unconditional: edges past the end of a row, and edges that
// leave the page, read the all-zero row with weight 0 (0 * 0: no NaN can be manufactured from someone else's Inf),
// and columns >= f were zero-filled by the TMA unit -- so all R*U*VV loads of a step are in flight together.
template <int G, int V, int VV, int R, bool MG>
__device__ __forceinline__ void pk_row_pass(const PkRowArgs& A, int32_t rl0) {
  constexpr int CS = G * V * 4;
  constexpr int ROW_BYTES = CS * 4;
  constexpr int NG = PK_CONSUMERS / G;
  constexpr int U = 2;
  const int lane = threadIdx.x % G;
  const PkItem& cur = A.it;
  int col[VV];
  bool on[VV];
#pragma unroll
  for (int v = 0; v < VV; ++v) {
    col[v] = cur.c0 + (lane + v * G) * 4;
    on[v] = col[v] < A.f;
  }
  int64_t row[R];
  int32_t beg[R], end[R];
#pragma unroll
  for (int q = 0; q < R; ++q) {
    const int32_t rl = rl0 + q * NG;
    row[q] = (int64_t)cur.n0 + rl;
    if (cur.staged) {
      beg[q] = A.sptr[rl] - cur.e0;
      end[q] = A.sptr[rl + 1] - cur.e0;
    } else {
      beg[q] = __ldg(A.indptr + row[q]) - cur.e0;
      end[q] = __ldg(A.indptr + row[q] + 1) - cur.e0;
    }
  }
  // row-end operands first: their latency overlaps the neighbour loop
  float4 av[R][VV];
  float nrm[R];
#pragma unroll
  for (int q = 0; q < R; ++q) {
#pragma unroll
    for (int v = 0; v < VV; ++v) {
      av[q][v] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (A.addend && on[v]) av[q][v] = __ldg(reinterpret_cast<const float4*>(A.addend + row[q] * A.ldadd + col[v]));
    }
    nrm[q] = 1.0f;
    if (A.mode == GTE_AGG_SUM_NORM) nrm[q] = cur.staged ? A.snrm[rl0 + q * NG] : __ldg(A.row_norm + row[q]);
  }
  float4 acc[R][VV];
#pragma unroll
  for (int q = 0; q < R; ++q)
#pragma unroll
    for (int v = 0; v < VV; ++v) acc[q][v] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (cur.staged) {
    int32_t len = end[0] - beg[0];
    if (R == 2) len = max(len, end[R - 1] - beg[R - 1]);
    auto load_meta = [&](int32_t j, uint2 (&m)[R][U]) {
#pragma unroll
      for (int q = 0; q < R; ++q)
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int32_t e = beg[q] + j + u;
          m[q][u] = make_uint2(PK_OUTSIDE, 0u);
          if (e < end[q]) m[q][u] = MG ? __ldg(A.gpk + e) : A.spk[e];
        }
    };
    auto step = [&](const uint2 (&m)[R][U]) {
      float4 xv[R][U][VV];
#pragma unroll
      for (int q = 0; q < R; ++q)
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const uint8_t* xr = A.xb + min(m[q][u].x, A.zrow) * ROW_BYTES;  // PK_OUTSIDE -> the zero row
#pragma unroll
          for (int v = 0; v < VV; ++v) xv[q][u][v] = *reinterpret_cast<const float4*>(xr + v * (G * 16));
        }
#pragma unroll
      for (int u = 0; u < U; ++u)  // edge order inside each row is preserved
#pragma unroll
        for (int q = 0; q < R; ++q)
#pragma unroll
          for (int v = 0; v < VV; ++v) fma4(acc[q][v], __uint_as_float(m[q][u].y), xv[q][u][v]);
    };
    // two metadata buffers alternate (no register rotation): the next step's metadata is in flight under this
    // step's gathers
    uint2 ma[R][U], mb[R][U];
    load_meta(0, ma);
    for (int32_t j = 0; j < len; j += 2 * U) {
      load_meta(j + U, mb);
      step(ma);
      if (j + U >= len) break;
      load_meta(j + 2 * U, ma);
      step(mb);
    }
  }
  if (A.slow) {  // rare: edges leaving the page (not block diagonal) or a page larger than the staging capacity
#pragma unroll 1
    for (int q = 0; q < R; ++q) {
      for (int32_t j = beg[q]; j < end[q]; ++j) {
        const int32_t c = __ldg(A.indices + cur.e0 + j);
        const int32_t sl = c - cur.n0;
        if (cur.staged && sl >= 0 && sl < cur.np) continue;  // already accumulated from shared memory
        float wt = A.w ? __ldg(A.w + (A.eid ? __ldg(A.eid + cur.e0 + j) : cur.e0 + j)) : 1.0f;
        if (A.pre_scale) wt *= __ldg(A.pre_scale + c);
#pragma unroll
        for (int v = 0; v < VV; ++v)
          if (on[v]) {
            const float4 xg = __ldg(reinterpret_cast<const float4*>(A.x + (int64_t)c * A.ldx + col[v]));
            if (q == 0) fma4(acc[0][v], wt, xg);
            else fma4(acc[R - 1][v], wt, xg);
          }
      }
    }
  }
#pragma unroll
  for (int q = 0; q < R; ++q) {
    const int32_t deg = end[q] - beg[q];
    const float d = (float)(deg > 1 ? deg : 1);
#pragma unroll
    for (int v = 0; v < VV; ++v) {
      if (!on[v]) continue;
      float4 r = acc[q][v];
      if (A.mode == GTE_AGG_MEAN) {
        r.x /= d; r.y /= d; r.z /= d; r.w /= d;
      } else if (A.mode == GTE_AGG_SUM_NORM) {
        r.x *= nrm[q]; r.y *= nrm[q]; r.z *= nrm[q]; r.w *= nrm[q];
      }
      if (A.addend) {
        r.x += av[q][v].x; r.y += av[q][v].y; r.z += av[q][v].z; r.w += av[q][v].w;
      }
      *reinterpret_cast<float4*>(A.y + row[q] * A.ldy + col[v]) = r;
    }
  }
}

template <int G, int V, int VV, bool MG>
__device__ __forceinline__ void pk_rows(const PkRowArgs& A) {
  constexpr int NG = PK_CONSUMERS / G;
  const int grp = threadIdx.x / G;
  for (int32_t rl0 = grp; rl0 < A.it.np; rl0 += 2 * NG) {
    if (rl0 + NG < A.it.np)
      pk_row_pass<G, V, VV, 2, MG>(A, rl0);
    else
      pk_row_pass<G, V, VV, 1, MG>(A, rl0);  // odd row out: no padded second row (its gathers would be pure waste)
  }
}

// Warp-specialised: warps 0..15 reduce rows (consumers), warp 16 stages items (producer).  Two shared-memory
// stages cycle through full[s] (producer -> consumers: TMA bytes landed + small copies stored) and empty[s]
// (consumer warps -> producer: stage may be overwritten) mbarriers; there is no CTA-wide barrier in the loop, so a
// warp that finishes its rows early starts on the next item at once and the warps drift out of lock step.
// MG: the packed edges are NOT staged (pages with many edges): consumers read them from global memory through L1
// (a row's entries are contiguous, 16 per cache line) and the stages hold only the x slice, so the 64-column
// configuration fits whatever the degree.
template <int G, int V, bool MG>
__global__ void __launch_bounds__(PK_THREADS, 1)
    k_spmm_paged_pk(const __grid_constant__ PkMaps maps, const int32_t* __restrict__ indptr,
                    const uint2* __restrict__ packed, const int32_t* __restrict__ page_flag,
                    const int32_t* __restrict__ indices, const int32_t* __restrict__ eid, const float* __restrict__ w,
                    const float* __restrict__ pre_scale, const float* __restrict__ row_norm, int mode,
                    const float* __restrict__ x, int64_t ldx, const float* __restrict__ addend, int64_t ldadd,
                    float* __restrict__ y, int64_t ldy, const int32_t* __restrict__ page_off, int32_t f, int32_t num_items,
                    int32_t nslices, int32_t items_per_cta, int32_t np_cap, int32_t ne_cap) {
  extern __shared__ __align__(128) uint8_t pk_smem[];
  constexpr int CS = G * V * 4;            // columns per slice
  constexpr int ROW_BYTES = CS * 4;
  const PkStageLayout L = pk_layout(CS, np_cap, MG ? 0 : ne_cap);
  const uint32_t stage_bytes = L.stage_bytes();
  const uint32_t smem0 = (uint32_t)__cvta_generic_to_shared(pk_smem);
  const uint32_t bars = smem0 + 2 * stage_bytes;  // full[0], full[1], empty[0], empty[1]
  const uint32_t off_pk = L.x_bytes, off_ptr = off_pk + L.pk_bytes, off_nrm = off_ptr + L.ptr_bytes,
                 off_info = off_nrm + L.nrm_bytes;
  const int tid = threadIdx.x;

  const int item_beg = blockIdx.x * items_per_cta;
  const int item_end = min(num_items, item_beg + items_per_cta);
  if (item_beg >= item_end) return;
  if (tid == 0) {
    mbar_init(bars, 2);        // producer: expect_tx arrive + "small copies stored" arrive
    mbar_init(bars + 8, 2);
    mbar_init(bars + 16, PK_CONSUMERS / 32);  // one arrive per consumer warp
    mbar_init(bars + 24, PK_CONSUMERS / 32);
    fence_barrier_init();
    tma_prefetch_desc(&maps.big);
    tma_prefetch_desc(&maps.small);
  }
  for (int i = tid; i < 2 * (ROW_BYTES / 4); i += PK_THREADS) {  // the all-zero row of both stages
    const int st = i / (ROW_BYTES / 4), c = i % (ROW_BYTES / 4);
    reinterpret_cast<float*>(pk_smem + (size_t)st * stage_bytes + L.x_bytes - ROW_BYTES)[c] = 0.f;
  }
  __syncthreads();

  if (tid >= PK_CONSUMERS) {
    // ================================== producer warp ==================================
    const int pl = tid - PK_CONSUMERS;  // lane
    auto load_item = [&](int item) {
      PkItem it = {0, 0, 0, 0, 0, 0, 0, 0};
      if (item < item_end) {
        const int page = item / nslices;
        it.c0 = (item - page * nslices) * CS;
        it.n0 = __ldg(page_off + page);
        it.np = __ldg(page_off + page + 1) - it.n0;
        it.e0 = __ldg(indptr + it.n0);
        it.ne = __ldg(indptr + it.n0 + it.np) - it.e0;
        it.flag = __ldg(page_flag + page);
        it.staged = (it.np <= np_cap && (MG || it.ne <= ne_cap)) ? 1 : 0;
      }
      return it;
    };
    PkItem it = load_item(item_beg);
    for (int item = item_beg, s = 0, k = 0; item < item_end; ++item, s ^= 1, ++k) {
      const PkItem nxt = load_item(item + 1);  // in flight while this item is staged
      if (k >= 2) mbar_wait_backoff(bars + 16 + s * 8, (uint32_t)((k >> 1) - 1) & 1u);  // consumers released stage s
      uint8_t* sbase = pk_smem + (size_t)s * stage_bytes;
      const uint32_t sx = smem0 + s * stage_bytes;
      const uint32_t bar = bars + s * 8;
      if (pl == 0) {
        *reinterpret_cast<PkItem*>(sbase + off_info) = it;
        if (it.staged) {
          const int nbig = it.np / PK_BOX_BIG;
          const int nsmall = (it.np - nbig * PK_BOX_BIG + PK_BOX_SMALL - 1) / PK_BOX_SMALL;
          const int e_lo = it.e0 & ~1;  // 16-byte aligned start of the bulk copy
          const uint32_t pk_copy = (!MG && it.ne > 0) ? (uint32_t)((it.e0 + it.ne - e_lo + 1) & ~1) * 8u : 0u;
          mbar_expect_tx(bar, (uint32_t)(nbig * PK_BOX_BIG + nsmall * PK_BOX_SMALL) * ROW_BYTES + pk_copy);
          for (int b = 0; b < nbig; ++b)
            tma_load_2d(sx + b * PK_BOX_BIG * ROW_BYTES, &maps.big, bar, it.c0, it.n0 + b * PK_BOX_BIG);
          for (int b = 0; b < nsmall; ++b)
            tma_load_2d(sx + (nbig * PK_BOX_BIG + b * PK_BOX_SMALL) * ROW_BYTES, &maps.small, bar, it.c0,
                        it.n0 + nbig * PK_BOX_BIG + b * PK_BOX_SMALL);
          if (pk_copy) bulk_load_1d(sx + off_pk, packed + e_lo, pk_copy, bar);
        } else {
          mbar_arrive(bar);  // nothing in flight: the page runs from global memory
        }
      }
      if (it.staged) {
        // row pointers and normalisers: 4-byte cp.async by the 32 producer lanes, completion tracked by full[s].
        // (Plain loads + shared stores cost the producer one global round trip per 4 entries and lane -- about six
        // per 300-row page -- and that chain, not the ring depth, set the time of the narrow slices.)
        const int32_t* ip = indptr + it.n0;
        for (int i = pl; i <= it.np; i += 32) cp_async_4(sx + off_ptr + 4u * i, ip + i);
        if (mode == GTE_AGG_SUM_NORM) {
          const float* nr = row_norm + it.n0;
          for (int i = pl; i < it.np; i += 32) cp_async_4(sx + off_nrm + 4u * i, nr + i);
        }
        cp_async_mbar_arrive(bar);
      }
      if (addend) {  // pull the addend rows of this slice into L2 ahead of the consumers
        for (int i = pl; i < it.np * 2; i += 32) {
          const int col = it.c0 + (i & 1) * 32;
          if (col < f) asm volatile("prefetch.global.L2 [%0];" ::"l"(addend + (int64_t)(it.n0 + (i >> 1)) * ldadd + col));
        }
      }
      __syncwarp();
      if (pl == 0) mbar_arrive(bar);  // release: item info + small copies are in shared memory
      it = nxt;
    }
  } else {
    // ================================== consumer warps ==================================
    const int lane = tid % G;
    PkRowArgs A;
    A.zrow = L.x_bytes / ROW_BYTES - 1;
    A.indptr = indptr; A.indices = indices; A.eid = eid; A.w = w; A.pre_scale = pre_scale; A.row_norm = row_norm;
    A.mode = mode; A.x = x; A.ldx = ldx; A.addend = addend; A.ldadd = ldadd; A.y = y; A.ldy = ldy; A.f = f;
    for (int item = item_beg, s = 0, k = 0; item < item_end; ++item, s ^= 1, ++k) {
      mbar_wait(bars + s * 8, (uint32_t)(k >> 1) & 1u);
      const uint8_t* sbase = pk_smem + (size_t)s * stage_bytes;
      A.it = *reinterpret_cast<const PkItem*>(sbase + off_info);
      A.xb = sbase + lane * 16;
      A.spk = reinterpret_cast<const uint2*>(sbase + off_pk) + (A.it.e0 & 1);  // entry j of the page: spk[j]
      A.gpk = packed + A.it.e0;
      A.sptr = reinterpret_cast<const int32_t*>(sbase + off_ptr);
      A.snrm = reinterpret_cast<const float*>(sbase + off_nrm);
      A.slow = !A.it.staged || A.it.flag != 0;
      // the last slice of a row may need only the first of the two column chunks (F = 218: 7 of 16 chunks)
      if (V == 2 && A.it.c0 + G * 4 >= f)
        pk_rows<G, V, 1, MG>(A);
      else
        pk_rows<G, V, V, MG>(A);
      __syncwarp();
      if ((tid & 31) == 0) mbar_arrive(bars + 16 + s * 8);  // this warp is done with stage s
    }
  }
}

static size_t pk_smem_bytes(int cs, int32_t np_cap, int32_t ne_cap) {
  return 2 * (size_t)pk_layout(cs, np_cap, ne_cap).stage_bytes() + 32;
}

constexpr size_t PK_SMEM_MAX = 227 * 1024;

// (G, V, MG) for feature width f and page capacity, or G = 0 when two stages do not fit in shared memory.
// The slice width follows f; for that width the packed edges are staged when they fit and read through L1
// otherwise; only then a narrower slice is tried.
static void pk_pick(int32_t f, int32_t np_cap, int32_t ne_cap, int* G, int* V, int* MG) {
  const int fv = (f + 3) / 4;
  *G = 0;
  *V = 0;
  *MG = 0;
  // measured order of preference (conv sweep, F = 218): staged edges beat L1 edges even at half the slice width
  // (degree 20: 35 % vs 26 % of the HBM roofline); L1 edges are for pages whose edges fit no stage (degree 40)
  struct Cand { int cs, mg; };
  const Cand wide[] = {{64, 0}, {32, 0}, {64, 1}, {32, 1}, {16, 0}, {16, 1}};
  const Cand mid[] = {{32, 0}, {32, 1}, {16, 0}, {16, 1}};
  const Cand narrow[] = {{16, 0}, {16, 1}};
  const Cand* c = fv > 8 ? wide : (fv > 4 ? mid : narrow);
  const int nc = fv > 8 ? 6 : (fv > 4 ? 4 : 2);
  for (int i = 0; i < nc; ++i) {
    if (pk_smem_bytes(c[i].cs, np_cap, c[i].mg ? 0 : ne_cap) <= PK_SMEM_MAX) {
      *G = c[i].cs == 16 ? 4 : 8;
      *V = c[i].cs == 64 ? 2 : 1;
      *MG = c[i].mg;
      return;
    }
  }
}

template <int G, int V, bool MG>
static int launch_spmm_paged_pk(const int32_t* indptr, const uint2* packed, const int32_t* page_flag,
                                const int32_t* indices, const int32_t* eid, const float* w, const float* pre_scale,
                                const float* row_norm, int mode, const float* x, int64_t ldx, const float* addend,
                                int64_t ldadd, float* y, int64_t ldy, const int32_t* page_off, int32_t num_pages,
                                int32_t np_cap, int32_t ne_cap, int32_t n_rows, int32_t f, cudaStream_t st) {
  constexpr int CS = G * V * 4;
  const size_t smem = pk_smem_bytes(CS, np_cap, MG ? 0 : ne_cap);
  if (int rc = ensure_dynamic_smem(reinterpret_cast<const void*>(&k_spmm_paged_pk<G, V, MG>), smem, "k_spmm_paged_pk")) return rc;
  // resident CTAs per SM for this shared-memory size (a host-side query, no cache: the answer depends on the device
  // and on smem, and a process-wide static would be wrong for both and racy)
  int occ = 1;
  GTE_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_spmm_paged_pk<G, V, MG>, PK_THREADS, smem),
                 "k_spmm_paged_pk(occupancy)");
  if (occ < 1) occ = 1;
  PkMaps maps;
  {
    int rc = make_tmap_2d(&maps.big, x, n_rows, f, ldx, CS, PK_BOX_BIG, CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;
    rc = make_tmap_2d(&maps.small, x, n_rows, f, ldx, CS, PK_BOX_SMALL, CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;
  }
  const int nslices = (int)ceil_div64((f + 3) / 4, G * V);
  const int64_t items = (int64_t)num_pages * nslices;
  GTE_CHECK_ARG(items < (int64_t)1 << 31, "gte_spmm_paged_packed: too many (page, slice) items");
  int grid = (int)(items < (int64_t)sm_count() * occ ? items : (int64_t)sm_count() * occ);
  const int per = (int)ceil_div64(items, grid);
  grid = (int)ceil_div64(items, per);
  k_spmm_paged_pk<G, V, MG><<<grid, PK_THREADS, smem, st>>>(maps, indptr, packed, page_flag, indices, eid, w, pre_scale, row_norm,
                                                       mode, x, ldx, addend, ldadd, y, ldy, page_off, f, (int32_t)items,
                                                       nslices, per, np_cap, ne_cap);
  GTE_CHECK_LAUNCH("k_spmm_paged_pk");
  return GTE_OK;
}

}  // namespace gte

using namespace gte;

extern "C" int gte_spmm(const int32_t* indptr, const int32_t* indices, const float* w, const float* pre_scale,
                        const float* row_norm, int mode, const float* x, int64_t ldx, const float* addend,
                        int64_t ldadd, float* y, int64_t ldy, int32_t n_rows, int32_t f, gte_stream_t stream) {
  GTE_CHECK_ARG(n_rows >= 0 && f >= 0, "gte_spmm: negative size");
  GTE_CHECK_ARG(mode == GTE_AGG_SUM || mode == GTE_AGG_SUM_NORM || mode == GTE_AGG_MEAN, "gte_spmm: bad mode %d", mode);
  if (n_rows == 0 || f == 0) return GTE_OK;
  GTE_CHECK_ARG(indptr && indices && x && y, "gte_spmm: null argument");
  GTE_CHECK_ARG(mode != GTE_AGG_SUM_NORM || row_norm, "gte_spmm: SUM_NORM needs row_norm");
  GTE_CHECK_ARG(ldx >= f && ldy >= f && (!addend || ldadd >= f), "gte_spmm: leading dimension < f");
  GTE_CHECK_ARG(x != y, "gte_spmm: x and y must not alias");
  cudaStream_t st = as_stream(stream);
  const bool vec = aligned16(x) && aligned16(y) && (ldx % 4 == 0) && (ldy % 4 == 0) &&
                   (!addend || (aligned16(addend) && ldadd % 4 == 0));
#define GTE_SPMM_GO(VEC, G, C) \
  return launch_spmm<VEC, G, C>(indptr, indices, w, pre_scale, row_norm, mode, x, ldx, addend, ldadd, y, ldy, n_rows, f, st)
  if (vec) {
    const int nv = (f + 3) / 4;  // 128-bit chunks per row (padding columns in [f, ld) are touched, never interpreted)
    if (nv <= 4) GTE_SPMM_GO(4, 4, 1);
    if (nv <= 8) GTE_SPMM_GO(4, 8, 1);
    if (nv <= 16) GTE_SPMM_GO(4, 16, 1);
    if (nv <= 32) GTE_SPMM_GO(4, 32, 1);
    if (nv <= 64) GTE_SPMM_GO(4, 32, 2);
    if (nv <= 96) GTE_SPMM_GO(4, 32, 3);
    GTE_SPMM_GO(4, 32, 4);  // wider rows tile over grid.y in blocks of 512 columns
  } else {
    if (f <= 4) GTE_SPMM_GO(1, 4, 1);
    if (f <= 8) GTE_SPMM_GO(1, 8, 1);
    if (f <= 16) GTE_SPMM_GO(1, 16, 1);
    if (f <= 32) GTE_SPMM_GO(1, 32, 1);
    if (f <= 64) GTE_SPMM_GO(1, 32, 2);
    GTE_SPMM_GO(1, 32, 4);  // blocks of 128 columns over grid.y
  }
#undef GTE_SPMM_GO
}

extern "C" int gte_spmm_paged(const int32_t* indptr, const int32_t* indices, const float* w, const float* pre_scale,
                              const float* row_norm, int mode, const float* x, int64_t ldx, const float* addend,
                              int64_t ldadd, float* y, int64_t ldy, const int32_t* page_off, int32_t num_pages,
                              int32_t max_page_nodes, int32_t max_page_edges, int32_t n_rows, int32_t f,
                              gte_stream_t stream) {
  GTE_CHECK_ARG(n_rows >= 0 && f >= 0 && num_pages >= 0 && max_page_nodes >= 0 && max_page_edges >= 0,
                "gte_spmm_paged: negative size");
  GTE_CHECK_ARG(mode == GTE_AGG_SUM || mode == GTE_AGG_SUM_NORM || mode == GTE_AGG_MEAN, "gte_spmm_paged: bad mode %d", mode);
  if (n_rows == 0 || f == 0 || num_pages == 0) return GTE_OK;
  GTE_CHECK_ARG(indptr && indices && x && y && page_off, "gte_spmm_paged: null argument");
  GTE_CHECK_ARG(mode != GTE_AGG_SUM_NORM || row_norm, "gte_spmm_paged: SUM_NORM needs row_norm");
  GTE_CHECK_ARG(ldx >= f && ldy >= f && (!addend || ldadd >= f), "gte_spmm_paged: leading dimension < f");
  GTE_CHECK_ARG(x != y, "gte_spmm_paged: x and y must not alias");
  const bool vec = aligned16(x) && aligned16(y) && (ldx % 4 == 0) && (ldy % 4 == 0) &&
                   (!addend || (aligned16(addend) && ldadd % 4 == 0));
  // widest column slice whose page working set fits ~110 KB of shared memory (2 CTAs per SM)
  const size_t budget = 110 * 1024;
  int G = 0;
  const int fv = (f + 3) / 4;  // 16-byte chunks per row
  for (int g : {32, 16, 8}) {
    if (paged_smem_bytes(g, max_page_nodes, max_page_edges) <= budget) {
      G = g;
      break;
    }
  }
  while (G > 8 && G / 2 >= fv) G /= 2;  // narrow rows: do not stage padding
  if (!vec || G == 0)  // unaligned operands or pages too large to stage: generic L2-gather kernel
    return gte_spmm(indptr, indices, w, pre_scale, row_norm, mode, x, ldx, addend, ldadd, y, ldy, n_rows, f, stream);
  cudaStream_t st = as_stream(stream);
#define GTE_PAGED_GO(GG)                                                                                               \
  return launch_spmm_paged<GG>(indptr, indices, w, pre_scale, row_norm, mode, x, ldx, addend, ldadd, y, ldy, page_off, \
                               num_pages, max_page_nodes, max_page_edges, f, st)
  if (G == 32) GTE_PAGED_GO(32);
  if (G == 16) GTE_PAGED_GO(16);
  GTE_PAGED_GO(8);
#undef GTE_PAGED_GO
}

extern "C" int gte_paged_pack_edges(const int32_t* indptr, const int32_t* indices, const int32_t* eid, const float* w,
                                    const float* pre_scale, const int32_t* page_off, int32_t num_pages,
                                    uint64_t* packed, int32_t* page_flag, gte_stream_t stream) {
  GTE_CHECK_ARG(num_pages >= 0, "gte_paged_pack_edges: negative size");
  if (num_pages == 0) return GTE_OK;
  GTE_CHECK_ARG(indptr && indices && page_off && packed && page_flag, "gte_paged_pack_edges: null argument");
  GTE_CHECK_ARG((reinterpret_cast<uintptr_t>(packed) & 7u) == 0, "gte_paged_pack_edges: packed must be 8-byte aligned");
  k_paged_pack_edges<<<num_pages, 256, 0, as_stream(stream)>>>(indptr, indices, eid, w, pre_scale, page_off,
                                                              reinterpret_cast<uint2*>(packed), page_flag);
  GTE_CHECK_LAUNCH("k_paged_pack_edges");
  return GTE_OK;
}

extern "C" size_t gte_spmm_paged_packed_smem_bytes(int32_t max_page_nodes, int32_t max_page_edges, int32_t f) {
  if (max_page_nodes < 0 || max_page_edges < 0 || f <= 0) return 0;
  int G, V, MG;
  pk_pick(f, max_page_nodes, max_page_edges, &G, &V, &MG);
  return G ? pk_smem_bytes(G * V * 4, max_page_nodes, MG ? 0 : max_page_edges) : 0;
}

extern "C" int gte_spmm_paged_packed(const int32_t* indptr, const uint64_t* packed, const int32_t* page_flag,
                                     const int32_t* indices, const int32_t* eid, const float* w, const float* pre_scale,
                                     const float* row_norm, int mode, const float* x, int64_t ldx, const float* addend,
                                     int64_t ldadd, float* y, int64_t ldy, const int32_t* page_off, int32_t num_pages,
                                     int32_t max_page_nodes, int32_t max_page_edges, int32_t n_rows, int32_t f,
                                     gte_stream_t stream) {
  GTE_CHECK_ARG(n_rows >= 0 && f >= 0 && num_pages >= 0 && max_page_nodes >= 0 && max_page_edges >= 0,
                "gte_spmm_paged_packed: negative size");
  GTE_CHECK_ARG(mode == GTE_AGG_SUM || mode == GTE_AGG_SUM_NORM || mode == GTE_AGG_MEAN, "gte_spmm_paged_packed: bad mode %d",
                mode);
  if (n_rows == 0 || f == 0 || num_pages == 0) return GTE_OK;
  GTE_CHECK_ARG(indptr && packed && page_flag && indices && x && y && page_off, "gte_spmm_paged_packed: null argument");
  GTE_CHECK_ARG(mode != GTE_AGG_SUM_NORM || row_norm, "gte_spmm_paged_packed: SUM_NORM needs row_norm");
  GTE_CHECK_ARG(ldx >= f && ldy >= f && (!addend || ldadd >= f), "gte_spmm_paged_packed: leading dimension < f");
  GTE_CHECK_ARG(x != y, "gte_spmm_paged_packed: x and y must not alias");
  const bool vec = aligned16(x) && aligned16(y) && (ldx % 4 == 0) && (ldy % 4 == 0) &&
                   (!addend || (aligned16(addend) && ldadd % 4 == 0));
  int G, V, MG;
  pk_pick(f, max_page_nodes, max_page_edges, &G, &V, &MG);
  if (!vec || G == 0)
    return fail(GTE_ERR_UNSUPPORTED,
                "gte_spmm_paged_packed: operands not 16-byte aligned or pages too large to stage (query "
                "gte_spmm_paged_packed_smem_bytes first); use gte_spmm_paged");
  cudaStream_t st = as_stream(stream);
  const uint2* pk = reinterpret_cast<const uint2*>(packed);
#define GTE_PK_GO(GG, VV, MM)                                                                                              \
  return launch_spmm_paged_pk<GG, VV, MM>(indptr, pk, page_flag, indices, eid, w, pre_scale, row_norm, mode, x, ldx,     \
                                          addend, ldadd, y, ldy, page_off, num_pages, max_page_nodes, max_page_edges,    \
                                          n_rows, f, st)
  if (G == 8 && V == 2 && !MG) GTE_PK_GO(8, 2, false);
  if (G == 8 && V == 2) GTE_PK_GO(8, 2, true);
  if (G == 8 && !MG) GTE_PK_GO(8, 1, false);
  if (G == 8) GTE_PK_GO(8, 1, true);
  if (!MG) GTE_PK_GO(4, 1, false);
  GTE_PK_GO(4, 1, true);
#undef GTE_PK_GO
}
