// The two steps either side of the layers that SURVEY.md section 8(f) ranks next:
//
//   k_page_predictions : `preds = logits.argmax(dim=1)` and the per-page accuracy
//                        `sum(preds == labels) / g.num_nodes()` of the predict loop
//                        (/root/reference/src/models/model_predict.py:144-154), for a whole batch of pages at once:
//                        int32 predictions (first maximal index, like torch.argmax) and per-page correct counts.
//   k_bbox_features    : the 13 BBOX node features of /root/reference/src/components/nlp/bbox.py:49-54,57-111:
//                        9 shape values from the integer box [x0, y0, x1, y1] and the 4-bin character-class
//                        histogram from per-box (letters, digits, others) counts -- float64 arithmetic like the
//                        Python original, cast to float32 at the end (model_train.py:295 `.float()`).
//
// Both are integer / tiny-arithmetic streams; results are bit-exact against the reference semantics.
#include "gte_common.cuh"

namespace gte {

__device__ __forceinline__ int64_t page_label(const void* labels, int dtype, int64_t i) {
  if (dtype == GTE_LABEL_I64) return static_cast<const int64_t*>(labels)[i];
  if (dtype == GTE_LABEL_I32) return static_cast<const int32_t*>(labels)[i];
  return (int64_t)static_cast<const float*>(labels)[i];  // float32 labels, `.long()` truncation (model_train.py:327)
}

// one CTA per page: predictions of its nodes + the page's number of correct predictions
__global__ void __launch_bounds__(256)
    k_page_predictions(const float* __restrict__ logits, int64_t ld, int32_t c, const void* __restrict__ labels,
                       int label_dtype, const int32_t* __restrict__ page_off, int32_t* __restrict__ preds,
                       int32_t* __restrict__ page_correct) {
  __shared__ int red[8];
  const int page = blockIdx.x;
  const int32_t n0 = page_off[page], n1 = page_off[page + 1];
  int correct = 0;
  for (int32_t i = n0 + threadIdx.x; i < n1; i += blockDim.x) {
    const int arg = row_argmax(logits + (int64_t)i * ld, c);
    preds[i] = arg;
    if (labels && page_label(labels, label_dtype, i) == arg) ++correct;
  }
  if (page_correct) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) correct += __shfl_xor_sync(0xffffffffu, correct, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = correct;
    __syncthreads();
    if (threadIdx.x == 0) {
      int s = 0;
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
      page_correct[page] = s;
    }
  }
}

// bbox.py:49-54 get_shape + bbox.py:57-111 get_histogram, one thread per text box
__global__ void k_bbox_features(const int32_t* __restrict__ boxes /*[n,4]*/, const int32_t* __restrict__ counts /*[n,3]*/,
                                float* __restrict__ out, int64_t ldo, int32_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t x0 = boxes[4 * i], y0 = boxes[4 * i + 1], x1 = boxes[4 * i + 2], y1 = boxes[4 * i + 3];
  const int32_t w = x1 - x0, h = y1 - y0;
  // int(width/2): Python true division, then truncation toward zero
  const int32_t hw = (int32_t)((double)w / 2.0), hh = (int32_t)((double)h / 2.0);
  float* o = out + i * ldo;
  o[0] = (float)w;
  o[1] = (float)h;
  o[2] = (float)(x1 - hw);
  o[3] = (float)(y1 - hh);
  o[4] = (float)((double)w * (double)h);
  o[5] = (float)x0;
  o[6] = (float)y0;
  o[7] = (float)x1;
  o[8] = (float)y1;
  double hist[4] = {0.0, 0.0, 0.0, 0.0};
  const int32_t lit = counts[3 * i], num = counts[3 * i + 1], oth = counts[3 * i + 2];
  const int32_t tot = lit + num + oth;
  if (tot != 0) {
    hist[0] = (double)lit / (double)tot;
    hist[1] = (double)num / (double)tot;
    hist[2] = (double)oth / (double)tot;
    // "keep sum 1 after truncate": Python sum() adds left to right starting from 0 (bbox.py:100-103)
    const double s = ((0.0 + hist[0]) + hist[1]) + hist[2] + hist[3];
    if (s != 1.0) {
      const double diff = 1.0 - s;
      double mxv = hist[0];
      int mi = 0;  // list.index(max(...)): first maximal entry
      for (int k = 1; k < 4; ++k)
        if (hist[k] > mxv) {
          mxv = hist[k];
          mi = k;
        }
      hist[mi] = mxv + diff;
    }
  }
  if (hist[0] == 0.0 && hist[1] == 0.0 && hist[2] == 0.0) hist[3] = 1.0;
  o[9] = (float)hist[0];
  o[10] = (float)hist[1];
  o[11] = (float)hist[2];
  o[12] = (float)hist[3];
}

}  // namespace gte

using namespace gte;

extern "C" int gte_page_predictions(const float* logits, int64_t ld, int32_t n, int32_t c, const void* labels,
                                    int label_dtype, const int32_t* page_off, int32_t num_pages, int32_t* preds,
                                    int32_t* page_correct, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0 && c > 0 && num_pages >= 0, "gte_page_predictions: bad size");
  GTE_CHECK_ARG(label_dtype >= GTE_LABEL_I64 && label_dtype <= GTE_LABEL_F32, "gte_page_predictions: bad label dtype");
  if (n == 0 || num_pages == 0) return GTE_OK;
  GTE_CHECK_ARG(logits && page_off && preds && ld >= c, "gte_page_predictions: bad argument");
  GTE_CHECK_ARG(!page_correct || labels, "gte_page_predictions: page_correct needs labels");
  k_page_predictions<<<num_pages, 256, 0, as_stream(stream)>>>(logits, ld, c, labels, label_dtype, page_off, preds,
                                                              page_correct);
  GTE_CHECK_LAUNCH("k_page_predictions");
  return GTE_OK;
}

extern "C" int gte_bbox_features(const int32_t* boxes, const int32_t* counts, int32_t n, float* out, int64_t ldo,
                                 gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0, "gte_bbox_features: negative size");
  if (n == 0) return GTE_OK;
  GTE_CHECK_ARG(boxes && counts && out && ldo >= 13, "gte_bbox_features: bad argument");
  k_bbox_features<<<(unsigned)ceil_div64(n, 256), 256, 0, as_stream(stream)>>>(boxes, counts, out, ldo, n);
  GTE_CHECK_LAUNCH("k_bbox_features");
  return GTE_OK;
}

// ---------------------------------------------------------------------------------------------------
// Batch assembly of a page batch in ONE kernel (SURVEY.md section 8(f) row 1; replaces `dgl.batch(...)`'s lazy
// COO -> CSC and COO -> CSR builds of /root/reference/src/models/model_train.py:297 + the per-layer
// `in_degrees` / `get_norm` of models.py:74-78):  one CTA per page sorts the page's edges by destination (CSC,
// forward) and by source (CSR, backward) entirely in shared memory -- stable, i.e. bit-identical to
// gte_csx_from_coo / a stable argsort of the batched COO -- and emits, in the same pass, the degree normaliser
// and the packed edge entries the conv-layer kernel stages (gte_paged_pack_edges' output for both directions).
// dgl.batch's contract is assumed: nodes and edges of page p occupy [page_off[p], page_off[p+1]) and
// [edge_off[p], edge_off[p+1]); an edge with an endpoint outside its page raises *bad (results undefined).
namespace gte {

constexpr int PF_THREADS = 256;

struct PfOut {
  int32_t *indptr, *indices, *eid;
  uint2* packed;
};

__global__ void __launch_bounds__(PF_THREADS)
    k_build_page_formats(const int32_t* __restrict__ src, const int32_t* __restrict__ dst, const float* __restrict__ w,
                         const int32_t* __restrict__ page_off, const int32_t* __restrict__ edge_off, int32_t num_pages,
                         int32_t np_cap, int32_t ne_cap, PfOut csc, PfOut csr, float* __restrict__ norm,
                         int* __restrict__ bad) {
  extern __shared__ __align__(16) int32_t pf_smem[];
  int32_t* s_src = pf_smem;                 // [ne_cap] page-local source of edge i
  int32_t* s_dst = s_src + ne_cap;          // [ne_cap]
  int32_t* slot_in = s_dst + ne_cap;        // [ne_cap] edge index per CSC position
  int32_t* slot_out = slot_in + ne_cap;     // [ne_cap]
  int32_t* ptr_in = slot_out + ne_cap;      // [np_cap + 1]
  int32_t* ptr_out = ptr_in + np_cap + 1;   // [np_cap + 1]
  int32_t* cur_in = ptr_out + np_cap + 1;   // [np_cap] counts, then fill cursors
  int32_t* cur_out = cur_in + np_cap;       // [np_cap]
  float* s_norm = reinterpret_cast<float*>(cur_out + np_cap);  // [np_cap]
  __shared__ int32_t warp_tot[2][PF_THREADS / 32];
  __shared__ int32_t carry[2];
  const int tid = threadIdx.x;
  const int page = blockIdx.x;
  const int32_t n0 = page_off[page], np = page_off[page + 1] - n0;
  const int32_t e0 = edge_off[page], ne = edge_off[page + 1] - e0;
  if (np > np_cap || ne > ne_cap) {  // cannot happen when the caller's maxima are right
    if (tid == 0) *bad = 2;
    return;
  }
  for (int i = tid; i < np; i += PF_THREADS) cur_in[i] = cur_out[i] = 0;
  __syncthreads();
  // 1. local ids + in/out degree counts
  for (int i = tid; i < ne; i += PF_THREADS) {
    const int32_t s = src[e0 + i] - n0, d = dst[e0 + i] - n0;
    const bool ok = s >= 0 && s < np && d >= 0 && d < np;
    if (!ok) *bad = 1;
    // an edge that leaves its page breaks the contract (*bad = 1, results meaningless) but must stay memory safe:
    // it is kept with its endpoints clamped to local node 0, so every count / cursor / slot below stays consistent
    const int32_t sl = ok ? s : 0, dl = ok ? d : 0;
    s_src[i] = sl;
    s_dst[i] = dl;
    atomicAdd(&cur_in[dl], 1);
    atomicAdd(&cur_out[sl], 1);
  }
  __syncthreads();
  // 2. exclusive scans of both degree arrays (block scan, PF_THREADS entries per round)
  if (tid < 2) carry[tid] = 0;
  __syncthreads();
  for (int base = 0; base < np; base += PF_THREADS) {
    const int i = base + tid;
    int32_t v[2] = {i < np ? cur_in[i] : 0, i < np ? cur_out[i] : 0};
    int32_t incl[2] = {v[0], v[1]};
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int32_t t0 = __shfl_up_sync(0xffffffffu, incl[0], o), t1 = __shfl_up_sync(0xffffffffu, incl[1], o);
      if ((tid & 31) >= o) {
        incl[0] += t0;
        incl[1] += t1;
      }
    }
    if ((tid & 31) == 31) {
      warp_tot[0][tid >> 5] = incl[0];
      warp_tot[1][tid >> 5] = incl[1];
    }
    __syncthreads();
    int32_t woff[2] = {0, 0};
    for (int k = 0; k < (tid >> 5); ++k) {
      woff[0] += warp_tot[0][k];
      woff[1] += warp_tot[1][k];
    }
    const int32_t ex0 = carry[0] + woff[0] + incl[0] - v[0], ex1 = carry[1] + woff[1] + incl[1] - v[1];
    if (i < np) {
      ptr_in[i] = ex0;
      ptr_out[i] = ex1;
    }
    __syncthreads();
    if (tid == PF_THREADS - 1) {
      carry[0] = ex0 + v[0];
      carry[1] = ex1 + v[1];
    }
    __syncthreads();
  }
  if (tid == 0) {
    ptr_in[np] = ne;
    ptr_out[np] = ne;
  }
  // 3. row pointers, normaliser; reset the cursors
  for (int i = tid; i < np; i += PF_THREADS) {
    const int32_t deg = cur_in[i];
    const float nv = deg > 0 ? 1.0f / (float)deg : 0.0f;  // 1./in_degree, inf -> 0 (models.py:75-76)
    s_norm[i] = nv;
    norm[n0 + i] = nv;
    csc.indptr[n0 + i] = e0 + ptr_in[i];
    csr.indptr[n0 + i] = e0 + ptr_out[i];
    cur_in[i] = 0;
    cur_out[i] = 0;
  }
  if (page == num_pages - 1 && tid == 0) {
    csc.indptr[n0 + np] = e0 + ne;
    csr.indptr[n0 + np] = e0 + ne;
  }
  __syncthreads();
  // 4. scatter edge indices into their rows (any order inside a row) ...
  for (int i = tid; i < ne; i += PF_THREADS) {
    const int32_t s = s_src[i], d = s_dst[i];
    slot_in[ptr_in[d] + atomicAdd(&cur_in[d], 1)] = i;
    slot_out[ptr_out[s] + atomicAdd(&cur_out[s], 1)] = i;
  }
  __syncthreads();
  // 5. ... then order every row by edge index (= stable sort of the COO): rows are short, one thread per row
  for (int r = tid; r < 2 * np; r += PF_THREADS) {
    int32_t* slot = r < np ? slot_in : slot_out;
    const int32_t* ptr = r < np ? ptr_in : ptr_out;
    const int rr = r < np ? r : r - np;
    const int b = ptr[rr], e = ptr[rr + 1];
    for (int a = b + 1; a < e; ++a) {
      const int32_t v = slot[a];
      int c = a - 1;
      while (c >= b && slot[c] > v) {
        slot[c + 1] = slot[c];
        --c;
      }
      slot[c + 1] = v;
    }
  }
  __syncthreads();
  // 6. write both formats and their packed entries
  for (int j = tid; j < ne; j += PF_THREADS) {
    const int32_t i = slot_in[j];
    const float wv = w ? __ldg(w + e0 + i) : 1.0f;
    csc.indices[e0 + j] = n0 + s_src[i];
    csc.eid[e0 + j] = e0 + i;
    csc.packed[e0 + j] = make_uint2((uint32_t)s_src[i], __float_as_uint(wv));
    const int32_t k = slot_out[j];
    float wk = w ? __ldg(w + e0 + k) : 1.0f;
    wk *= s_norm[s_dst[k]];  // source-side scale of the backward aggregation: norm[dst]
    csr.indices[e0 + j] = n0 + s_dst[k];
    csr.eid[e0 + j] = e0 + k;
    csr.packed[e0 + j] = make_uint2((uint32_t)s_dst[k], __float_as_uint(wk));
  }
}

static size_t pf_smem_bytes(int32_t np_cap, int32_t ne_cap) {
  return ((size_t)4 * ne_cap + 2 * ((size_t)np_cap + 1) + 3 * (size_t)np_cap) * 4 + 16;
}

}  // namespace gte

extern "C" size_t gte_build_page_formats_smem_bytes(int32_t max_page_nodes, int32_t max_page_edges) {
  if (max_page_nodes < 0 || max_page_edges < 0) return 0;
  const size_t b = gte::pf_smem_bytes(max_page_nodes, max_page_edges);
  return b <= 227 * 1024 ? b : 0;
}

extern "C" int gte_build_page_formats(const int32_t* src, const int32_t* dst, const float* w, const int32_t* page_off,
                                      const int32_t* edge_off, int32_t num_pages, int32_t n, int64_t e,
                                      int32_t max_page_nodes, int32_t max_page_edges, int32_t* csc_indptr,
                                      int32_t* csc_indices, int32_t* csc_eid, uint64_t* csc_packed, int32_t* csr_indptr,
                                      int32_t* csr_indices, int32_t* csr_eid, uint64_t* csr_packed, float* norm,
                                      int32_t* page_flag, int32_t* bad, gte_stream_t stream) {
  GTE_CHECK_ARG(num_pages >= 0 && n >= 0 && e >= 0 && max_page_nodes >= 0 && max_page_edges >= 0,
                "gte_build_page_formats: negative size");
  const size_t smem = gte_build_page_formats_smem_bytes(max_page_nodes, max_page_edges);
  if (smem == 0)
    return fail(GTE_ERR_UNSUPPORTED, "gte_build_page_formats: a page of %d nodes / %d edges does not fit in shared memory",
                max_page_nodes, max_page_edges);
  GTE_CHECK_ARG(page_off && edge_off && csc_indptr && csr_indptr && norm && bad && page_flag,
                "gte_build_page_formats: null argument");
  GTE_CHECK_ARG(e == 0 || (src && dst && csc_indices && csc_eid && csc_packed && csr_indices && csr_eid && csr_packed),
                "gte_build_page_formats: null edge argument");
  cudaStream_t st = as_stream(stream);
  GTE_CHECK_CUDA(cudaMemsetAsync(bad, 0, 4, st), "gte_build_page_formats(memset bad)");
  if (num_pages == 0) {
    GTE_CHECK_CUDA(cudaMemsetAsync(csc_indptr, 0, 4, st), "gte_build_page_formats(memset)");
    GTE_CHECK_CUDA(cudaMemsetAsync(csr_indptr, 0, 4, st), "gte_build_page_formats(memset)");
    return GTE_OK;
  }
  GTE_CHECK_CUDA(cudaMemsetAsync(page_flag, 0, (size_t)num_pages * 4, st), "gte_build_page_formats(memset flags)");
  if (int rc = ensure_dynamic_smem(reinterpret_cast<const void*>(&k_build_page_formats), smem, "k_build_page_formats")) return rc;
  PfOut a{csc_indptr, csc_indices, csc_eid, reinterpret_cast<uint2*>(csc_packed)};
  PfOut b{csr_indptr, csr_indices, csr_eid, reinterpret_cast<uint2*>(csr_packed)};
  k_build_page_formats<<<num_pages, PF_THREADS, smem, st>>>(src, dst, w, page_off, edge_off, num_pages, max_page_nodes,
                                                           max_page_edges, a, b, norm, bad);
  GTE_CHECK_LAUNCH("k_build_page_formats");
  return GTE_OK;
}

// ---------------------------------------------------------------------------------------------------
// Padding of a page batch to a fixed capacity shape, on the device (the first kernel of a capacity-captured step).
// The reference trains on shuffled batches of real pages whose node / edge totals change every step
// (/root/reference/src/models/model_train.py:283-297) and predicts on streams ending with a short batch
// (model_predict.py:130-154); a CUDA graph needs one shape.  The host copies only the real prefix (n nodes, e edges,
// P pages) into buffers sized [n_cap] / [e_cap]; this kernel turns the tail into padding that is itself a legal
// dgl.batch, so every later kernel runs on it unchanged:
//   feat[n, n_cap) = 0, label[n, n_cap) = -1 (weight 0 in the loss, never counted correct),
//   edges [e, e_cap): weight 0, src = dst = a padding node of the page that owns the edge (a self-loop).
// The page table is written by the HOST: page_off / edge_off hold all p_cap + 1 entries (real pages, then padding
// pages of at most the capacity's page sizes, then empty pages), so this kernel only reads it to find the page of a
// padding edge (binary search over edge_off).  `word` = (n, e, P) of the batch, copied with it.  The grid is fixed by
// the capacity; grid-stride loops are bounded by the counts read from `word`.  A word outside the capacity, or a
// page table that gives a padding edge no padding node, raises *bad (1 / 2); the kernel then clamps, so it never
// writes outside [0, n_cap) rows / [0, e_cap) edges (an out-of-page self-loop is left for gte_build_page_formats to
// report).
namespace gte {

constexpr int PAD_THREADS = 256;

__global__ void __launch_bounds__(PAD_THREADS)
    k_pad_batch(const int32_t* __restrict__ word, int32_t n_cap, int32_t e_cap, int32_t p_cap,
                const int32_t* __restrict__ page_off, const int32_t* __restrict__ edge_off, int32_t* __restrict__ src,
                int32_t* __restrict__ dst, float* __restrict__ w, float* __restrict__ feat, int64_t ldf, int32_t f,
                float* __restrict__ label, int* __restrict__ bad) {
  int32_t n = word[0], e = word[1];
  const int32_t p = word[2];
  if (n < 0 || n > n_cap || e < 0 || e > e_cap || p < 0 || p > p_cap) {
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(bad, 1);
    n = min(max(n, 0), n_cap);
    e = min(max(e, 0), e_cap);
  }
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t nf = (int64_t)(n_cap - n) * f;
  for (int64_t k = t0; k < nf; k += stride) feat[(n + k / f) * ldf + k % f] = 0.0f;
  for (int64_t i = n + t0; i < n_cap; i += stride) label[i] = -1.0f;
  for (int64_t i = e + t0; i < e_cap; i += stride) {
    // page of edge i: the last page whose first edge is <= i
    int32_t lo = 0, hi = p_cap - 1;
    while (lo < hi) {
      const int32_t mid = (lo + hi + 1) >> 1;
      if (edge_off[mid] <= i) lo = mid; else hi = mid - 1;
    }
    const int32_t n0 = page_off[lo], cnt = page_off[lo + 1] - n0;
    const int64_t j = i - edge_off[lo];
    int32_t v;
    if (cnt > 0 && n0 >= n && n0 + cnt <= n_cap && j >= 0) {
      v = n0 + (int32_t)(j % cnt);
    } else {
      atomicOr(bad, 2);
      v = n_cap - 1;
    }
    src[i] = v;
    dst[i] = v;
    w[i] = 0.0f;
  }
}

}  // namespace gte

extern "C" int gte_pad_batch(const int32_t* word, int32_t n_cap, int64_t e_cap, int32_t p_cap, const int32_t* page_off,
                             const int32_t* edge_off, int32_t* src, int32_t* dst, float* weight, float* feat, int64_t ldf,
                             int32_t f, float* label, int32_t* bad, gte_stream_t stream) {
  GTE_CHECK_ARG(n_cap > 0 && e_cap >= 0 && e_cap < ((int64_t)1 << 31) && p_cap > 0 && f > 0 && ldf >= f,
                "gte_pad_batch: bad capacity");
  GTE_CHECK_ARG(word && page_off && edge_off && feat && label && bad, "gte_pad_batch: null argument");
  GTE_CHECK_ARG(e_cap == 0 || (src && dst && weight), "gte_pad_batch: null edge argument");
  cudaStream_t st = as_stream(stream);
  GTE_CHECK_CUDA(cudaMemsetAsync(bad, 0, 4, st), "gte_pad_batch(memset bad)");
  const int64_t work = (int64_t)n_cap * f > e_cap ? (int64_t)n_cap * f : e_cap;
  const int64_t cap_blocks = 4 * (int64_t)sm_count();
  int64_t blocks = ceil_div64(work, PAD_THREADS);
  if (blocks > cap_blocks) blocks = cap_blocks;
  if (blocks < 1) blocks = 1;
  k_pad_batch<<<(unsigned)blocks, PAD_THREADS, 0, st>>>(word, n_cap, (int32_t)e_cap, p_cap, page_off, edge_off, src, dst, weight,
                                              feat, ldf, f, label, bad);
  GTE_CHECK_LAUNCH("k_pad_batch");
  return GTE_OK;
}

// ---------------------------------------------------------------------------------------------------
// Batches gathered from a device-resident page pool (the first kernels of a resident capacity-captured pass).
// The reference builds every training batch on the host (`dgl.batch(train_batch).to(device)`,
// /root/reference/src/models/model_train.py:279-297) and every predict batch the same way (model_predict.py:130-154);
// here the pages stay in HBM (PagePool) and the captured pass itself assembles the next batch of an epoch plan:
//   k_gather_plan   : one CTA; reads the plan cursor, checks the batch against the capacity and writes the static
//                     set's `meta` = (n, e, P, start | padded page table) -- what the host uploads for a host-fed batch;
//   k_gather_pages  : copies the batch's pages (features, labels, weights, page-local src / dst + node offset) into the
//                     real prefix of the static set; gte_pad_batch then pads it as for a host-fed batch.
// Plan layout (int32): [cursor, flag, nfit, B, L, 0, 0, 0 | ids[L] | starts[nfit]]: slice k of the plan is
// ids[starts[k], min(starts[k] + B, L)).
namespace gte {

constexpr int PLAN_HDR = 8;
constexpr int PLAN_THREADS = 1024;
constexpr int GATHER_THREADS = 256;

struct GatherCap {
  int32_t nodes, pages, page_nodes, page_edges;
  int64_t edges;
  int32_t n_cap, e_cap, p_cap;
};

// inclusive block scan of two int32 values (PLAN_THREADS threads); returns the block totals in tot[2]
__device__ __forceinline__ void block_scan2(int32_t& a, int32_t& b, int32_t* warp_a, int32_t* warp_b, int32_t* tot) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int32_t ta = __shfl_up_sync(0xffffffffu, a, o), tb = __shfl_up_sync(0xffffffffu, b, o);
    if (lane >= o) {
      a += ta;
      b += tb;
    }
  }
  if (lane == 31) {
    warp_a[w] = a;
    warp_b[w] = b;
  }
  __syncthreads();
  if (w == 0) {
    int32_t xa = lane < PLAN_THREADS / 32 ? warp_a[lane] : 0, xb = lane < PLAN_THREADS / 32 ? warp_b[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int32_t ta = __shfl_up_sync(0xffffffffu, xa, o), tb = __shfl_up_sync(0xffffffffu, xb, o);
      if (lane >= o) {
        xa += ta;
        xb += tb;
      }
    }
    warp_a[lane] = xa;  // inclusive warp prefixes
    warp_b[lane] = xb;
    if (lane == 31) {
      tot[0] = xa;
      tot[1] = xb;
    }
  }
  __syncthreads();
  if (w > 0) {
    a += warp_a[w - 1];
    b += warp_b[w - 1];
  }
  __syncthreads();
}

__global__ void __launch_bounds__(PLAN_THREADS)
    k_gather_plan(int32_t* __restrict__ plan, const int32_t* __restrict__ pool_n, const int32_t* __restrict__ pool_e,
                  int32_t pool_pages, GatherCap cap, int32_t* __restrict__ meta) {
  __shared__ int32_t hdr[3];  // start, P, status
  __shared__ unsigned long long s_n, s_e;
  __shared__ int32_t s_mn, s_me, s_badid;
  __shared__ int32_t warp_a[PLAN_THREADS / 32], warp_b[PLAN_THREADS / 32], tot[2];
  const int tid = threadIdx.x;
  if (tid == 0) {
    const int32_t cur = plan[0], nfit = plan[2], b = plan[3], l = plan[4];
    int32_t status = 0, start = 0, p = 0;
    if (cur < 0 || cur >= nfit || b < 1 || l < 1 || l > pool_pages || nfit > l) {  // reads stay in 8 + 2 * pool_pages words
      status = 1;
    } else {
      start = plan[PLAN_HDR + l + cur];
      if (start < 0 || start >= l) status = 1;
      else p = min(b, l - start);
    }
    if (status == 0 && p > cap.pages) status = 2;
    hdr[0] = start;
    hdr[1] = p;
    hdr[2] = status;
    s_n = s_e = 0ull;
    s_mn = s_me = 0;
    s_badid = 0;
    plan[0] = cur + 1;  // one planned batch per launch
    if (status) atomicOr(plan + 1, status);
  }
  __syncthreads();
  if (hdr[2]) return;
  const int32_t start = hdr[0], p = hdr[1];
  const int32_t* ids = plan + PLAN_HDR + start;
  // 1. totals and largest page of the batch: nothing is written before it is known to fit
  unsigned long long ln = 0, le = 0;
  int32_t mn = 0, me = 0;
  for (int j = tid; j < p; j += PLAN_THREADS) {
    const int32_t id = ids[j];
    if (id < 0 || id >= pool_pages) {
      s_badid = 1;
      continue;
    }
    const int32_t a = pool_n[id], b = pool_e[id];
    ln += (unsigned long long)max(a, 0);
    le += (unsigned long long)max(b, 0);
    mn = max(mn, a);
    me = max(me, b);
  }
  atomicAdd(&s_n, ln);
  atomicAdd(&s_e, le);
  atomicMax(&s_mn, mn);
  atomicMax(&s_me, me);
  __syncthreads();
  const int64_t n64 = (int64_t)s_n, e64 = (int64_t)s_e;
  // BatchCapacity.check: pages, nodes, edges, largest page
  if (s_badid || n64 > cap.nodes || e64 > cap.edges || s_mn > cap.page_nodes || s_me > cap.page_edges) {
    if (tid == 0) atomicOr(plan + 1, 2);
    return;
  }
  const int32_t n = (int32_t)n64, e = (int32_t)e64;
  int32_t* po = meta + 4;
  int32_t* eo = meta + 5 + cap.p_cap;
  // 2. offsets of the real pages
  int32_t carry_n = 0, carry_e = 0;
  for (int base = 0; base < p; base += PLAN_THREADS) {
    const int j = base + tid;
    int32_t a = 0, b = 0;
    if (j < p) {
      const int32_t id = ids[j];
      a = pool_n[id];
      b = pool_e[id];
    }
    block_scan2(a, b, warp_a, warp_b, tot);
    if (j < p) {
      po[j + 1] = carry_n + a;
      eo[j + 1] = carry_e + b;
    }
    carry_n += tot[0];
    carry_e += tot[1];
    __syncthreads();
  }
  // 3. padding pages and empty pages, as engine.padded_page_table
  const int32_t s = min(cap.p_cap - p, cap.n_cap - n);
  for (int j = p + 1 + tid; j <= cap.p_cap; j += PLAN_THREADS) {
    const int64_t k = j - p;  // 1-based padding slot
    if (k <= s) {
      po[j] = (int32_t)(n + k * (int64_t)(cap.n_cap - n) / s);
      eo[j] = (int32_t)(e + k * (int64_t)(cap.e_cap - e) / s);
    } else {
      po[j] = cap.n_cap;
      eo[j] = cap.e_cap;
    }
  }
  if (tid == 0) {
    po[0] = 0;
    eo[0] = 0;
    meta[0] = n;
    meta[1] = e;
    meta[2] = p;
    meta[3] = start;
  }
}

// dst[i] = src[i] + add over `count` 32-bit words; float4 / int4 accesses where both sides share their 16-byte phase
template <typename T>
__device__ __forceinline__ void copy_words(T* __restrict__ dst, const T* __restrict__ src, int64_t count, int32_t add) {
  static_assert(sizeof(T) == 4, "32-bit words");
  int64_t head = 0;
  const bool vec = ((reinterpret_cast<uintptr_t>(dst) ^ reinterpret_cast<uintptr_t>(src)) & 15u) == 0;
  if (vec) {
    head = (int64_t)(((16u - (reinterpret_cast<uintptr_t>(dst) & 15u)) & 15u) >> 2);
    if (head > count) head = count;
    const int64_t nv = (count - head) >> 2;
    const int4* s4 = reinterpret_cast<const int4*>(src + head);
    int4* d4 = reinterpret_cast<int4*>(dst + head);
    for (int64_t k = threadIdx.x; k < nv; k += blockDim.x) {
      int4 v = __ldg(s4 + k);
      if (add) {
        v.x += add;
        v.y += add;
        v.z += add;
        v.w += add;
      }
      d4[k] = v;
    }
    for (int64_t k = head + 4 * nv + threadIdx.x; k < count; k += blockDim.x) {
      if (add) dst[k] = (T)(__ldg(src + k) + add);
      else dst[k] = __ldg(src + k);
    }
    if (threadIdx.x < head) {
      if (add) dst[threadIdx.x] = (T)(__ldg(src + threadIdx.x) + add);
      else dst[threadIdx.x] = __ldg(src + threadIdx.x);
    }
    return;
  }
  for (int64_t k = threadIdx.x; k < count; k += blockDim.x) {
    if (add) dst[k] = (T)(__ldg(src + k) + add);
    else dst[k] = __ldg(src + k);
  }
}

__global__ void __launch_bounds__(GATHER_THREADS)
    k_gather_pages(int32_t* __restrict__ plan, const int32_t* __restrict__ meta, int32_t n_cap, int32_t e_cap,
                   int32_t p_cap, const int64_t* __restrict__ pool_node_off, const int64_t* __restrict__ pool_edge_off,
                   int32_t pool_pages, const int32_t* __restrict__ pool_src, const int32_t* __restrict__ pool_dst,
                   const float* __restrict__ pool_w, const float* __restrict__ pool_feat,
                   const float* __restrict__ pool_label, int32_t f, int32_t* __restrict__ src, int32_t* __restrict__ dst,
                   float* __restrict__ w, float* __restrict__ feat, float* __restrict__ label) {
  // a flagged plan (the plan kernel refused this batch, so meta still describes an earlier one): copy nothing
  if (plan[1] != 0) return;
  const int32_t p = meta[2], start = meta[3], l = plan[4];
  if (p < 0 || p > p_cap || start < 0 || l > pool_pages || (int64_t)start + p > l) {
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(plan + 1, 4);
    return;
  }
  const int32_t* ids = plan + PLAN_HDR + start;
  const int32_t* po = meta + 4;
  const int32_t* eo = meta + 5 + p_cap;
  for (int32_t j = blockIdx.x; j < p; j += gridDim.x) {
    const int32_t id = ids[j];
    const int32_t nb = po[j], ni = po[j + 1] - nb, eb = eo[j], ei = eo[j + 1] - eb;
    // the page table must describe exactly these pool pages (it does unless the plan buffer was rewritten after
    // k_gather_plan ran): otherwise skip the page and flag, never copy out of bounds
    bool ok = id >= 0 && id < pool_pages && nb >= 0 && ni >= 0 && (int64_t)nb + ni <= n_cap && eb >= 0 && ei >= 0 &&
              (int64_t)eb + ei <= e_cap;
    int64_t pn = 0, pe = 0;
    if (ok) {
      pn = pool_node_off[id];
      pe = pool_edge_off[id];
      ok = pool_node_off[id + 1] - pn == ni && pool_edge_off[id + 1] - pe == ei;
    }
    if (!ok) {
      if (threadIdx.x == 0) atomicOr(plan + 1, 4);
      continue;
    }
    copy_words(feat + (int64_t)nb * f, pool_feat + pn * f, (int64_t)ni * f, 0);
    copy_words(label + nb, pool_label + pn, ni, 0);
    copy_words(w + eb, pool_w + pe, ei, 0);
    copy_words(src + eb, pool_src + pe, ei, nb);
    copy_words(dst + eb, pool_dst + pe, ei, nb);
  }
}

}  // namespace gte

extern "C" int gte_gather_plan(int32_t* plan, const int32_t* pool_num_nodes, const int32_t* pool_num_edges,
                               int32_t pool_pages, int32_t cap_nodes, int64_t cap_edges, int32_t cap_pages,
                               int32_t cap_page_nodes, int32_t cap_page_edges, int32_t n_cap, int64_t e_cap, int32_t p_cap,
                               int32_t* meta, gte_stream_t stream) {
  GTE_CHECK_ARG(plan && pool_num_nodes && pool_num_edges && meta, "gte_gather_plan: null argument");
  GTE_CHECK_ARG(pool_pages > 0 && cap_nodes > 0 && cap_edges >= 0 && cap_pages > 0 && cap_page_nodes > 0 &&
                    cap_page_edges > 0, "gte_gather_plan: bad pool or capacity");
  GTE_CHECK_ARG(n_cap > cap_nodes && e_cap >= cap_edges && e_cap < ((int64_t)1 << 31) && p_cap > cap_pages,
                "gte_gather_plan: padded shape below the capacity");
  GatherCap cap{cap_nodes, cap_pages, cap_page_nodes, cap_page_edges, cap_edges, n_cap, (int32_t)e_cap, p_cap};
  k_gather_plan<<<1, PLAN_THREADS, 0, as_stream(stream)>>>(plan, pool_num_nodes, pool_num_edges, pool_pages, cap, meta);
  GTE_CHECK_LAUNCH("k_gather_plan");
  return GTE_OK;
}

extern "C" int gte_gather_pages(int32_t* plan, const int32_t* meta, int32_t n_cap, int64_t e_cap, int32_t p_cap,
                                int32_t max_pages, const int64_t* pool_node_off, const int64_t* pool_edge_off,
                                int32_t pool_pages, const int32_t* pool_src, const int32_t* pool_dst,
                                const float* pool_weight, const float* pool_feat, const float* pool_label, int32_t f,
                                int32_t* src, int32_t* dst, float* weight, float* feat, float* label,
                                gte_stream_t stream) {
  GTE_CHECK_ARG(plan && meta && pool_node_off && pool_edge_off && pool_feat && pool_label && feat && label,
                "gte_gather_pages: null argument");
  GTE_CHECK_ARG(e_cap == 0 || (src && dst && weight), "gte_gather_pages: null edge argument");
  GTE_CHECK_ARG(pool_pages > 0 && f > 0 && n_cap > 0 && e_cap >= 0 && e_cap < ((int64_t)1 << 31) && p_cap > 0 &&
                    max_pages > 0 && max_pages <= p_cap, "gte_gather_pages: bad size");
  int64_t blocks = 4 * (int64_t)sm_count();
  if (blocks > max_pages) blocks = max_pages;
  k_gather_pages<<<(unsigned)blocks, GATHER_THREADS, 0, as_stream(stream)>>>(
      plan, meta, n_cap, (int32_t)e_cap, p_cap, pool_node_off, pool_edge_off, pool_pages, pool_src, pool_dst, pool_weight,
      pool_feat, pool_label, f, src, dst, weight, feat, label);
  GTE_CHECK_LAUNCH("k_gather_pages");
  return GTE_OK;
}
