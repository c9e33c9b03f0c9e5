/*
 * gte.h -- C ABI of libgte_b200.so: the B200-native (sm_100a) graph-convolution
 * hot path of AILab-UniFI/GNN-TableExtraction.
 *
 * The reference has no FFI of its own: the path sits behind the Python
 * nn.Module API of /root/reference/src/components/graphs/models.py and reaches
 * its arithmetic through DGL (`g.update_all`, `g.in_degrees`) and ATen
 * (`nn.Linear`, `nn.LayerNorm`, `F.relu`).  Each entry point below names the
 * reference call site (file:line under /root/reference) that it replaces.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer into caller-owned (PyTorch) storage,
 *     unless the parameter name ends in `_host`;
 *   - the library never allocates or frees user-visible memory and keeps no
 *     reference after return; scratch space is passed in (`ws`, `ws_bytes`,
 *     sizes from the matching `*_workspace_bytes` query);
 *   - every launch goes to the `stream` passed in (a cudaStream_t); nothing
 *     synchronises the device, so all entries are CUDA-graph capturable;
 *   - every entry returns 0 on success and a negative GTE_ERR_* otherwise;
 *     `gte_last_error_string()` (thread-local) explains the failure.  No C++
 *     exception crosses the ABI.  There is NO CPU fallback: host pointers are
 *     rejected where detectable, and the Python host layer refuses to run
 *     without this library;
 *   - node / edge ids are int32 (builder.py:425), row offsets are computed in
 *     64-bit; features, weights and parameters are fp32 (model_train.py:295);
 *   - feature matrices are row-major with an explicit leading dimension `ld*`
 *     (in floats).  Kernels vectorise to 128-bit accesses when the pointers are
 *     16-byte aligned and the leading dimensions are multiples of 4; columns in
 *     [f, ld) are padding and are never interpreted.
 */
#ifndef GTE_H_
#define GTE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* gte_stream_t; /* cudaStream_t */

#define GTE_ABI_VERSION 2

#define GTE_OK 0
#define GTE_ERR_INVALID (-1)     /* bad argument (null pointer, negative size, bad enum) */
#define GTE_ERR_UNSUPPORTED (-2) /* shape / device not supported by this build */
#define GTE_ERR_CUDA (-3)        /* a CUDA runtime call or launch failed */
#define GTE_ERR_WORKSPACE (-4)   /* workspace missing or too small */

/* aggregation modes of gte_spmm */
#define GTE_AGG_SUM 0       /* y = sum_e w_e x[src]                      (models.py:53-54) */
#define GTE_AGG_SUM_NORM 1  /* y = norm[v] * sum_e w_e x[src]            (models.py:69-71) */
#define GTE_AGG_MEAN 2      /* y = (sum_e w_e x[src]) / max(deg[v], 1)   (models.py:149)   */

/* degree-normaliser modes of gte_degree_norm */
#define GTE_NORM_INV_DEG_ZERO 0 /* 1/deg, 0 where deg == 0  (models.py:74-78 get_norm)     */
#define GTE_NORM_INV_DEG_CLAMP 1 /* 1/max(deg,1)            (DGL fn.mean, models.py:149)   */

/* label dtypes of the cross-entropy entries */
#define GTE_LABEL_I64 0
#define GTE_LABEL_I32 1
#define GTE_LABEL_F32 2 /* the reference stores labels as float32 (loader.py:350-354) */

/* ---------------------------------------------------------------- misc -- */
int gte_abi_version(void);
const char* gte_last_error_string(void);
/* Kernels launched by this library since it was loaded (process-wide diagnostic counter). */
int64_t gte_launch_count(void);

/*
 * Process-wide A/B switches for tests and measurements (NOT a configuration surface: the defaults are the product
 * path; every value computes the same results through a different kernel).
 *   GTE_TUNE_UMMA_PAIR   1 (default): tensor-core projections run on CTA pairs (tcgen05 cta_group::2) when the shape
 *                        allows it; 0: always the single-CTA kernel
 *   GTE_TUNE_DW_PAIR     reserved, no effect (the weight-gradient kernel has one form: a CTA-pair variant would not raise
 *                        its MMA rate and was not built -- DESIGN.md section d)
 *   GTE_TUNE_UMMA_SPLIT  1 (default): contractions of more than two k-blocks keep the 3xTF32 cross terms in their own
 *                        TMEM accumulator; 0: one accumulator (and two accumulator stages) for every shape
 *   GTE_TUNE_EPI_STORE   0 (default): the pair kernel's epilogue leaves through TMA stores; 1: through the epilogue
 *                        warps' own row-contiguous 128-bit global stores
 */
#define GTE_TUNE_UMMA_PAIR 0
#define GTE_TUNE_DW_PAIR 1
#define GTE_TUNE_EPI_STORE 2
#define GTE_TUNE_UMMA_SPLIT 3
#define GTE_TUNE_COUNT 4
int gte_set_tuning(int key, int value);
int gte_get_tuning(int key);
/* SM count and compute capability of the current device. */
int gte_device_info(int* sm_count_host, int* cc_major_host, int* cc_minor_host);

/* ----------------------------------------------------- graph formats ---- */
/*
 * Stable COO -> compressed rows over `key` (key = dst gives the CSC that
 * `update_all` aggregates over, models.py:53-54; key = src gives the CSR that
 * autograd's reverse-graph SpMM needs).  Replaces DGL's lazy per-batch format
 * build.  Output is bit-identical to a stable sort of the COO by `key`:
 *   indptr [n+1], indices [e] (= `other` in row order), eid [e] (= original
 *   edge position; ties inside a row ascending by eid).
 */
size_t gte_csx_from_coo_workspace_bytes(int32_t n, int64_t e);
int gte_csx_from_coo(const int32_t* key, const int32_t* other, int32_t n, int64_t e,
                     int32_t* indptr, int32_t* indices, int32_t* eid,
                     void* ws, size_t ws_bytes, gte_stream_t stream);
/*
 * Same build with the id check exposed (DGL raises on out-of-range node ids when the graph is created,
 * builder.py:425): `*bad_ids` (device int32, caller-cleared, only ever raised -- one flag can collect the CSC and the
 * CSR build) becomes 1 when a `key` lies outside [0, n) (the edge is dropped) or an `other` outside [0, n_other)
 * (stored as 0, so that no later gather leaves the feature matrix).  The caller reads the flag when it chooses to
 * synchronise (PageGraphBatch.validate()).  bad_ids NULL = flag kept in the workspace (gte_csx_from_coo).
 */
int gte_csx_from_coo_checked(const int32_t* key, const int32_t* other, int32_t n, int32_t n_other, int64_t e,
                             int32_t* indptr, int32_t* indices, int32_t* eid, int32_t* bad_ids,
                             void* ws, size_t ws_bytes, gte_stream_t stream);

/*
 * Batch assembly from device-resident per-page compressed rows: replaces
 * `dgl.batch(train_batch).to(device)` + the lazy format build
 * (model_train.py:297).  `pool_*` hold every page of the dataset back to back
 * with page-local ids (`pool_indptr` has n_i+1 entries per page).  Page p of the
 * batch is dataset page `page_ids[p]`; `pool_node_off/pool_edge_off` index the
 * pools ([num_pool_pages+1], with pool_indptr offset = node_off + page index),
 * `batch_node_off/batch_edge_off` ([num_pages+1]) are the exclusive scans of
 * the batch's page sizes.  Result equals gte_csx_from_coo on the batched COO.
 * `pool_w`/`w_out` (row-order edge weights) may both be NULL.
 */
int gte_batch_concat_csx(const int32_t* pool_indptr, const int32_t* pool_indices,
                         const int32_t* pool_eid, const float* pool_w,
                         const int64_t* pool_node_off, const int64_t* pool_edge_off,
                         const int32_t* page_ids, const int64_t* batch_node_off,
                         const int64_t* batch_edge_off, int32_t num_pages,
                         int32_t* indptr, int32_t* indices, int32_t* eid, float* w_out,
                         gte_stream_t stream);

/* out[i] = in[idx[i]]  (edge weights into row order: w_row = edata['feat'][eid]) */
int gte_gather_f32(const float* in, const int32_t* idx, float* out, int64_t count, gte_stream_t stream);

/* norm[v] from in-degrees (indptr differences).  models.py:74-78 */
int gte_degree_norm(const int32_t* indptr, int32_t n, int mode, float* norm, gte_stream_t stream);

/* ------------------------------------------------------- aggregation ---- */
/*
 * Gather + segment-reduce SpMM over compressed rows (forward on the CSC,
 * backward on the CSR of the same graph -- deterministic, no atomics):
 *
 *   y[r,:] = post(r) * sum_{j in [indptr[r], indptr[r+1])} w[j] * pre[c_j] * x[c_j,:]  (+ addend[r,:])
 *
 * with c_j = indices[j]; `w` (row order) NULL = 1; `pre_scale` [n_cols-side]
 * NULL = 1; post(r) by `mode`: SUM -> 1, SUM_NORM -> row_norm[r], MEAN ->
 * 1/max(deg r,1) (true division).  `addend` NULL = 0.
 * Forward  (models.py:53-54,69-71): mode SUM_NORM, row_norm = norm.
 * Backward (DGL GSpMM.backward on the reversed graph): CSR rows, w in CSR
 * order, pre_scale = norm (d(ah*norm)), addend = the self-path gradient.
 */
int gte_spmm(const int32_t* indptr, const int32_t* indices, const float* w,
             const float* pre_scale, const float* row_norm, int mode,
             const float* x, int64_t ldx, const float* addend, int64_t ldadd,
             float* y, int64_t ldy, int32_t n_rows, int32_t f, gte_stream_t stream);

/*
 * Same contract as gte_spmm for a batch of independent page graphs (block-diagonal adjacency):
 * `page_off` [num_pages+1] (int32, device) are the node offsets of the pages
 * (dgl.batch's batch_num_nodes prefix sums), `max_page_nodes` / `max_page_edges` the largest page.
 * Each page's operand slice is staged in shared memory so gathers never leave the SM.
 * Falls back to gte_spmm when pages are too large to stage or operands are unaligned;
 * indices outside a page's own range are still handled correctly (slow path).
 */
int gte_spmm_paged(const int32_t* indptr, const int32_t* indices, const float* w,
                   const float* pre_scale, const float* row_norm, int mode,
                   const float* x, int64_t ldx, const float* addend, int64_t ldadd,
                   float* y, int64_t ldy, const int32_t* page_off, int32_t num_pages,
                   int32_t max_page_nodes, int32_t max_page_edges, int32_t n_rows, int32_t f,
                   gte_stream_t stream);

/*
 * The headline conv-layer kernel: same contract and same sums (row order, deterministic) as
 * gte_spmm_paged, on edges pre-packed per (graph, direction) by gte_paged_pack_edges:
 *   packed[j] = (page-local source row of edge j | bits of w[j] * pre_scale[c_j]) as one 64-bit word,
 *   page_flag[p] = 1 when page p has an edge whose source lies outside the page (served by a slow
 *   global path from the raw `indices` / `w` / `eid` / `pre_scale`, so the result stays correct).
 * `w` is either in row order (`eid` NULL) or in original edge order with `eid` the row-order -> edge
 * map from gte_csx_from_coo (w_row[j] = w[eid[j]]: the edge-weight permutation `edata['feat'][eid]`
 * is folded into the packing).  The kernel is persistent (one CTA per SM over a contiguous range of
 * (page, 64-column slice) items) and double buffered: the cp.async staging of the next item overlaps
 * the shared-memory gather/reduce of the current one.  gte_spmm_paged_packed_smem_bytes returns 0
 * when two stages of the largest page do not fit in shared memory (use gte_spmm_paged then);
 * gte_spmm_paged_packed itself returns GTE_ERR_UNSUPPORTED in that case or for unaligned operands.
 * Workspaces (caller-owned): packed [E + 1] uint64, 16-byte aligned (the 16-byte bulk copies that stage a page's
 * edges may read one entry past the last edge), page_flag [num_pages] int32.
 */
int gte_paged_pack_edges(const int32_t* indptr, const int32_t* indices, const int32_t* eid,
                         const float* w, const float* pre_scale, const int32_t* page_off,
                         int32_t num_pages, uint64_t* packed, int32_t* page_flag, gte_stream_t stream);
size_t gte_spmm_paged_packed_smem_bytes(int32_t max_page_nodes, int32_t max_page_edges, int32_t f);
int gte_spmm_paged_packed(const int32_t* indptr, const uint64_t* packed, const int32_t* page_flag,
                          const int32_t* indices, const int32_t* eid, const float* w,
                          const float* pre_scale, const float* row_norm, int mode,
                          const float* x, int64_t ldx, const float* addend, int64_t ldadd,
                          float* y, int64_t ldy, const int32_t* page_off, int32_t num_pages,
                          int32_t max_page_nodes, int32_t max_page_edges, int32_t n_rows, int32_t f,
                          gte_stream_t stream);

/* ---------------------------------- narrow dense operands (streams) ----- */
/*
 * `nn.Linear` and its autograd (models.py:27,63) where one operand is at most 32 columns wide -- the
 * input layer (2 x 13 features) and the class layer (9 classes): HBM streams on CUDA cores (exact fp32
 * FMA), not tensor-core tiles.
 *
 * gte_gram_stream:  C[a][b] = sum_r P[r,a] * Q[r,b],  P [n, wide <= 256] (16-byte aligned rows),
 *   Q = [Q1 | Q2] with nq1 + nq2 <= 32 columns.  Block b < nq1 goes to out1[a*sa1 + b*sb1], block
 *   b >= nq1 to out2[a*sa2 + (b-nq1)*sb2] (strides in floats, so either orientation of the weight
 *   gradient can be written); `qsum` (may be NULL) receives the column sums of Q1 (the bias gradient when
 *   Q1 = dz).  Row ranges are reduced in fixed order: deterministic.  Weight gradients of
 *   the input layer: P = dz, Q = [h | ah]; of the class layer: P = h, Q = [dz | A^T dz].
 *
 * gte_wide_out:  z[r,c] = (sum_j A1[r,j] B1(j,c) + sum_j A2[r,j] B2(j,c) + bias[c]) * row_scale[r],
 *   element B(j,c) at B[j*sj + c*sc]; k1, k2 <= 16, C <= 256; with fuse_ln also
 *   y = relu?(LayerNorm(z) * gamma + beta) and the per-row mean / rstd (two-pass statistics held in
 *   registers).  Input-layer forward: A = [h | ah], B1 = W, B2 = W + k1, sj = 1, sc = ldw.  Class-layer
 *   input gradient: A = [dz | A^T dz], B1 = W, B2 = W + fin, sj = ldw, sc = 1.
 */
size_t gte_gram_stream_workspace_bytes(int32_t n, int32_t wide);
int gte_gram_stream(const float* P, int64_t ldp, int32_t wide, const float* Q1, int64_t ldq1, int32_t nq1,
                    const float* Q2, int64_t ldq2, int32_t nq2, int32_t n,
                    float* out1, int64_t sa1, int64_t sb1, float* out2, int64_t sa2, int64_t sb2,
                    float* qsum, int accumulate, void* ws, size_t ws_bytes, gte_stream_t stream);
int gte_wide_out(const float* A1, int64_t lda1, int32_t k1, const float* A2, int64_t lda2, int32_t k2,
                 const float* B1, const float* B2, int64_t sj, int64_t sc, const float* bias,
                 const float* gamma, const float* beta, float eps, int relu, int fuse_ln,
                 const float* row_scale, float* z, int64_t ldz, float* y, int64_t ldy,
                 float* mean, float* rstd, int32_t n, int32_t C, gte_stream_t stream);

/* ------------------------------------------------- dense projection ----- */
/*
 * z[n,fo] = x1[n,k1] W[:, 0:k1]^T + x2[n,k2] W[:, k1:k1+k2]^T + bias
 * = nn.Linear over cat(h, ah*norm) without materialising the concatenation
 * (models.py:63,69-72; W is [fo, k1+k2] row-major with leading dimension ldw;
 * the self block comes first).  x2 may be NULL (k2 = 0); bias may be NULL.
 */
int gte_linear_fwd(const float* x1, int64_t ldx1, int32_t k1,
                   const float* x2, int64_t ldx2, int32_t k2,
                   const float* W, int64_t ldw, const float* bias,
                   float* z, int64_t ldz, int32_t n, int32_t fo, gte_stream_t stream);

/*
 * dx[n,k] (+)= (dz[n,fo] W[:, col0:col0+k]) * row_scale[r]   (autograd of nn.Linear
 * w.r.t. its input, one column block at a time; row_scale NULL = 1;
 * accumulate != 0 adds into dx).
 */
int gte_linear_bwd_data(const float* dz, int64_t lddz, int32_t fo,
                        const float* W, int64_t ldw, int32_t col0, int32_t k,
                        const float* row_scale, float* dx, int64_t lddx, int32_t n,
                        int accumulate, gte_stream_t stream);
/*
 * Two-term form used by the project-then-aggregate layers:
 * dx (+)= (dz1 W[:, col1:col1+k] + dz2 W[:, col2:col2+k]) * row_scale[r]   (dz2 may be NULL).
 */
int gte_linear_bwd_data2(const float* dz1, int64_t lddz1, int32_t col1,
                         const float* dz2, int64_t lddz2, int32_t col2, int32_t fo,
                         const float* W, int64_t ldw, int32_t k, const float* row_scale,
                         float* dx, int64_t lddx, int32_t n, int accumulate, gte_stream_t stream);

/*
 * dW[fo, k1+k2] = dz^T [x1 | x2]  and  db[fo] = column sums of dz (db may be
 * NULL).  Deterministic: fixed-shape split over the rows + fixed-order
 * reduction, no atomics.  `accumulate` != 0 adds into dW/db (autograd .grad
 * semantics), otherwise overwrites.
 */
size_t gte_linear_bwd_weight_workspace_bytes(int32_t n, int32_t fo, int32_t k1, int32_t k2);
int gte_linear_bwd_weight(const float* dz, int64_t lddz, int32_t fo,
                          const float* x1, int64_t ldx1, int32_t k1,
                          const float* x2, int64_t ldx2, int32_t k2,
                          float* dW, int64_t lddw, float* db, int accumulate, int32_t n,
                          void* ws, size_t ws_bytes, gte_stream_t stream);

/*
 * Two gradient blocks against the SAME input in one pass (project-then-aggregate layers):
 * dW[:, col1:col1+k] (+)= dz1^T x ; dW[:, col2:col2+k] (+)= dz2^T x ; db (+)= colsum(dz1).
 * Workspace: gte_linear_bwd_weight_workspace_bytes(n, fo, k, k).
 */
int gte_linear_bwd_weight2(const float* dz1, int64_t lddz1, const float* dz2, int64_t lddz2, int32_t fo,
                           const float* x, int64_t ldx, int32_t k, float* dW, int64_t lddw,
                           int32_t col1, int32_t col2, float* db, int accumulate, int32_t n,
                           void* ws, size_t ws_bytes, gte_stream_t stream);

/* ------------------------------------ tensor-core route (tcgen05, 3xTF32) -- */
/*
 * Same contractions as gte_linear_fwd / gte_linear_bwd_data for the wide hidden
 * layers (fin, fo <= 256), on tcgen05.mma kind::tf32 with the
 * error-compensated 3xTF32 operand split (fp32-level accuracy: a_lo*b_hi +
 * a_hi*b_lo + a_hi*b_hi accumulated in fp32 TMEM), TMA-staged operands and the
 * bias / LayerNorm / ReLU epilogue of models.py:63-66 fused.  Activations must be
 * 16-byte aligned with leading dimensions that are multiples of 4 floats.
 *
 * gte_umma_pack_weights splits W [fo, nseg*fin] into tf32 hi/lo halves, zero pads
 * them to the tile shape and stores both the forward (W) and the backward (W^T)
 * operand layouts into `pack` (gte_umma_pack_bytes bytes, 16-byte aligned).
 * It must be re-run whenever W changes.
 */
int gte_umma_supported(int32_t fo, int32_t fin);
size_t gte_umma_pack_bytes(int32_t fo, int32_t fin, int32_t nseg);
/* Several matrices in ONE launch (the train step packs all its layers at once): `descs` is a HOST array. */
#define GTE_PACK_BATCH_MAX 8
typedef struct {
  const float* W;
  int64_t ldw;
  int32_t fo, fin, nseg;
  float* pack;
} gte_pack_desc_t;
int gte_umma_pack_weights_batch(const gte_pack_desc_t* descs, int32_t count, gte_stream_t stream);
int gte_umma_pack_weights(const float* W, int64_t ldw, int32_t fo, int32_t fin, int32_t nseg,
                          float* pack, gte_stream_t stream);
/*
 * z = x1 W[:, :fin]^T (+ x2 W[:, fin:]^T) + bias ; y = act(LayerNorm(z)) when
 * fuse_ln (mean/rstd [n] saved), else y = act(z) when y != NULL.  x2 may be NULL.
 */
int gte_umma_linear_fwd(const float* x1, int64_t ldx1, const float* x2, int64_t ldx2, int32_t fin,
                        const float* pack, const float* bias, const float* gamma, const float* beta,
                        float eps, int relu, int fuse_ln, float* z, int64_t ldz, float* y, int64_t ldy,
                        float* mean, float* rstd, int32_t n, int32_t fo, gte_stream_t stream);
/* dx1 = dz W[:, :fin] and (nseg == 2) dx2 = dz W[:, fin:2*fin]. */
int gte_umma_linear_bwd_data(const float* dz, int64_t lddz, int32_t fo, const float* pack, int32_t nseg,
                             float* dx1, int64_t lddx1, float* dx2, int64_t lddx2, int32_t n, int32_t fin,
                             gte_stream_t stream);

/* Diagnostic (-DGTE_EXPERIMENTS builds; GTE_ERR_UNSUPPORTED otherwise): role timestamps (clock64) of the last tensor-core
 * projection launched with GTE_UMMA_DBG=1; which: 0 = single-CTA kernel, 1 = CTA-pair kernel. */
int gte_umma_debug_times(int32_t which, int64_t* out_host, int32_t count);

/*
 * Class-layer (fo <= 16) forms of the project-then-aggregate strategy.  `pack` from
 * gte_umma_pack_weights(W, fo, fin, nseg = 2).
 *   fwd_stacked: out[n, 32]: columns [0, fo) = x W[:, :fin]^T + bias, columns [16, 16+fo) = x W[:, fin:]^T
 *                (one pass over x; the aggregation then reads the two column blocks as views)
 *   bwd_data2:   dx = dz1 W[:, :fin] + dz2 W[:, fin:2 fin]
 */
int gte_umma_linear_fwd_stacked(const float* x, int64_t ldx, int32_t fin, const float* pack,
                                const float* bias, int32_t fo, float* out, int64_t ldo, int32_t n,
                                gte_stream_t stream);
int gte_umma_linear_bwd_data2(const float* dz1, int64_t lddz1, const float* dz2, int64_t lddz2,
                              int32_t fo, const float* pack, float* dx, int64_t lddx, int32_t n,
                              int32_t fin, gte_stream_t stream);

/*
 * Weight gradients on the tensor cores (MN-major tcgen05.mma operands straight from the row-major
 * activations, 3xTF32, row chunks reduced in fixed order).  Same results contract as
 * gte_linear_bwd_weight / gte_linear_bwd_weight2; fo, k1, k2 <= 256 (fo <= 32 for the *2 form);
 * operands 16-byte aligned with ld % 4 == 0.  db is produced from the same pass through an
 * all-ones padding column: it needs k1 % 32 != 0 (k % 128 != 0 for the *2 form), otherwise pass
 * db = NULL and obtain it elsewhere (gte_layernorm_act_bwd's dz_colsum).
 */
int gte_umma_bwd_weight_supported(int32_t fo, int32_t k1, int32_t k2);
size_t gte_umma_bwd_weight_workspace_bytes(int32_t n, int32_t fo, int32_t k1, int32_t k2);
int gte_umma_linear_bwd_weight(const float* dz, int64_t lddz, int32_t fo, const float* x1, int64_t ldx1,
                               int32_t k1, const float* x2, int64_t ldx2, int32_t k2, float* dW,
                               int64_t lddw, float* db, int accumulate, int32_t n, void* ws,
                               size_t ws_bytes, gte_stream_t stream);
size_t gte_umma_bwd_weight2_workspace_bytes(int32_t n, int32_t fo, int32_t k);
int gte_umma_linear_bwd_weight2(const float* dz1, int64_t lddz1, const float* dz2, int64_t lddz2,
                                int32_t fo, const float* x, int64_t ldx, int32_t k, float* dW,
                                int64_t lddw, int32_t col1, int32_t col2, float* db, int accumulate,
                                int32_t n, void* ws, size_t ws_bytes, gte_stream_t stream);

/*
 * Combined-operand forms for the narrow sides of the model (the 13-wide input layer, the 9-wide class
 * layer): the self block and the neighbour block live side by side in ONE [n, 32] matrix, columns
 * [0, w) and [16, 16+w), every other column FINITE (zero): the narrow side of each contraction is then
 * a single k-block / a single full-row TMA box.  Same results contract as the two-operand forms they
 * replace (models.py:47-62 with `pool` aggregation; concat order self | neighbour):
 *   fwd_comb          (fin <= 16)  z = [xc[:, :fin] | xc[:, 16:16+fin]] W^T + b, epilogue as gte_umma_linear_fwd
 *   bwd_data_comb     (fo  <= 16)  dx = dc[:, :fo] W[:, :fin] + dc[:, 16:16+fo] W[:, fin:2 fin]
 *   bwd_weight_comb   (w   <= 16)  dW[:, :w] (+)= dz^T xc[:, :w] ; dW[:, w:2w] (+)= dz^T xc[:, 16:16+w] ;
 *                                  db (+)= colsum(dz) (needs w < 16)
 *   bwd_weight2_comb  (fo  <= 16)  dW[:, col1:col1+k] (+)= dc[:, :fo]^T x ; dW[:, col2:col2+k] (+)=
 *                                  dc[:, 16:16+fo]^T x ; db (+)= colsum(dc[:, :fo]) (needs k % 32 != 0)
 * pack = gte_umma_pack_weights(..., nseg = 2) of the same W.  Workspace of the two weight-gradient forms:
 * gte_umma_bwd_weight_workspace_bytes(n, fo, 256, 0) is sufficient.  In both, the narrow operand is the A side of
 * the MMA (one real 32-column box of a 128-row tile) and the wide one the B side (N up to 256 in one instruction).
 */
int gte_umma_linear_fwd_comb(const float* xc, int64_t ldx, int32_t fin, const float* pack,
                             const float* bias, const float* gamma, const float* beta, float eps,
                             int relu, int fuse_ln, float* z, int64_t ldz, float* y, int64_t ldy,
                             float* mean, float* rstd, int32_t n, int32_t fo, gte_stream_t stream);
int gte_umma_linear_bwd_data_comb(const float* dc, int64_t lddc, int32_t fo, const float* pack,
                                  float* dx, int64_t lddx, int32_t n, int32_t fin,
                                  gte_stream_t stream);
int gte_umma_linear_bwd_weight_comb(const float* dz, int64_t lddz, int32_t fo, const float* xc,
                                    int64_t ldx, int32_t w, float* dW, int64_t lddw, float* db,
                                    int accumulate, int32_t n, void* ws, size_t ws_bytes,
                                    gte_stream_t stream);
int gte_umma_linear_bwd_weight2_comb(const float* dc, int64_t lddc, int32_t fo, const float* x,
                                     int64_t ldx, int32_t k, float* dW, int64_t lddw, int32_t col1,
                                     int32_t col2, float* db, int accumulate, int32_t n, void* ws,
                                     size_t ws_bytes, gte_stream_t stream);

/* ------------------------------------------- row normalisation + act ---- */
/*
 * y = act(LayerNorm(z; gamma, beta, eps)) per row over the first f columns
 * (models.py:64-66; nn.LayerNorm biased variance).  relu != 0 applies F.relu.
 * Saves mean/rstd [n] for the backward.  y may alias z.
 */
int gte_layernorm_act_fwd(const float* z, int64_t ldz, const float* gamma, const float* beta,
                          float eps, int relu, float* y, int64_t ldy, float* mean, float* rstd,
                          int32_t n, int32_t f, gte_stream_t stream);
size_t gte_layernorm_act_bwd_workspace_bytes(int32_t n, int32_t f);
/* dz may alias dy.  dgamma/dbeta [f]: deterministic two-stage reduction.  dz_colsum [f]
 * (may be NULL) receives the column sums of dz = the gradient of the preceding nn.Linear's bias. */
int gte_layernorm_act_bwd(const float* dy, int64_t lddy, const float* z, int64_t ldz,
                          const float* mean, const float* rstd, const float* gamma,
                          const float* beta, int relu, float* dz, int64_t lddz,
                          float* dgamma, float* dbeta, float* dz_colsum, int accumulate,
                          int32_t n, int32_t f, void* ws, size_t ws_bytes, gte_stream_t stream);

/* y = normalize(relu(z)) : F.relu + F.normalize(p=2, dim=1, eps) (models.py:168-169) */
int gte_relu_l2norm_fwd(const float* z, int64_t ldz, float eps, float* y, int64_t ldy,
                        int32_t n, int32_t f, gte_stream_t stream);
int gte_relu_l2norm_bwd(const float* dy, int64_t lddy, const float* z, int64_t ldz, float eps,
                        float* dz, int64_t lddz, int32_t n, int32_t f, gte_stream_t stream);
/* elementwise relu helpers for activation=F.relu without LayerNorm */
int gte_relu_fwd(const float* z, int64_t ldz, float* y, int64_t ldy, int32_t n, int32_t f, gte_stream_t stream);

/*
 * nn.Dropout(p) in training mode on the concatenation [x1 | x2] that the layers never materialise (models.py:30-33,
 * 60-61: `h = self.dropout(concat(h, ah * norm))`; models.py:113: the input features, then x2 = NULL, f2 = 0):
 *   y[r, c] = keep(r, c) ? x[r, c] / (1 - p) : 0,   keep ~ Bernoulli(1 - p)
 * keep(r, c) is a pure function of (seed, offset, r * (f1 + f2) + c) through Philox4x32-10, so the backward pass calls
 * the same entry on the gradients with the same (seed, offset) -- the mask is recomputed, never stored.  Statistically
 * (not bitwise) equal to ATen's mask.  One launch consumes ceil(n (f1 + f2) / 4) counters starting at `offset`.
 * `rng_dev` (device int64[2] = {seed, base offset}, may be NULL): when given, seed = rng_dev[0] and the offset is
 * rng_dev[1] + `offset` -- a captured CUDA graph then draws fresh masks on every replay after gte_rng_advance.
 * In-place use (y = x) is allowed.
 */
int gte_dropout_concat(const float* x1, int64_t ldx1, int32_t f1, const float* x2, int64_t ldx2, int32_t f2, int32_t n,
                       float p, uint64_t seed, uint64_t offset, const int64_t* rng_dev, float* y1, int64_t ldy1, float* y2,
                       int64_t ldy2, gte_stream_t stream);
/* rng_dev[1] += by  (one launch; graph-replay safe like the optimiser's step counter) */
int gte_rng_advance(int64_t* rng_dev, int64_t by, gte_stream_t stream);
int gte_relu_bwd(const float* dy, int64_t lddy, const float* z, int64_t ldz, float* dz, int64_t lddz,
                 int32_t n, int32_t f, gte_stream_t stream);

/* ------------------------------------------------ loss and optimiser ---- */
/*
 * nn.CrossEntropyLoss(weight=class_w) forward statistics (model_train.py:171,327-328):
 * stats[0] = sum_i w[y_i] * nll_i, stats[1] = sum_i w[y_i], stats[2] = #(argmax == y).
 * The loss is stats[0]/stats[1].  class_w NULL = all ones.  Deterministic.
 */
size_t gte_cross_entropy_workspace_bytes(int32_t n);
int gte_cross_entropy_fwd(const float* logits, int64_t ld, const void* labels, int label_dtype,
                          const float* class_w, int32_t n, int32_t c, float* stats,
                          void* ws, size_t ws_bytes, gte_stream_t stream);
/* dlogits[i,:] = w[y_i] * (softmax(logits[i]) - onehot(y_i)) / *denominator   (device scalar:
 * the GLOBAL sum of w[y_i]; single GPU: &stats[1]; data parallel: its all-reduce). */
int gte_cross_entropy_bwd(const float* logits, int64_t ld, const void* labels, int label_dtype,
                          const float* class_w, int32_t n, int32_t c, const float* denominator,
                          float* dlogits, int64_t lddl, gte_stream_t stream);
/* The same, and columns [c, zero_to) of every dlogits row are set to zero (zero_to % 4 == 0, rows 16-byte
 * aligned): the self block of the class layer's combined [n, 32] gradient operand, written in place. */
int gte_cross_entropy_bwd_padded(const float* logits, int64_t ld, const void* labels, int label_dtype,
                                 const float* class_w, int32_t n, int32_t c, const float* denominator,
                                 float* dlogits, int64_t lddl, int32_t zero_to, gte_stream_t stream);
/*
 * Validation statistics of one batch, ADDED to a float64 buffer totals[2 + c*c] (the validation step of
 * model_train.py:349-364 and the confusion matrix of model_predict.py:159-169):
 *   totals[0] += sum_i w[y_i] * nll_i and totals[1] += sum_i w[y_i]  (log-sum-exp and class weights of
 *                gte_cross_entropy_fwd; the validation loss is totals[0] / totals[1]),
 *   totals[2 + y_i*c + p_i] += 1  (confusion matrix: rows are true classes, columns predictions), p_i = torch.argmax
 *                of row i: the first maximal index, NaN counting as maximal (as gte_page_predictions).
 * Rows whose label lies outside [0, c) -- the -1 padding of gte_pad_batch -- are skipped.  c <= GTE_EVAL_MAX_CLASSES.
 * Deterministic: the counts are exact integer sums, the loss partials are reduced in a fixed order and added in
 * double.  n == 0 is a no-op.  Two launches.
 */
#define GTE_EVAL_MAX_CLASSES 64
size_t gte_eval_workspace_bytes(int32_t n);
int gte_eval_accumulate(const float* logits, int64_t ld, const void* labels, int label_dtype, const float* class_w,
                        int32_t n, int32_t c, double* totals, void* ws, size_t ws_bytes, gte_stream_t stream);
/* Self block of a combined [n, 32] operand (see the *_comb entries): out[r, 0:w] = x[r, 0:w] (x rows may be
 * unaligned, e.g. the raw [N, 13] BBOX features), every other column of the 32 zero; w <= 16. */
int gte_comb_fill(const float* x, int64_t ldx, int32_t w, float* out, int64_t ldo, int64_t n,
                  gte_stream_t stream);

/*
 * torch.optim.Adam(lr, betas, eps, weight_decay) with L2-in-gradient decay over
 * a flat parameter buffer (model_train.py:168,332).  The 1-based step count is
 * `step_host`, or -- when `step_dev` is non-NULL -- a device counter that this
 * call increments first and then uses (CUDA-graph replay safe).  grad_scale
 * multiplies the gradient first; `grad_den` (device float, may be NULL) divides it:
 * the data-parallel step sums UN-normalised gradients together with the loss
 * statistics in ONE all-reduce and normalises here by the global label-weight sum.
 */
int gte_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq,
                  int64_t count, float lr, float beta1, float beta2, float eps,
                  float weight_decay, int64_t step_host, int64_t* step_dev, float grad_scale,
                  const float* grad_den, gte_stream_t stream);

/*
 * Data-parallel step tail in ONE kernel: one-shot all-reduce of the flat gradient buffers over NVLink peer memory
 * (P2P loads, summed in rank order => bit-identical replicas) fused with the Adam update of gte_adam_step (device step
 * counter, division by the global label-weight sum found at stats_off + 1).  Replaces `ncclAllReduce` + optimizer.step()
 * of a data-parallel model_train.py:330-332; capturable in a CUDA graph with the rest of the step.
 *   peer_grad_ptrs_dev / peer_signal_ptrs_dev: DEVICE arrays [world] of device pointers -- every rank's flat gradient
 *     buffer ([count parameters ... stats_off: sum w*nll, sum w, #correct]) and the 2*world uint32 words this library
 *     owns inside every rank's signal pad (zero before the first call).  Both come from a symmetric-memory rendezvous
 *     (torch.distributed._symmetric_memory); the entry itself never allocates or maps memory.
 *   local_words: [4] uint32 device words of this rank, zero before the first call.
 *   stats_out [3]: the global statistics.
 * Every rank must call it once per step on the stream that produced its gradients.
 */
int gte_dp_allreduce_adam(const void* peer_grad_ptrs_dev, const void* peer_signal_ptrs_dev, int32_t rank, int32_t world,
                          int64_t count, int64_t stats_off, float* param, float* exp_avg, float* exp_avg_sq,
                          float* stats_out, float lr, float beta1, float beta2, float eps, float weight_decay,
                          int64_t* step_dev, uint32_t* local_words, gte_stream_t stream);

/* ---------------------------------------- either side of the layers ---- */
/*
 * Batched predict tail (model_predict.py:144-154): preds[i] = argmax_j logits[i, j] (first maximal index; NaN
 * counts as maximal, like torch.argmax) as int32, and -- when `labels` is given -- page_correct[p] =
 * #(preds == labels) over the nodes [page_off[p], page_off[p+1]) of page p, from which the reference's per-page
 * accuracy `correct / g.num_nodes()` and its mean over pages follow.  `page_correct` may be NULL.
 */
int gte_page_predictions(const float* logits, int64_t ld, int32_t n, int32_t c, const void* labels,
                         int label_dtype, const int32_t* page_off, int32_t num_pages, int32_t* preds,
                         int32_t* page_correct, gte_stream_t stream);

/*
 * Batch assembly of a page batch in ONE kernel (SURVEY 8(f) row 1): everything the layers need from
 * `dgl.batch(train_batch).to(device)` (model_train.py:297) and `get_norm` (models.py:74-78).  One CTA per page
 * sorts the page's edges by destination (CSC) and by source (CSR) in shared memory; outputs are bit-identical to
 * gte_csx_from_coo on the batched COO (stable), gte_degree_norm(INV_DEG_ZERO) and gte_paged_pack_edges
 * (CSC: weights; CSR: weights * norm[dst]).  Contract of dgl.batch: nodes / edges of page p occupy
 * [page_off[p], page_off[p+1]) / [edge_off[p], edge_off[p+1]) and no edge leaves its page; *bad (device int) is set to
 * 1 otherwise (results undefined) -- page_flag[] is cleared (no out-of-page edges by contract).  `w` NULL = all ones.
 * Rows are put in edge order by a per-row insertion sort in shared memory (one thread per row): meant for the
 * bounded degrees of page graphs (k-NN / visibility edges); a hub row of degree d costs O(d^2) steps of one thread.
 * packed arrays need e + 1 entries (see gte_spmm_paged_packed).  gte_build_page_formats_smem_bytes returns 0 when the
 * largest page does not fit in shared memory (use gte_csx_from_coo + gte_degree_norm + gte_paged_pack_edges then).
 */
size_t gte_build_page_formats_smem_bytes(int32_t max_page_nodes, int32_t max_page_edges);
int gte_build_page_formats(const int32_t* src, const int32_t* dst, const float* w, const int32_t* page_off,
                           const int32_t* edge_off, int32_t num_pages, int32_t n, int64_t e,
                           int32_t max_page_nodes, int32_t max_page_edges,
                           int32_t* csc_indptr, int32_t* csc_indices, int32_t* csc_eid, uint64_t* csc_packed,
                           int32_t* csr_indptr, int32_t* csr_indices, int32_t* csr_eid, uint64_t* csr_packed,
                           float* norm, int32_t* page_flag, int32_t* bad, gte_stream_t stream);

/*
 * Pads a page batch to a capacity shape in place, so that one captured CUDA graph serves batches of any size up to
 * the capacity: the shuffled training batches of model_train.py:283-297 and the streamed predict batches of
 * model_predict.py:130-154 (whose last batch is short) change their node / edge totals from batch to batch.
 * The caller fills the real prefix of src / dst / weight [e_cap], feat [n_cap, f] (row stride ldf) and label [n_cap],
 * the device word `word` = (n, e, P) of that prefix, and the whole page table page_off / edge_off [p_cap + 1]:
 * the P real pages, then padding pages, then empty pages (0 nodes, 0 edges) up to p_cap.  The kernel writes
 *   feat rows [n, n_cap) = 0, label [n, n_cap) = -1, weight [e, e_cap) = 0,
 *   src = dst over [e, e_cap) = a node of the padding page that owns the edge (a weight-0 self-loop),
 * which makes the padded batch a valid dgl.batch whose padding adds nothing to the loss statistics or any
 * gradient.  *bad (device int, cleared first): bit 0 = the word lies outside the capacity, bit 1 = the page table
 * leaves a padding edge without a padding node; the kernel then clamps and writes nothing outside the buffers.
 */
int gte_pad_batch(const int32_t* word, int32_t n_cap, int64_t e_cap, int32_t p_cap, const int32_t* page_off,
                  const int32_t* edge_off, int32_t* src, int32_t* dst, float* weight, float* feat, int64_t ldf,
                  int32_t f, float* label, int32_t* bad, gte_stream_t stream);

/*
 * Batches gathered from a device-resident page pool, so that a captured pass assembles its own next batch: the
 * host-side `dgl.batch(train_batch).to(device)` of model_train.py:279-297 and the per-page batches of
 * model_predict.py:130-154 become one small upload of page ids per epoch.  Both entries are graph-capturable.
 *
 * The pool (PagePool) holds every page with page-local ids: COO src / dst [E_pool] int32, weights [E_pool], features
 * [N_pool, f] (row-major, stride f), labels [N_pool] fp32, node / edge offsets [pool_pages + 1] int64 and the per-page
 * node / edge counts [pool_pages] int32.  `plan` is an int32 device buffer of 8 + 2 * pool_pages words:
 *   [cursor, flag, nfit, B, L, 0, 0, 0 | ids[L] | starts[nfit]],
 * the epoch's page ids and the start offsets of its slices that fit; slice k is ids[starts[k], min(starts[k] + B, L)).
 *
 * gte_gather_plan (one CTA) runs slice `cursor` and advances the cursor by one.  It writes the capacity static set's
 * `meta` = [n, e, P, start | page_off (p_cap + 1) | edge_off (p_cap + 1)]: the batch's totals, its start offset in
 * ids, and the padded page table of gte_pad_batch -- the real pages, then s = min(p_cap - P, n_cap - n) padding
 * pages at n + j (n_cap - n) / s nodes (64-bit; edges likewise), then empty pages.  The batch must fit the capacity
 * (cap_*: total nodes, total edges, pages, largest page in nodes / edges, as BatchCapacity.check) with n_cap >
 * cap_nodes, p_cap > cap_pages.  Otherwise `flag` gains bit 0 (cursor past the plan, or a malformed header) or bit 1
 * (the batch does not fit, or an id lies outside the pool) and `meta` is left as it was.
 * gte_gather_pages copies the pages of the batch in `meta` into the real prefix of src / dst / weight [e_cap], feat
 * [n_cap, f] (contiguous) and label [n_cap]: features, labels and weights as they are, src / dst plus the page's node
 * offset in the batch.  It copies nothing while `flag` is non-zero (the plan kernel refused the batch, so `meta`
 * still describes an earlier one); a page the page table does not describe sets flag bit 2 and is skipped.  Its grid is
 * min(4 * SMs, max_pages) CTAs (max_pages = the capacity's page count), looping over the pages.
 */
int gte_gather_plan(int32_t* plan, const int32_t* pool_num_nodes, const int32_t* pool_num_edges, int32_t pool_pages,
                    int32_t cap_nodes, int64_t cap_edges, int32_t cap_pages, int32_t cap_page_nodes,
                    int32_t cap_page_edges, int32_t n_cap, int64_t e_cap, int32_t p_cap, int32_t* meta,
                    gte_stream_t stream);
int gte_gather_pages(int32_t* plan, const int32_t* meta, int32_t n_cap, int64_t e_cap, int32_t p_cap,
                     int32_t max_pages, const int64_t* pool_node_off, const int64_t* pool_edge_off,
                     int32_t pool_pages, const int32_t* pool_src, const int32_t* pool_dst, const float* pool_weight,
                     const float* pool_feat, const float* pool_label, int32_t f, int32_t* src, int32_t* dst,
                     float* weight, float* feat, float* label, gte_stream_t stream);

/*
 * BBOX node features on the device (src/components/nlp/bbox.py:49-54 get_shape, :57-111 get_histogram, called
 * per batch at model_train.py:293): boxes [n, 4] int32 = [x0, y0, x1, y1]; counts [n, 3] int32 = (letters,
 * digits, other symbols) of the box text with blanks removed (str.isalpha / str.isdigit are host string
 * operations and stay on the host).  out [n, 13] fp32 = [w, h, cx, cy, w*h, x0, y0, x1, y1, hist0..hist3],
 * computed in float64 like the Python original and cast to float32 (model_train.py:295).
 */
int gte_bbox_features(const int32_t* boxes, const int32_t* counts, int32_t n, float* out, int64_t ldo,
                      gte_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* GTE_H_ */
