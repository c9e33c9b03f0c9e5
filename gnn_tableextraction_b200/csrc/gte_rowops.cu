// Row-wise epilogues of the GraphSAGE layers and the train-step tail:
//   LayerNorm + ReLU        /root/reference/src/components/graphs/models.py:34-37,64-66
//   ReLU + L2 row normalise models.py:167-169 (MeanSAGE)
//   weighted cross entropy  /root/reference/src/models/model_train.py:171,327-328
//   Adam with L2 decay      model_train.py:168,330-332
// All HBM-bound, one warp per row, fixed-order reductions (no atomics).
#include "gte_common.cuh"
#include <stdlib.h>

#include <math.h>

namespace gte {

constexpr int ROW_THREADS = 256;
constexpr int ROW_WARPS = ROW_THREADS / 32;

// ------------------------------------------------------------ LayerNorm ---
template <int MAXC>
__global__ void __launch_bounds__(ROW_THREADS)
    k_layernorm_act_fwd(const float* __restrict__ z, int64_t ldz, const float* __restrict__ gamma,
                        const float* __restrict__ beta, float eps, int relu, float* __restrict__ y, int64_t ldy,
                        float* __restrict__ mean_out, float* __restrict__ rstd_out, int32_t n, int32_t f) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * ROW_WARPS + (threadIdx.x >> 5);
  if (row >= n) return;
  const float* zr = z + row * ldz;
  float v[MAXC];
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    const int col = lane + 32 * c;
    v[c] = col < f ? zr[col] : 0.f;
    s += v[c];
  }
  const float mean = warp_sum(s) / (float)f;
  float q = 0.f;
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    const int col = lane + 32 * c;
    const float d = col < f ? v[c] - mean : 0.f;
    q = fmaf(d, d, q);
  }
  const float var = warp_sum(q) / (float)f;  // biased, like nn.LayerNorm
  const float rstd = 1.0f / sqrtf(var + eps);
  if (lane == 0) {
    mean_out[row] = mean;
    rstd_out[row] = rstd;
  }
  float* yr = y + row * ldy;
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    const int col = lane + 32 * c;
    if (col < f) {
      float o = (v[c] - mean) * rstd * __ldg(gamma + col) + __ldg(beta + col);
      if (relu) o = fmaxf(o, 0.f);
      yr[col] = o;
    }
  }
}

// dz per row + per-block partial sums of dgamma / dbeta / colsum(dz): partial[block][3][f]
template <int MAXC>
__global__ void __launch_bounds__(ROW_THREADS)
    k_layernorm_act_bwd(const float* __restrict__ dy, int64_t lddy, const float* __restrict__ z, int64_t ldz,
                        const float* __restrict__ mean, const float* __restrict__ rstd,
                        const float* __restrict__ gamma, const float* __restrict__ beta, int relu,
                        float* __restrict__ dz, int64_t lddz, float* __restrict__ partial, int32_t n, int32_t f) {
  extern __shared__ float sm[];  // [ROW_WARPS][3][f]
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  float gam[MAXC], bet[MAXC], dg[MAXC], db[MAXC], dl[MAXC];
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    const int col = lane + 32 * c;
    gam[c] = col < f ? __ldg(gamma + col) : 0.f;
    bet[c] = col < f ? __ldg(beta + col) : 0.f;
    dg[c] = 0.f;
    db[c] = 0.f;
    dl[c] = 0.f;
  }
  const float inv_f = 1.0f / (float)f;
  for (int64_t row = (int64_t)blockIdx.x * ROW_WARPS + warp; row < n; row += (int64_t)gridDim.x * ROW_WARPS) {
    const float mu = mean[row], rs = rstd[row];
    const float* zr = z + row * ldz;
    const float* gr = dy + row * lddy;
    float xh[MAXC], a[MAXC];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      const int col = lane + 32 * c;
      float g = 0.f;
      xh[c] = 0.f;
      if (col < f) {
        xh[c] = (zr[col] - mu) * rs;
        g = gr[col];
        if (relu && !(xh[c] * gam[c] + bet[c] > 0.f)) g = 0.f;
      }
      db[c] += g;
      dg[c] = fmaf(g, xh[c], dg[c]);
      a[c] = g * gam[c];
      s1 += a[c];
      s2 = fmaf(a[c], xh[c], s2);
    }
    const float c1 = warp_sum(s1) * inv_f;
    const float c2 = warp_sum(s2) * inv_f;
    float* dr = dz + row * lddz;
#pragma unroll
    for (int c = 0; c < MAXC; ++c) {
      const int col = lane + 32 * c;
      if (col < f) {
        const float o = rs * (a[c] - c1 - xh[c] * c2);
        dr[col] = o;
        dl[c] += o;
      }
    }
  }
  // block combine, warps in fixed order
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    const int col = lane + 32 * c;
    if (col < f) {
      sm[(warp * 3 + 0) * f + col] = dg[c];
      sm[(warp * 3 + 1) * f + col] = db[c];
      sm[(warp * 3 + 2) * f + col] = dl[c];
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * f; i += ROW_THREADS) {
    const int which = i / f, col = i % f;
    float s = 0.f;
    for (int w = 0; w < ROW_WARPS; ++w) s += sm[(w * 3 + which) * f + col];
    partial[(int64_t)blockIdx.x * 3 * f + i] = s;
  }
}

// 128-bit variant: lane owns float4 chunks lane, lane+32, ... of the row; two rows in flight per warp.
// Same arithmetic and the same fixed reduction order as the scalar kernel above.
template <int MAXV>
__global__ void __launch_bounds__(ROW_THREADS)
    k_layernorm_act_bwd_v4(const float* __restrict__ dy, int64_t lddy, const float* __restrict__ z, int64_t ldz,
                           const float* __restrict__ mean, const float* __restrict__ rstd,
                           const float* __restrict__ gamma, const float* __restrict__ beta, int relu,
                           float* __restrict__ dz, int64_t lddz, float* __restrict__ partial, int32_t n, int32_t f) {
  extern __shared__ float sm[];  // [ROW_WARPS][3][f]
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  float gam[MAXV][4], bet[MAXV][4], dg[MAXV][4], db[MAXV][4], dl[MAXV][4];
#pragma unroll
  for (int c = 0; c < MAXV; ++c)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int col = 4 * (lane + 32 * c) + e;
      gam[c][e] = col < f ? __ldg(gamma + col) : 0.f;
      bet[c][e] = col < f ? __ldg(beta + col) : 0.f;
      dg[c][e] = 0.f;
      db[c][e] = 0.f;
      dl[c][e] = 0.f;
    }
  const float inv_f = 1.0f / (float)f;
  const int64_t stride = (int64_t)gridDim.x * ROW_WARPS;
  for (int64_t row0 = (int64_t)blockIdx.x * ROW_WARPS + warp; row0 < n; row0 += 2 * stride) {
    float4 zv[2][MAXV], gv[2][MAXV];
    float mu[2], rs[2];
    bool live[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int64_t row = row0 + u * stride;
      live[u] = row < n;
      mu[u] = live[u] ? mean[row] : 0.f;
      rs[u] = live[u] ? rstd[row] : 0.f;
#pragma unroll
      for (int c = 0; c < MAXV; ++c) {
        const int col = 4 * (lane + 32 * c);
        const bool ok = live[u] && col < f;  // padding columns [f, ld) are readable, never interpreted
        zv[u][c] = ok ? *reinterpret_cast<const float4*>(z + row * ldz + col) : make_float4(0.f, 0.f, 0.f, 0.f);
        gv[u][c] = ok ? *reinterpret_cast<const float4*>(dy + row * lddy + col) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if (!live[u]) continue;  // warp-uniform
      const int64_t row = row0 + u * stride;
      float xh[MAXV][4], a[MAXV][4];
      float s1 = 0.f, s2 = 0.f;
#pragma unroll
      for (int c = 0; c < MAXV; ++c) {
        const float zz[4] = {zv[u][c].x, zv[u][c].y, zv[u][c].z, zv[u][c].w};
        const float gg[4] = {gv[u][c].x, gv[u][c].y, gv[u][c].z, gv[u][c].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int col = 4 * (lane + 32 * c) + e;
          float g = 0.f;
          xh[c][e] = 0.f;
          if (col < f) {
            xh[c][e] = (zz[e] - mu[u]) * rs[u];
            g = gg[e];
            if (relu && !(xh[c][e] * gam[c][e] + bet[c][e] > 0.f)) g = 0.f;
          }
          db[c][e] += g;
          dg[c][e] = fmaf(g, xh[c][e], dg[c][e]);
          a[c][e] = g * gam[c][e];
          s1 += a[c][e];
          s2 = fmaf(a[c][e], xh[c][e], s2);
        }
      }
      const float c1 = warp_sum(s1) * inv_f;
      const float c2 = warp_sum(s2) * inv_f;
#pragma unroll
      for (int c = 0; c < MAXV; ++c) {
        const int col = 4 * (lane + 32 * c);
        if (col < f) {
          float4 o;
          o.x = rs[u] * (a[c][0] - c1 - xh[c][0] * c2);
          o.y = rs[u] * (a[c][1] - c1 - xh[c][1] * c2);
          o.z = rs[u] * (a[c][2] - c1 - xh[c][2] * c2);
          o.w = rs[u] * (a[c][3] - c1 - xh[c][3] * c2);
          *reinterpret_cast<float4*>(dz + row * lddz + col) = o;
          dl[c][0] += o.x;  // columns >= f carry a = xh = 0, i.e. o = -rs*c1: never read back (col < f below)
          dl[c][1] += o.y;
          dl[c][2] += o.z;
          dl[c][3] += o.w;
        }
      }
    }
  }
#pragma unroll
  for (int c = 0; c < MAXV; ++c)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int col = 4 * (lane + 32 * c) + e;
      if (col < f) {
        sm[(warp * 3 + 0) * f + col] = dg[c][e];
        sm[(warp * 3 + 1) * f + col] = db[c][e];
        sm[(warp * 3 + 2) * f + col] = dl[c][e];
      }
    }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * f; i += ROW_THREADS) {
    const int which = i / f, col = i % f;
    float s = 0.f;
    for (int w = 0; w < ROW_WARPS; ++w) s += sm[(w * 3 + which) * f + col];
    partial[(int64_t)blockIdx.x * 3 * f + i] = s;
  }
}

// out[i] (+)= sum_b partial[b*stride + i] in a fixed order; 32 outputs per block (T = double: added in double)
template <typename T>
__global__ void __launch_bounds__(RED_THREADS)
    k_reduce_partials(const float* __restrict__ partial, int nb, int64_t stride, int32_t count, T* __restrict__ out,
                      int accumulate) {
  __shared__ float red[RED_THREADS];
  const int i = blockIdx.x * 32 + (threadIdx.x & 31);
  const bool valid = i < count;
  const float s = reduce_partials_block(partial, nb, stride, i, valid, red);
  if ((threadIdx.x >> 5) != 0 || !valid) return;
  T r = s;
  if (accumulate) r += out[i];
  out[i] = r;
}

// three reductions over one partial matrix [nb][3 * f] in one launch: out_k[i] (+)= sum_b partial[b * 3f + k * f + i]
__global__ void __launch_bounds__(RED_THREADS)
    k_reduce_partials3(const float* __restrict__ partial, int nb, int32_t f, float* __restrict__ out0, float* __restrict__ out1,
                       float* __restrict__ out2, int accumulate) {
  __shared__ float red[RED_THREADS];
  const int i = blockIdx.x * 32 + (threadIdx.x & 31);
  const int nout = (out2 ? 3 : 2) * f;
  const bool valid = i < nout;
  float s = reduce_partials_block(partial, nb, 3 * (int64_t)f, i, valid, red);
  if ((threadIdx.x >> 5) != 0 || !valid) return;
  float* out = i < f ? out0 + i : (i < 2 * f ? out1 + (i - f) : out2 + (i - 2 * f));
  if (accumulate) s += *out;
  *out = s;
}

static int ln_bwd_grid(int32_t n) {
  int64_t b = ceil_div64(n, ROW_WARPS);
  // 128 registers x 256 threads: two CTAs are resident per SM; one wave (measured 90 us vs 99 us with four CTAs per SM
  // queued in two waves at N = 153600, F = 218)
  const int cap = 2 * sm_count();
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

// ------------------------------------------------- ReLU + L2 normalise ----
template <int MAXC>
__global__ void __launch_bounds__(ROW_THREADS)
    k_relu_l2norm_fwd(const float* __restrict__ z, int64_t ldz, float eps, float* __restrict__ y, int64_t ldy,
                      int32_t n, int32_t f) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * ROW_WARPS + (threadIdx.x >> 5);
  if (row >= n) return;
  const float* zr = z + row * ldz;
  float v[MAXC];
  float q = 0.f;
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    const int col = lane + 32 * c;
    v[c] = col < f ? fmaxf(zr[col], 0.f) : 0.f;
    q = fmaf(v[c], v[c], q);
  }
  const float nrm = fmaxf(sqrtf(warp_sum(q)), eps);  // F.normalize: x / max(||x||_2, eps)
  float* yr = y + row * ldy;
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    const int col = lane + 32 * c;
    if (col < f) yr[col] = v[c] / nrm;
  }
}

// One warp per row: dz of row `row`; returns nothing, adds dz to cs[] when COLSUM
template <int MAXC, bool COLSUM>
__device__ __forceinline__ void relu_l2norm_bwd_row(const float* __restrict__ dy, int64_t lddy, const float* __restrict__ z,
                                                    int64_t ldz, float eps, float* __restrict__ dz, int64_t lddz,
                                                    int64_t row, int32_t f, int lane, float (&cs)[MAXC]) {
  const float* zr = z + row * ldz;
  const float* gr = dy + row * lddy;
  float r[MAXC], g[MAXC];
  float q = 0.f;
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    const int col = lane + 32 * c;
    r[c] = col < f ? fmaxf(zr[col], 0.f) : 0.f;
    g[c] = col < f ? gr[col] : 0.f;
    q = fmaf(r[c], r[c], q);
  }
  const float nrm_raw = sqrtf(warp_sum(q));
  // F.normalize divides by norm.clamp_min(eps), whose gradient passes where norm >= eps: only a norm strictly below
  // eps drops the second term
  const bool clamped = nrm_raw < eps;
  const float nrm = clamped ? eps : nrm_raw;
  // d r = (g - y (y.g)) / nrm with y = r / nrm: no power of the norm is formed, so neither overflows nor underflows
  // where the norm itself is finite and normal
  float y[MAXC];
  float dot_y = 0.f;
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    y[c] = r[c] / nrm;
    dot_y = fmaf(y[c], g[c], dot_y);
  }
  dot_y = warp_sum(dot_y);
  if (clamped) dot_y = 0.f;
  float* dr = dz + row * lddz;
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    const int col = lane + 32 * c;
    if (col < f) {
      const float o = r[c] > 0.f ? (g[c] - y[c] * dot_y) / nrm : 0.f;
      dr[col] = o;
      if constexpr (COLSUM) cs[c] += o;
    }
  }
}

template <int MAXC>
__global__ void __launch_bounds__(ROW_THREADS)
    k_relu_l2norm_bwd(const float* __restrict__ dy, int64_t lddy, const float* __restrict__ z, int64_t ldz, float eps,
                      float* __restrict__ dz, int64_t lddz, int32_t n, int32_t f) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * ROW_WARPS + (threadIdx.x >> 5);
  if (row >= n) return;
  float unused[MAXC];
  relu_l2norm_bwd_row<MAXC, false>(dy, lddy, z, ldz, eps, dz, lddz, row, f, lane, unused);
}

// the same rows, grid-stride, plus the column sums of dz (the linear-bias gradient): every lane keeps the sums of its
// columns, the block writes partial[block][f] (warps added in fixed order) for k_reduce_partials
template <int MAXC>
__global__ void __launch_bounds__(ROW_THREADS)
    k_relu_l2norm_bwd_colsum(const float* __restrict__ dy, int64_t lddy, const float* __restrict__ z, int64_t ldz,
                             float eps, float* __restrict__ dz, int64_t lddz, float* __restrict__ partial, int32_t n,
                             int32_t f) {
  extern __shared__ float sm[];  // [ROW_WARPS][f]
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  float cs[MAXC];
#pragma unroll
  for (int c = 0; c < MAXC; ++c) cs[c] = 0.f;
#pragma unroll 1
  for (int64_t row = (int64_t)blockIdx.x * ROW_WARPS + warp; row < n; row += (int64_t)gridDim.x * ROW_WARPS)
    relu_l2norm_bwd_row<MAXC, true>(dy, lddy, z, ldz, eps, dz, lddz, row, f, lane, cs);
#pragma unroll
  for (int c = 0; c < MAXC; ++c) {
    const int col = lane + 32 * c;
    if (col < f) sm[warp * f + col] = cs[c];
  }
  __syncthreads();
  for (int col = threadIdx.x; col < f; col += ROW_THREADS) {
    float s = 0.f;
    for (int w = 0; w < ROW_WARPS; ++w) s += sm[w * f + col];
    partial[(int64_t)blockIdx.x * f + col] = s;
  }
}

__global__ void k_relu_fwd(const float* __restrict__ z, int64_t ldz, float* __restrict__ y, int64_t ldy, int32_t n,
                           int32_t f) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)n * f;
  for (; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / f;
    const int c = (int)(i % f);
    y[r * ldy + c] = fmaxf(z[r * ldz + c], 0.f);
  }
}

__global__ void k_relu_bwd(const float* __restrict__ dy, int64_t lddy, const float* __restrict__ z, int64_t ldz,
                           float* __restrict__ dz, int64_t lddz, int32_t n, int32_t f) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = (int64_t)n * f;
  for (; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / f;
    const int c = (int)(i % f);
    dz[r * lddz + c] = z[r * ldz + c] > 0.f ? dy[r * lddy + c] : 0.f;
  }
}

// -------------------------------------------------------- cross entropy ---
__device__ __forceinline__ int64_t load_label(const void* labels, int dtype, int64_t i) {
  if (dtype == GTE_LABEL_I64) return static_cast<const int64_t*>(labels)[i];
  if (dtype == GTE_LABEL_I32) return static_cast<const int32_t*>(labels)[i];
  return (int64_t)static_cast<const float*>(labels)[i];  // `.type(torch.long)` truncation, model_train.py:327
}

constexpr int CE_THREADS = 256;

// per-block partials: [block][3] = {sum w*nll, sum w, #correct}.
// EVAL (gte_eval_accumulate): no #correct (its partial is 0); the block counts (label, torch.argmax) pairs of the rows
// with a label in [0, c) in a c x c int32 histogram in dynamic shared memory and adds it to cm[c * c] (float64) at
// the end: integral sums below 2^53 are exact in any order.
template <bool EVAL>
__global__ void __launch_bounds__(CE_THREADS)
    k_ce_fwd(const float* __restrict__ logits, int64_t ld, const void* __restrict__ labels, int label_dtype,
             const float* __restrict__ class_w, int32_t n, int32_t c, float* __restrict__ partial,
             double* __restrict__ cm) {
  __shared__ float red[3][CE_THREADS / 32];
  extern __shared__ int hist[];
  if constexpr (EVAL) {
    for (int k = threadIdx.x; k < c * c; k += CE_THREADS) hist[k] = 0;
    __syncthreads();
  }
  float loss = 0.f, wsum = 0.f, correct = 0.f;
  for (int64_t i = (int64_t)blockIdx.x * CE_THREADS + threadIdx.x; i < n; i += (int64_t)gridDim.x * CE_THREADS) {
    const float* lr = logits + i * ld;
    const int64_t yv = load_label(labels, label_dtype, i);
    // torch.argmax and the row maximum in one pass: a NaN row picks a NaN maximum, its se and nll are NaN either way
    const int arg = row_argmax(lr, c);
    const float mx = lr[arg];
    float se = 0.f;
    for (int j = 0; j < c; ++j) se += expf(lr[j] - mx);
    if (yv >= 0 && yv < c) {
      const float wv = class_w ? __ldg(class_w + yv) : 1.0f;
      // log-sum-exp minus the label's distance below the maximum: both terms are independent of a common offset of the
      // row (the form mx + logf(se) - lr[y] rounds at the scale of |mx|)
      const float nll = logf(se) - (lr[yv] - mx);
      loss = fmaf(wv, nll, loss);
      wsum += wv;
      if constexpr (EVAL) atomicAdd(&hist[(int)yv * c + arg], 1);
    }
    if constexpr (!EVAL) correct += (arg == (int)yv) ? 1.f : 0.f;
  }
  loss = warp_sum(loss);
  wsum = warp_sum(wsum);
  correct = warp_sum(correct);
  if ((threadIdx.x & 31) == 0) {
    red[0][threadIdx.x >> 5] = loss;
    red[1][threadIdx.x >> 5] = wsum;
    red[2][threadIdx.x >> 5] = correct;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    float s = 0.f;
    for (int w = 0; w < CE_THREADS / 32; ++w) s += red[threadIdx.x][w];
    partial[(int64_t)blockIdx.x * 3 + threadIdx.x] = s;
  }
  if constexpr (EVAL) {
    for (int k = threadIdx.x; k < c * c; k += CE_THREADS)  // after the __syncthreads above: the histogram is complete
      if (hist[k] != 0) atomicAdd(cm + k, (double)hist[k]);
  }
}

__global__ void k_ce_bwd(const float* __restrict__ logits, int64_t ld, const void* __restrict__ labels,
                         int label_dtype, const float* __restrict__ class_w, int32_t n, int32_t c,
                         const float* __restrict__ denominator, float* __restrict__ dl, int64_t lddl) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* lr = logits + i * ld;
  float* dr = dl + i * lddl;
  const int64_t yv = load_label(labels, label_dtype, i);
  const bool valid = yv >= 0 && yv < c;
  const float den = *denominator;
  const float wv = valid ? (class_w ? __ldg(class_w + yv) : 1.0f) : 0.f;
  const float scale = wv / den;
  float mx = -INFINITY;
  for (int j = 0; j < c; ++j) mx = fmaxf(mx, lr[j]);
  float se = 0.f;
  for (int j = 0; j < c; ++j) se += expf(lr[j] - mx);
  const float inv = 1.0f / se;
  for (int j = 0; j < c; ++j) {
    float p = expf(lr[j] - mx) * inv;
    if (j == (int)yv) p -= 1.0f;
    dr[j] = p * scale;
  }
}

// the same, for a class layer that consumes [d logits | A_hat^T d logits] as one combined operand: the thread also
// zeroes columns [c, zero_to) of its row (rows 16-byte aligned), so the caller needs no separate fill
__global__ void k_ce_bwd_padded(const float* __restrict__ logits, int64_t ld, const void* __restrict__ labels,
                                int label_dtype, const float* __restrict__ class_w, int32_t n, int32_t c,
                                const float* __restrict__ denominator, float* __restrict__ dl, int64_t lddl,
                                int32_t zero_to) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* lr = logits + i * ld;
  float* dr = dl + i * lddl;
  const int64_t yv = load_label(labels, label_dtype, i);
  const bool valid = yv >= 0 && yv < c;
  const float den = *denominator;
  const float wv = valid ? (class_w ? __ldg(class_w + yv) : 1.0f) : 0.f;
  const float scale = wv / den;
  float mx = -INFINITY;
  for (int j = 0; j < c; ++j) mx = fmaxf(mx, lr[j]);
  float se = 0.f;
  for (int j = 0; j < c; ++j) se += expf(lr[j] - mx);
  const float inv = 1.0f / se;
  for (int j0 = 0; j0 < zero_to; j0 += 4) {
    float v[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int j = j0 + e;
      float p = 0.f;
      if (j < c) {
        p = expf(lr[j] - mx) * inv;
        if (j == (int)yv) p -= 1.0f;
        p *= scale;
      }
      v[e] = p;
    }
    *reinterpret_cast<float4*>(dr + j0) = make_float4(v[0], v[1], v[2], v[3]);
  }
}

// zero_to == lddl == 32 (the combined operand itself): the 256 rows of a block are one contiguous 32 KB piece of the
// output, so the rows go through a swizzled shared-memory tile and leave as fully coalesced 128-bit stores (the
// thread-per-row stores of the general kernel touch 32 lines per warp instruction: 15 us instead of 6 at config 2)
__global__ void __launch_bounds__(256) k_ce_bwd_comb32(const float* __restrict__ logits, int64_t ld,
                                                      const void* __restrict__ labels, int label_dtype,
                                                      const float* __restrict__ class_w, int32_t n, int32_t c,
                                                      const float* __restrict__ denominator, float* __restrict__ dl) {
  __shared__ float4 tile[256 * 8];
  const int64_t row0 = (int64_t)blockIdx.x * 256;
  const int64_t i = row0 + threadIdx.x;
  float v[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) v[j] = 0.f;
  if (i < n) {
    const float* lr = logits + i * ld;
    const int64_t yv = load_label(labels, label_dtype, i);
    const bool valid = yv >= 0 && yv < c;
    const float den = *denominator;
    const float wv = valid ? (class_w ? __ldg(class_w + yv) : 1.0f) : 0.f;
    const float scale = wv / den;
    float mx = -INFINITY;
    for (int j = 0; j < c; ++j) mx = fmaxf(mx, lr[j]);
    float se = 0.f;
    for (int j = 0; j < c; ++j) se += expf(lr[j] - mx);
    const float inv = 1.0f / se;
#pragma unroll
    for (int j = 0; j < 16; ++j) {  // c <= 16 on this path
      if (j < c) {
        float p = expf(lr[j] - mx) * inv;
        if (j == (int)yv) p -= 1.0f;
        v[j] = p * scale;
      }
    }
  }
  const int r = threadIdx.x;
#pragma unroll
  for (int q = 0; q < 8; ++q) tile[r * 8 + (q ^ (r & 7))] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
  __syncthreads();
  float4* out = reinterpret_cast<float4*>(dl + row0 * 32);
  const int64_t lim = (n - row0 < 256 ? n - row0 : 256) * 8;  // float4 slots of the real rows
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int slot = k * 256 + threadIdx.x;  // row = slot / 8, quad = slot % 8
    if (slot < lim) {
      const int rr = slot >> 3, qq = slot & 7;
      out[slot] = tile[rr * 8 + (qq ^ (rr & 7))];
    }
  }
}

// Combined [n, 32] operand, self block: out[r, 0:w] = x[r, 0:w], every other column of the 32 zero (the neighbour block
// [16, 16+w) is written afterwards by the aggregation).  One thread per (row, 4-column slot): 128-byte rows, coalesced.
__global__ void k_comb_fill(const float* __restrict__ x, int64_t ldx, int32_t w, float* __restrict__ out, int64_t ldo,
                            int64_t n) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t r = t >> 3;
  if (r >= n) return;
  const int c0 = (int)(t & 7) * 4;
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (c0 < w) {
    const float* xr = x + r * ldx;
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (c0 + e < w) v[e] = __ldg(xr + c0 + e);
  }
  *reinterpret_cast<float4*>(out + r * ldo + c0) = make_float4(v[0], v[1], v[2], v[3]);
}

static int ce_grid(int32_t n) {
  int64_t b = ceil_div64(n, CE_THREADS);
  if (b > 296) b = 296;
  if (b < 1) b = 1;
  return (int)b;
}

// ----------------------------------------------------------------- Adam ---
// ---------------------------------------------------------------- dropout ----
// nn.Dropout on the (never materialised) concatenation [x1 | x2] (models.py:30-33,60-61,113): element (row, c) of the
// concatenation -- c < f1 in x1, else in x2 -- is kept with probability 1 - p and scaled by 1 / (1 - p).  The keep
// decision is a pure function of (seed, offset, row * (f1 + f2) + c) through Philox4x32-10 (the generator family torch's
// CUDA dropout uses; the stream layout is this library's own, so masks are statistically, not bitwise, equal to ATen's):
// counter = (element >> 2) + offset, the element's word = element & 3.  The backward pass calls the same kernel on the
// gradients with the same (seed, offset): the mask is recomputed, never stored.
__device__ __forceinline__ uint2 mulhilo32(uint32_t a, uint32_t b) {
  const uint64_t p = (uint64_t)a * b;
  return make_uint2((uint32_t)p, (uint32_t)(p >> 32));
}
__device__ __forceinline__ uint4 philox4x32_10(uint64_t counter, uint64_t seed) {
  uint32_t c0 = (uint32_t)counter, c1 = (uint32_t)(counter >> 32), c2 = 0u, c3 = 0u;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint2 m0 = mulhilo32(0xD2511F53u, c0), m1 = mulhilo32(0xCD9E8D57u, c2);
    const uint32_t n0 = m1.y ^ c1 ^ k0, n2 = m0.y ^ c3 ^ k1;
    c0 = n0; c1 = m1.x; c2 = n2; c3 = m0.x;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}

__global__ void k_dropout2(const float* __restrict__ x1, int64_t ldx1, int32_t f1, const float* __restrict__ x2, int64_t ldx2,
                           int32_t f2, int64_t n, float p, uint64_t seed_host, uint64_t offset_host,
                           const int64_t* __restrict__ rng_dev, float* __restrict__ y1, int64_t ldy1, float* __restrict__ y2,
                           int64_t ldy2) {
  const uint64_t seed = rng_dev ? (uint64_t)rng_dev[0] : seed_host;
  const uint64_t offset = rng_dev ? (uint64_t)rng_dev[1] + offset_host : offset_host;
  const int64_t ft = (int64_t)f1 + f2;
  const int64_t groups = (n * ft + 3) >> 2;  // one Philox call per 4 consecutive elements of the concatenation
  const float scale = 1.0f / (1.0f - p);
  // keep iff u >= p with u = word * 2^-32 (uniform in [0, 1)): integer threshold, no float rounding of the uniform
  const uint32_t thresh = (uint32_t)fminf(fmaxf(p * 4294967296.0f, 0.f), 4294967040.0f);
  int64_t gidx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; gidx < groups; gidx += (int64_t)gridDim.x * blockDim.x) {
    const uint4 r = philox4x32_10((uint64_t)gidx + offset, seed);
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int64_t el = gidx * 4 + e;
      if (el >= n * ft) break;
      const int64_t row = el / ft;
      const int32_t c = (int32_t)(el - row * ft);
      const bool keep = w[e] >= thresh;
      if (c < f1) y1[row * ldy1 + c] = keep ? x1[row * ldx1 + c] * scale : 0.f;
      else y2[row * ldy2 + (c - f1)] = keep ? x2[row * ldx2 + (c - f1)] * scale : 0.f;
    }
  }
}

__global__ void k_rng_advance(int64_t* rng, int64_t by) { rng[1] += by; }

__global__ void k_step_inc(int64_t* step) { *step += 1; }

// hp (may be NULL): device [lr, beta1, beta2, eps, weight_decay], read once per CTA in place of the by-value arguments
__global__ void k_adam(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                       float* __restrict__ v, int64_t count, float lr, float b1, float b2, float eps, float wd,
                       const float* __restrict__ hp, int64_t step_host, const int64_t* __restrict__ step_dev,
                       float grad_scale, const float* __restrict__ grad_den) {
  if (hp) {
    __shared__ float s_hp[5];
    if (threadIdx.x < 5) s_hp[threadIdx.x] = hp[threadIdx.x];
    __syncthreads();
    lr = s_hp[0]; b1 = s_hp[1]; b2 = s_hp[2]; eps = s_hp[3]; wd = s_hp[4];
  }
  const int64_t t = step_dev ? *step_dev : step_host;
  if (grad_den) {
    // data parallel: gradients were summed un-normalised.  A step without any weighted label (every label out of
    // range / ignored, or class weight 0) has no defined gradient: leave parameters and moments untouched instead of
    // dividing by zero (NaN moments would poison every later step).
    const float den = *grad_den;
    if (!(den > 0.f)) return;
    grad_scale = grad_scale / den;
  }
  // bias corrections exactly as torch.optim.Adam's single-tensor path (double maths, then fp32 use)
  const double bc1 = 1.0 - pow((double)b1, (double)t);
  const double bc2 = 1.0 - pow((double)b2, (double)t);
  const float step_size = (float)((double)lr / bc1);
  const float bc2_sqrt = (float)sqrt(bc2);
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i < count; i += (int64_t)gridDim.x * blockDim.x) {
    const float pi = p[i];
    float gi = g[i] * grad_scale;
    gi = fmaf(wd, pi, gi);  // grad = grad + weight_decay * param
    const float mi = m[i] + (gi - m[i]) * (1.0f - b1);  // exp_avg.lerp_(grad, 1 - beta1)
    const float vi = v[i] * b2 + (1.0f - b2) * gi * gi;  // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = pi - step_size * (mi / denom);
  }
}

}  // namespace gte

using namespace gte;

#define GTE_ROW_DISPATCH(KERNEL, F, ...)                                                            \
  do {                                                                                              \
    if ((F) <= 32) KERNEL<1> __VA_ARGS__;                                                           \
    else if ((F) <= 64) KERNEL<2> __VA_ARGS__;                                                      \
    else if ((F) <= 128) KERNEL<4> __VA_ARGS__;                                                     \
    else if ((F) <= 256) KERNEL<8> __VA_ARGS__;                                                     \
    else if ((F) <= 512) KERNEL<16> __VA_ARGS__;                                                    \
    else KERNEL<32> __VA_ARGS__;                                                                    \
  } while (0)
extern "C" {

int gte_layernorm_act_fwd(const float* z, int64_t ldz, const float* gamma, const float* beta, float eps, int relu,
                          float* y, int64_t ldy, float* mean, float* rstd, int32_t n, int32_t f,
                          gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0 && f > 0, "gte_layernorm_act_fwd: bad size");
  if (f > 1024) return fail(GTE_ERR_UNSUPPORTED, "gte_layernorm_act_fwd: f=%d > 1024 not supported", f);
  if (n == 0) return GTE_OK;
  GTE_CHECK_ARG(z && gamma && beta && y && mean && rstd, "gte_layernorm_act_fwd: null argument");
  GTE_CHECK_ARG(ldz >= f && ldy >= f, "gte_layernorm_act_fwd: leading dimension < f");
  cudaStream_t st = as_stream(stream);
  const unsigned grid = (unsigned)ceil_div64(n, ROW_WARPS);
  GTE_ROW_DISPATCH(k_layernorm_act_fwd, f,
                   <<<grid, ROW_THREADS, 0, st>>>(z, ldz, gamma, beta, eps, relu, y, ldy, mean, rstd, n, f));
  GTE_CHECK_LAUNCH("k_layernorm_act_fwd");
  return GTE_OK;
}

size_t gte_layernorm_act_bwd_workspace_bytes(int32_t n, int32_t f) {
  if (n < 0 || f <= 0) return 0;
  return (size_t)ln_bwd_grid(n) * 3 * (size_t)f * 4 + 256;
}

int gte_layernorm_act_bwd(const float* dy, int64_t lddy, const float* z, int64_t ldz, const float* mean,
                          const float* rstd, const float* gamma, const float* beta, int relu, float* dz,
                          int64_t lddz, float* dgamma, float* dbeta, float* dz_colsum, int accumulate, int32_t n,
                          int32_t f, void* ws, size_t ws_bytes, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0 && f > 0, "gte_layernorm_act_bwd: bad size");
  if (f > 1024) return fail(GTE_ERR_UNSUPPORTED, "gte_layernorm_act_bwd: f=%d > 1024 not supported", f);
  GTE_CHECK_ARG(dgamma && dbeta, "gte_layernorm_act_bwd: null dgamma/dbeta");
  GTE_CHECK_ARG(n == 0 || (dy && z && mean && rstd && gamma && beta && dz), "gte_layernorm_act_bwd: null argument");
  GTE_CHECK_ARG(lddy >= f && ldz >= f && lddz >= f, "gte_layernorm_act_bwd: leading dimension < f");
  const size_t need = gte_layernorm_act_bwd_workspace_bytes(n, f);
  if (ws == nullptr || ws_bytes < need)
    return fail(GTE_ERR_WORKSPACE, "gte_layernorm_act_bwd: workspace %zu < required %zu", ws_bytes, need);
  cudaStream_t st = as_stream(stream);
  float* partial = static_cast<float*>(ws);
  const int grid = ln_bwd_grid(n);
  const bool vec4 = aligned16(dy) && aligned16(z) && aligned16(dz) && lddy % 4 == 0 && ldz % 4 == 0 && lddz % 4 == 0 && f <= 480;  // 8 warps x 3 x f floats of shared memory stay under 48 KB
  if (n > 0 && vec4) {
    const size_t smem = (size_t)ROW_WARPS * 3 * f * 4;
    const int nv = (f + 3) / 4;
    if (nv <= 32)
      k_layernorm_act_bwd_v4<1><<<grid, ROW_THREADS, smem, st>>>(dy, lddy, z, ldz, mean, rstd, gamma, beta, relu, dz, lddz, partial, n, f);
    else if (nv <= 64)
      k_layernorm_act_bwd_v4<2><<<grid, ROW_THREADS, smem, st>>>(dy, lddy, z, ldz, mean, rstd, gamma, beta, relu, dz, lddz, partial, n, f);
    else
      k_layernorm_act_bwd_v4<4><<<grid, ROW_THREADS, smem, st>>>(dy, lddy, z, ldz, mean, rstd, gamma, beta, relu, dz, lddz, partial, n, f);
    GTE_CHECK_LAUNCH("k_layernorm_act_bwd_v4");
  } else if (n > 0) {
    const size_t smem = (size_t)ROW_WARPS * 3 * f * 4;
    if (smem > 48 * 1024)
      GTE_CHECK_CUDA(cudaFuncSetAttribute(k_layernorm_act_bwd<32>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)smem),
                     "gte_layernorm_act_bwd(smem attr)");
    GTE_ROW_DISPATCH(k_layernorm_act_bwd, f,
                     <<<grid, ROW_THREADS, smem, st>>>(dy, lddy, z, ldz, mean, rstd, gamma, beta, relu, dz, lddz,
                                                      partial, n, f));
    GTE_CHECK_LAUNCH("k_layernorm_act_bwd");
  }
  const int nb = n > 0 ? grid : 0;
  // dgamma, dbeta and (optionally) the column sums of dz live side by side in every partial row: one launch
  k_reduce_partials3<<<(unsigned)ceil_div64((dz_colsum ? 3 : 2) * (int64_t)f, 32), RED_THREADS, 0, st>>>(partial, nb, f, dgamma, dbeta,
                                                                                                   dz_colsum, accumulate);
  GTE_CHECK_LAUNCH("k_reduce_partials3");
  return GTE_OK;
}

int gte_relu_l2norm_fwd(const float* z, int64_t ldz, float eps, float* y, int64_t ldy, int32_t n, int32_t f,
                        gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0 && f > 0, "gte_relu_l2norm_fwd: bad size");
  if (f > 1024) return fail(GTE_ERR_UNSUPPORTED, "gte_relu_l2norm_fwd: f=%d > 1024 not supported", f);
  if (n == 0) return GTE_OK;
  GTE_CHECK_ARG(z && y && ldz >= f && ldy >= f, "gte_relu_l2norm_fwd: bad argument");
  const unsigned grid = (unsigned)ceil_div64(n, ROW_WARPS);
  cudaStream_t st = as_stream(stream);
  GTE_ROW_DISPATCH(k_relu_l2norm_fwd, f, <<<grid, ROW_THREADS, 0, st>>>(z, ldz, eps, y, ldy, n, f));
  GTE_CHECK_LAUNCH("k_relu_l2norm_fwd");
  return GTE_OK;
}

int gte_relu_l2norm_bwd(const float* dy, int64_t lddy, const float* z, int64_t ldz, float eps, float* dz,
                        int64_t lddz, int32_t n, int32_t f, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0 && f > 0, "gte_relu_l2norm_bwd: bad size");
  if (f > 1024) return fail(GTE_ERR_UNSUPPORTED, "gte_relu_l2norm_bwd: f=%d > 1024 not supported", f);
  if (n == 0) return GTE_OK;
  GTE_CHECK_ARG(dy && z && dz && lddy >= f && ldz >= f && lddz >= f, "gte_relu_l2norm_bwd: bad argument");
  const unsigned grid = (unsigned)ceil_div64(n, ROW_WARPS);
  cudaStream_t st = as_stream(stream);
  GTE_ROW_DISPATCH(k_relu_l2norm_bwd, f, <<<grid, ROW_THREADS, 0, st>>>(dy, lddy, z, ldz, eps, dz, lddz, n, f));
  GTE_CHECK_LAUNCH("k_relu_l2norm_bwd");
  return GTE_OK;
}

size_t gte_relu_l2norm_bwd_colsum_workspace_bytes(int32_t n, int32_t f) {
  if (n < 0 || f <= 0) return 0;
  return (size_t)ln_bwd_grid(n) * (size_t)f * 4 + 256;
}

int gte_relu_l2norm_bwd_colsum(const float* dy, int64_t lddy, const float* z, int64_t ldz, float eps, float* dz,
                               int64_t lddz, float* dz_colsum, int accumulate, int32_t n, int32_t f, void* ws,
                               size_t ws_bytes, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0 && f > 0, "gte_relu_l2norm_bwd_colsum: bad size");
  if (f > 1024) return fail(GTE_ERR_UNSUPPORTED, "gte_relu_l2norm_bwd_colsum: f=%d > 1024 not supported", f);
  GTE_CHECK_ARG(dz_colsum, "gte_relu_l2norm_bwd_colsum: null dz_colsum");
  GTE_CHECK_ARG(n == 0 || (dy && z && dz), "gte_relu_l2norm_bwd_colsum: null argument");
  GTE_CHECK_ARG(lddy >= f && ldz >= f && lddz >= f, "gte_relu_l2norm_bwd_colsum: leading dimension < f");
  const size_t need = gte_relu_l2norm_bwd_colsum_workspace_bytes(n, f);
  if (ws == nullptr || ws_bytes < need)
    return fail(GTE_ERR_WORKSPACE, "gte_relu_l2norm_bwd_colsum: workspace %zu < required %zu", ws_bytes, need);
  cudaStream_t st = as_stream(stream);
  float* partial = static_cast<float*>(ws);
  const int grid = ln_bwd_grid(n);
  if (n > 0) {
    const size_t smem = (size_t)ROW_WARPS * f * 4;  // 32 KB at f = 1024
    GTE_ROW_DISPATCH(k_relu_l2norm_bwd_colsum, f,
                     <<<grid, ROW_THREADS, smem, st>>>(dy, lddy, z, ldz, eps, dz, lddz, partial, n, f));
    GTE_CHECK_LAUNCH("k_relu_l2norm_bwd_colsum");
  }
  // fixed-order second stage over the per-block partials (none when n == 0: zeros, or dz_colsum unchanged)
  k_reduce_partials<float><<<(unsigned)ceil_div64(f, 32), RED_THREADS, 0, st>>>(partial, n > 0 ? grid : 0, f, f,
                                                                               dz_colsum, accumulate);
  GTE_CHECK_LAUNCH("k_reduce_partials");
  return GTE_OK;
}

static unsigned ew_grid(int64_t total) {
  int64_t b = ceil_div64(total, 256);
  const int64_t cap = (int64_t)sm_count() * 16;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (unsigned)b;
}

int gte_relu_fwd(const float* z, int64_t ldz, float* y, int64_t ldy, int32_t n, int32_t f, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0 && f >= 0, "gte_relu_fwd: bad size");
  if (n == 0 || f == 0) return GTE_OK;
  GTE_CHECK_ARG(z && y && ldz >= f && ldy >= f, "gte_relu_fwd: bad argument");
  k_relu_fwd<<<ew_grid((int64_t)n * f), 256, 0, as_stream(stream)>>>(z, ldz, y, ldy, n, f);
  GTE_CHECK_LAUNCH("k_relu_fwd");
  return GTE_OK;
}

int gte_relu_bwd(const float* dy, int64_t lddy, const float* z, int64_t ldz, float* dz, int64_t lddz, int32_t n,
                 int32_t f, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0 && f >= 0, "gte_relu_bwd: bad size");
  if (n == 0 || f == 0) return GTE_OK;
  GTE_CHECK_ARG(dy && z && dz && lddy >= f && ldz >= f && lddz >= f, "gte_relu_bwd: bad argument");
  k_relu_bwd<<<ew_grid((int64_t)n * f), 256, 0, as_stream(stream)>>>(dy, lddy, z, ldz, dz, lddz, n, f);
  GTE_CHECK_LAUNCH("k_relu_bwd");
  return GTE_OK;
}

size_t gte_cross_entropy_workspace_bytes(int32_t n) {
  if (n < 0) return 0;
  return (size_t)ce_grid(n) * 3 * 4 + 256;
}

int gte_cross_entropy_fwd(const float* logits, int64_t ld, const void* labels, int label_dtype, const float* class_w,
                          int32_t n, int32_t c, float* stats, void* ws, size_t ws_bytes, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0 && c > 0, "gte_cross_entropy_fwd: bad size");
  GTE_CHECK_ARG(label_dtype >= GTE_LABEL_I64 && label_dtype <= GTE_LABEL_F32, "gte_cross_entropy_fwd: bad label dtype");
  GTE_CHECK_ARG(stats != nullptr, "gte_cross_entropy_fwd: stats is null");
  GTE_CHECK_ARG(n == 0 || (logits && labels && ld >= c), "gte_cross_entropy_fwd: bad argument");
  const size_t need = gte_cross_entropy_workspace_bytes(n);
  if (ws == nullptr || ws_bytes < need)
    return fail(GTE_ERR_WORKSPACE, "gte_cross_entropy_fwd: workspace %zu < required %zu", ws_bytes, need);
  cudaStream_t st = as_stream(stream);
  float* partial = static_cast<float*>(ws);
  const int grid = ce_grid(n);
  if (n > 0) {
    k_ce_fwd<false><<<grid, CE_THREADS, 0, st>>>(logits, ld, labels, label_dtype, class_w, n, c, partial, nullptr);
    GTE_CHECK_LAUNCH("k_ce_fwd");
  }
  k_reduce_partials<float><<<1, RED_THREADS, 0, st>>>(partial, n > 0 ? grid : 0, 3, 3, stats, 0);
  GTE_CHECK_LAUNCH("k_reduce_partials(ce)");
  return GTE_OK;
}

size_t gte_eval_workspace_bytes(int32_t n) { return gte_cross_entropy_workspace_bytes(n); }

int gte_eval_accumulate(const float* logits, int64_t ld, const void* labels, int label_dtype, const float* class_w,
                        int32_t n, int32_t c, double* totals, void* ws, size_t ws_bytes, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0 && c > 0 && c <= GTE_EVAL_MAX_CLASSES, "gte_eval_accumulate: need 0 < c <= %d classes (got %d)",
                GTE_EVAL_MAX_CLASSES, c);
  GTE_CHECK_ARG(label_dtype >= GTE_LABEL_I64 && label_dtype <= GTE_LABEL_F32, "gte_eval_accumulate: bad label dtype");
  if (n == 0) return GTE_OK;
  GTE_CHECK_ARG(logits && labels && totals && ld >= c, "gte_eval_accumulate: bad argument");
  const size_t need = gte_eval_workspace_bytes(n);
  if (ws == nullptr || ws_bytes < need)
    return fail(GTE_ERR_WORKSPACE, "gte_eval_accumulate: workspace %zu < required %zu", ws_bytes, need);
  cudaStream_t st = as_stream(stream);
  float* partial = static_cast<float*>(ws);
  const int grid = ce_grid(n);
  k_ce_fwd<true><<<grid, CE_THREADS, (size_t)c * c * sizeof(int), st>>>(logits, ld, labels, label_dtype, class_w, n, c,
                                                                       partial, totals + 2);
  GTE_CHECK_LAUNCH("k_ce_fwd(eval)");
  k_reduce_partials<double><<<1, RED_THREADS, 0, st>>>(partial, grid, 3, 2, totals, 1);
  GTE_CHECK_LAUNCH("k_reduce_partials(eval)");
  return GTE_OK;
}

int gte_cross_entropy_bwd(const float* logits, int64_t ld, const void* labels, int label_dtype, const float* class_w,
                          int32_t n, int32_t c, const float* denominator, float* dlogits, int64_t lddl,
                          gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0 && c > 0, "gte_cross_entropy_bwd: bad size");
  GTE_CHECK_ARG(label_dtype >= GTE_LABEL_I64 && label_dtype <= GTE_LABEL_F32, "gte_cross_entropy_bwd: bad label dtype");
  if (n == 0) return GTE_OK;
  GTE_CHECK_ARG(logits && labels && denominator && dlogits && ld >= c && lddl >= c, "gte_cross_entropy_bwd: bad argument");
  k_ce_bwd<<<(unsigned)ceil_div64(n, 256), 256, 0, as_stream(stream)>>>(logits, ld, labels, label_dtype, class_w, n, c,
                                                                       denominator, dlogits, lddl);
  GTE_CHECK_LAUNCH("k_ce_bwd");
  return GTE_OK;
}

int gte_cross_entropy_bwd_padded(const float* logits, int64_t ld, const void* labels, int label_dtype, const float* class_w,
                                 int32_t n, int32_t c, const float* denominator, float* dlogits, int64_t lddl,
                                 int32_t zero_to, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0 && c >= 1, "gte_cross_entropy_bwd_padded: bad size");
  if (n == 0) return GTE_OK;
  GTE_CHECK_ARG(logits && labels && denominator && dlogits && ld >= c, "gte_cross_entropy_bwd_padded: bad argument");
  GTE_CHECK_ARG(zero_to >= c && zero_to % 4 == 0 && lddl >= zero_to && lddl % 4 == 0 && aligned16(dlogits),
                "gte_cross_entropy_bwd_padded: zero_to must be a multiple of 4 in [c, lddl], rows 16-byte aligned");
  if (zero_to == 32 && lddl == 32 && c <= 16) {
    k_ce_bwd_comb32<<<(unsigned)ceil_div64(n, 256), 256, 0, as_stream(stream)>>>(logits, ld, labels, label_dtype, class_w, n,
                                                                                c, denominator, dlogits);
    GTE_CHECK_LAUNCH("k_ce_bwd_comb32");
    return GTE_OK;
  }
  k_ce_bwd_padded<<<(unsigned)ceil_div64(n, 256), 256, 0, as_stream(stream)>>>(logits, ld, labels, label_dtype, class_w, n, c,
                                                                              denominator, dlogits, lddl, zero_to);
  GTE_CHECK_LAUNCH("k_ce_bwd_padded");
  return GTE_OK;
}

int gte_comb_fill(const float* x, int64_t ldx, int32_t w, float* out, int64_t ldo, int64_t n, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0 && w >= 0 && w <= 16, "gte_comb_fill: bad size (w <= 16)");
  if (n == 0) return GTE_OK;
  GTE_CHECK_ARG(out && (w == 0 || (x && ldx >= w)) && ldo >= 32 && ldo % 4 == 0 && aligned16(out),
                "gte_comb_fill: out must be a 16-byte aligned [n, >= 32] matrix");
  k_comb_fill<<<(unsigned)ceil_div64(n * 8, 256), 256, 0, as_stream(stream)>>>(x, ldx, w, out, ldo, n);
  GTE_CHECK_LAUNCH("k_comb_fill");
  return GTE_OK;
}

static int adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t count, float lr,
                     float beta1, float beta2, float eps, float weight_decay, const float* hparams, int64_t step_host,
                     int64_t* step_dev, float grad_scale, const float* grad_den, gte_stream_t stream) {
  GTE_CHECK_ARG(count >= 0, "gte_adam_step: negative count");
  GTE_CHECK_ARG(step_dev != nullptr || step_host >= 1, "gte_adam_step: step must be >= 1");
  if (count == 0) return GTE_OK;
  GTE_CHECK_ARG(param && grad && exp_avg && exp_avg_sq, "gte_adam_step: null argument");
  cudaStream_t st = as_stream(stream);
  if (step_dev) {
    k_step_inc<<<1, 1, 0, st>>>(step_dev);
    GTE_CHECK_LAUNCH("k_step_inc");
  }
  k_adam<<<ew_grid(count), 256, 0, st>>>(param, grad, exp_avg, exp_avg_sq, count, lr, beta1, beta2, eps, weight_decay,
                                        hparams, step_host, step_dev, grad_scale, grad_den);
  GTE_CHECK_LAUNCH("k_adam");
  return GTE_OK;
}

int gte_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t count, float lr,
                  float beta1, float beta2, float eps, float weight_decay, int64_t step_host, int64_t* step_dev,
                  float grad_scale, const float* grad_den, gte_stream_t stream) {
  return adam_step(param, grad, exp_avg, exp_avg_sq, count, lr, beta1, beta2, eps, weight_decay, nullptr, step_host,
                   step_dev, grad_scale, grad_den, stream);
}

int gte_adam_step_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t count,
                      const float* hparams, int64_t step_host, int64_t* step_dev, float grad_scale, const float* grad_den,
                      gte_stream_t stream) {
  GTE_CHECK_ARG(hparams != nullptr, "gte_adam_step_dev: null hparams");
  return adam_step(param, grad, exp_avg, exp_avg_sq, count, 0.f, 0.f, 0.f, 0.f, 0.f, hparams, step_host, step_dev,
                   grad_scale, grad_den, stream);
}

int gte_dropout_concat(const float* x1, int64_t ldx1, int32_t f1, const float* x2, int64_t ldx2, int32_t f2, int32_t n,
                       float p, uint64_t seed, uint64_t offset, const int64_t* rng_dev, float* y1, int64_t ldy1, float* y2,
                       int64_t ldy2, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0 && f1 >= 0 && f2 >= 0, "gte_dropout_concat: bad size");
  GTE_CHECK_ARG(p >= 0.f && p < 1.f, "gte_dropout_concat: p must be in [0, 1) (p = 1 zeroes everything: use a memset)");
  if (n == 0 || f1 + f2 == 0) return GTE_OK;
  GTE_CHECK_ARG((f1 == 0 || (x1 && y1 && ldx1 >= f1 && ldy1 >= f1)) && (f2 == 0 || (x2 && y2 && ldx2 >= f2 && ldy2 >= f2)),
                "gte_dropout_concat: bad argument");
  const int64_t groups = ((int64_t)n * (f1 + f2) + 3) / 4;
  k_dropout2<<<ew_grid(groups), 256, 0, as_stream(stream)>>>(x1, ldx1, f1, x2, ldx2, f2, n, p, seed, offset, rng_dev, y1, ldy1,
                                                            y2, ldy2);
  GTE_CHECK_LAUNCH("k_dropout2");
  return GTE_OK;
}

int gte_rng_advance(int64_t* rng_dev, int64_t by, gte_stream_t stream) {
  GTE_CHECK_ARG(rng_dev && by >= 0, "gte_rng_advance: bad argument");
  k_rng_advance<<<1, 1, 0, as_stream(stream)>>>(rng_dev, by);
  GTE_CHECK_LAUNCH("k_rng_advance");
  return GTE_OK;
}

}  // extern "C"
