// Arguments and small device helpers shared by the two tensor-core projection kernels:
//   gte_umma.cu   k_umma_gemm       one CTA per SM, cta_group::1 (any shape the route supports)
//   gte_umma2.cu  k_umma_gemm_pair  CTA pairs, cta_group::2 (the product path for >= 2 row tiles)
#pragma once
#include "gte_common.cuh"
#include "gte_umma_ptx.cuh"

namespace gte {

constexpr int UM_BM = 128;
constexpr int UM_BK = 32;               // floats per k block = one 128-byte swizzle row
constexpr int UM_A_BYTES = UM_BM * 128;  // 16 KB
constexpr int UM_MAX_BN = 256;
constexpr int UM_ACC_STRIDE = 256;       // TMEM columns per accumulator stage

// UmmaArgs::fuse_ln: the forward epilogue that turns z into y
constexpr int UM_EPI_NONE = 0;  // y = act(z)
constexpr int UM_EPI_LN = 1;    // y = act(LayerNorm(z)), mean / rstd per row
constexpr int UM_EPI_L2 = 2;    // y = relu(z) / max(||relu(z)||_2, eps), nothing saved per row

struct UmmaArgs {
  CUtensorMap tmA[2];       // per K segment: activations [M, K_s], box 32 x 128
  CUtensorMap tmBhi[2][2];  // [group][segment]: packed weights hi [BN, Kpad], box 32 x BN (pair kernel: 32 x BN/2)
  CUtensorMap tmBlo[2][2];
  CUtensorMap tmOut[2];     // per group: z / dx, box 32 x 32 (TMA store)
  CUtensorMap tmY;          // y (TMA store)
  const float* bhi[2][2];   // the packed tiles behind tmBhi / tmBlo ([BN, b_cols] row-major): the launcher encodes
  const float* blo[2][2];   //   the maps with the box its kernel needs
  int32_t b_cols;
  int32_t nseg, ngroups;
  int32_t kblocks[2];
  int32_t M, N, BN;
  float* out[2];            // per group: pre-activation output (z / dx); out[0] may be null when only y is wanted
  int64_t ldo[2];
  float* y;                 // LayerNorm/ReLU output (forward only), may be null
  int64_t ldy;
  const float* bias;
  const float* gamma;
  const float* beta;
  float* mean;
  float* rstd;
  float eps;
  int32_t fuse_ln, relu;    // fuse_ln: UM_EPI_NONE / UM_EPI_LN / UM_EPI_L2
  int32_t tma_store;  // outputs are TMA-store compatible (16-byte aligned, ld % 4 == 0)
  int32_t epi_bufs;   // store tiles per epilogue warp (single-CTA kernel: 2 unless shared memory is tight)
  int32_t bias_n;     // number of valid bias entries (the stacked class-layer output is wider than its bias)
  int32_t stages;     // operand ring depth (pair kernel)
};

// launchers (host): return GTE_OK or a recorded failure
int launch_umma_single(UmmaArgs& a, cudaStream_t st);
int launch_umma_pair(UmmaArgs& a, cudaStream_t st);
bool umma_pair_supported(const UmmaArgs& a);
int setup_weight_maps(UmmaArgs& a, int box_rows);  // tmBhi / tmBlo with the box the chosen kernel stages

// x[j] = accumulator (main [+ cross-term accumulator]) + bias for the 32 columns of one chunk of this thread's row.
// Everything is compile-time indexed so the 32-register TMEM load windows stay in registers (no local memory).
template <bool SPLIT>
__device__ __forceinline__ void epi_load_chunk(uint32_t taddr, const float* bias_c, float (&x)[32]) {
  uint32_t v[32];
  tmem_ld_32x32b_x32_nowait(taddr, v);
  if constexpr (SPLIT) {
    uint32_t v2[32];
    tmem_ld_32x32b_x32_nowait(taddr + UM_ACC_STRIDE, v2);
    tmem_wait_ld();
#pragma unroll
    for (int j = 0; j < 32; ++j) x[j] = __uint_as_float(v[j]) + __uint_as_float(v2[j]);
  } else {
    tmem_wait_ld();
#pragma unroll
    for (int j = 0; j < 32; ++j) x[j] = __uint_as_float(v[j]);
  }
  const float4* b4 = reinterpret_cast<const float4*>(bias_c);
#pragma unroll
  for (int qd = 0; qd < 8; ++qd) {
    const float4 b = b4[qd];
    x[4 * qd] += b.x; x[4 * qd + 1] += b.y; x[4 * qd + 2] += b.z; x[4 * qd + 3] += b.w;
  }
}

// y = act(LayerNorm(x)) for one 32-column chunk (gamma / beta staged in shared memory)
__device__ __forceinline__ void epi_norm_act(float (&x)[32], const float* gamma_c, const float* beta_c, bool ln, bool relu,
                                             float mean, float rstd) {
  const float4* g4 = reinterpret_cast<const float4*>(gamma_c);
  const float4* e4 = reinterpret_cast<const float4*>(beta_c);
#pragma unroll
  for (int qd = 0; qd < 8; ++qd) {
    const float4 gm = g4[qd], bt = e4[qd];
    const float gv[4] = {gm.x, gm.y, gm.z, gm.w}, bv[4] = {bt.x, bt.y, bt.z, bt.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float o = x[4 * qd + e];
      if (ln) o = (o - mean) * rstd * gv[e] + bv[e];
      if (relu) o = fmaxf(o, 0.f);
      x[4 * qd + e] = o;
    }
  }
}

// sum of relu(x)^2 over the first nv columns of one chunk, added to q in column order
__device__ __forceinline__ float epi_relu_sq_sum(const float (&x)[32], int nv, float q) {
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    const float r = (j < nv) ? fmaxf(x[j], 0.f) : 0.f;
    q = fmaf(r, r, q);
  }
  return q;
}

// y = relu(x) / nrm for one chunk (nrm = max(||relu(z)||_2, eps): a division, as k_relu_l2norm_fwd and F.normalize)
__device__ __forceinline__ void epi_relu_div(float (&x)[32], float nrm) {
#pragma unroll
  for (int j = 0; j < 32; ++j) x[j] = fmaxf(x[j], 0.f) / nrm;
}

}  // namespace gte
