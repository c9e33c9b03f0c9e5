// Tensor-core route for the wide hidden layers (Fin, Fout ~ 218): tcgen05.mma
// kind::tf32 with fp32 accumulators in TMEM, operands staged by TMA, and the
// error-compensated 3xTF32 split so that the result stays within fp32 parity
// (1e-5 rel) of the reference's `nn.Linear` (models.py:63):
//
//     a = a_hi + a_lo,  b = b_hi + b_lo   (hi = top 19 bits, lo = remainder)
//     a*b ~= a_lo*b_hi + a_hi*b_lo + a_hi*b_hi          (drops a_lo*b_lo ~ 2^-22)
//
// One persistent CTA per SM, 12 warps, warp-specialised:
//   warp 0      TMA producer: raw A tile [128 x 32] + packed W_hi/W_lo tiles [BN x 32]
//               (SWIZZLE_128B, K-major) into a 2-stage smem ring
//   warps 2-7   split A in place (hi) + side buffer (lo) -- position preserving, so
//               the swizzle does not matter -- then fence.proxy.async + arrive
//   warp 1      elected lane issues 12 tcgen05.mma (M=128, N=BN, K=8) per 32-wide k block
//               into one of two TMEM accumulator stages; tcgen05.commit frees smem / signals
//   warps 8-11  epilogue: tcgen05.ld (thread = row), + bias, optional fused
//               LayerNorm + ReLU (row statistics are thread-local), smem transpose,
//               coalesced stores of z (saved for backward) and y
//
// Used for   z = [h | ah] W^T + b  (+ LayerNorm + ReLU)      -> gte_umma_linear_fwd
//            [dh_self | d_ah] = dz W                         -> gte_umma_linear_bwd_data
// Weights are re-packed (split, zero padded, transposed for the backward) by
// gte_umma_pack_weights every step: 95k elements, negligible.
//
// Roofline: tensor pipe (3 * 2*M*N*K flops at the TF32 rate) vs. L2->SM operand
// traffic (W tiles are re-read per 128-row tile); HBM traffic is compulsory
// (read A once, write z and y once).
#include "gte_umma_args.cuh"

#include <cuda.h>

namespace gte {

constexpr int PK_PLANES = 2;  // packed weight tiles: tf32 hi, tf32 lo
constexpr int UM_THREADS = 384;
constexpr int UM_STAGES = 2;
constexpr int UM_SPLIT_THREADS = 192;     // warps 2..7 split the A operand
constexpr int UM_PREFETCH = 8;            // k-blocks of L2 prefetch lookahead for the activation tiles
// per epilogue warp: one or two 32x32 fp32 store tiles (TMA store, 1024-byte aligned); the legacy
// [32][36] transposition tile (4608 B) must fit as well
__host__ __device__ constexpr int um_epi_bytes(int nbuf) { return nbuf == 2 ? 8192 : 5120; }

// ------------------------------------------------------------ the kernel ---
template <bool SPLIT>
__global__ void __launch_bounds__(UM_THREADS, 1) k_umma_gemm(const __grid_constant__ UmmaArgs P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // carve-up (all operand tiles 1024-byte aligned)
  // keep the shared address space visible to the compiler (pointer arithmetic only): LDS/STS, not generic LD/ST
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int b_bytes = P.BN * 128;
  const int stage_bytes = 2 * UM_A_BYTES + 2 * b_bytes;
  uint8_t* const tiles = base;
  auto sA_hi_p = [&](int s) { return tiles + s * stage_bytes; };
  auto sA_lo_p = [&](int s) { return tiles + s * stage_bytes + UM_A_BYTES; };
  auto sB_hi_p = [&](int s) { return tiles + s * stage_bytes + 2 * UM_A_BYTES; };
  auto sB_lo_p = [&](int s) { return tiles + s * stage_bytes + 2 * UM_A_BYTES + b_bytes; };
  base = tiles + UM_STAGES * stage_bytes;
  uint8_t* s_stage = base;                                         // [4 warps][2][4096 B], 1024-byte aligned
  float* s_bias = reinterpret_cast<float*>(s_stage + 4 * um_epi_bytes(P.epi_bufs));  // [256]
  float* s_gamma = s_bias + UM_MAX_BN;
  float* s_beta = s_gamma + UM_MAX_BN;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_beta + UM_MAX_BN);  // 8-byte aligned by construction
  uint64_t* bar_full = bars;                  // [STAGES] TMA landed
  uint64_t* bar_ready = bars + UM_STAGES;     // [STAGES] A split done
  uint64_t* bar_empty = bars + 2 * UM_STAGES; // [STAGES] MMAs finished reading the stage
  uint64_t* bar_tfull = bars + 3 * UM_STAGES; // [2] accumulator complete
  uint64_t* bar_tempty = bar_tfull + 2;       // [2] accumulator drained
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bar_tempty + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int m_tiles = (P.M + UM_BM - 1) / UM_BM;
  const int total_tiles = m_tiles * P.ngroups;
  const int kb_total = P.kblocks[0] + (P.nseg > 1 ? P.kblocks[1] : 0);

  for (int i = threadIdx.x; i < UM_MAX_BN; i += UM_THREADS) {
    s_bias[i] = (P.bias && i < P.bias_n) ? P.bias[i] : 0.f;
    s_gamma[i] = (P.gamma && i < P.N) ? P.gamma[i] : 1.f;
    s_beta[i] = (P.beta && i < P.N) ? P.beta[i] : 0.f;
  }
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < UM_STAGES; ++s) {
      mbar_init(smem_u32(&bar_full[s]), 1);
      mbar_init(smem_u32(&bar_ready[s]), UM_SPLIT_THREADS);
      mbar_init(smem_u32(&bar_empty[s]), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(smem_u32(&bar_tfull[a]), 1);
      mbar_init(smem_u32(&bar_tempty[a]), 128);
    }
    fence_barrier_init();
    for (int s = 0; s < P.nseg; ++s) tma_prefetch_desc(&P.tmA[s]);
    for (int gq = 0; gq < P.ngroups; ++gq)
      for (int s = 0; s < P.nseg; ++s) {
        tma_prefetch_desc(&P.tmBhi[gq][s]);
        tma_prefetch_desc(&P.tmBlo[gq][s]);
      }
  }
  if (warp == 1) tmem_alloc(smem_u32(s_tmem), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;

  if (warp == 0) {
    // ================================ TMA producer ================================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      // L2 prefetch cursor for the activation tiles, UM_PREFETCH k-blocks ahead (the packed weights are L2 resident)
      int pf_tile = blockIdx.x, pf_seg = 0, pf_kb = 0;
      auto pf_step = [&]() {
        if (pf_tile >= total_tiles) return;
        tma_prefetch_2d(&P.tmA[pf_seg], pf_kb * UM_BK, (pf_tile / P.ngroups) * UM_BM);
        if (++pf_kb >= P.kblocks[pf_seg]) {
          pf_kb = 0;
          if (++pf_seg >= P.nseg) {
            pf_seg = 0;
            pf_tile += gridDim.x;
          }
        }
      };
      for (int i = 0; i < UM_PREFETCH; ++i) pf_step();
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int mt = tile / P.ngroups, grp = tile % P.ngroups;
        for (int seg = 0; seg < P.nseg; ++seg) {
          for (int kb = 0; kb < P.kblocks[seg]; ++kb) {
            pf_step();
            mbar_wait_backoff(smem_u32(&bar_empty[stage]), phase ^ 1);
            const uint32_t fb = smem_u32(&bar_full[stage]);
            mbar_expect_tx(fb, (uint32_t)(UM_A_BYTES + 2 * b_bytes));
            tma_load_2d(smem_u32(sA_hi_p(stage)), &P.tmA[seg], fb, kb * UM_BK, mt * UM_BM);
            tma_load_2d(smem_u32(sB_hi_p(stage)), &P.tmBhi[grp][seg], fb, kb * UM_BK, 0);
            tma_load_2d(smem_u32(sB_lo_p(stage)), &P.tmBlo[grp][seg], fb, kb * UM_BK, 0);
            if (++stage == UM_STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ==================================
    if (lane == 0) {
      // instruction descriptor: D=f32, A=B=tf32, both K-major, N=BN, M=128
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(P.BN >> 3) << 17) | ((uint32_t)(UM_BM >> 4) << 24);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      constexpr bool split_acc = SPLIT;
      constexpr int nacc = SPLIT ? 1 : 2;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        mbar_wait_backoff(smem_u32(&bar_tempty[acc]), acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * UM_ACC_STRIDE);
        const uint32_t d_cross = split_acc ? tmem_base + UM_ACC_STRIDE : d_tmem;
        for (int kb = 0; kb < kb_total; ++kb) {
          mbar_wait(smem_u32(&bar_full[stage]), phase);
          mbar_wait(smem_u32(&bar_ready[stage]), phase);
          tc_fence_after();
          const uint64_t dah = make_desc_k_sw128(smem_u32(sA_hi_p(stage)));
          const uint64_t dal = make_desc_k_sw128(smem_u32(sA_lo_p(stage)));
          const uint64_t dbh = make_desc_k_sw128(smem_u32(sB_hi_p(stage)));
          const uint64_t dbl = make_desc_k_sw128(smem_u32(sB_lo_p(stage)));
#pragma unroll
          for (int k = 0; k < UM_BK / 8; ++k) {
            const uint64_t adv = (uint64_t)((k * 8 * 4) >> 4);  // 32 bytes per K=8 step inside the 128 B swizzle row
            umma_tf32(d_cross, dal + adv, dbh + adv, idesc, (kb | k) != 0 ? 1u : 0u);
            umma_tf32(d_cross, dah + adv, dbl + adv, idesc, 1u);
            umma_tf32(d_tmem, dah + adv, dbh + adv, idesc, (split_acc && (kb | k) == 0) ? 0u : 1u);
          }
          umma_commit(smem_u32(&bar_empty[stage]));
          if (++stage == UM_STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(smem_u32(&bar_tfull[acc]));
        if (++acc == nacc) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp >= 2 && warp < 8) {
    // ================================ operand split (6 warps: 2..7) ================
    const int t = threadIdx.x - 64;
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      for (int kb = 0; kb < kb_total; ++kb) {
        mbar_wait_backoff(smem_u32(&bar_full[stage]), phase);
        float4* hi = reinterpret_cast<float4*>(sA_hi_p(stage));
        float4* lo = reinterpret_cast<float4*>(sA_lo_p(stage));
#pragma unroll
        for (int i = 0; i < (UM_A_BYTES / 16 + UM_SPLIT_THREADS - 1) / UM_SPLIT_THREADS; ++i) {
          const int idx = t + UM_SPLIT_THREADS * i;
          if (idx >= UM_A_BYTES / 16) break;
          // hi stays as TMA wrote it: kind::tf32 reads the top 19 bits of the fp32 word, i.e. a_hi = trunc(a);
          // only the remainder a - trunc(a) (exact in fp32, rounded to tf32) is written
          const float4 v = hi[idx];
          float4 l;
          l.x = tf32_rna(v.x - tf32_hi(v.x)); l.y = tf32_rna(v.y - tf32_hi(v.y));
          l.z = tf32_rna(v.z - tf32_hi(v.z)); l.w = tf32_rna(v.w - tf32_hi(v.w));
          lo[idx] = l;
        }
        fence_proxy_async();  // generic-proxy writes -> visible to the tensor-core (async) proxy
        mbar_arrive(smem_u32(&bar_ready[stage]));
        if (++stage == UM_STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp >= 8) {
    // ================================ epilogue ====================================
    const int q = warp & 3;                     // TMEM lane quarter this warp may touch
    uint8_t* stb = s_stage + q * um_epi_bytes(P.epi_bufs);
    float* st = reinterpret_cast<float*>(stb);  // legacy store path: [32][EPI_LD] floats fit the same buffer
    int store_seq = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    constexpr int nacc = SPLIT ? 1 : 2;
    const int nchunks = (P.N + 31) / 32;
    const float inv_n = 1.0f / (float)P.N;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int mt = tile / P.ngroups, grp = tile % P.ngroups;
      mbar_wait(smem_u32(&bar_tfull[acc]), acc_phase);
      tc_fence_after();
      const uint32_t t_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * UM_ACC_STRIDE);
      const int64_t row0 = (int64_t)mt * UM_BM + q * 32;  // first global row of this warp
      float* outp = P.out[grp];
      const int64_t ldo = P.ldo[grp];
      const bool vec_out = ((reinterpret_cast<uintptr_t>(outp) & 15) == 0) && (ldo % 4 == 0);
      const bool vec_y = P.y != nullptr && ((reinterpret_cast<uintptr_t>(P.y) & 15) == 0) && (P.ldy % 4 == 0);
      float x[32];
#define load_chunk(c) epi_load_chunk<SPLIT>(t_base + (c) * 32, s_bias + (c) * 32, x)
      float mean = 0.f, rstd = 1.f, nrm = 1.f;
      if (P.fuse_ln == UM_EPI_L2) {
        // one pass over TMEM for ||relu(z)||^2 (column order), y below divides by max(||relu(z)||, eps)
        float ss = 0.f;
        for (int c = 0; c < nchunks; ++c) {
          load_chunk(c);
          ss = epi_relu_sq_sum(x, min(32, P.N - c * 32), ss);
        }
        nrm = fmaxf(sqrtf(ss), P.eps);
      } else if (P.fuse_ln == UM_EPI_LN) {
        // two passes over TMEM (mean, then centred second moment): exact like nn.LayerNorm; the last chunk
        // is the only one that needs per-column predicates
        const int nfull = P.N / 32, ntail = P.N % 32;
        float s1 = 0.f;
        for (int c = 0; c < nfull; ++c) {
          load_chunk(c);
#pragma unroll
          for (int j = 0; j < 32; ++j) s1 += x[j];
        }
        if (ntail) {
          load_chunk(nfull);
#pragma unroll
          for (int j = 0; j < 32; ++j) s1 += (j < ntail) ? x[j] : 0.f;
        }
        mean = s1 * inv_n;
        float s2 = 0.f;
        for (int c = 0; c < nfull; ++c) {
          load_chunk(c);
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float d = x[j] - mean;
            s2 = fmaf(d, d, s2);
          }
        }
        if (ntail) {
          load_chunk(nfull);
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float d = (j < ntail) ? x[j] - mean : 0.f;
            s2 = fmaf(d, d, s2);
          }
        }
        rstd = 1.0f / sqrtf(s2 * inv_n + P.eps);
        const int64_t grow = row0 + lane;
        if (grow < P.M) {
          P.mean[grow] = mean;
          P.rstd[grow] = rstd;
        }
      }
      const int rows_valid = (int)min((int64_t)32, (int64_t)P.M - row0);
      for (int c = 0; c < nchunks; ++c) {
        load_chunk(c);
        if (outp != nullptr) {  // z / dx (not wanted by inference-only callers)
          if (P.tma_store)
            epi_store_chunk_tma(stb, P.epi_bufs, store_seq, x, &P.tmOut[grp], c * 32, (int32_t)row0);
          else if (rows_valid > 0)
            epi_store_chunk(st, x, outp + row0 * ldo + c * 32, ldo, rows_valid, P.N - c * 32, vec_out);
        }
        if (P.y != nullptr) {
          if (P.fuse_ln == UM_EPI_L2)
            epi_relu_div(x, nrm);
          else
            epi_norm_act(x, s_gamma + c * 32, s_beta + c * 32, P.fuse_ln == UM_EPI_LN, P.relu != 0, mean, rstd);
          if (P.tma_store)
            epi_store_chunk_tma(stb, P.epi_bufs, store_seq, x, &P.tmY, c * 32, (int32_t)row0);
          else if (rows_valid > 0)
            epi_store_chunk(st, x, P.y + row0 * P.ldy + c * 32, P.ldy, rows_valid, P.N - c * 32, vec_y);
        }
      }
#undef load_chunk
      tc_fence_before();
      mbar_arrive(smem_u32(&bar_tempty[acc]));
      if (++acc == nacc) { acc = 0; acc_phase ^= 1; }
    }
  }
  if (warp >= 8 && lane == 0) tma_store_wait_all();  // shared store tiles must outlive their TMA reads
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------- weight packing ----
// fwd pack:  Pf[seg][half][BN][Kp]   Pf[seg][.][o][k] = W[o, seg*fin + k]          (K-major B of z = x W^T)
// bwd pack:  Pb[grp][half][BNb][Kpb] Pb[grp][.][j][o] = W[o, grp*fin + j]          (K-major B of dx = dz W)
// half 0 = tf32 hi, half 1 = tf32(lo); zero padded.
// stacked pack (narrow layers, fo <= 16, nseg == 2): Ps[half][32][Kp], row o = W[o, 0:fin] (self block),
//            row 16+o = W[o, fin:2fin] (neighbour block): ONE pass over x gives [x Ws^T | x Wn^T] side by side.
// combined packs (nseg == 2) for operands stored side by side in ONE 32-column matrix (columns [0, w) = self block,
//            [16, 16+w) = neighbour block, the rest zero), so that the whole contraction is a single k-block:
//   Pc[half][BN][32]   (fin <= 16)  Pc[o][k] = W[o, k] (k < fin), W[o, fin + k-16] (16 <= k < 16+fin)     z = [h|ah] W^T
//   Pd[half][BNb][32]  (fo <= 16)   Pd[j][k] = W[k, j] (k < fo),  W[k-16, fin + j] (16 <= k < 16+fo)      dx = [dz|gq] W
__device__ __forceinline__ void pack_one(const float* __restrict__ W, int64_t ldw, int32_t fo, int32_t fin, int32_t nseg,
                            float* __restrict__ Pf, int32_t BN, int32_t Kp, float* __restrict__ Pb, int32_t BNb,
                            int32_t Kpb, float* __restrict__ Ps, float* __restrict__ Pc, float* __restrict__ Pd) {
  const int64_t per_f = (int64_t)BN * Kp, per_b = (int64_t)BNb * Kpb;
  const int64_t total_f = (int64_t)nseg * per_f, total_b = (int64_t)nseg * per_b;
  const int64_t total_s = Ps ? (int64_t)32 * Kp : 0;
  const int64_t total_c = Pc ? (int64_t)BN * 32 : 0;
  const int64_t total_d = Pd ? (int64_t)BNb * 32 : 0;
  const int64_t end_b = total_f + total_b, end_s = end_b + total_s, end_c = end_s + total_c;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;  // (gridDim.x only: blockIdx.y selects the matrix in the batch form)
  for (; i < end_c + total_d; i += stride) {
    float w = 0.f;
    float* dst;
    int64_t half_stride;
    if (i >= end_c) {
      const int64_t r = i - end_c;
      const int j = (int)(r >> 5), k = (int)(r & 31);
      const int o = k & 15, blk = k >> 4;
      if (o < fo && j < fin) w = W[(int64_t)o * ldw + (int64_t)blk * fin + j];
      dst = Pd + r;
      half_stride = total_d;
    } else if (i >= end_s) {
      const int64_t r = i - end_s;
      const int o = (int)(r >> 5), k = (int)(r & 31);
      const int kk = k & 15, blk = k >> 4;
      if (o < fo && kk < fin) w = W[(int64_t)o * ldw + (int64_t)blk * fin + kk];
      dst = Pc + r;
      half_stride = total_c;
    } else if (i >= end_b) {
      const int64_t r = i - end_b;
      const int row = (int)(r / Kp), k = (int)(r % Kp);
      const int o = row & 15, blk = row >> 4;
      if (o < fo && k < fin) w = W[(int64_t)o * ldw + (int64_t)blk * fin + k];
      dst = Ps + r;
      half_stride = total_s;
    } else if (i < total_f) {
      const int seg = (int)(i / per_f);
      const int64_t r = i % per_f;
      const int o = (int)(r / Kp), k = (int)(r % Kp);
      if (o < fo && k < fin) w = W[(int64_t)o * ldw + (int64_t)seg * fin + k];
      dst = Pf + (int64_t)seg * PK_PLANES * per_f + r;
      half_stride = per_f;
    } else {
      const int64_t ib = i - total_f;
      const int grp = (int)(ib / per_b);
      const int64_t r = ib % per_b;
      const int j = (int)(r / Kpb), o = (int)(r % Kpb);
      if (o < fo && j < fin) w = W[(int64_t)o * ldw + (int64_t)grp * fin + j];
      dst = Pb + (int64_t)grp * PK_PLANES * per_b + r;
      half_stride = per_b;
    }
    const float h = tf32_rna(w);  // round-to-nearest split of the (small, packed once per step) weight operand
    dst[0] = h;
    dst[half_stride] = tf32_rna(w - h);
  }
}

__global__ void k_umma_pack(const float* __restrict__ W, int64_t ldw, int32_t fo, int32_t fin, int32_t nseg,
                            float* __restrict__ Pf, int32_t BN, int32_t Kp, float* __restrict__ Pb, int32_t BNb,
                            int32_t Kpb, float* __restrict__ Ps, float* __restrict__ Pc, float* __restrict__ Pd) {
  pack_one(W, ldw, fo, fin, nseg, Pf, BN, Kp, Pb, BNb, Kpb, Ps, Pc, Pd);
}

// several weight matrices in one launch (blockIdx.y = matrix): the train step packs all its layers at once
struct PackOne {
  const float* W;
  int64_t ldw;
  int32_t fo, fin, nseg, BN, Kp, BNb, Kpb;
  float *Pf, *Pb, *Ps, *Pc, *Pd;
};
struct PackBatch {
  PackOne m[GTE_PACK_BATCH_MAX];
};
__global__ void k_umma_pack_batch(const PackBatch B) {
  const PackOne& p = B.m[blockIdx.y];
  pack_one(p.W, p.ldw, p.fo, p.fin, p.nseg, p.Pf, p.BN, p.Kp, p.Pb, p.BNb, p.Kpb, p.Ps, p.Pc, p.Pd);
}

// ------------------------------------------------------------ host side ----
// 2-D fp32 row-major [rows, cols] with leading dimension ld (floats); box = 32 cols x box_rows, SWIZZLE_128B
static int make_map(CUtensorMap* m, const float* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  return make_tmap_2d(m, ptr, rows, cols, ld, UM_BK, box_rows);
}

static int round_up(int v, int m) { return (v + m - 1) / m * m; }

struct PackDims {
  int BN, Kp, BNb, Kpb;
  size_t fwd_floats, bwd_floats, stacked_floats, combf_floats, combb_floats;
  size_t off_stacked() const { return fwd_floats + bwd_floats; }
  size_t off_combf() const { return off_stacked() + stacked_floats; }
  size_t off_combb() const { return off_combf() + combf_floats; }
  size_t total() const { return off_combb() + combb_floats; }
};
static PackDims pack_dims(int fo, int fin, int nseg) {
  PackDims d;
  d.BN = round_up(fo, 16);
  d.Kp = round_up(fin, UM_BK);
  d.BNb = round_up(fin, 16);
  d.Kpb = round_up(fo, UM_BK);
  d.fwd_floats = (size_t)nseg * PK_PLANES * d.BN * d.Kp;
  d.bwd_floats = (size_t)nseg * PK_PLANES * d.BNb * d.Kpb;
  d.stacked_floats = (fo <= 16 && nseg == 2) ? (size_t)PK_PLANES * 32 * d.Kp : 0;
  d.combf_floats = (fin <= 16 && nseg == 2) ? (size_t)PK_PLANES * d.BN * 32 : 0;
  d.combb_floats = (fo <= 16 && nseg == 2) ? (size_t)PK_PLANES * d.BNb * 32 : 0;
  return d;
}

static size_t umma_smem_bytes(int BN, int epi_bufs) {
  return 1024 + (size_t)UM_STAGES * (2 * UM_A_BYTES + 2 * (size_t)BN * 128) + 4 * (size_t)um_epi_bytes(epi_bufs) +
         3 * UM_MAX_BN * 4 + (3 * UM_STAGES + 4) * 8 + 16;
}

// TMA-store descriptors for the outputs (used when every output is 16-byte aligned with ld % 4 == 0)
static int setup_output_maps(UmmaArgs& a) {
  bool ok = true;
  for (int g = 0; g < a.ngroups; ++g) ok = ok && (a.out[g] == nullptr || (aligned16(a.out[g]) && a.ldo[g] % 4 == 0));
  if (a.y) ok = ok && aligned16(a.y) && a.ldy % 4 == 0;
  a.tma_store = ok ? 1 : 0;
  if (!ok) return GTE_OK;
  for (int g = 0; g < a.ngroups; ++g) {
    if (a.out[g] == nullptr) continue;
    int rc = make_tmap_2d(&a.tmOut[g], a.out[g], a.M, a.N, a.ldo[g], 32, 32);
    if (rc) return rc;
  }
  if (a.y) {
    int rc = make_tmap_2d(&a.tmY, a.y, a.M, a.N, a.ldy, 32, 32);
    if (rc) return rc;
  }
  return GTE_OK;
}

// weight-tile maps with the box of the kernel that will run: BN rows (single CTA) or BN/2 rows (each CTA of a pair
// stages half of the B rows)
int setup_weight_maps(UmmaArgs& a, int box_rows) {
  for (int g = 0; g < a.ngroups; ++g)
    for (int s = 0; s < a.nseg; ++s) {
      int rc = make_map(&a.tmBhi[g][s], a.bhi[g][s], a.BN, a.b_cols, a.b_cols, box_rows);
      if (rc) return rc;
      rc = make_map(&a.tmBlo[g][s], a.blo[g][s], a.BN, a.b_cols, a.b_cols, box_rows);
      if (rc) return rc;
    }
  return GTE_OK;
}

int launch_umma_single(UmmaArgs& a, cudaStream_t st) {
  if (int rc = setup_weight_maps(a, a.BN)) return rc;
  a.epi_bufs = umma_smem_bytes(a.BN, 2) <= 227 * 1024 ? 2 : 1;
  const size_t smem = umma_smem_bytes(a.BN, a.epi_bufs);
  if (int rc = ensure_dynamic_smem(reinterpret_cast<const void*>(&k_umma_gemm<true>), smem, "k_umma_gemm")) return rc;
  if (int rc = ensure_dynamic_smem(reinterpret_cast<const void*>(&k_umma_gemm<false>), smem, "k_umma_gemm")) return rc;
  const int tiles = ((a.M + UM_BM - 1) / UM_BM) * a.ngroups;
  int grid = sm_count();
  if (grid > tiles) grid = tiles;
  if (grid < 1) return GTE_OK;
  // The cross-term accumulator exists to keep the long main accumulation chain free of the small terms (the
  // tensor core truncates when it accumulates).  A contraction of one or two k-blocks (the input layer: K = 26,
  // the class-layer input gradient: K = 18) has no long chain: one accumulator is just as exact, and it frees
  // TMEM for a second accumulator stage (epilogue of tile i overlaps the MMAs of tile i+1) and halves the
  // epilogue's TMEM reads.
  const int kb_total = a.kblocks[0] + (a.nseg > 1 ? a.kblocks[1] : 0);
  if (kb_total > 2)
    k_umma_gemm<true><<<grid, UM_THREADS, smem, st>>>(a);
  else
    k_umma_gemm<false><<<grid, UM_THREADS, smem, st>>>(a);
  GTE_CHECK_LAUNCH("k_umma_gemm");
  return GTE_OK;
}

// CTA pairs (cta_group::2) whenever the shape allows it: the pair halves the weight-tile traffic per SM, which is what
// bounds the 3xTF32 contraction (see gte_umma2.cu); gte_set_tuning(GTE_TUNE_UMMA_PAIR, 0) forces the single-CTA kernel.
static int launch_umma(UmmaArgs& a, cudaStream_t st) {
  if (int rc = setup_output_maps(a)) return rc;
  if (tuning(GTE_TUNE_UMMA_PAIR) != 0 && umma_pair_supported(a)) return launch_umma_pair(a, st);
  return launch_umma_single(a, st);
}

}  // namespace gte

using namespace gte;

extern "C" {

int gte_umma_supported(int32_t fo, int32_t fin) {
  return (fo >= 1 && fo <= UM_MAX_BN && fin >= 1 && fin <= UM_MAX_BN) ? 1 : 0;
}

size_t gte_umma_pack_bytes(int32_t fo, int32_t fin, int32_t nseg) {
  if (!gte_umma_supported(fo, fin) || nseg < 1 || nseg > 2) return 0;
  PackDims d = pack_dims(fo, fin, nseg);
  return d.total() * 4;
}

int gte_umma_pack_weights(const float* W, int64_t ldw, int32_t fo, int32_t fin, int32_t nseg, float* pack,
                          gte_stream_t stream) {
  GTE_CHECK_ARG(W && pack, "gte_umma_pack_weights: null argument");
  GTE_CHECK_ARG(nseg >= 1 && nseg <= 2 && ldw >= (int64_t)nseg * fin, "gte_umma_pack_weights: bad nseg/ldw");
  if (!gte_umma_supported(fo, fin)) return fail(GTE_ERR_UNSUPPORTED, "gte_umma_pack_weights: fo=%d fin=%d unsupported", fo, fin);
  GTE_CHECK_ARG(aligned16(pack), "gte_umma_pack_weights: pack buffer must be 16-byte aligned");
  PackDims d = pack_dims(fo, fin, nseg);
  const int64_t total = (int64_t)(d.total() / PK_PLANES);
  k_umma_pack<<<(unsigned)ceil_div64(total, 256), 256, 0, as_stream(stream)>>>(
      W, ldw, fo, fin, nseg, pack, d.BN, d.Kp, pack + d.fwd_floats, d.BNb, d.Kpb,
      d.stacked_floats ? pack + d.off_stacked() : nullptr, d.combf_floats ? pack + d.off_combf() : nullptr,
      d.combb_floats ? pack + d.off_combb() : nullptr);
  GTE_CHECK_LAUNCH("k_umma_pack");
  return GTE_OK;
}

int gte_umma_pack_weights_batch(const gte_pack_desc_t* descs, int32_t count, gte_stream_t stream) {
  GTE_CHECK_ARG(count >= 0 && count <= GTE_PACK_BATCH_MAX && (count == 0 || descs), "gte_umma_pack_weights_batch: 0 <= count <= %d", GTE_PACK_BATCH_MAX);
  if (count == 0) return GTE_OK;
  PackBatch B{};
  int64_t max_total = 0;
  for (int i = 0; i < count; ++i) {
    const gte_pack_desc_t& q = descs[i];
    GTE_CHECK_ARG(q.W && q.pack, "gte_umma_pack_weights_batch: null argument");
    GTE_CHECK_ARG(q.nseg >= 1 && q.nseg <= 2 && q.ldw >= (int64_t)q.nseg * q.fin, "gte_umma_pack_weights_batch: bad nseg/ldw");
    if (!gte_umma_supported(q.fo, q.fin))
      return fail(GTE_ERR_UNSUPPORTED, "gte_umma_pack_weights_batch: fo=%d fin=%d unsupported", q.fo, q.fin);
    GTE_CHECK_ARG(aligned16(q.pack), "gte_umma_pack_weights_batch: pack buffer must be 16-byte aligned");
    PackDims d = pack_dims(q.fo, q.fin, q.nseg);
    PackOne& m = B.m[i];
    m.W = q.W; m.ldw = q.ldw; m.fo = q.fo; m.fin = q.fin; m.nseg = q.nseg;
    m.BN = d.BN; m.Kp = d.Kp; m.BNb = d.BNb; m.Kpb = d.Kpb;
    m.Pf = q.pack;
    m.Pb = q.pack + d.fwd_floats;
    m.Ps = d.stacked_floats ? q.pack + d.off_stacked() : nullptr;
    m.Pc = d.combf_floats ? q.pack + d.off_combf() : nullptr;
    m.Pd = d.combb_floats ? q.pack + d.off_combb() : nullptr;
    const int64_t total = (int64_t)(d.total() / PK_PLANES);
    if (total > max_total) max_total = total;
  }
  dim3 grid((unsigned)ceil_div64(max_total, 256), (unsigned)count);
  k_umma_pack_batch<<<grid, 256, 0, as_stream(stream)>>>(B);
  GTE_CHECK_LAUNCH("k_umma_pack_batch");
  return GTE_OK;
}

int gte_umma_linear_fwd(const float* x1, int64_t ldx1, const float* x2, int64_t ldx2, int32_t fin, const float* pack,
                        const float* bias, const float* gamma, const float* beta, float eps, int relu, int fuse_ln,
                        float* z, int64_t ldz, float* y, int64_t ldy, float* mean, float* rstd, int32_t n, int32_t fo,
                        gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0, "gte_umma_linear_fwd: negative n");
  if (!gte_umma_supported(fo, fin)) return fail(GTE_ERR_UNSUPPORTED, "gte_umma_linear_fwd: fo=%d fin=%d unsupported", fo, fin);
  if (n == 0) return GTE_OK;
  GTE_CHECK_ARG(x1 && pack && (z || y), "gte_umma_linear_fwd: null argument (z may be NULL only when y is given)");
  GTE_CHECK_ARG(fuse_ln >= UM_EPI_NONE && fuse_ln <= UM_EPI_L2, "gte_umma_linear_fwd: fuse_ln must be 0 (none), 1 (LayerNorm) or 2 (ReLU + L2-normalise)");
  GTE_CHECK_ARG(fuse_ln != UM_EPI_LN || (gamma && beta && mean && rstd && y), "gte_umma_linear_fwd: fused LayerNorm needs gamma/beta/mean/rstd/y");
  GTE_CHECK_ARG(fuse_ln != UM_EPI_L2 || y, "gte_umma_linear_fwd: fused ReLU + L2-normalise needs y");
  GTE_CHECK_ARG(aligned16(x1) && ldx1 % 4 == 0 && ldx1 >= fin, "gte_umma_linear_fwd: x1 must be 16-byte aligned with ld %% 4 == 0");
  GTE_CHECK_ARG(!x2 || (aligned16(x2) && ldx2 % 4 == 0 && ldx2 >= fin), "gte_umma_linear_fwd: x2 must be 16-byte aligned with ld %% 4 == 0");
  GTE_CHECK_ARG((!z || ldz >= fo) && (!y || ldy >= fo), "gte_umma_linear_fwd: output leading dimension < fo");
  const int nseg = x2 ? 2 : 1;
  PackDims d = pack_dims(fo, fin, nseg);
  UmmaArgs a{};
  a.nseg = nseg;
  a.ngroups = 1;
  a.M = n;
  a.N = fo;
  a.BN = d.BN;
  const float* xs[2] = {x1, x2};
  const int64_t lds[2] = {ldx1, ldx2};
  const size_t per = (size_t)d.BN * d.Kp;
  for (int s = 0; s < nseg; ++s) {
    a.kblocks[s] = d.Kp / UM_BK;
    int rc = make_map(&a.tmA[s], xs[s], n, fin, lds[s], UM_BM);
    if (rc) return rc;
    a.bhi[0][s] = pack + (size_t)s * PK_PLANES * per;
    a.blo[0][s] = a.bhi[0][s] + per;
  }
  a.b_cols = d.Kp;
  a.out[0] = z;
  a.ldo[0] = ldz;
  a.y = y;
  a.ldy = ldy;
  a.bias = bias;
  a.bias_n = fo;
  a.gamma = gamma;
  a.beta = beta;
  a.mean = mean;
  a.rstd = rstd;
  a.eps = eps;
  a.fuse_ln = fuse_ln;
  a.relu = (relu && fuse_ln != UM_EPI_L2) ? 1 : 0;  // the L2 mode applies its own ReLU
  return launch_umma(a, as_stream(stream));
}

int gte_umma_linear_bwd_data(const float* dz, int64_t lddz, int32_t fo, const float* pack, int32_t nseg, float* dx1,
                             int64_t lddx1, float* dx2, int64_t lddx2, int32_t n, int32_t fin, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0, "gte_umma_linear_bwd_data: negative n");
  if (!gte_umma_supported(fo, fin)) return fail(GTE_ERR_UNSUPPORTED, "gte_umma_linear_bwd_data: fo=%d fin=%d unsupported", fo, fin);
  if (n == 0) return GTE_OK;
  GTE_CHECK_ARG(dz && pack && dx1 && nseg >= 1 && nseg <= 2 && (nseg == 1 || dx2), "gte_umma_linear_bwd_data: null argument");
  GTE_CHECK_ARG(aligned16(dz) && lddz % 4 == 0 && lddz >= fo, "gte_umma_linear_bwd_data: dz must be 16-byte aligned with ld %% 4 == 0");
  GTE_CHECK_ARG(lddx1 >= fin && (nseg == 1 || lddx2 >= fin), "gte_umma_linear_bwd_data: output leading dimension < fin");
  PackDims d = pack_dims(fo, fin, nseg);
  const float* pb = pack + d.fwd_floats;
  UmmaArgs a{};
  a.nseg = 1;
  a.ngroups = nseg;
  a.M = n;
  a.N = fin;
  a.BN = d.BNb;
  a.kblocks[0] = d.Kpb / UM_BK;
  int rc = make_map(&a.tmA[0], dz, n, fo, lddz, UM_BM);
  if (rc) return rc;
  const size_t per = (size_t)d.BNb * d.Kpb;
  for (int gq = 0; gq < nseg; ++gq) {
    a.bhi[gq][0] = pb + (size_t)gq * PK_PLANES * per;
    a.blo[gq][0] = a.bhi[gq][0] + per;
  }
  a.b_cols = d.Kpb;
  a.out[0] = dx1;
  a.ldo[0] = lddx1;
  a.out[1] = dx2;
  a.ldo[1] = lddx2;
  return launch_umma(a, as_stream(stream));
}

// Narrow (class) layer, project-then-aggregate: out[n, 32] = x [Ws | . | Wn | .]^T (+ bias on the first fo columns):
// columns [0, fo) = x Ws^T + b, columns [16, 16+fo) = x Wn^T.  One pass over x.
int gte_umma_linear_fwd_stacked(const float* x, int64_t ldx, int32_t fin, const float* pack, const float* bias, int32_t fo,
                                float* out, int64_t ldo, int32_t n, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0, "gte_umma_linear_fwd_stacked: negative n");
  if (fo < 1 || fo > 16 || !gte_umma_supported(fo, fin))
    return fail(GTE_ERR_UNSUPPORTED, "gte_umma_linear_fwd_stacked: fo=%d fin=%d unsupported (fo <= 16)", fo, fin);
  if (n == 0) return GTE_OK;
  GTE_CHECK_ARG(x && pack && out, "gte_umma_linear_fwd_stacked: null argument");
  GTE_CHECK_ARG(aligned16(x) && ldx % 4 == 0 && ldx >= fin && ldo >= 32,
                "gte_umma_linear_fwd_stacked: x must be 16-byte aligned with ld %% 4 == 0; out needs ld >= 32");
  PackDims d = pack_dims(fo, fin, 2);
  const float* ps = pack + d.fwd_floats + d.bwd_floats;
  UmmaArgs a{};
  a.nseg = 1;
  a.ngroups = 1;
  a.M = n;
  a.N = 32;
  a.BN = 32;
  a.kblocks[0] = d.Kp / UM_BK;
  int rc = make_map(&a.tmA[0], x, n, fin, ldx, UM_BM);
  if (rc) return rc;
  a.bhi[0][0] = ps;
  a.blo[0][0] = ps + (size_t)32 * d.Kp;
  a.b_cols = d.Kp;
  a.out[0] = out;
  a.ldo[0] = ldo;
  a.bias = bias;
  a.bias_n = fo;
  return launch_umma(a, as_stream(stream));
}

// dx = dz1 W[:, :fin] + dz2 W[:, fin:2fin]   (two K segments, one output; class layer backward)
int gte_umma_linear_bwd_data2(const float* dz1, int64_t lddz1, const float* dz2, int64_t lddz2, int32_t fo,
                              const float* pack, float* dx, int64_t lddx, int32_t n, int32_t fin, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0, "gte_umma_linear_bwd_data2: negative n");
  if (!gte_umma_supported(fo, fin)) return fail(GTE_ERR_UNSUPPORTED, "gte_umma_linear_bwd_data2: fo=%d fin=%d unsupported", fo, fin);
  if (n == 0) return GTE_OK;
  GTE_CHECK_ARG(dz1 && dz2 && pack && dx, "gte_umma_linear_bwd_data2: null argument");
  GTE_CHECK_ARG(aligned16(dz1) && lddz1 % 4 == 0 && lddz1 >= fo && aligned16(dz2) && lddz2 % 4 == 0 && lddz2 >= fo,
                "gte_umma_linear_bwd_data2: dz must be 16-byte aligned with ld %% 4 == 0");
  GTE_CHECK_ARG(lddx >= fin, "gte_umma_linear_bwd_data2: output leading dimension < fin");
  PackDims d = pack_dims(fo, fin, 2);
  const float* pb = pack + d.fwd_floats;
  const size_t per = (size_t)d.BNb * d.Kpb;
  UmmaArgs a{};
  a.nseg = 2;
  a.ngroups = 1;
  a.M = n;
  a.N = fin;
  a.BN = d.BNb;
  const float* dzs[2] = {dz1, dz2};
  const int64_t lds[2] = {lddz1, lddz2};
  for (int s = 0; s < 2; ++s) {
    a.kblocks[s] = d.Kpb / UM_BK;
    int rc = make_map(&a.tmA[s], dzs[s], n, fo, lds[s], UM_BM);
    if (rc) return rc;
    a.bhi[0][s] = pb + (size_t)s * PK_PLANES * per;
    a.blo[0][s] = a.bhi[0][s] + per;
  }
  a.b_cols = d.Kpb;
  a.out[0] = dx;
  a.ldo[0] = lddx;
  return launch_umma(a, as_stream(stream));
}

// Narrow-INPUT layer (fin <= 16, the input layer) on a combined operand: xc[n, 32] holds h in columns [0, fin) and
// A_hat h in columns [16, 16+fin), every other column finite (they meet zero weights): z = [h | ah] W^T + b is a
// single k-block instead of two segments of one k-block each; same epilogue as gte_umma_linear_fwd.
int gte_umma_linear_fwd_comb(const float* xc, int64_t ldx, int32_t fin, const float* pack, const float* bias,
                             const float* gamma, const float* beta, float eps, int relu, int fuse_ln, float* z,
                             int64_t ldz, float* y, int64_t ldy, float* mean, float* rstd, int32_t n, int32_t fo,
                             gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0, "gte_umma_linear_fwd_comb: negative n");
  if (fin < 1 || fin > 16 || !gte_umma_supported(fo, fin))
    return fail(GTE_ERR_UNSUPPORTED, "gte_umma_linear_fwd_comb: fo=%d fin=%d unsupported (fin <= 16)", fo, fin);
  if (n == 0) return GTE_OK;
  GTE_CHECK_ARG(xc && pack && (z || y), "gte_umma_linear_fwd_comb: null argument (z may be NULL only when y is given)");
  GTE_CHECK_ARG(fuse_ln >= UM_EPI_NONE && fuse_ln <= UM_EPI_L2, "gte_umma_linear_fwd_comb: fuse_ln must be 0 (none), 1 (LayerNorm) or 2 (ReLU + L2-normalise)");
  GTE_CHECK_ARG(fuse_ln != UM_EPI_LN || (gamma && beta && mean && rstd && y), "gte_umma_linear_fwd_comb: fused LayerNorm needs gamma/beta/mean/rstd/y");
  GTE_CHECK_ARG(fuse_ln != UM_EPI_L2 || y, "gte_umma_linear_fwd_comb: fused ReLU + L2-normalise needs y");
  GTE_CHECK_ARG(aligned16(xc) && ldx % 4 == 0 && ldx >= 32, "gte_umma_linear_fwd_comb: xc must be 16-byte aligned with ld %% 4 == 0, ld >= 32");
  GTE_CHECK_ARG((!z || ldz >= fo) && (!y || ldy >= fo), "gte_umma_linear_fwd_comb: output leading dimension < fo");
  PackDims d = pack_dims(fo, fin, 2);
  const float* pc = pack + d.off_combf();
  UmmaArgs a{};
  a.nseg = 1;
  a.ngroups = 1;
  a.M = n;
  a.N = fo;
  a.BN = d.BN;
  a.kblocks[0] = 1;
  int rc = make_map(&a.tmA[0], xc, n, 32, ldx, UM_BM);
  if (rc) return rc;
  a.bhi[0][0] = pc;
  a.blo[0][0] = pc + (size_t)d.BN * 32;
  a.b_cols = 32;
  a.out[0] = z;
  a.ldo[0] = ldz;
  a.y = y;
  a.ldy = ldy;
  a.bias = bias;
  a.bias_n = fo;
  a.gamma = gamma;
  a.beta = beta;
  a.mean = mean;
  a.rstd = rstd;
  a.eps = eps;
  a.fuse_ln = fuse_ln;
  a.relu = (relu && fuse_ln != UM_EPI_L2) ? 1 : 0;  // the L2 mode applies its own ReLU
  return launch_umma(a, as_stream(stream));
}

// Narrow-OUTPUT (class) layer backward on a combined operand: dc[n, 32] holds dz in columns [0, fo) and A_hat^T dz in
// columns [16, 16+fo), every other column finite: dx = dz Ws + gq Wn as a single k-block (gte_umma_linear_bwd_data2
// runs the same contraction as two segments).
int gte_umma_linear_bwd_data_comb(const float* dc, int64_t lddc, int32_t fo, const float* pack, float* dx, int64_t lddx,
                                  int32_t n, int32_t fin, gte_stream_t stream) {
  GTE_CHECK_ARG(n >= 0, "gte_umma_linear_bwd_data_comb: negative n");
  if (fo < 1 || fo > 16 || !gte_umma_supported(fo, fin))
    return fail(GTE_ERR_UNSUPPORTED, "gte_umma_linear_bwd_data_comb: fo=%d fin=%d unsupported (fo <= 16)", fo, fin);
  if (n == 0) return GTE_OK;
  GTE_CHECK_ARG(dc && pack && dx, "gte_umma_linear_bwd_data_comb: null argument");
  GTE_CHECK_ARG(aligned16(dc) && lddc % 4 == 0 && lddc >= 32, "gte_umma_linear_bwd_data_comb: dc must be 16-byte aligned with ld %% 4 == 0, ld >= 32");
  GTE_CHECK_ARG(lddx >= fin, "gte_umma_linear_bwd_data_comb: output leading dimension < fin");
  PackDims d = pack_dims(fo, fin, 2);
  const float* pd = pack + d.off_combb();
  UmmaArgs a{};
  a.nseg = 1;
  a.ngroups = 1;
  a.M = n;
  a.N = fin;
  a.BN = d.BNb;
  a.kblocks[0] = 1;
  int rc = make_map(&a.tmA[0], dc, n, 32, lddc, UM_BM);
  if (rc) return rc;
  a.bhi[0][0] = pd;
  a.blo[0][0] = pd + (size_t)d.BNb * 32;
  a.b_cols = 32;
  a.out[0] = dx;
  a.ldo[0] = lddx;
  return launch_umma(a, as_stream(stream));
}

}  // extern "C"
