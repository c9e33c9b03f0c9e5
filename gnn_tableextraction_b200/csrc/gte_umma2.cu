// Tensor-core projection on CTA PAIRS (tcgen05 cta_group::2) -- the product path of gte_umma_linear_fwd /
// _bwd_data / _fwd_stacked / _bwd_data2 whenever the batch has at least two 128-row tiles.
//
// Why pairs: each SM stages only HALF of the weight tile (the hardware shares the halves of a cta_group::2 MMA), and the
// operand split writes only the low part (the tensor core truncates the raw fp32 word to tf32 by itself).
//
// What bounds it (role timestamps, profiles/r02_umma_pair_experiments.md): NOT the tensor pipe
// (issuing one of the three MMAs changes nothing; the 3x pattern alone runs at 1350-1500 clocks per k-block) but the
// SM <-> L2 traffic: per 128-row tile 616 KB of operand tiles come in (224 KB activations + 392 KB weight tiles, which do
// not fit in shared memory next to the operand ring and are re-read per tile) and 229 KB of z / y go out, ~1 GB per
// launch at config 2 against ~550 MB of HBM traffic.  Variants measured and NOT kept (same results, slower or equal):
// weight tile staged as one fp32 plane with the low part derived on chip (-23 % bytes, but the split then sits on the
// critical path of a 3-stage ring: 1100 clocks per k-block); epilogue draining its row slice into registers
// (setmaxnreg 56/200) to overlap the next tile's MMAs (the stores then contend with the operand loads: +8 k clocks on
// the MMA phase for 11 k saved); thread-per-row 256-bit global stores instead of TMA stores (2x slower: every warp
// instruction touches 32 lines).
//
// Per CTA, 14 warps:
//   warp 0          TMA producer: raw A tile [128 x 32] of its own row tile + its half of W_hi / W_lo
//                   (SWIZZLE_128B, K-major) into an S-stage ring (S = 3 at N = 224); full[s] is CTA local
//   warps 2,3,12,13 operand split: a_lo = rna(a - trunc(a)) into the side tile (position preserving), then ONE
//                   arrive per warp on the LEADER's ready[s] (remote for the peer CTA)
//   warp 1          leader CTA only: elected lane issues 12 tcgen05.mma.cta_group::2 (M = 256, N = BN, K = 8) per
//                   k-block; tcgen05.commit multicasts "stage free" / "accumulator complete" to both CTAs
//   warps 4-11      epilogue, TWO warps per TMEM lane quarter.  Split accumulator (long k loops, one TMEM stage): the two
//                   share a tile, each takes half of the column chunks -- bias, LayerNorm statistics in ONE TMEM pass
//                   (shifted sums per half, merged with the parallel-variance formula through shared memory), second
//                   pass normalises + ReLU (the ReLU + L2-normalise epilogue merges the halves' sums of relu(z)^2 the
//                   same way).  One accumulator (k loops of one or two k-blocks, two TMEM stages): each
//                   group of four warps owns a stage and takes every second tile, whole rows, no exchange.  z and y
//                   leave through swizzled shared tiles and TMA stores; one arrive per warp on the leader's tempty
//
// Results contract, packing and the SPLIT (separate cross-term accumulator) rule are those of gte_umma.cu.
#include "gte_umma_args.cuh"

#include <cuda.h>

namespace gte {

constexpr int U2_THREADS = 448;
constexpr int U2_EPI_WARP0 = 4;   // epilogue warps 4..11
constexpr int U2_EPI_WARPS = 8;
constexpr int U2_SPLIT_WARPS = 4;  // warps 2, 3, 12, 13
constexpr int U2_PREFETCH = 8;     // k-blocks of L2 prefetch lookahead for the activation tiles
constexpr int U2_EPI_BUF = 4096;   // one 32 x 32 fp32 store tile per epilogue warp
constexpr int U2_MAX_STAGES = 6;
constexpr size_t U2_SMEM_MAX = 227 * 1024;

struct U2Layout {
  uint32_t bh_bytes, stage_bytes, epi_off, par_off, stat_off, bar_off, tmem_off, total;
};
__host__ __device__ inline U2Layout u2_layout(int BN, int stages, int epi_bufs) {
  U2Layout L;
  L.bh_bytes = (uint32_t)(BN / 2) * 128u;                  // this CTA's half of one weight tile (hi or lo)
  L.stage_bytes = 2u * UM_A_BYTES + 2u * L.bh_bytes;       // A raw + A lo + W_hi half + W_lo half (multiples of 1024)
  L.epi_off = (uint32_t)stages * L.stage_bytes;
  L.par_off = L.epi_off + U2_EPI_WARPS * U2_EPI_BUF * (uint32_t)epi_bufs;  // bias / gamma / beta
  L.stat_off = L.par_off + 3u * UM_MAX_BN * 4u;            // [parity][half][128 rows] float2 (mean, M2)
  L.bar_off = L.stat_off + 2u * 2u * 128u * 8u;
  L.tmem_off = L.bar_off + (3u * U2_MAX_STAGES + 4u) * 8u;
  L.total = L.tmem_off + 16u;
  return L;
}

template <bool SPLIT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(U2_THREADS, 1)
    k_umma_gemm_pair(const __grid_constant__ UmmaArgs P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // identical carve-up in both CTAs of the pair (same kernel, same dynamic shared-memory offset): the MMA descriptors
  // and the multicast barrier offsets are valid in either CTA
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const U2Layout L = u2_layout(P.BN, P.stages, P.epi_bufs);
  const int S = P.stages;
  uint8_t* const tiles = base;
  auto sA_hi_p = [&](int s) { return tiles + s * L.stage_bytes; };
  auto sA_lo_p = [&](int s) { return tiles + s * L.stage_bytes + UM_A_BYTES; };
  auto sB_hi_p = [&](int s) { return tiles + s * L.stage_bytes + 2 * UM_A_BYTES; };
  auto sB_lo_p = [&](int s) { return tiles + s * L.stage_bytes + 2 * UM_A_BYTES + L.bh_bytes; };
  uint8_t* const s_stage = base + L.epi_off;
  float* const s_bias = reinterpret_cast<float*>(base + L.par_off);
  float* const s_gamma = s_bias + UM_MAX_BN;
  float* const s_beta = s_gamma + UM_MAX_BN;
  float2* const s_stat = reinterpret_cast<float2*>(base + L.stat_off);
  uint64_t* const bars = reinterpret_cast<uint64_t*>(base + L.bar_off);
  uint64_t* const bar_full = bars;                          // [S] local: TMA landed
  uint64_t* const bar_ready = bars + U2_MAX_STAGES;         // [S] leader: both CTAs split their A tile
  uint64_t* const bar_empty = bars + 2 * U2_MAX_STAGES;     // [S] local (multicast commit): MMAs finished reading
  uint64_t* const bar_tfull = bars + 3 * U2_MAX_STAGES;     // [2] local (multicast commit): accumulator complete
  uint64_t* const bar_tempty = bar_tfull + 2;               // [2] leader: both CTAs' epilogues drained it
  uint32_t* const s_tmem = reinterpret_cast<uint32_t*>(base + L.tmem_off);

  const uint32_t rank = cluster_ctarank();
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int m_tiles = (P.M + UM_BM - 1) / UM_BM;
  const int m_pairs = (m_tiles + 1) / 2;
  const int total = m_pairs * P.ngroups;
  const int cluster_id = blockIdx.x >> 1, nclusters = gridDim.x >> 1;
  const int kb_total = P.kblocks[0] + (P.nseg > 1 ? P.kblocks[1] : 0);

  for (int i = threadIdx.x; i < UM_MAX_BN; i += U2_THREADS) {
    s_bias[i] = (P.bias && i < P.bias_n) ? P.bias[i] : 0.f;
    s_gamma[i] = (P.gamma && i < P.N) ? P.gamma[i] : 1.f;
    s_beta[i] = (P.beta && i < P.N) ? P.beta[i] : 0.f;
  }
  if (warp == 0 && lane == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(smem_u32(&bar_full[s]), 1);
      mbar_init(smem_u32(&bar_ready[s]), 2 * U2_SPLIT_WARPS);
      mbar_init(smem_u32(&bar_empty[s]), 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(smem_u32(&bar_tfull[a]), 1);
      // SPLIT: all eight epilogue warps of both CTAs drain the one accumulator stage; otherwise every stage has its own
      // group of four warps per CTA (see the epilogue)
      mbar_init(smem_u32(&bar_tempty[a]), SPLIT ? 2 * U2_EPI_WARPS : U2_EPI_WARPS);
    }
    fence_barrier_init();
    for (int s = 0; s < P.nseg; ++s) tma_prefetch_desc(&P.tmA[s]);
    for (int gq = 0; gq < P.ngroups; ++gq)
      for (int s = 0; s < P.nseg; ++s) {
        tma_prefetch_desc(&P.tmBhi[gq][s]);
        tma_prefetch_desc(&P.tmBlo[gq][s]);
      }
  }
  if (warp == 1) tmem_alloc_pair(smem_u32(s_tmem), 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // the peer's barriers are initialised before anything arrives on them remotely
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;

  if (warp == 0) {
    // ================================ TMA producer (both CTAs) ================================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const int b_row0 = (int)rank * (P.BN >> 1);
      // L2 prefetch cursor for this CTA's activation tiles, U2_PREFETCH k-blocks ahead (the packed weights are L2 resident)
      int pf_t = cluster_id, pf_seg = 0, pf_kb = 0;
      auto pf_step = [&]() {
        if (pf_t >= total) return;
        tma_prefetch_2d(&P.tmA[pf_seg], pf_kb * UM_BK, (2 * (pf_t / P.ngroups) + (int)rank) * UM_BM);
        if (++pf_kb >= P.kblocks[pf_seg]) {
          pf_kb = 0;
          if (++pf_seg >= P.nseg) {
            pf_seg = 0;
            pf_t += nclusters;
          }
        }
      };
      for (int i = 0; i < U2_PREFETCH; ++i) pf_step();
      for (int t = cluster_id; t < total; t += nclusters) {
        const int mt = 2 * (t / P.ngroups) + (int)rank, grp = t % P.ngroups;
        for (int seg = 0; seg < P.nseg; ++seg) {
          for (int kb = 0; kb < P.kblocks[seg]; ++kb) {
            pf_step();
            mbar_wait_cluster_backoff(smem_u32(&bar_empty[stage]), phase ^ 1);
            const uint32_t fb = smem_u32(&bar_full[stage]);
            mbar_expect_tx(fb, (uint32_t)UM_A_BYTES + 2u * L.bh_bytes);
            tma_load_2d(smem_u32(sA_hi_p(stage)), &P.tmA[seg], fb, kb * UM_BK, mt * UM_BM);
            tma_load_2d(smem_u32(sB_hi_p(stage)), &P.tmBhi[grp][seg], fb, kb * UM_BK, b_row0);
            tma_load_2d(smem_u32(sB_lo_p(stage)), &P.tmBlo[grp][seg], fb, kb * UM_BK, b_row0);
            if (++stage == S) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer (leader CTA) =================================
    if (rank == 0 && lane == 0) {
      // instruction descriptor: D=f32, A=B=tf32, both K-major, N=BN, M=256 (128 rows in each CTA)
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(P.BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      constexpr int nacc = SPLIT ? 1 : 2;
      for (int t = cluster_id; t < total; t += nclusters) {
        mbar_wait_cluster(smem_u32(&bar_tempty[acc]), acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * UM_ACC_STRIDE);
        const uint32_t d_cross = SPLIT ? tmem_base + UM_ACC_STRIDE : d_tmem;
        for (int kb = 0; kb < kb_total; ++kb) {
          mbar_wait_cluster(smem_u32(&bar_ready[stage]), phase);
          tc_fence_after();
          const uint64_t dah = make_desc_k_sw128(smem_u32(sA_hi_p(stage)));
          const uint64_t dal = make_desc_k_sw128(smem_u32(sA_lo_p(stage)));
          const uint64_t dbh = make_desc_k_sw128(smem_u32(sB_hi_p(stage)));
          const uint64_t dbl = make_desc_k_sw128(smem_u32(sB_lo_p(stage)));
#pragma unroll
          for (int k = 0; k < UM_BK / 8; ++k) {
            const uint64_t adv = (uint64_t)((k * 8 * 4) >> 4);  // 32 bytes per K=8 step inside the 128 B swizzle row
            umma_tf32_pair(d_cross, dal + adv, dbh + adv, idesc, (kb | k) != 0 ? 1u : 0u);
            umma_tf32_pair(d_cross, dah + adv, dbl + adv, idesc, 1u);
            umma_tf32_pair(d_tmem, dah + adv, dbh + adv, idesc, (SPLIT && (kb | k) == 0) ? 0u : 1u);
          }
          umma_commit_pair(smem_u32(&bar_empty[stage]));
          if (++stage == S) { stage = 0; phase ^= 1; }
        }
        umma_commit_pair(smem_u32(&bar_tfull[acc]));
        if (++acc == nacc) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else if (warp < U2_EPI_WARP0 || warp >= U2_EPI_WARP0 + U2_EPI_WARPS) {
    // ================================ operand split (warps 2, 3, 12, 13) ======================
    const int t = ((warp < U2_EPI_WARP0) ? warp - 2 : warp - (U2_EPI_WARP0 + U2_EPI_WARPS) + 2) * 32 + lane;  // 0..127
    const uint32_t ready_leader = mapa_shared(smem_u32(&bar_ready[0]), 0);
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = cluster_id; tile < total; tile += nclusters) {
      for (int kb = 0; kb < kb_total; ++kb) {
        mbar_wait_backoff(smem_u32(&bar_full[stage]), phase);
        const float4* hi = reinterpret_cast<const float4*>(sA_hi_p(stage));
        float4* lo = reinterpret_cast<float4*>(sA_lo_p(stage));
        // hi stays as TMA wrote it: kind::tf32 reads the top 19 bits of the fp32 word, i.e. a_hi = trunc(a); only the
        // remainder a - trunc(a) (exact in fp32, then rounded to tf32) is written
#pragma unroll
        for (int i = 0; i < UM_A_BYTES / 16 / (U2_SPLIT_WARPS * 32); ++i) {
          const int idx = t + U2_SPLIT_WARPS * 32 * i;
          const float4 v = hi[idx];
          float4 l;
          l.x = tf32_rna(v.x - tf32_hi(v.x)); l.y = tf32_rna(v.y - tf32_hi(v.y));
          l.z = tf32_rna(v.z - tf32_hi(v.z)); l.w = tf32_rna(v.w - tf32_hi(v.w));
          lo[idx] = l;
        }
        fence_proxy_async();  // generic-proxy writes -> visible to the tensor-core (async) proxy
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(ready_leader + (uint32_t)stage * 8u);
        if (++stage == S) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ================================ epilogue (warps 4..11) ===================================
    const int ew = warp - U2_EPI_WARP0;
    const int q = warp & 3;      // TMEM lane quarter this warp may touch
    const int half = ew >> 2;    // which half of the column chunks
    uint8_t* const stb = s_stage + ew * U2_EPI_BUF * P.epi_bufs;
    const int nbuf = P.epi_bufs;
    const uint32_t tempty_leader = mapa_shared(smem_u32(&bar_tempty[0]), 0);
    int store_seq = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    int par = 0;
    constexpr int nacc = SPLIT ? 1 : 2;
    // SPLIT (one accumulator stage): the two warps of a lane quarter share a tile, each takes half of the column chunks
    // and the LayerNorm statistics of the halves are merged through shared memory.
    // !SPLIT (two accumulator stages, the store-bound one- and two-k-block shapes): warp group `half` owns accumulator
    // stage `half` -- it takes every second tile, whole rows, no exchange and no barrier inside a tile (the named
    // barrier between unevenly loaded halves was 40 % of the epilogue warps' stall samples).
    const int nchunks = (P.N + 31) / 32;
    const int c_split = SPLIT ? (nchunks + 1) / 2 : nchunks;
    const int c_beg = (SPLIT && half) ? c_split : 0, c_end = (SPLIT && half) ? nchunks : c_split;
    const int cols_a = min(P.N, c_split * 32);
    const float n_a = (float)cols_a, n_b = (float)(P.N - cols_a), n_all = (float)P.N;
    const float my_n = (SPLIT && half) ? n_b : n_a;
    int it = 0;
    for (int t = cluster_id; t < total; t += nclusters, ++it) {
      const int mt = 2 * (t / P.ngroups) + (int)rank, grp = t % P.ngroups;
      if constexpr (!SPLIT) {
        if ((it & 1) != half) continue;  // the other warp group's tile
        acc = half;
        acc_phase = (uint32_t)(it >> 1) & 1u;
      }
      mbar_wait_cluster_backoff(smem_u32(&bar_tfull[acc]), acc_phase);
      tc_fence_after();
      const uint32_t t_base = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * UM_ACC_STRIDE);
      const int64_t row0 = (int64_t)mt * UM_BM + q * 32;  // first global row of this warp
      const bool rows_live = row0 < (int64_t)P.M;           // the odd tail tile of the peer CTA has no rows at all
      const bool store_z = P.out[grp] != nullptr && rows_live;
      const bool store_y = P.y != nullptr && rows_live;
      float x[32];
      // one 32 x 32 chunk of this warp's rows (z / dx or y) leaves as a TMA store of the swizzled tile
      auto put_chunk = [&](const CUtensorMap* map, int c) {
        epi_store_chunk_tma(stb, nbuf, store_seq, x, map, c * 32, (int32_t)row0);
      };
#define load_chunk(c) epi_load_chunk<SPLIT>(t_base + (c) * 32, s_bias + (c) * 32, x)
      if (P.fuse_ln == UM_EPI_L2) {
        // pass 1: z leaves, and this warp's columns add relu(z)^2 in column order
        float ss = 0.f;
        for (int c = c_beg; c < c_end; ++c) {
          load_chunk(c);
          ss = epi_relu_sq_sum(x, min(32, P.N - c * 32), ss);
          if (store_z) put_chunk(&P.tmOut[grp], c);
        }
        if constexpr (SPLIT) {
          // the two halves meet through shared memory; both warps add them in the same order, so hold the same bits
          float2* const st = s_stat + (par * 2) * 128 + q * 32 + lane;
          st[half * 128] = make_float2(ss, 0.f);
          asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");  // the two warps of this lane quarter
          ss = st[0].x + st[128].x;
          par ^= 1;
        }
        const float nrm = fmaxf(sqrtf(ss), P.eps);
        // pass 2: y = relu(z) / max(||relu(z)||, eps)
        for (int c = c_beg; c < c_end; ++c) {
          load_chunk(c);
          epi_relu_div(x, nrm);
          if (store_y) put_chunk(&P.tmY, c);
        }
      } else if (P.fuse_ln == UM_EPI_LN) {
        // pass 1: z leaves, and this warp's columns are summed around a shift (the mean of its first chunk), which
        // keeps the one-pass variance as accurate as the two-pass form
        float shift = 0.f, s1 = 0.f, s2 = 0.f;
        for (int c = c_beg; c < c_end; ++c) {
          load_chunk(c);
          const int nv = min(32, P.N - c * 32);
          if (c == c_beg) {
            float s0 = 0.f;
#pragma unroll
            for (int j = 0; j < 32; ++j) s0 += (j < nv) ? x[j] : 0.f;
            shift = s0 / (float)nv;
          }
          if (nv == 32) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const float d = x[j] - shift;
              s1 += d;
              s2 = fmaf(d, d, s2);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const float d = (j < nv) ? x[j] - shift : 0.f;
              s1 += d;
              s2 = fmaf(d, d, s2);
            }
          }
          if (store_z) put_chunk(&P.tmOut[grp], c);
        }
        float mh = 0.f, m2h = 0.f;
        if (my_n > 0.f) {
          mh = shift + s1 / my_n;
          m2h = fmaxf(s2 - s1 * s1 / my_n, 0.f);
        }
        float mean = mh, m2 = m2h;
        if constexpr (SPLIT) {
          float2* const st = s_stat + (par * 2) * 128 + q * 32 + lane;
          st[half * 128] = make_float2(mh, m2h);
          asm volatile("bar.sync %0, 64;" ::"r"(1 + q) : "memory");  // the two warps of this lane quarter
          const float2 pa = st[0], pb = st[128];
          par ^= 1;
          // parallel-variance merge of the two halves (both warps compute the same bits: fixed operand order)
          mean = pa.x;
          m2 = pa.y;
          if (n_b > 0.f) {
            const float delta = pb.x - pa.x;
            mean = pa.x + delta * (n_b / n_all);
            m2 = pa.y + pb.y + delta * delta * (n_a * n_b / n_all);
          }
        }
        const float rstd = 1.0f / sqrtf(m2 / n_all + P.eps);
        if (!SPLIT || half == 0) {
          const int64_t grow = row0 + lane;
          if (grow < P.M) {
            P.mean[grow] = mean;
            P.rstd[grow] = rstd;
          }
        }
        // pass 2: normalise + activation
        for (int c = c_beg; c < c_end; ++c) {
          load_chunk(c);
          epi_norm_act(x, s_gamma + c * 32, s_beta + c * 32, true, P.relu != 0, mean, rstd);
          if (store_y) put_chunk(&P.tmY, c);
        }
      } else {
        for (int c = c_beg; c < c_end; ++c) {
          load_chunk(c);
          if (store_z) put_chunk(&P.tmOut[grp], c);
          if (P.y != nullptr) {
            epi_norm_act(x, s_gamma + c * 32, s_beta + c * 32, false, P.relu != 0, 0.f, 1.f);
            if (store_y) put_chunk(&P.tmY, c);
          }
        }
      }
#undef load_chunk
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(tempty_leader + (uint32_t)acc * 8u);
      if constexpr (SPLIT) {
        if (++acc == nacc) { acc = 0; acc_phase ^= 1; }
      }
    }
    if (lane == 0) tma_store_wait_all();  // shared store tiles must outlive their TMA reads
  }
  tc_fence_before();
  __syncwarp();
  __syncthreads();
  cluster_sync_all();  // nobody leaves (or frees TMEM) while the peer may still signal its barriers / read its tiles
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, 512);
  }
}

// Ring depth and store tiles per epilogue warp.  A tile's k loop of one or two k-blocks (input layer, class-layer input
// gradient) never has more than two stages in flight and is bound by its epilogue's TMA stores: two stages, and the
// shared memory goes to up to four store tiles per warp.  Long k loops take the deepest ring that fits with one tile.
static void u2_pick(int BN, int kb_total, int* stages, int* epi_bufs) {
  *stages = 0;
  *epi_bufs = 1;
  if (kb_total <= 2) {
    for (int b = 4; b >= 1; --b)
      if (1024 + (size_t)u2_layout(BN, 2, b).total <= U2_SMEM_MAX) {
        *stages = 2;
        *epi_bufs = b;
        return;
      }
    return;
  }
  for (int s = U2_MAX_STAGES; s >= 2; --s)
    if (1024 + (size_t)u2_layout(BN, s, 1).total <= U2_SMEM_MAX) {
      *stages = s;
      // leftover shared memory: a second store tile per warp
      if (1024 + (size_t)u2_layout(BN, s, 2).total <= U2_SMEM_MAX) *epi_bufs = 2;
      return;
    }
}

bool umma_pair_supported(const UmmaArgs& a) {
  const int m_tiles = (a.M + UM_BM - 1) / UM_BM;
  int st = 0, eb = 0;
  u2_pick(a.BN, 3, &st, &eb);
  return a.tma_store != 0 && m_tiles >= 2 && a.BN % 16 == 0 && a.BN >= 16 && a.BN <= UM_MAX_BN && sm_count() >= 2 && st >= 2;
}

int launch_umma_pair(UmmaArgs& a, cudaStream_t st) {
  if (int rc = setup_weight_maps(a, a.BN / 2)) return rc;
  const int kb_total = a.kblocks[0] + (a.nseg > 1 ? a.kblocks[1] : 0);
  int stages = 0, epi_bufs = 1;
  u2_pick(a.BN, kb_total, &stages, &epi_bufs);
  if (stages < 2) return fail(GTE_ERR_UNSUPPORTED, "k_umma_gemm_pair: BN=%d does not fit shared memory", a.BN);
  a.stages = stages;
  a.epi_bufs = epi_bufs;
  const size_t smem = 1024 + (size_t)u2_layout(a.BN, a.stages, a.epi_bufs).total;
  if (int rc = ensure_dynamic_smem(reinterpret_cast<const void*>(&k_umma_gemm_pair<true>), smem, "k_umma_gemm_pair")) return rc;
  if (int rc = ensure_dynamic_smem(reinterpret_cast<const void*>(&k_umma_gemm_pair<false>), smem, "k_umma_gemm_pair")) return rc;
  const int m_tiles = (a.M + UM_BM - 1) / UM_BM;
  const int total = ((m_tiles + 1) / 2) * a.ngroups;
  int clusters = sm_count() / 2;
  if (clusters > total) clusters = total;
  if (clusters < 1) return GTE_OK;
  // same SPLIT rule as the single-CTA kernel: contractions of one or two k-blocks keep one accumulator per TMEM stage
  // (two stages: the epilogue of tile i overlaps the MMAs of tile i+1)
  if (kb_total > 2)
    k_umma_gemm_pair<true><<<2 * clusters, U2_THREADS, smem, st>>>(a);
  else
    k_umma_gemm_pair<false><<<2 * clusters, U2_THREADS, smem, st>>>(a);
  GTE_CHECK_LAUNCH("k_umma_gemm_pair");
  return GTE_OK;
}

}  // namespace gte
