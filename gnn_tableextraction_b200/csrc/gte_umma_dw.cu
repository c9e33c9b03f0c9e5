// Weight gradients on the tensor cores: dW = dz^T [x1 | x2] (and the transposed, narrow-dz form of
// the class layer), the reduction over all N nodes of the batch.
//
//     out[m, j] = sum_r A[r, m] * B[r, j]          A: [n, M<=256]   B: boxes of 32 columns from up to 3 tensors
//
// Both operands are activations stored row-major [node, feature], i.e. "MN-major" for the MMA
// (the contraction index r is the slow axis), which tcgen05.mma kind::tf32 consumes directly through
// MN-major SWIZZLE_128B_BASE32B shared-memory descriptors -- no transposes are materialised.  TMA loads
// [32 rows x 32 floats] boxes; a 128-row A tile is 4 boxes, a B tile up to 8 boxes (N <= 256).
// 3xTF32 split as in gte_umma.cu (both operands are split in shared memory by the transform warps:
// hi = rna(x), lo = rna(x - hi)); the small cross terms (a_lo*b_hi + a_hi*b_lo) accumulate in
// their own TMEM accumulator so that the long main chain sees as few round-toward-zero steps as possible.
//
// Rows are processed in chunks (~512 rows = 64 MMA K-steps per accumulator, the in-TMEM chain stays short because
// tensor-core accumulation truncates).  Every persistent CTA owns ONE (group, m-tile) output tile and walks its share
// of the chunks in a fixed order; after each chunk it adds the accumulator to its private fp32 partial tile (plain
// coalesced read-modify-write, L2 resident: 148 tiles of 112 KB), so a launch writes one partial per CTA instead of one
// per chunk (r01: 145 MB of chunk partials written and read back).  A second kernel sums the <= 148 partials in a fixed
// order -- deterministic, no atomics.
// An all-ones column (B side) or row (A side) can be injected to obtain column sums (bias gradient)
// from the same pass.
//
// Pipeline: 4 stages of 16 contraction rows (r01: 2 stages of 32 rows -- the ring was latency bound: TMA + split + MMA
// of a stage ran almost back to back); every operand tile arrives as ONE TMA request through a 3-D blocked view of the
// row-major matrix (r01: one request per 32-column box, 11 per stage -- the TMA unit's request rate was a bound); the
// operand split writes only the low parts (hi = the raw fp32 word, which kind::tf32 truncates by itself) with batched
// shared-memory loads, on twelve worker warps that also run the per-chunk epilogue (role accounting of an instrumented
// build: with six split warps the MMA issuer waited 40 % of the time for split operands).
//
// Roofline: HBM (each activation byte is read once per use) -- the MMA work is 3*2*n*M*N flops.
#include "gte_common.cuh"
#include "gte_umma_ptx.cuh"

namespace gte {

constexpr int DW_THREADS = 448;                // producer, MMA issuer, 12 worker warps
constexpr int DW_KB = 16;                      // contraction rows per pipeline stage (two K = 8 MMA steps)
constexpr int DW_BOX_BYTES = DW_KB * 128;      // one TMA box: 16 rows x 32 floats
constexpr int DW_MAX_STAGES = 8;
constexpr int DW_WORKERS = 12;                 // warps 2..13: operand split per stage + epilogue per chunk
constexpr int DW_SPLIT_THREADS = DW_WORKERS * 32;
constexpr int DW_MAX_BOXES = 8;

struct DwRun {      // consecutive 32-column blocks of one B tensor, consecutive boxes of the shared-memory tile
  int32_t map;      // index into tmB
  int32_t blk0;     // first 32-column block
  int32_t nblk;
  int32_t blocked;  // 1: tmB[map] is a 3-D blocked map (one request for the run), 0: 2-D boxes, one request per block
};
struct DwGroup {
  int32_t a;       // index into tmA
  int32_t nboxes;  // N = 32 * nboxes
  int32_t nruns;
  DwRun run[2];
  int32_t pcol0;   // first column of this group's tile in the partial matrix
  int32_t ones_b_col;  // >= 0: tile column of B forced to 1 (column sums of A); -1: none
  int32_t ones_a_col;  // >= 0: column of A forced to 1 (column sums of B); -1: none
};
struct DwArgs {
  CUtensorMap tmA[2];
  CUtensorMap tmB[3];
  DwGroup grp[2];
  int32_t item_g[4], item_mt[4];  // (group, m-tile) pairs processed per row chunk
  int32_t items_per_chunk;
  int32_t n, chunk_rows, nchunks;
  int32_t max_boxes;
  int32_t a_blocked[2];  // tmA[i] is a 3-D blocked map (box = 4 blocks = one m-tile)
  int32_t a_real_boxes;  // 4, or fewer when A is a narrow operand: boxes [a_real_boxes, 4) of the A tile stay zero
  int32_t stages;        // operand ring depth (as many stages as fit: narrow operands get a deeper ring)
  float* partial;        // [gridDim.x] tiles of [32 * max_boxes columns][128 rows] floats (column-major: row fastest)
  int64_t tile_stride;   // floats per partial tile
};

// AREAL: real 32-column boxes of the A tile (4; 1 for a narrow A operand -- compile time, so that the operand split keeps
// constant bounds: with a run-time bound the hidden-layer launch measured 15 % slower)
template <int AREAL>
__global__ void __launch_bounds__(DW_THREADS, 1) k_umma_dw(const __grid_constant__ DwArgs P) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // keep the shared address space visible to the compiler (pointer arithmetic only): LDS/STS, not generic LD/ST
  uint8_t* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int a_bytes = 4 * DW_BOX_BYTES;
  const int b_bytes = P.max_boxes * DW_BOX_BYTES;
  const int stage_bytes = 2 * a_bytes + 2 * b_bytes;
  uint8_t* const tiles = base;
  auto sA_hi = [&](int s) { return tiles + s * stage_bytes; };
  auto sA_lo = [&](int s) { return tiles + s * stage_bytes + a_bytes; };
  auto sB_hi = [&](int s) { return tiles + s * stage_bytes + 2 * a_bytes; };
  auto sB_lo = [&](int s) { return tiles + s * stage_bytes + 2 * a_bytes + b_bytes; };
  const int DW_STAGES = P.stages;
  uint64_t* bars = reinterpret_cast<uint64_t*>(tiles + DW_STAGES * stage_bytes);
  uint64_t* bar_full = bars;
  uint64_t* bar_ready = bars + DW_MAX_STAGES;
  uint64_t* bar_empty = bars + 2 * DW_MAX_STAGES;
  uint64_t* bar_tfull = bars + 3 * DW_MAX_STAGES;
  uint64_t* bar_tempty = bar_tfull + 1;
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bar_tempty + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int kb_per_chunk = P.chunk_rows / DW_KB;
  // this CTA's output tile and its chunks: CTAs b, b + ipc, b + 2 ipc, ... share sub-item b % ipc and deal the chunks
  // round robin (fixed order => reproducible partials)
  const int ipc = P.items_per_chunk;
  const int sub = blockIdx.x % ipc;
  const int peers = ((int)gridDim.x - sub + ipc - 1) / ipc;  // CTAs working on this sub-item
  const int first_chunk = blockIdx.x / ipc;
  const DwGroup& G = P.grp[P.item_g[sub]];
  const int mt = P.item_mt[sub];

  if (warp == 0 && lane == 0) {
    for (int s = 0; s < DW_STAGES; ++s) {
      mbar_init(smem_u32(&bar_full[s]), 1);
      mbar_init(smem_u32(&bar_ready[s]), DW_WORKERS);
      mbar_init(smem_u32(&bar_empty[s]), 1);
    }
    mbar_init(smem_u32(bar_tfull), 1);
    mbar_init(smem_u32(bar_tempty), DW_WORKERS);
    fence_barrier_init();
    tma_prefetch_desc(&P.tmA[G.a]);
    for (int r = 0; r < G.nruns; ++r) tma_prefetch_desc(&P.tmB[G.run[r].map]);
  }
  if (AREAL < 4) {
    // narrow A operand: the unused 32-column boxes of every stage's A tile (hi and lo) are zero for the whole launch
    const int z0 = AREAL * DW_BOX_BYTES / 16, zn = a_bytes / 16;
    for (int s = 0; s < DW_STAGES; ++s)
      for (int i = z0 + threadIdx.x; i < zn; i += DW_THREADS) {
        reinterpret_cast<float4*>(sA_hi(s))[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        reinterpret_cast<float4*>(sA_lo(s))[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
    fence_proxy_async();
  }
  if (warp == 1) tmem_alloc(smem_u32(s_tmem), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;

  // number of K blocks of a chunk that contain at least one real row
  auto chunk_kblocks = [&](int chunk) {
    const int r0 = chunk * P.chunk_rows;
    const int rows = min(P.chunk_rows, P.n - r0);
    const int kb = (rows + DW_KB - 1) / DW_KB;
    return kb < 1 ? 1 : (kb > kb_per_chunk ? kb_per_chunk : kb);
  };

  if (warp == 0) {
    // ================================ TMA producer ================================
    // No L2 prefetch: both ways of doing it were measured to SLOW the kernel down at config 2 (hidden-layer dW 0.23 ms
    // without; 0.28 ms with cp.async.bulk.prefetch requests 12 stages ahead -- they queue in the TMA unit in front of the
    // real loads; 0.47 ms with prefetch.global.L2 from the producer warp's spare lanes).
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int chunk = first_chunk; chunk < P.nchunks; chunk += peers) {
        const int r0 = chunk * P.chunk_rows;
        const int nkb = chunk_kblocks(chunk);
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(smem_u32(&bar_empty[stage]), phase ^ 1);
          const uint32_t fb = smem_u32(&bar_full[stage]);
          mbar_expect_tx(fb, (uint32_t)((AREAL + G.nboxes) * DW_BOX_BYTES));
          const int row = r0 + kb * DW_KB;
          if (P.a_blocked[G.a]) tma_load_3d(smem_u32(sA_hi(stage)), &P.tmA[G.a], fb, 0, row, mt * 4);
          else for (int b = 0; b < AREAL; ++b)
            tma_load_2d(smem_u32(sA_hi(stage) + b * DW_BOX_BYTES), &P.tmA[G.a], fb, mt * 128 + b * 32, row);
          int box = 0;
          for (int r = 0; r < G.nruns; ++r) {
            const DwRun& R = G.run[r];
            if (R.blocked) tma_load_3d(smem_u32(sB_hi(stage) + box * DW_BOX_BYTES), &P.tmB[R.map], fb, 0, row, R.blk0);
            else for (int b = 0; b < R.nblk; ++b)
              tma_load_2d(smem_u32(sB_hi(stage) + (box + b) * DW_BOX_BYTES), &P.tmB[R.map], fb, (R.blk0 + b) * 32, row);
            box += R.nblk;
          }
          if (++stage == DW_STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer ==================================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0, acc_phase = 0;
      const int BN = G.nboxes * 32;
      // D=f32, A=B=tf32, both MN-major, N=BN, M=128
      const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(BN >> 3) << 17) |
                             ((uint32_t)(128 >> 4) << 24);
      const uint32_t d_main = tmem_base, d_cross = tmem_base + 256;
      for (int chunk = first_chunk; chunk < P.nchunks; chunk += peers) {
        mbar_wait_backoff(smem_u32(bar_tempty), acc_phase ^ 1);
        tc_fence_after();
        const int nkb = chunk_kblocks(chunk);
        for (int kb = 0; kb < nkb; ++kb) {
          mbar_wait(smem_u32(&bar_ready[stage]), phase);
          tc_fence_after();
          const uint64_t dah = make_desc_mn_sw128_32b(smem_u32(sA_hi(stage)), DW_BOX_BYTES);
          const uint64_t dal = make_desc_mn_sw128_32b(smem_u32(sA_lo(stage)), DW_BOX_BYTES);
          const uint64_t dbh = make_desc_mn_sw128_32b(smem_u32(sB_hi(stage)), DW_BOX_BYTES);
          const uint64_t dbl = make_desc_mn_sw128_32b(smem_u32(sB_lo(stage)), DW_BOX_BYTES);
#pragma unroll
          for (int k = 0; k < DW_KB / 8; ++k) {
            const uint64_t adv = (uint64_t)((k * 1024) >> 4);  // next 8-row atom inside every box
            const uint32_t first = (kb | k) == 0 ? 0u : 1u;
            umma_tf32(d_cross, dal + adv, dbh + adv, idesc, first);
            umma_tf32(d_cross, dah + adv, dbl + adv, idesc, 1u);
            umma_tf32(d_main, dah + adv, dbh + adv, idesc, first);
          }
          umma_commit(smem_u32(&bar_empty[stage]));
          if (++stage == DW_STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(smem_u32(bar_tfull));
        acc_phase ^= 1;
      }
    }
  } else {
    // ================================ worker warps (2..13) ========================
    // Per stage: the operand split.  hi stays as TMA wrote it (kind::tf32 truncates the raw fp32 word by itself); only
    // lo = rna(v - trunc(v)) is written, position preserving, so the swizzle does not matter.
    // Per chunk: the epilogue.  The same warps add the accumulator (main + cross) to this CTA's partial tile -- the MMA
    // issuer and the ring are idle then anyway (one accumulator pair fills TMEM), so twelve warps instead of four
    // shorten exactly the part that cannot overlap.  Warp w may touch TMEM lanes 32 (w % 4) ..: three warps per lane
    // quarter, which take the 32-column chunks c = j, j + 3, j + 6.  The partial tile is column major, so a warp's 32
    // rows of one column are one 128-byte line.
    const int t = threadIdx.x - 64;
    const int q = warp & 3, third = (warp - 2) >> 2;
    int stage = 0;
    uint32_t phase = 0, acc_phase = 0;
    constexpr int na4 = AREAL * DW_BOX_BYTES / 16;
    const int nb4 = G.nboxes * DW_BOX_BYTES / 16;
    const bool epi_rows = q < AREAL;  // narrow A: only the first lane quarters hold real rows
    const int ones_col = G.ones_b_col >= 0 ? G.ones_b_col : ((G.ones_a_col >= 0 && G.ones_a_col / 128 == mt) ? G.ones_a_col % 128 : -1);
    float* const ptile = P.partial + (int64_t)blockIdx.x * P.tile_stride + q * 32 + lane;
    bool first = true;
    for (int chunk = first_chunk; chunk < P.nchunks; chunk += peers) {
      const int r0 = chunk * P.chunk_rows;
      const int nkb = chunk_kblocks(chunk);
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(smem_u32(&bar_full[stage]), phase);
        constexpr int PER = ((4 + DW_MAX_BOXES) * DW_BOX_BYTES / 16 + DW_SPLIT_THREADS - 1) / DW_SPLIT_THREADS;  // 4
        float4 v[PER];
        const float4* a_hi = reinterpret_cast<const float4*>(sA_hi(stage));
        const float4* b_hi = reinterpret_cast<const float4*>(sB_hi(stage));
        float4* a_lo = reinterpret_cast<float4*>(sA_lo(stage));
        float4* b_lo = reinterpret_cast<float4*>(sB_lo(stage));
#pragma unroll
        for (int i = 0; i < PER; ++i) {  // all loads first: one shared-memory round trip
          const int idx = t + i * DW_SPLIT_THREADS;
          if (idx < na4) v[i] = a_hi[idx];
          else if (idx - na4 < nb4) v[i] = b_hi[idx - na4];
        }
#pragma unroll
        for (int i = 0; i < PER; ++i) {
          const int idx = t + i * DW_SPLIT_THREADS;
          float4 l;
          l.x = tf32_rna_fast(v[i].x - tf32_hi(v[i].x)); l.y = tf32_rna_fast(v[i].y - tf32_hi(v[i].y));
          l.z = tf32_rna_fast(v[i].z - tf32_hi(v[i].z)); l.w = tf32_rna_fast(v[i].w - tf32_hi(v[i].w));
          if (idx < na4) a_lo[idx] = l;
          else if (idx - na4 < nb4) b_lo[idx - na4] = l;
        }
        if (ones_col >= 0) {
          // all-ones column: element (row kk, tile column c) of an MN-major SW128 box tile.  It is a padding column: zero
          // filled by the 2-D maps, but whatever the row's padding holds with the 3-D blocked maps -- so hi := 1 and
          // lo := 0 are both patched, after every splitting thread wrote its low parts.  Rows past the end of the batch are
          // zero filled by either map and stay 0.
          asm volatile("bar.sync 1, %0;" ::"n"(DW_SPLIT_THREADS) : "memory");
          if (t < DW_KB) {
            const int kk = t;
            if (r0 + kb * DW_KB + kk < P.n) {
              const int box = ones_col / 32, cin = ones_col % 32;
              const int off = box * DW_BOX_BYTES + kk * 128 + (((cin >> 3) ^ (kk & 3)) << 5) + (cin & 7) * 4;  // 32-byte chunk swizzle
              *reinterpret_cast<float*>((G.ones_b_col >= 0 ? sB_hi(stage) : sA_hi(stage)) + off) = 1.0f;
              *reinterpret_cast<float*>((G.ones_b_col >= 0 ? sB_lo(stage) : sA_lo(stage)) + off) = 0.0f;
            }
          }
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&bar_ready[stage]));
        if (++stage == DW_STAGES) { stage = 0; phase ^= 1; }
      }
      // ---- epilogue of this chunk
      mbar_wait(smem_u32(bar_tfull), acc_phase);
      tc_fence_after();
      const uint32_t t_base = tmem_base + ((uint32_t)(q * 32) << 16);
      for (int c = third; c < G.nboxes && epi_rows; c += 3) {
        uint32_t v[32], v2[32];
        tmem_ld_32x32b_x32_nowait(t_base + c * 32, v);
        tmem_ld_32x32b_x32_nowait(t_base + 256 + c * 32, v2);
        float old[32];
        float* const pc = ptile + (int64_t)(c * 32) * 128;
        if (!first) {
#pragma unroll
          for (int j = 0; j < 32; ++j) old[j] = pc[j * 128];
        }
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float val = __uint_as_float(v[j]) + __uint_as_float(v2[j]);
          pc[j * 128] = first ? val : old[j] + val;
        }
      }
      first = false;
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(bar_tempty));
      acc_phase ^= 1;
    }
    if (first) {  // a CTA without any chunk still owns a partial tile: it must read as zero
      for (int c = third; c < G.nboxes && epi_rows; c += 3)
        for (int j = 0; j < 32; ++j) ptile[(int64_t)(c * 32 + j) * 128] = 0.f;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---- fixed-order reduction of the per-CTA partial tiles into up to four rectangular destinations ----------------
struct DwSeg {
  int32_t prow0, nrows, pcol0, ncols;  // rectangle of the conceptual [m-tiles * 128, sum of group widths] result
  float* dst;
  int64_t stride_row, stride_col;      // dst[row*stride_row + col*stride_col]
};
struct DwReduceArgs {
  DwSeg seg[4];
  int32_t nseg;
  const float* partial;
  int64_t tile_stride;
  int32_t grid, ipc;                   // CTAs of the k_umma_dw launch, sub-items per chunk
  int32_t item_g[4], item_mt[4];
  int32_t grp_pcol0[2], grp_ncols[2];
  int32_t accumulate;
};

// 32 consecutive output elements (rows fastest: consecutive threads read consecutive floats of the column-major partial
// tiles) x 8 slices of the <= 148 partials per block; slice s adds partials s, s + 8, ... in ascending order, then slice 0
// adds the slice sums in ascending order -- a fixed order, so the result is reproducible.
constexpr int DWR_SLICES = 8;
__global__ void __launch_bounds__(32 * DWR_SLICES) k_umma_dw_reduce(const DwReduceArgs R) {
  __shared__ float red[DWR_SLICES][32];
  const int ox = threadIdx.x & 31, sy = threadIdx.x >> 5;
  int64_t i = (int64_t)blockIdx.x * 32 + ox;
  int s = 0;
  bool valid = false;
  for (; s < R.nseg; ++s) {
    const int64_t cnt = (int64_t)R.seg[s].nrows * R.seg[s].ncols;
    if (i < cnt) {
      valid = true;
      break;
    }
    i -= cnt;
  }
  int row = 0, col = 0;
  float v = 0.f;
  if (valid) {
    col = (int)(i / R.seg[s].nrows);
    row = (int)(i % R.seg[s].nrows);
    const int prow = R.seg[s].prow0 + row, pcol = R.seg[s].pcol0 + col;
    const int mt = prow >> 7, r = prow & 127;
    int g = 0;
    if (pcol >= R.grp_pcol0[1] && R.grp_ncols[1] > 0) g = 1;
    const int c = pcol - R.grp_pcol0[g];
    int sub = 0;
    for (int k = 0; k < R.ipc; ++k)
      if (R.item_g[k] == g && R.item_mt[k] == mt) sub = k;
    const int nb = (R.grid - sub + R.ipc - 1) / R.ipc;  // CTAs sub, sub + ipc, ... hold the partials of this output tile
    const float* p = R.partial + (int64_t)sub * R.tile_stride + (int64_t)c * 128 + r;
    const int64_t stride = (int64_t)R.ipc * R.tile_stride;
    // four loads in flight per thread (the partials sit in L2: one dependent load at a time was a 600-clock chain per
    // partial); still a fixed order: slice s adds partials s, s + 8, ... four at a time, then the four sub-sums
    float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
    int b = sy;
    for (; b + 3 * DWR_SLICES < nb; b += 4 * DWR_SLICES) {
      const float a0 = p[(int64_t)b * stride], a1 = p[(int64_t)(b + DWR_SLICES) * stride];
      const float a2 = p[(int64_t)(b + 2 * DWR_SLICES) * stride], a3 = p[(int64_t)(b + 3 * DWR_SLICES) * stride];
      v0 += a0; v1 += a1; v2 += a2; v3 += a3;
    }
    for (; b < nb; b += DWR_SLICES) v0 += p[(int64_t)b * stride];
    v = (v0 + v1) + (v2 + v3);
  }
  red[sy][ox] = v;
  __syncthreads();
  if (sy != 0 || !valid) return;
  float t = 0.f;
#pragma unroll
  for (int k = 0; k < DWR_SLICES; ++k) t += red[k][ox];
  float* d = R.seg[s].dst + row * R.seg[s].stride_row + col * R.seg[s].stride_col;
  if (R.accumulate) t += *d;
  *d = t;
}

constexpr int DW_CHUNK_ROWS_DEFAULT = 512;

static size_t dw_smem_bytes(int max_boxes, int stages) {
  return 1024 + (size_t)stages * (2 * 4 * DW_BOX_BYTES + 2 * (size_t)max_boxes * DW_BOX_BYTES) + (3 * DW_MAX_STAGES + 2) * 8 + 16;
}

// partial tiles: one per CTA of the (at most sm_count) persistent grid
static size_t dw_workspace_bytes(int max_boxes) { return (size_t)sm_count() * 32 * max_boxes * 128 * 4 + 256; }

static int dw_launch(DwArgs& a, DwReduceArgs& r, cudaStream_t st) {
  if (a.a_real_boxes <= 0) a.a_real_boxes = 4;
  a.stages = DW_MAX_STAGES;
  while (a.stages > 2 && dw_smem_bytes(a.max_boxes, a.stages) > 227 * 1024) --a.stages;
  const size_t smem = dw_smem_bytes(a.max_boxes, a.stages);
  if (a.a_real_boxes != 4 && a.a_real_boxes != 1) return fail(GTE_ERR_INVALID, "k_umma_dw: a_real_boxes = %d", a.a_real_boxes);
  const void* kfn = a.a_real_boxes == 4 ? reinterpret_cast<const void*>(&k_umma_dw<4>) : reinterpret_cast<const void*>(&k_umma_dw<1>);
  if (int rc = ensure_dynamic_smem(kfn, smem, "k_umma_dw")) return rc;
  // Rows per accumulation chunk: 384..640 rows (the accuracy experiments behind the default of 512 hold for this whole
  // range), chosen so that the persistent CTAs finish together: every sub-item is shared by grid / ipc CTAs that deal
  // its chunks round robin, cost = rounds * k-blocks with rounds = ceil(chunks / (grid / ipc)).
  const int sms = sm_count();
  int grid = sms;
  if (a.n > 0) {
    const int lanes = sms / a.items_per_chunk > 0 ? sms / a.items_per_chunk : 1;
    int best_kb = DW_CHUNK_ROWS_DEFAULT / DW_KB;
    int64_t best_cost = -1;
    for (int kb = 384 / DW_KB; kb <= 640 / DW_KB; ++kb) {
      const int64_t chunks = ceil_div64(a.n, (int64_t)kb * DW_KB);
      const int64_t rounds = ceil_div64(chunks, lanes);
      const int64_t cost = rounds * kb;
      if (best_cost < 0 || cost < best_cost) {
        best_cost = cost;
        best_kb = kb;
      }
    }
    a.chunk_rows = best_kb * DW_KB;
    a.nchunks = (int)ceil_div64(a.n, a.chunk_rows);
    const int64_t items = (int64_t)a.nchunks * a.items_per_chunk;
    if (grid > items) grid = (int)items;
  } else {
    a.nchunks = 0;
    grid = 0;
  }
  a.tile_stride = (int64_t)32 * a.max_boxes * 128;
  r.tile_stride = a.tile_stride;
  r.grid = grid;
  r.ipc = a.items_per_chunk;
  for (int k = 0; k < 4; ++k) {
    r.item_g[k] = a.item_g[k];
    r.item_mt[k] = a.item_mt[k];
  }
  for (int g = 0; g < 2; ++g) {
    r.grp_pcol0[g] = a.grp[g].pcol0;
    r.grp_ncols[g] = a.grp[g].nboxes * 32;
  }
  if (grid >= 1) {
    if (a.a_real_boxes == 4) k_umma_dw<4><<<grid, DW_THREADS, smem, st>>>(a);
    else k_umma_dw<1><<<grid, DW_THREADS, smem, st>>>(a);
    GTE_CHECK_LAUNCH("k_umma_dw");
  }
  int64_t total = 0;
  for (int s = 0; s < r.nseg; ++s) total += (int64_t)r.seg[s].nrows * r.seg[s].ncols;
  if (total > 0) {
    k_umma_dw_reduce<<<(unsigned)ceil_div64(total, 32), 32 * DWR_SLICES, 0, st>>>(r);
    GTE_CHECK_LAUNCH("k_umma_dw_reduce");
  }
  return GTE_OK;
}

static int boxes_of(int k) { return (k + 31) / 32; }

// Operand map: the 3-D blocked view (one TMA request per run of 32-column blocks) when every block lies inside the row's
// leading dimension, 2-D boxes (one request per block, columns past `cols` zero filled) otherwise.
static int dw_make_map(CUtensorMap* m, int32_t* blocked, const float* p, int64_t rows, int64_t cols, int64_t ld, int box_blocks) {
  *blocked = (box_blocks > 1 && ld >= 32 * ((cols + 31) / 32)) ? 1 : 0;
  if (*blocked) {
    if (make_tmap_3d_blocks(m, p, rows, cols, ld, DW_KB, box_blocks, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B) == GTE_OK) return GTE_OK;
    *blocked = 0;  // a driver that refuses the overlapping strides: plain boxes
  }
  return make_tmap_2d(m, p, rows, cols, ld, 32, DW_KB, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B);
}

static bool tma_ok(const float* p, int64_t ld) { return p == nullptr || (aligned16(p) && ld % 4 == 0); }

}  // namespace gte

using namespace gte;

extern "C" {

// dW[:, 0:k1] (+)= dz^T x1 ; dW[:, k1:k1+k2] (+)= dz^T x2 ; db (+)= colsum(dz) when a padding column is free.
int gte_umma_bwd_weight_supported(int32_t fo, int32_t k1, int32_t k2) {
  return (fo >= 1 && fo <= 256 && k1 >= 1 && k1 <= 256 && k2 >= 0 && k2 <= 256) ? 1 : 0;
}

size_t gte_umma_bwd_weight_workspace_bytes(int32_t n, int32_t fo, int32_t k1, int32_t k2) {
  if (!gte_umma_bwd_weight_supported(fo, k1, k2) || n < 0) return 0;
  const int nb1 = boxes_of(k1), nb2 = boxes_of(k2);
  const int mb = nb1 + nb2 <= DW_MAX_BOXES ? nb1 + nb2 : (nb1 > nb2 ? nb1 : nb2);
  return dw_workspace_bytes(mb);  // one partial tile per persistent CTA, whatever n is
}

int gte_umma_linear_bwd_weight(const float* dz, int64_t lddz, int32_t fo, const float* x1, int64_t ldx1, int32_t k1,
                               const float* x2, int64_t ldx2, int32_t k2, float* dW, int64_t lddw, float* db,
                               int accumulate, int32_t n, void* ws, size_t ws_bytes, gte_stream_t stream) {
  if (!gte_umma_bwd_weight_supported(fo, k1, k2))
    return fail(GTE_ERR_UNSUPPORTED, "gte_umma_linear_bwd_weight: fo=%d k1=%d k2=%d unsupported", fo, k1, k2);
  GTE_CHECK_ARG(n >= 0 && dW && (n == 0 || (dz && x1 && (k2 == 0 || x2))), "gte_umma_linear_bwd_weight: bad argument");
  GTE_CHECK_ARG(tma_ok(dz, lddz) && tma_ok(x1, ldx1) && (k2 == 0 || tma_ok(x2, ldx2)),
                "gte_umma_linear_bwd_weight: operands must be 16-byte aligned with ld %% 4 == 0");
  GTE_CHECK_ARG(lddz >= fo && ldx1 >= k1 && (k2 == 0 || ldx2 >= k2) && lddw >= (int64_t)k1 + k2,
                "gte_umma_linear_bwd_weight: leading dimension too small");
  const size_t need = gte_umma_bwd_weight_workspace_bytes(n, fo, k1, k2);
  if (ws == nullptr || ws_bytes < need)
    return fail(GTE_ERR_WORKSPACE, "gte_umma_linear_bwd_weight: workspace %zu < required %zu", ws_bytes, need);
  const int nb1 = boxes_of(k1), nb2 = boxes_of(k2);
  DwArgs a{};
  DwReduceArgs r{};
  a.n = n;
  const int mtiles = (fo + 127) / 128;
  a.partial = static_cast<float*>(ws);
  int b_blocked[2] = {0, 0};
  if (n > 0) {
    int rc = dw_make_map(&a.tmA[0], &a.a_blocked[0], dz, n, fo, lddz, 4);
    if (rc) return rc;
    rc = dw_make_map(&a.tmB[0], &b_blocked[0], x1, n, k1, ldx1, nb1);
    if (rc) return rc;
    if (k2 > 0) {
      rc = dw_make_map(&a.tmB[1], &b_blocked[1], x2, n, k2, ldx2, nb2);
      if (rc) return rc;
    }
  }
  // one group when all boxes fit one accumulator (N <= 256), otherwise one group per input segment
  const bool one_group = nb1 + nb2 <= DW_MAX_BOXES;
  int ngroups = 0;
  auto add_boxes = [&](DwGroup& G, int map, int nb) {
    G.run[G.nruns++] = DwRun{map, 0, nb, b_blocked[map]};
    G.nboxes += nb;
  };
  DwGroup& G0 = a.grp[0];
  G0.a = 0; G0.nboxes = 0; G0.nruns = 0; G0.pcol0 = 0; G0.ones_b_col = -1; G0.ones_a_col = -1;
  add_boxes(G0, 0, nb1);
  ngroups = 1;
  if (k2 > 0) {
    if (one_group) {
      add_boxes(G0, 1, nb2);
    } else {
      DwGroup& G1 = a.grp[1];
      G1.a = 0; G1.nboxes = 0; G1.nruns = 0; G1.pcol0 = 32 * nb1; G1.ones_b_col = -1; G1.ones_a_col = -1;
      add_boxes(G1, 1, nb2);
      ngroups = 2;
    }
  }
  // bias gradient: a free padding column of the first segment carries the all-ones column
  bool db_fused = false;
  if (db && k1 % 32 != 0) {
    G0.ones_b_col = k1;
    db_fused = true;
  }
  a.max_boxes = 0;
  a.items_per_chunk = 0;
  for (int g = 0; g < ngroups; ++g) {
    if (a.grp[g].nboxes > a.max_boxes) a.max_boxes = a.grp[g].nboxes;
    for (int mt = 0; mt < mtiles; ++mt) {
      a.item_g[a.items_per_chunk] = g;
      a.item_mt[a.items_per_chunk] = mt;
      ++a.items_per_chunk;
    }
  }
  r.partial = a.partial;
  r.accumulate = accumulate;
  r.nseg = 0;
  r.seg[r.nseg++] = DwSeg{0, fo, 0, k1, dW, lddw, 1};
  if (k2 > 0) r.seg[r.nseg++] = DwSeg{0, fo, 32 * nb1, k2, dW + k1, lddw, 1};
  if (db_fused) r.seg[r.nseg++] = DwSeg{0, fo, k1, 1, db, 1, 0};
  int rc = dw_launch(a, r, as_stream(stream));
  if (rc) return rc;
  if (db && !db_fused) return fail(GTE_ERR_UNSUPPORTED, "gte_umma_linear_bwd_weight: db needs k1 %% 32 != 0 (no free padding column)");
  return GTE_OK;
}

// Narrow-dz form (class layer, project-then-aggregate): A = x [n, k<=256], B = [dz1 | dz2] (fo <= 32 each)
//   dW[:, col1:col1+k] (+)= dz1^T x ; dW[:, col2:col2+k] (+)= dz2^T x ; db (+)= colsum(dz1)
size_t gte_umma_bwd_weight2_workspace_bytes(int32_t n, int32_t fo, int32_t k) {
  if (n < 0 || fo < 1 || fo > 32 || k < 1 || k > 256) return 0;
  return dw_workspace_bytes(2);
}

int gte_umma_linear_bwd_weight2(const float* dz1, int64_t lddz1, const float* dz2, int64_t lddz2, int32_t fo,
                                const float* x, int64_t ldx, int32_t k, float* dW, int64_t lddw, int32_t col1,
                                int32_t col2, float* db, int accumulate, int32_t n, void* ws, size_t ws_bytes,
                                gte_stream_t stream) {
  if (fo < 1 || fo > 32 || k < 1 || k > 256)
    return fail(GTE_ERR_UNSUPPORTED, "gte_umma_linear_bwd_weight2: fo=%d k=%d unsupported", fo, k);
  GTE_CHECK_ARG(n >= 0 && dW && (n == 0 || (dz1 && dz2 && x)), "gte_umma_linear_bwd_weight2: bad argument");
  GTE_CHECK_ARG(tma_ok(dz1, lddz1) && tma_ok(dz2, lddz2) && tma_ok(x, ldx),
                "gte_umma_linear_bwd_weight2: operands must be 16-byte aligned with ld %% 4 == 0");
  GTE_CHECK_ARG(lddz1 >= fo && lddz2 >= fo && ldx >= k && lddw >= (int64_t)col1 + k && lddw >= (int64_t)col2 + k,
                "gte_umma_linear_bwd_weight2: leading dimension too small");
  const size_t need = gte_umma_bwd_weight2_workspace_bytes(n, fo, k);
  if (ws == nullptr || ws_bytes < need)
    return fail(GTE_ERR_WORKSPACE, "gte_umma_linear_bwd_weight2: workspace %zu < required %zu", ws_bytes, need);
  const bool db_fused = db != nullptr && (k % 128 != 0);
  if (db && !db_fused) return fail(GTE_ERR_UNSUPPORTED, "gte_umma_linear_bwd_weight2: db needs k %% 128 != 0");
  DwArgs a{};
  DwReduceArgs r{};
  a.n = n;
  const int mtiles = (k + (db_fused ? 1 : 0) + 127) / 128;
  a.partial = static_cast<float*>(ws);
  int b_blocked[2] = {0, 0};
  if (n > 0) {
    int rc = dw_make_map(&a.tmA[0], &a.a_blocked[0], x, n, k, ldx, 4);
    if (rc) return rc;
    rc = dw_make_map(&a.tmB[0], &b_blocked[0], dz1, n, fo, lddz1, 1);
    if (rc) return rc;
    rc = dw_make_map(&a.tmB[1], &b_blocked[1], dz2, n, fo, lddz2, 1);
    if (rc) return rc;
  }
  DwGroup& G = a.grp[0];
  G.a = 0; G.nboxes = 2; G.nruns = 2; G.pcol0 = 0; G.ones_b_col = -1; G.ones_a_col = db_fused ? k : -1;
  G.run[0] = DwRun{0, 0, 1, b_blocked[0]};
  G.run[1] = DwRun{1, 0, 1, b_blocked[1]};
  a.max_boxes = 2;
  a.items_per_chunk = 0;
  for (int mt = 0; mt < mtiles; ++mt) {
    a.item_g[a.items_per_chunk] = 0;
    a.item_mt[a.items_per_chunk] = mt;
    ++a.items_per_chunk;
  }
  r.partial = a.partial;
  r.accumulate = accumulate;
  r.nseg = 0;
  r.seg[r.nseg++] = DwSeg{0, k, 0, fo, dW + col1, 1, lddw};   // out[j][o] -> dW[o][col1 + j]
  r.seg[r.nseg++] = DwSeg{0, k, 32, fo, dW + col2, 1, lddw};
  if (db_fused) r.seg[r.nseg++] = DwSeg{k, 1, 0, fo, db, 0, 1};  // ones row: column sums of dz1
  return dw_launch(a, r, as_stream(stream));
}

// Combined-operand forms: the two narrow blocks live side by side in ONE 32-column matrix (columns [0, w) and
// [16, 16+w)).  The tcgen05.mma issue cost does not shrink with N, so the NARROW operand is the A side here (M = 128
// with one real 32-column box; the other three boxes of the A tile stay zero in shared memory and only the first TMEM
// lane quarter is read back) and the WIDE operand is the B side (N up to 256 in ONE MMA): one (group, m-tile) item
// per row chunk instead of two, half the MMA instructions, and the narrow side is one full-row TMA box.
//
// Narrow-x form (input layer): xc[n, 32] = [h | ah]:  dW[:, 0:w] (+)= dz^T xc[:, 0:w] ; dW[:, w:2w] (+)= dz^T xc[:, 16:16+w] ;
// db (+)= colsum(dz) through the free column w of xc (w < 16).
static int dw_narrow_a(const float* narrow, int64_t ldn, const float* wide, int64_t ldwide, int32_t kwide, int32_t n,
                       void* ws, DwArgs& a, DwReduceArgs& r) {
  a.n = n;
  a.partial = static_cast<float*>(ws);
  a.a_real_boxes = 1;
  const int nbw = boxes_of(kwide);
  int b_blocked = 0;
  if (n > 0) {
    int rc = dw_make_map(&a.tmA[0], &a.a_blocked[0], narrow, n, 32, ldn, 1);  // 2-D: one 32-column box per stage
    if (rc) return rc;
    rc = dw_make_map(&a.tmB[0], &b_blocked, wide, n, kwide, ldwide, nbw);
    if (rc) return rc;
  }
  DwGroup& G = a.grp[0];
  G.a = 0; G.nboxes = nbw; G.nruns = 1; G.pcol0 = 0; G.ones_b_col = -1; G.ones_a_col = -1;
  G.run[0] = DwRun{0, 0, nbw, b_blocked};
  a.max_boxes = nbw;
  a.items_per_chunk = 1;
  a.item_g[0] = 0;
  a.item_mt[0] = 0;
  r.partial = a.partial;
  r.nseg = 0;
  return GTE_OK;
}

int gte_umma_linear_bwd_weight_comb(const float* dz, int64_t lddz, int32_t fo, const float* xc, int64_t ldx, int32_t w,
                                    float* dW, int64_t lddw, float* db, int accumulate, int32_t n, void* ws,
                                    size_t ws_bytes, gte_stream_t stream) {
  if (fo < 1 || fo > 256 || w < 1 || w > 16)
    return fail(GTE_ERR_UNSUPPORTED, "gte_umma_linear_bwd_weight_comb: fo=%d w=%d unsupported", fo, w);
  GTE_CHECK_ARG(n >= 0 && dW && (n == 0 || (dz && xc)), "gte_umma_linear_bwd_weight_comb: bad argument");
  GTE_CHECK_ARG(tma_ok(dz, lddz) && tma_ok(xc, ldx), "gte_umma_linear_bwd_weight_comb: operands must be 16-byte aligned with ld %% 4 == 0");
  GTE_CHECK_ARG(lddz >= fo && ldx >= 32 && lddw >= 2 * (int64_t)w, "gte_umma_linear_bwd_weight_comb: leading dimension too small");
  if (db && w >= 16) return fail(GTE_ERR_UNSUPPORTED, "gte_umma_linear_bwd_weight_comb: db needs w < 16 (no free padding column)");
  const size_t need = dw_workspace_bytes(boxes_of(fo));
  if (ws == nullptr || ws_bytes < need)
    return fail(GTE_ERR_WORKSPACE, "gte_umma_linear_bwd_weight_comb: workspace %zu < required %zu", ws_bytes, need);
  DwArgs a{};
  DwReduceArgs r{};
  if (int rc = dw_narrow_a(xc, ldx, dz, lddz, fo, n, ws, a, r)) return rc;
  if (db) a.grp[0].ones_a_col = w;  // row w of the result = column sums of dz
  r.accumulate = accumulate;
  // result[i][o] = sum_rows xc[row][i] * dz[row][o]  ->  dW[o][i] (i < w), dW[o][w + i - 16] (16 <= i < 16 + w)
  r.seg[r.nseg++] = DwSeg{0, w, 0, fo, dW, 1, lddw};
  r.seg[r.nseg++] = DwSeg{16, w, 0, fo, dW + w, 1, lddw};
  if (db) r.seg[r.nseg++] = DwSeg{w, 1, 0, fo, db, 0, 1};
  return dw_launch(a, r, as_stream(stream));
}

// Narrow-dz form (class layer) on dc[n, 32] = [dz | gq]; x [n, k <= 256]:
//   dW[:, col1:col1+k] (+)= dc[:, 0:fo]^T x ; dW[:, col2:col2+k] (+)= dc[:, 16:16+fo]^T x ; db (+)= colsum(dc[:, 0:fo])
// (db through an all-ones padding column of x: needs k % 32 != 0)
int gte_umma_linear_bwd_weight2_comb(const float* dc, int64_t lddc, int32_t fo, const float* x, int64_t ldx, int32_t k,
                                     float* dW, int64_t lddw, int32_t col1, int32_t col2, float* db, int accumulate,
                                     int32_t n, void* ws, size_t ws_bytes, gte_stream_t stream) {
  if (fo < 1 || fo > 16 || k < 1 || k > 256)
    return fail(GTE_ERR_UNSUPPORTED, "gte_umma_linear_bwd_weight2_comb: fo=%d k=%d unsupported", fo, k);
  GTE_CHECK_ARG(n >= 0 && dW && (n == 0 || (dc && x)), "gte_umma_linear_bwd_weight2_comb: bad argument");
  GTE_CHECK_ARG(tma_ok(dc, lddc) && tma_ok(x, ldx), "gte_umma_linear_bwd_weight2_comb: operands must be 16-byte aligned with ld %% 4 == 0");
  GTE_CHECK_ARG(lddc >= 32 && ldx >= k && lddw >= (int64_t)col1 + k && lddw >= (int64_t)col2 + k,
                "gte_umma_linear_bwd_weight2_comb: leading dimension too small");
  const size_t need = dw_workspace_bytes(boxes_of(k));
  if (ws == nullptr || ws_bytes < need)
    return fail(GTE_ERR_WORKSPACE, "gte_umma_linear_bwd_weight2_comb: workspace %zu < required %zu", ws_bytes, need);
  if (db && k % 32 == 0) return fail(GTE_ERR_UNSUPPORTED, "gte_umma_linear_bwd_weight2_comb: db needs k %% 32 != 0");
  DwArgs a{};
  DwReduceArgs r{};
  if (int rc = dw_narrow_a(dc, lddc, x, ldx, k, n, ws, a, r)) return rc;
  if (db) a.grp[0].ones_b_col = k;  // column k of the result = column sums of dc
  r.accumulate = accumulate;
  // result[i][j] = sum_rows dc[row][i] * x[row][j]  ->  dW[i][col1 + j] (i < fo), dW[i - 16][col2 + j] (16 <= i < 16 + fo)
  r.seg[r.nseg++] = DwSeg{0, fo, 0, k, dW + col1, lddw, 1};
  r.seg[r.nseg++] = DwSeg{16, fo, 0, k, dW + col2, lddw, 1};
  if (db) r.seg[r.nseg++] = DwSeg{0, fo, k, 1, db, 1, 0};
  return dw_launch(a, r, as_stream(stream));
}

}  // extern "C"
