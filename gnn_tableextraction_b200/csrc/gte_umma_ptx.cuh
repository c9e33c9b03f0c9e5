// Inline-PTX wrappers for the Blackwell (sm_100a) async machinery used by the tensor-core kernels:
// mbarrier, TMA (cp.async.bulk.tensor), TMEM allocation, tcgen05.mma / commit / ld, proxy fences.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "gte_common.cuh"

namespace gte {

// ------------------------------------------------------------ PTX helpers --
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (!done);
}
// Same wait with exponential nanosleep backoff: for roles that routinely wait a long time (whole warps
// spinning on try_wait steal issue slots from the epilogue warps sharing their scheduler).
__device__ __forceinline__ void mbar_wait_backoff(uint32_t bar, uint32_t parity) {
  uint32_t done, ns = 32;
  while (true) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) break;
    __nanosleep(ns);
    if (ns < 512) ns <<= 1;
  }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int32_t c0, int32_t c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int32_t c0, int32_t c1, int32_t c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_3d(const CUtensorMap* map, int32_t c0, int32_t c1, int32_t c2) {
  asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(reinterpret_cast<uint64_t>(map)),
               "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
// DRAM -> L2 prefetch of one tensor box (no shared memory, no barrier): issued a few k-blocks ahead so that
// the real TMA load finds its data in L2
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* map, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global.tile [%0, {%1, %2}];" ::"l"(reinterpret_cast<uint64_t>(map)),
               "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc], kind::tf32, fp32 accumulate
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// K-major, SWIZZLE_128B operand tile: rows of 128 B, 8-row atoms 1024 B apart (SBO), version 1 (sm_100)
__device__ __forceinline__ uint64_t make_desc_k_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);        // start address, 16-byte units, bits [0,14)
  d |= (uint64_t)1 << 16;                          // leading byte offset (ignored for swizzled K-major), bits [16,30)
  d |= (uint64_t)(1024 >> 4) << 32;                // stride byte offset = 1024 B, bits [32,46)
  d |= (uint64_t)1 << 46;                          // descriptor version, bits [46,48)
  d |= (uint64_t)2 << 61;                          // layout type SWIZZLE_128B, bits [61,64)
  return d;
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// issue-only variant: several TMEM loads can be in flight before one tmem_wait_ld()
__device__ __forceinline__ void tmem_ld_32x32b_x32_nowait(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16_nowait(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Warp-group register re-allocation (all four warps of a warp group execute it together)
template <int N>
__device__ __forceinline__ void setmaxnreg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void setmaxnreg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

// ------------------------------------------------------------ CTA pairs (cta_group::2) ----
// Two CTAs of one cluster (two SMs of a TPC) run ONE tcgen05.mma: each holds 128 rows of A and half of the B rows in
// its own shared memory, and its own 128 TMEM lanes of the accumulator.  The leader CTA (cluster rank 0) issues.
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address of this CTA -> shared::cluster address of the same offset in CTA `rank`
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// Arrive on a barrier that may live in the peer CTA (address from mapa_shared).  Default semantics (.release.cta), as
// CUTLASS's ClusterBarrier::arrive does for the same purpose: what the peer must see was either written through the
// async proxy (TMA, tcgen05) or fenced to it (fence.proxy.async) before this arrive.  The explicit .release.cluster /
// .acquire.cluster forms were measured to cost 60 % of all stall samples of the pair kernel (ncu source page: every
// arrive became MEMBAR.ALL.GPU + ERRBAR + CGAERRBAR, every wait iteration a CCTL.IVALL that invalidates L1).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// waits on barriers whose arrivals come from the peer CTA / from multicast tcgen05.commit: the plain try_wait loops
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) { mbar_wait(bar, parity); }
__device__ __forceinline__ void mbar_wait_cluster_backoff(uint32_t bar, uint32_t parity) { mbar_wait_backoff(bar, parity); }
__device__ __forceinline__ void tmem_alloc_pair(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// completion of all MMAs issued so far by this thread -> one arrive on the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}
// D[tmem, 2 x 128 lanes] (+)= A[2 x 128 rows, smem of each CTA] * B[N rows: N/2 in each CTA], kind::tf32
__device__ __forceinline__ void umma_tf32_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// smem tile -> global, element-wise fp32 ADD performed by the memory system (L2): partial accumulation without
// reading the old value into the SM
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* map, uint32_t src_smem, int32_t c0, int32_t c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(src_smem), "r"(c0), "r"(c1)
               : "memory");
}

__device__ __forceinline__ float tf32_hi(float v) { return __uint_as_float(__float_as_uint(v) & 0xFFFFE000u); }
// round-to-nearest (ties away from zero) to tf32 with two integer ops: adds half an ulp of the 10-bit mantissa and
// clears the 13 low bits -- same result as cvt.rna.tf32.f32 for finite values, at full ALU rate
__device__ __forceinline__ float tf32_rna_fast(float v) { return __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xFFFFE000u); }
// 256-bit global store (one full 32-byte sector per thread)
__device__ __forceinline__ void st_global_v8(float* p, const float* v) {
  asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(v[0]), "f"(v[1]), "f"(v[2]), "f"(v[3]),
               "f"(v[4]), "f"(v[5]), "f"(v[6]), "f"(v[7])
               : "memory");
}
__device__ __forceinline__ float tf32_rna(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}


// MN-major tf32 operand tile built from TMA boxes of [rows(K) x 32 floats(MN)].  For 32-bit MN-major
// operands the only legal shared-memory layout is SWIZZLE_128B_BASE32B (layout type 1, Swizzle<2,5,2>):
// rows of 128 B, 32-byte chunks XOR-ed with (row & 3), K atoms of 4 rows = 512 B (SBO); boxes along MN are
// `lbo_bytes` apart.  The matching TMA mode is CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B.
__device__ __forceinline__ uint64_t make_desc_mn_sw128_32b(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes = 512) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;  // SWIZZLE_128B_BASE32B
  return d;
}

}  // namespace gte

namespace gte {

// ------------------------------------------------------------ TMA stores (smem -> global) ----
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src_smem, int32_t c0, int32_t c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
               "r"(src_smem), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// One 32-row x 32-column accumulator chunk (thread = row) -> dense, 128B-swizzled shared tile [32][32] floats
// -> one asynchronous TMA store (bounds clipped by the tensor map).  `bufs` is 1024-byte aligned and warp private;
// `seq` counts this warp's stores; nbuf (1..4) tiles of 4096 bytes rotate.
__device__ __forceinline__ void epi_store_chunk_tma(uint8_t* bufs, int nbuf, int& seq, const float (&v)[32],
                                                    const CUtensorMap* map, int32_t col0, int32_t row0) {
  const int lane = threadIdx.x & 31;
  uint8_t* buf = bufs + (seq % nbuf) * 4096;  // nbuf store tiles rotate: nbuf - 1 older stores may still be reading theirs
  if (seq >= nbuf) {
    if (lane == 0) {
      if (nbuf == 1) tma_store_wait_read<0>();
      else if (nbuf == 2) tma_store_wait_read<1>();
      else if (nbuf == 3) tma_store_wait_read<2>();
      else tma_store_wait_read<3>();
    }
    __syncwarp();
  }
  float* rowp = reinterpret_cast<float*>(buf) + lane * 32;
#pragma unroll
  for (int q = 0; q < 8; ++q)
    *reinterpret_cast<float4*>(rowp + ((q ^ (lane & 7)) << 2)) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
  fence_proxy_async();
  __syncwarp();
  if (lane == 0) {
    tma_store_2d(map, smem_u32(buf), col0, row0);
    tma_store_commit();
  }
  ++seq;
}

// ------------------------------------------------------------ epilogue store helper ----
// Transposes one 32-row x 32-column accumulator chunk (thread = row, v[] = its 32 columns) through a
// per-warp shared-memory tile and writes it to global memory with 128-bit, row-contiguous stores:
// 8 lanes cover one 128-byte row segment, 4 rows per instruction.  `st` = warp-private [32][EPI_LD] floats.
constexpr int EPI_LD = 36;  // 16-byte aligned rows; STS.128 / LDS.128 below are bank-conflict free
__device__ __forceinline__ void epi_store_chunk(float* st, const float (&v)[32], float* out, int64_t ld, int rows_valid,
                                                int cols_valid, bool vec_ok) {
  const int lane = threadIdx.x & 31;
  __syncwarp();
#pragma unroll
  for (int q = 0; q < 8; ++q)
    *reinterpret_cast<float4*>(st + lane * EPI_LD + q * 4) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
  __syncwarp();
  const int r_in = lane >> 3, c4 = (lane & 7) * 4;
  if (c4 >= cols_valid) return;
#pragma unroll
  for (int it = 0; it < 8; ++it) {
    const int row = it * 4 + r_in;
    if (row >= rows_valid) break;
    const float4 val = *reinterpret_cast<const float4*>(st + row * EPI_LD + c4);
    float* p = out + (int64_t)row * ld + c4;
    if (vec_ok) {
      *reinterpret_cast<float4*>(p) = val;  // may touch padding columns [N, ld): never interpreted
    } else {
      p[0] = val.x;
      if (c4 + 1 < cols_valid) p[1] = val.y;
      if (c4 + 2 < cols_valid) p[2] = val.z;
      if (c4 + 3 < cols_valid) p[3] = val.w;
    }
  }
}

// ------------------------------------------------------------ host: TMA descriptors ----
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<PFN_encodeTiled>(p);
  return fn;
}

// 2-D fp32 row-major [rows, cols], leading dimension ld floats; box = box_cols (<= 32) x box_rows, SWIZZLE_128B,
// out-of-bounds elements read as zero.
static inline int make_tmap_2d(CUtensorMap* m, const float* ptr, int64_t rows, int64_t cols, int64_t ld, int box_cols,
                               int box_rows, CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) return fail(GTE_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)ld * 4};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(GTE_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return GTE_OK;
}

// The same row-major matrix seen as [column block][row][32 columns]: ONE request then brings `box_blocks` 32-column
// blocks of `box_rows` rows, laid out block after block in shared memory -- exactly the MN-major operand tile the
// weight-gradient kernel builds from 2-D boxes, at a fraction of the TMA requests (the unit handles one request per
// ~160-220 clocks, which bounded that kernel at 11 boxes per stage).  Needs ld >= 32 * ceil(cols / 32): the last block
// is read to its full width (padding columns of the row; they only reach outputs nobody reads).  Blocks past the last
// one are zero filled.
static inline int make_tmap_3d_blocks(CUtensorMap* m, const float* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows,
                                      int box_blocks, CUtensorMapSwizzle swizzle) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) return fail(GTE_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  cuuint64_t gdim[3] = {32, (cuuint64_t)rows, (cuuint64_t)((cols + 31) / 32)};
  cuuint64_t gstr[2] = {(cuuint64_t)ld * 4, 128};
  cuuint32_t box[3] = {32, (cuuint32_t)box_rows, (cuuint32_t)box_blocks};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(ptr), gdim, gstr, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(GTE_ERR_CUDA, "cuTensorMapEncodeTiled(3d) failed (%d)", (int)r);
  return GTE_OK;
}

}  // namespace gte
