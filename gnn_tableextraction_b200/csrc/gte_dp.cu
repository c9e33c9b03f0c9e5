// Data-parallel gradient exchange fused with the optimiser: ONE kernel per step that (1) meets the other ranks on
// flags in NVLink-mapped peer memory, (2) reads every rank's flat gradient buffer through peer pointers (NVLink 5 /
// NVSwitch, P2P loads) and sums them in rank order, (3) applies Adam (with L2 weight decay) to the local replica and
// (4) waits until every peer has finished reading this rank's gradients.
//
// It replaces `ncclAllReduce(flat_grad)` + the Adam kernels behind `loss.backward(); optimizer.step()`
// (/root/reference/src/models/model_train.py:330-332) for the data-parallel run north_star asks for (pages are
// independent, gradients are the only exchange).  The exchange is 424 KB per rank (latency bound): a one-shot
// all-reduce -- every rank reads all peers and reduces redundantly -- is a single NVLink round trip, the sum order is
// the same on every rank (replicas stay bit-identical), and the whole step becomes capturable in one CUDA graph (a
// NCCL call between two graphs plus two eager launches cost ~47 us per step in round 1).
//
// Gradients arrive UN-normalised together with the loss statistics [sum w*nll, sum w, #correct] in the tail of the flat
// buffer (see gte_adam_step): the kernel divides by the global label-weight sum it finds there.
//
// Memory: the flat gradient buffers and the signal pads are torch symmetric-memory allocations (cudaMalloc'ed /
// fabric-exported by PyTorch, rendezvoused once); this file only sees raw device pointers.
#include "gte_common.cuh"

namespace gte {

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_release_gpu(uint32_t* p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// peer memory must not be served from this SM's L1 (it holds last step's values of the same addresses)
__device__ __forceinline__ float4 ld_peer_v4(const float* p) {
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_peer(const float* p) {
  float v;
  asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

constexpr int DP_MAX_WORLD = 16;
constexpr int DP_THREADS = 256;
// signal pad layout (uint32 words, inside this library's region of the pad): [0, W) "gradients of step s ready" written
// by rank r into slot r of every peer; [W, 2W) "done reading" likewise; the local words live in `local` (device memory)
struct DpArgs {
  const float* const* peer_grad;   // device array [world] of device pointers (symmetric memory buffer_ptrs_dev)
  uint32_t* const* peer_signal;    // device array [world] of device pointers to this library's words of each signal pad
  int32_t rank, world;
  int64_t count;                   // parameter floats (multiple of 4)
  int64_t stats_off;               // offset of [sum w*nll, sum w, #correct] in the flat gradient buffer
  float* param;
  float* exp_avg;
  float* exp_avg_sq;
  float* stats_out;                // [4] global statistics
  float lr, b1, b2, eps, wd;
  const float* hparams;            // NULL, or device [lr, b1, b2, eps, wd] read in place of the five values above
  int64_t* step_dev;               // optimiser step counter (incremented here)
  uint32_t* local;                 // [4] device words: 0 = sequence number of the last finished call, 1 = "peers ready" flag,
                                   //     2 = finished-blocks counter
};

__global__ void __launch_bounds__(DP_THREADS) k_dp_allreduce_adam(const DpArgs A) {
  __shared__ float s_den;
  __shared__ float s_hp[5];
  const int tid = threadIdx.x;
  const uint32_t seq = A.local[0] + 1;  // written only by the LAST block of the previous call: every block reads the same value
  const int64_t t = *A.step_dev + 1;    // likewise
  uint32_t* const my_pad = A.peer_signal[A.rank];

  // ---- (1) start barrier: every rank's gradients of this step are complete (stream order on that rank) -------------
  if (blockIdx.x == 0) {
    if (tid < A.world) st_release_sys(A.peer_signal[tid] + A.rank, seq);
    if (tid < A.world)
      while (ld_acquire_sys(my_pad + tid) < seq) __nanosleep(20);
    __syncthreads();
    if (tid == 0) st_release_gpu(A.local + 1, seq);
  } else {
    if (tid == 0)
      while (ld_acquire_gpu(A.local + 1) < seq) __nanosleep(20);
    __syncthreads();
  }

  // ---- (2) one-shot all-reduce in rank order + Adam on the local replica ---------------------------------------------
  // all peer loads of a batch are issued before the first one is used: one NVLink round trip, not `world` of them
  if (tid < 32) {
    float v = 0.f, w3 = 0.f;
    if (tid < A.world) {
      v = ld_peer(A.peer_grad[tid] + A.stats_off + 1);
      if (blockIdx.x == 0) w3 = v;
    }
    // rank-order sum of the `world` values held by lanes 0..world-1 (fixed order: lane 0 adds them one by one)
    float den = 0.f;
    for (int r = 0; r < A.world; ++r) den += __shfl_sync(0xffffffffu, v, r);
    if (tid == 0) s_den = den;
    if (blockIdx.x == 0) {  // global loss statistics for the caller
      float a0 = 0.f, a2 = 0.f;
      if (tid < A.world) {
        a0 = ld_peer(A.peer_grad[tid] + A.stats_off);
        a2 = ld_peer(A.peer_grad[tid] + A.stats_off + 2);
      }
      float s0 = 0.f, s2 = 0.f;
      for (int r = 0; r < A.world; ++r) {
        s0 += __shfl_sync(0xffffffffu, a0, r);
        s2 += __shfl_sync(0xffffffffu, a2, r);
      }
      if (tid == 0) {
        A.stats_out[0] = s0;
        A.stats_out[1] = den;
        A.stats_out[2] = s2;
      }
      (void)w3;
    }
  }
  if (A.hparams && tid < 5) s_hp[tid] = A.hparams[tid];
  __syncthreads();
  const float den = s_den;
  const float lr = A.hparams ? s_hp[0] : A.lr, b1 = A.hparams ? s_hp[1] : A.b1, b2 = A.hparams ? s_hp[2] : A.b2;
  const float eps = A.hparams ? s_hp[3] : A.eps, wd = A.hparams ? s_hp[4] : A.wd;
  if (den > 0.f) {  // a step without any weighted label has no defined gradient: leave the replica untouched
    const float gscale = 1.0f / den;
    // bias corrections exactly as torch.optim.Adam's single-tensor path (double maths, then fp32 use)
    const double bc1 = 1.0 - pow((double)b1, (double)t);
    const double bc2 = 1.0 - pow((double)b2, (double)t);
    const float step_size = (float)((double)lr / bc1);
    const float bc2_sqrt = (float)sqrt(bc2);
    const int64_t n4 = A.count >> 2;
    for (int64_t i = (int64_t)blockIdx.x * DP_THREADS + tid; i < n4; i += (int64_t)gridDim.x * DP_THREADS) {
      float4 q[DP_MAX_WORLD];
#pragma unroll
      for (int r = 0; r < DP_MAX_WORLD; ++r)  // every peer's load in flight before the first add
        if (r < A.world) q[r] = ld_peer_v4(A.peer_grad[r] + 4 * i);
      float4 g = q[0];
#pragma unroll
      for (int r = 1; r < DP_MAX_WORLD; ++r)
        if (r < A.world) { g.x += q[r].x; g.y += q[r].y; g.z += q[r].z; g.w += q[r].w; }
      float4 p = reinterpret_cast<float4*>(A.param)[i];
      float4 m = reinterpret_cast<float4*>(A.exp_avg)[i];
      float4 v = reinterpret_cast<float4*>(A.exp_avg_sq)[i];
      float* gp = &g.x; float* pp = &p.x; float* mp = &m.x; float* vp = &v.x;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float gi = fmaf(wd, pp[e], gp[e] * gscale);      // grad = grad + weight_decay * param
        const float mi = mp[e] + (gi - mp[e]) * (1.0f - b1);   // exp_avg.lerp_(grad, 1 - beta1)
        const float vi = vp[e] * b2 + (1.0f - b2) * gi * gi;
        mp[e] = mi;
        vp[e] = vi;
        pp[e] = pp[e] - step_size * (mi / (sqrtf(vi) / bc2_sqrt + eps));
      }
      reinterpret_cast<float4*>(A.param)[i] = p;
      reinterpret_cast<float4*>(A.exp_avg)[i] = m;
      reinterpret_cast<float4*>(A.exp_avg_sq)[i] = v;
    }
  }

  // ---- (3) end barrier: nobody overwrites its gradient buffer (next step's backward) while a peer still reads it ----
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    const uint32_t prev = atomicAdd(A.local + 2, 1u);
    if (prev == gridDim.x - 1) {  // last block of this rank: all local reads of peer memory are done
      A.local[2] = 0;
      for (int r = 0; r < A.world; ++r) st_release_sys(A.peer_signal[r] + A.world + A.rank, seq);
      for (int r = 0; r < A.world; ++r)
        while (ld_acquire_sys(my_pad + A.world + r) < seq) __nanosleep(20);
      *A.step_dev = t;
      __threadfence();
      A.local[0] = seq;
    }
  }
}

}  // namespace gte

using namespace gte;

static int dp_allreduce_adam(const void* peer_grad_ptrs_dev, const void* peer_signal_ptrs_dev, int32_t rank, int32_t world,
                             int64_t count, int64_t stats_off, float* param, float* exp_avg, float* exp_avg_sq,
                             float* stats_out, float lr, float beta1, float beta2, float eps, float weight_decay,
                             const float* hparams, int64_t* step_dev, uint32_t* local_words, gte_stream_t stream) {
  GTE_CHECK_ARG(world >= 1 && world <= DP_MAX_WORLD && rank >= 0 && rank < world, "gte_dp_allreduce_adam: bad rank/world");
  GTE_CHECK_ARG(count >= 0 && count % 4 == 0 && stats_off >= count, "gte_dp_allreduce_adam: count must be a multiple of 4 and the statistics behind the parameters");
  GTE_CHECK_ARG(peer_grad_ptrs_dev && peer_signal_ptrs_dev && param && exp_avg && exp_avg_sq && stats_out && step_dev && local_words,
                "gte_dp_allreduce_adam: null argument");
  DpArgs a;
  a.peer_grad = static_cast<const float* const*>(peer_grad_ptrs_dev);
  a.peer_signal = static_cast<uint32_t* const*>(peer_signal_ptrs_dev);
  a.rank = rank; a.world = world; a.count = count; a.stats_off = stats_off;
  a.param = param; a.exp_avg = exp_avg; a.exp_avg_sq = exp_avg_sq; a.stats_out = stats_out;
  a.lr = lr; a.b1 = beta1; a.b2 = beta2; a.eps = eps; a.wd = weight_decay; a.hparams = hparams;
  a.step_dev = step_dev; a.local = local_words;
  // all blocks must be resident at once (they wait for block 0): a fraction of the SMs is plenty for <= tens of MB
  int grid = sm_count() / 2;
  const int64_t need = (count / 4 + DP_THREADS - 1) / DP_THREADS;
  if (grid > need) grid = (int)need;
  if (grid < 1) grid = 1;
  k_dp_allreduce_adam<<<grid, DP_THREADS, 0, as_stream(stream)>>>(a);
  GTE_CHECK_LAUNCH("k_dp_allreduce_adam");
  return GTE_OK;
}

extern "C" int gte_dp_allreduce_adam(const void* peer_grad_ptrs_dev, const void* peer_signal_ptrs_dev, int32_t rank,
                                     int32_t world, int64_t count, int64_t stats_off, float* param, float* exp_avg,
                                     float* exp_avg_sq, float* stats_out, float lr, float beta1, float beta2, float eps,
                                     float weight_decay, int64_t* step_dev, uint32_t* local_words, gte_stream_t stream) {
  return dp_allreduce_adam(peer_grad_ptrs_dev, peer_signal_ptrs_dev, rank, world, count, stats_off, param, exp_avg,
                           exp_avg_sq, stats_out, lr, beta1, beta2, eps, weight_decay, nullptr, step_dev, local_words,
                           stream);
}

extern "C" int gte_dp_allreduce_adam_dev(const void* peer_grad_ptrs_dev, const void* peer_signal_ptrs_dev, int32_t rank,
                                         int32_t world, int64_t count, int64_t stats_off, float* param, float* exp_avg,
                                         float* exp_avg_sq, float* stats_out, const float* hparams, int64_t* step_dev,
                                         uint32_t* local_words, gte_stream_t stream) {
  GTE_CHECK_ARG(hparams != nullptr, "gte_dp_allreduce_adam_dev: null hparams");
  return dp_allreduce_adam(peer_grad_ptrs_dev, peer_signal_ptrs_dev, rank, world, count, stats_off, param, exp_avg,
                           exp_avg_sq, stats_out, 0.f, 0.f, 0.f, 0.f, 0.f, hparams, step_dev, local_words, stream);
}
