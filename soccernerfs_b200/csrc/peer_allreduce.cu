// Gradient all-reduce over NVLink / NVSwitch peer memory (sm_100a), for the data-parallel training step
// (SURVEY.md 8e: ray-sharded data parallelism; replaces the NCCL all-reduce that DDP issues for the reference,
// NS/engine/trainer.py:382-412 under torch DDP).
//
// Every rank keeps its flat gradient bucket in a cudaMalloc'ed arena whose CUDA-IPC handle is opened by all other
// ranks of the node, so every GPU can load from and store to every other GPU's bucket through NVLink.
// One kernel per rank does the whole all-reduce IN PLACE ("two-shot", pull-reduce + push-broadcast):
//     rank r owns the r-th 1/N of the range.  For every 16-byte element of its part it loads the N copies
//     (N-1 of them over NVLink), adds them in rank order 0..N-1 (so the result is bit-identical everywhere and
//     independent of which rank computed it) and stores the sum into all N buckets (N-1 stores over NVLink).
// Nobody else touches that part of any bucket, so no staging buffer is needed.  NVLink carries (N-1)/N of the
// bucket in each direction per GPU, which is the minimum for an all-reduce without in-switch reduction.
// Cross-GPU ordering uses per-block flag words in the arenas (release/acquire at system scope): a start barrier
// ("every rank's backward has written its gradients") and an end barrier ("every push has landed").  The flags are
// monotonically increasing and the counter lives in device memory, so the kernel can be replayed from a CUDA graph.
#include <math.h>
#include <string.h>

#include "common.cuh"

namespace kp {

constexpr int kPeerMaxWorld = KP_PEER_MAX_WORLD;
constexpr int kPeerMaxBlocks = KP_PEER_MAX_BLOCKS;
constexpr int kPeerThreads = 512;
// signal region layout (uint32 words), at the start of every arena:
//   [0 .. 2*B*W)          flags[phase][block][src_rank]    written by the peers
//   [2*B*W .. 2*B*W + B)  counter[block]                   written by the owner only
//   [2*B*W + B]           error word (non-zero: a barrier timed out)
constexpr int kSigFlags = 2 * kPeerMaxBlocks * kPeerMaxWorld;
constexpr int kSigCounter = kSigFlags;
constexpr int kSigError = kSigFlags + kPeerMaxBlocks;
static_assert((kSigError + 1) * 4 <= KP_PEER_SIGNAL_BYTES, "signal region too small");

struct PeerArgs {
  float* buf[kPeerMaxWorld];      // data region of every rank's arena (index = rank)
  uint32_t* sig[kPeerMaxWorld];   // signal region of every rank's arena
  int rank, world;
  int64_t begin4, n4;             // range in float4 units
  int64_t tail_begin, tail_n;     // < 4 trailing floats, reduced by rank 0
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float4 ld_peer_v4(const float* p) {
  float4 v;
  asm volatile("ld.volatile.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void st_peer_v4(float* p, float4 v) {
  asm volatile("st.volatile.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// All ranks' block `blockIdx.x` meet here.  A bounded spin (tens of seconds) turns a lost peer into an error word plus
// a trapped kernel instead of a hung GPU -- never into a reduction over incomplete buckets.
__device__ __forceinline__ void peer_barrier(const PeerArgs& a, int phase, uint32_t flag) {
  __threadfence_system();
  __syncthreads();
  if ((int)threadIdx.x < a.world) {
    const int slot = (phase * kPeerMaxBlocks + (int)blockIdx.x) * kPeerMaxWorld;
    st_release_sys(a.sig[threadIdx.x] + slot + a.rank, flag);
    const uint32_t* mine = a.sig[a.rank] + slot + threadIdx.x;
    unsigned long long spins = 0;
    while ((int32_t)(ld_acquire_sys(mine) - flag) < 0) {
      if (++spins > (1ull << 27)) {
        // A peer never arrived.  Reducing anyway would sum buckets that are still being written and let the replicas
        // diverge silently, so: record it (kp_peer_error / TrainStep.check_collective_health) and abort the kernel --
        // the host sees a launch failure at its next synchronisation, like a failed NCCL collective.
        a.sig[a.rank][kSigError] = 1u + (uint32_t)phase;
        __threadfence_system();
        __trap();
      }
    }
  }
  __syncthreads();
}

template <int N>
__global__ void __launch_bounds__(kPeerThreads) peer_allreduce_kernel(const __grid_constant__ PeerArgs a) {
  __shared__ uint32_t s_flag;
  uint32_t* counter = a.sig[a.rank] + kSigCounter + blockIdx.x;
  if (threadIdx.x == 0) s_flag = *counter + 1u;
  __syncthreads();
  const uint32_t flag = s_flag;
  peer_barrier(a, 0, flag);  // everybody's gradients are in memory

  const int64_t lo = a.begin4 + a.n4 * a.rank / N, hi = a.begin4 + a.n4 * (a.rank + 1) / N;
  const int64_t stride = (int64_t)gridDim.x * kPeerThreads;
  constexpr int U = N <= 4 ? 4 : 2;  // independent elements in flight per thread: U*N 16-byte loads (<= 64 registers)
  for (int64_t i0 = lo + (int64_t)blockIdx.x * kPeerThreads + threadIdx.x; i0 < hi; i0 += U * stride) {
    float4 v[U][N];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = i0 + u * stride;
      if (i < hi) {
#pragma unroll
        for (int p = 0; p < N; ++p) v[u][p] = ld_peer_v4(a.buf[p] + 4 * i);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = i0 + u * stride;
      if (i < hi) {
        float4 s = v[u][0];
#pragma unroll
        for (int p = 1; p < N; ++p) {
          s.x += v[u][p].x; s.y += v[u][p].y; s.z += v[u][p].z; s.w += v[u][p].w;
        }
#pragma unroll
        for (int p = 0; p < N; ++p) st_peer_v4(a.buf[p] + 4 * i, s);
      }
    }
  }
  if (a.rank == 0 && blockIdx.x == 0 && (int64_t)threadIdx.x < a.tail_n) {
    const int64_t i = a.tail_begin + threadIdx.x;
    float s = 0.f;
    for (int p = 0; p < N; ++p) s += *(volatile float*)(a.buf[p] + i);
    for (int p = 0; p < N; ++p) *(volatile float*)(a.buf[p] + i) = s;
  }
  peer_barrier(a, 1, flag);  // every push has landed
  if (threadIdx.x == 0) *counter = flag;
}

// ---------------------------------------------------------------------------------------------------------------
// Sharded optimizer step fused with its collectives (reduce-scatter -> Adam -> all-gather in ONE kernel):
//   rank r owns the r-th 1/N of a parameter group.  For every 16-byte element of its shard it loads the N ranks'
//   gradients (N-1 over NVLink), sums them in rank order, applies torch.optim.Adam's update to ITS OWN copy of the
//   moments (which therefore only exist for the shard: 1/N of the optimizer state per GPU) and stores the new
//   parameter value into all N ranks' parameter buffers (N-1 stores over NVLink).  Same NVLink bytes as the
//   all-reduce above, but Adam's memory traffic per GPU drops from 7 x the group to 7/N x, and no rank ever
//   materialises the reduced gradient.  Every parameter element is computed by exactly one rank and broadcast, so the
//   replicas stay bit-identical.  Parameters and gradients live in the peer arenas at the same element offsets
//   relative to their region.  Barriers as above: start = "every rank's backward has written its gradients AND no rank
//   still reads the parameters", end = "every pushed parameter has landed".
// ---------------------------------------------------------------------------------------------------------------
struct ShardedAdamArgs {
  float* grad[kPeerMaxWorld];    // gradient region of every rank's arena, at the group's first element
  float* param[kPeerMaxWorld];   // parameter region of every rank's arena, at the group's first element
  uint32_t* sig[kPeerMaxWorld];
  float* m;                      // this rank's moments for its shard: index 0 = first owned element
  float* v;
  int rank, world;
  int64_t n4;                    // group size in float4 units
  const float* hyper_dev;        // optional, see with_hyper_dev
  AdamScalars adam;
  uint8_t* touched[kPeerMaxWorld];  // sparse variant: one byte per 128-byte line of every rank's gradient region
};

template <int N>
__global__ void __launch_bounds__(kPeerThreads) peer_sharded_adam_kernel(const __grid_constant__ ShardedAdamArgs a) {
  __shared__ uint32_t s_flag;
  PeerArgs b;  // barrier view of the same arenas
#pragma unroll
  for (int p = 0; p < kPeerMaxWorld; ++p) b.sig[p] = a.sig[p];
  b.rank = a.rank;
  b.world = a.world;
  uint32_t* counter = a.sig[a.rank] + kSigCounter + blockIdx.x;
  if (threadIdx.x == 0) s_flag = *counter + 1u;
  __syncthreads();
  const uint32_t flag = s_flag;
  peer_barrier(b, 0, flag);
  const AdamScalars adam = with_hyper_dev(a.adam, a.hyper_dev);
  const int64_t lo = a.n4 * a.rank / N, hi = a.n4 * (a.rank + 1) / N;
  const int64_t stride = (int64_t)gridDim.x * kPeerThreads;
  constexpr int U = 2;
  for (int64_t i0 = lo + (int64_t)blockIdx.x * kPeerThreads + threadIdx.x; i0 < hi; i0 += U * stride) {
    float4 g[U][N], pp[U], mm[U], vv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = i0 + u * stride;
      if (i < hi) {
#pragma unroll
        for (int p = 0; p < N; ++p) g[u][p] = ld_peer_v4(a.grad[p] + 4 * i);
        pp[u] = *reinterpret_cast<const float4*>(a.param[a.rank] + 4 * i);
        mm[u] = *reinterpret_cast<const float4*>(a.m + 4 * (i - lo));
        vv[u] = *reinterpret_cast<const float4*>(a.v + 4 * (i - lo));
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = i0 + u * stride;
      if (i < hi) {
        float4 s = g[u][0];
#pragma unroll
        for (int p = 1; p < N; ++p) { s.x += g[u][p].x; s.y += g[u][p].y; s.z += g[u][p].z; s.w += g[u][p].w; }
        adam_update4(scale4(s, adam.grad_scale), pp[u], mm[u], vv[u], adam);
        *reinterpret_cast<float4*>(a.m + 4 * (i - lo)) = mm[u];
        *reinterpret_cast<float4*>(a.v + 4 * (i - lo)) = vv[u];
#pragma unroll
        for (int p = 0; p < N; ++p) st_peer_v4(a.param[p] + 4 * i, pp[u]);
      }
    }
  }
  peer_barrier(b, 1, flag);
  if (threadIdx.x == 0) *counter = flag;
}


// ---------------------------------------------------------------------------------------------------------------
// Sparse variant for HBM-resident plane groups (the 32x preset: 2.3 GB of planes, of which one step's 4096 rays touch
// ~15-30 % of the 128-byte lines of the fine scales).  A dense reduce-scatter pulls (N-1)/N of the group over NVLink
// although most of it is zeros.  Here every rank keeps one "touched" byte per 128-byte line of its gradient region:
//   0 = the line is all zeros (nobody reads it),  1 = the scatter reduced into it this step,  2 = always dense (MLP
//   weights).  The owner of a shard reads its OWN lines unconditionally (the regularisers' gradient for the shard is
//   dense and is written, pre-multiplied by N, only into the owner's bucket) and a peer's line only if that peer marked
//   it.  After the end barrier every rank clears its marked lines outside its own shard (zero the line, flag back to 0),
//   so the bucket needs no memset.  The all-gather of the new parameters stays dense: Adam moves every parameter.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ld_peer_u8(const uint8_t* p) {
  uint32_t v;
  asm volatile("ld.volatile.global.u8 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

template <int N>
__global__ void __launch_bounds__(kPeerThreads) peer_sharded_adam_sparse_kernel(const __grid_constant__ ShardedAdamArgs a) {
  __shared__ uint32_t s_flag;
  PeerArgs b;
#pragma unroll
  for (int p = 0; p < kPeerMaxWorld; ++p) b.sig[p] = a.sig[p];
  b.rank = a.rank;
  b.world = a.world;
  uint32_t* counter = a.sig[a.rank] + kSigCounter + blockIdx.x;
  if (threadIdx.x == 0) s_flag = *counter + 1u;
  __syncthreads();
  const uint32_t flag = s_flag;
  peer_barrier(b, 0, flag);
  const AdamScalars adam = with_hyper_dev(a.adam, a.hyper_dev);
  const int64_t lo = a.n4 * a.rank / N, hi = a.n4 * (a.rank + 1) / N;
  const int64_t stride = (int64_t)gridDim.x * kPeerThreads;
  constexpr int U = N <= 4 ? 4 : 2;  // elements in flight per thread (U*N 16-byte peer loads)
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int64_t i0 = lo + (int64_t)blockIdx.x * kPeerThreads + threadIdx.x; i0 < hi; i0 += U * stride) {
    uint32_t t[U][N];
    float4 s[U], pp[U], mm[U], vv[U];
    // 1. the peers' marks (N-1 bytes per element over NVLink; 8 lanes share a byte)
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = i0 + u * stride;
#pragma unroll
      for (int p = 0; p < N; ++p) t[u][p] = (i < hi && p != a.rank) ? ld_peer_u8(a.touched[p] + (i >> 3)) : 0u;
    }
    // 2. own gradient + optimizer state (local), and the marked lines of the peers
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = i0 + u * stride;
      if (i < hi) {
        s[u] = *reinterpret_cast<const float4*>(a.grad[a.rank] + 4 * i);
        pp[u] = *reinterpret_cast<const float4*>(a.param[a.rank] + 4 * i);
        mm[u] = *reinterpret_cast<const float4*>(a.m + 4 * (i - lo));
        vv[u] = *reinterpret_cast<const float4*>(a.v + 4 * (i - lo));
      }
    }
    float4 g[U][N];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = i0 + u * stride;
#pragma unroll
      for (int p = 0; p < N; ++p) g[u][p] = t[u][p] ? ld_peer_v4(a.grad[p] + 4 * i) : zero;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t i = i0 + u * stride;
      if (i < hi) {
        float4 sum = s[u];
#pragma unroll
        for (int p = 0; p < N; ++p) { sum.x += g[u][p].x; sum.y += g[u][p].y; sum.z += g[u][p].z; sum.w += g[u][p].w; }
        adam_update4(scale4(sum, adam.grad_scale), pp[u], mm[u], vv[u], adam);
        *reinterpret_cast<float4*>(a.m + 4 * (i - lo)) = mm[u];
        *reinterpret_cast<float4*>(a.v + 4 * (i - lo)) = vv[u];
#pragma unroll
        for (int p = 0; p < N; ++p) st_peer_v4(a.param[p] + 4 * i, pp[u]);
      }
    }
  }
  peer_barrier(b, 1, flag);  // every pushed parameter has landed
  if (threadIdx.x == 0) *counter = flag;
}

// Clean-up of this rank's own bucket outside its shard: marked lines back to zero, marks back to 0.  A SEPARATE launch
// after the exchange kernel: the in-kernel barriers pair block k of every rank with block k of the others, so only the
// completion of the whole exchange kernel (all of this rank's blocks past their end barrier, hence all of every peer's
// blocks past their reads) guarantees that nobody still reads the lines being zeroed.
// One thread per line, four lines in flight per thread: the marks are read as consecutive bytes across the warp and only
// marked lines are touched, each with eight 16-byte stores that cover the whole 128-byte line (the first version walked
// every float4 of the bucket with a dependent mark load per step: 0.27 ms for 2.3 GB).
__global__ void __launch_bounds__(kPeerThreads) peer_touched_cleanup_kernel(float* __restrict__ gown, uint8_t* __restrict__ town,
                                                                            int64_t n4, int64_t lo, int64_t hi) {
  const int64_t n_lines = (n4 + 7) >> 3;
  const int64_t stride = (int64_t)gridDim.x * kPeerThreads;
  const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
  constexpr int U = 4;
  for (int64_t l0 = (int64_t)blockIdx.x * kPeerThreads + threadIdx.x; l0 < n_lines; l0 += stride * U) {
    uint8_t f[U];
#pragma unroll
    for (int u = 0; u < U; ++u) f[u] = (l0 + u * stride < n_lines) ? town[l0 + u * stride] : (uint8_t)0;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (f[u] != 1u) continue;
      const int64_t line = l0 + u * stride, j0 = line << 3;
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int64_t j = j0 + q;
        if (j < n4 && !(j >= lo && j < hi)) *reinterpret_cast<float4*>(gown + 4 * j) = zero;
      }
      if (!(j0 >= lo && j0 < hi)) town[line] = 0;  // the mark goes with the line's first float4, like the reduction's own clean-up
    }
  }
}

}  // namespace kp

using namespace kp;

template <int N>
static void launch_sharded_adam(bool sparse, int blocks, cudaStream_t st, const ShardedAdamArgs& a) {
  if (sparse) peer_sharded_adam_sparse_kernel<N><<<blocks, kPeerThreads, 0, st>>>(a);
  else peer_sharded_adam_kernel<N><<<blocks, kPeerThreads, 0, st>>>(a);
}

// The part both sharded launchers share: checks, kernel arguments, the launch for world 1..8 and, for the sparse variant,
// the clean-up.  touched_begin is read by the sparse variant only.
static int peer_sharded_adam_impl(bool sparse, void* const* arenas, int rank, int world, int64_t grad_begin, int64_t param_begin,
                                  int64_t touched_begin, int64_t count, float* exp_avg_shard, float* exp_avg_sq_shard, float lr,
                                  float beta1, float beta2, float eps, float weight_decay, int64_t step, float grad_scale,
                                  const float* hyper_dev, int blocks, void* stream) {
  const char* name = sparse ? "peer_sharded_adam_sparse" : "peer_sharded_adam";
  KP_CHECK(arenas != nullptr && exp_avg_shard != nullptr && exp_avg_sq_shard != nullptr, "%s: NULL argument", name);
  KP_CHECK(world >= 1 && world <= kPeerMaxWorld && rank >= 0 && rank < world, "%s: rank %d / world %d", name, rank, world);
  KP_CHECK(step >= 1, "%s: step is 1-based", name);
  if (count == 0) return 0;
  if (blocks <= 0) blocks = 64;
  KP_CHECK(blocks <= kPeerMaxBlocks, "%s: blocks=%d > %d", name, blocks, kPeerMaxBlocks);
  ShardedAdamArgs a = {};
  for (int p = 0; p < world; ++p) {
    KP_CHECK(arenas[p] != nullptr, "%s: arena %d is NULL", name, p);
    a.sig[p] = reinterpret_cast<uint32_t*>(arenas[p]);
    float* data = reinterpret_cast<float*>(reinterpret_cast<char*>(arenas[p]) + KP_PEER_SIGNAL_BYTES);
    a.grad[p] = data + grad_begin;
    a.param[p] = data + param_begin;
    if (sparse) a.touched[p] = reinterpret_cast<uint8_t*>(data + touched_begin);
  }
  a.m = exp_avg_shard;
  a.v = exp_avg_sq_shard;
  a.rank = rank;
  a.world = world;
  a.n4 = count / 4;
  a.hyper_dev = hyper_dev;
  a.adam = adam_scalars(lr, beta1, beta2, eps, weight_decay, step, grad_scale);
  cudaStream_t st = as_stream(stream);
  switch (world) {  // 1..kPeerMaxWorld, checked above
    case 1: launch_sharded_adam<1>(sparse, blocks, st, a); break;
    case 2: launch_sharded_adam<2>(sparse, blocks, st, a); break;
    case 3: launch_sharded_adam<3>(sparse, blocks, st, a); break;
    case 4: launch_sharded_adam<4>(sparse, blocks, st, a); break;
    case 5: launch_sharded_adam<5>(sparse, blocks, st, a); break;
    case 6: launch_sharded_adam<6>(sparse, blocks, st, a); break;
    case 7: launch_sharded_adam<7>(sparse, blocks, st, a); break;
    case 8: launch_sharded_adam<8>(sparse, blocks, st, a); break;
  }
  if (sparse) {
    kp::g_launches += 1;
    const int64_t lo = a.n4 * rank / world, hi = a.n4 * (rank + 1) / world;
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    peer_touched_cleanup_kernel<<<sms * 8, kPeerThreads, 0, st>>>(a.grad[rank], a.touched[rank], a.n4, lo, hi);
  }
  KP_LAUNCH_CHECK(name);
  return 0;
}

extern "C" int kp_peer_sharded_adam(void* const* arenas, int rank, int world, int64_t grad_begin, int64_t param_begin,
                                    int64_t count, float* exp_avg_shard, float* exp_avg_sq_shard, float lr, float beta1,
                                    float beta2, float eps, float weight_decay, int64_t step, float grad_scale,
                                    const float* hyper_dev, int blocks, void* stream) {
  KP_CHECK(grad_begin >= 0 && param_begin >= 0 && count >= 0 && grad_begin % 4 == 0 && param_begin % 4 == 0 && count % 4 == 0,
           "peer_sharded_adam: offsets / count must be multiples of 4 floats");
  return peer_sharded_adam_impl(false, arenas, rank, world, grad_begin, param_begin, 0, count, exp_avg_shard, exp_avg_sq_shard,
                                lr, beta1, beta2, eps, weight_decay, step, grad_scale, hyper_dev, blocks, stream);
}

extern "C" int kp_peer_sharded_adam_sparse(void* const* arenas, int rank, int world, int64_t grad_begin, int64_t param_begin,
                                           int64_t touched_begin, int64_t count, float* exp_avg_shard, float* exp_avg_sq_shard,
                                           float lr, float beta1, float beta2, float eps, float weight_decay, int64_t step,
                                           float grad_scale, const float* hyper_dev, int blocks, void* stream) {
  KP_CHECK(grad_begin >= 0 && param_begin >= 0 && touched_begin >= 0 && count >= 0 && grad_begin % 32 == 0 && param_begin % 4 == 0 &&
               touched_begin % 4 == 0 && count % 32 == 0,
           "peer_sharded_adam_sparse: the gradient region must start and end on a 128-byte line");
  return peer_sharded_adam_impl(true, arenas, rank, world, grad_begin, param_begin, touched_begin, count, exp_avg_shard,
                                exp_avg_sq_shard, lr, beta1, beta2, eps, weight_decay, step, grad_scale, hyper_dev, blocks, stream);
}

extern "C" int kp_peer_alloc(int64_t data_bytes, void** arena, void* ipc_handle64) {
  KP_CHECK(data_bytes > 0 && arena != nullptr && ipc_handle64 != nullptr, "peer_alloc: bad arguments");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  void* p = nullptr;
  const size_t total = (size_t)KP_PEER_SIGNAL_BYTES + (size_t)data_bytes;
  cudaError_t e = cudaMalloc(&p, total);
  KP_CHECK(e == cudaSuccess, "peer_alloc: cudaMalloc(%zu) failed: %s", total, cudaGetErrorString(e));
  e = cudaMemset(p, 0, total);
  KP_CHECK(e == cudaSuccess, "peer_alloc: cudaMemset failed: %s", cudaGetErrorString(e));
  e = cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(ipc_handle64), p);
  if (e != cudaSuccess) {
    cudaFree(p);
    set_error("peer_alloc: cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
    return 1;
  }
  e = cudaDeviceSynchronize();
  KP_CHECK(e == cudaSuccess, "peer_alloc: sync failed: %s", cudaGetErrorString(e));
  *arena = p;
  return 0;
}

extern "C" int kp_peer_open(const void* ipc_handle64, void** arena) {
  KP_CHECK(ipc_handle64 != nullptr && arena != nullptr, "peer_open: bad arguments");
  cudaIpcMemHandle_t h;
  memcpy(&h, ipc_handle64, sizeof(h));
  cudaError_t e = cudaIpcOpenMemHandle(arena, h, cudaIpcMemLazyEnablePeerAccess);
  KP_CHECK(e == cudaSuccess, "peer_open: cudaIpcOpenMemHandle failed: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" int kp_peer_close(void* arena) {
  cudaError_t e = cudaIpcCloseMemHandle(arena);
  KP_CHECK(e == cudaSuccess, "peer_close: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" int kp_peer_free(void* arena) {
  cudaError_t e = cudaFree(arena);
  KP_CHECK(e == cudaSuccess, "peer_free: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" int kp_peer_error(const void* arena, uint32_t* error_word) {
  KP_CHECK(arena != nullptr && error_word != nullptr, "peer_error: bad arguments");
  cudaError_t e = cudaMemcpy(error_word, reinterpret_cast<const uint32_t*>(arena) + kSigError, 4, cudaMemcpyDeviceToHost);
  KP_CHECK(e == cudaSuccess, "peer_error: %s", cudaGetErrorString(e));
  return 0;
}

extern "C" int kp_peer_allreduce(void* const* arenas, int rank, int world, int64_t begin, int64_t count, int blocks,
                                 void* stream) {
  KP_CHECK(arenas != nullptr, "peer_allreduce: arenas is NULL");
  KP_CHECK(world >= 1 && world <= kPeerMaxWorld && rank >= 0 && rank < world, "peer_allreduce: rank %d / world %d", rank, world);
  KP_CHECK(begin >= 0 && count >= 0 && begin % 4 == 0, "peer_allreduce: begin=%lld must be a multiple of 4", (long long)begin);
  if (count == 0 || world == 1) return 0;
  if (blocks <= 0) blocks = 64;
  KP_CHECK(blocks <= kPeerMaxBlocks, "peer_allreduce: blocks=%d > %d", blocks, kPeerMaxBlocks);
  PeerArgs a;
  for (int p = 0; p < world; ++p) {
    KP_CHECK(arenas[p] != nullptr, "peer_allreduce: arena %d is NULL", p);
    a.sig[p] = reinterpret_cast<uint32_t*>(arenas[p]);
    a.buf[p] = reinterpret_cast<float*>(reinterpret_cast<char*>(arenas[p]) + KP_PEER_SIGNAL_BYTES);
  }
  a.rank = rank;
  a.world = world;
  a.begin4 = begin / 4;
  a.n4 = count / 4;
  a.tail_begin = begin + (count / 4) * 4;
  a.tail_n = count % 4;
  cudaStream_t st = as_stream(stream);
  switch (world) {
    case 2: peer_allreduce_kernel<2><<<blocks, kPeerThreads, 0, st>>>(a); break;
    case 3: peer_allreduce_kernel<3><<<blocks, kPeerThreads, 0, st>>>(a); break;
    case 4: peer_allreduce_kernel<4><<<blocks, kPeerThreads, 0, st>>>(a); break;
    case 5: peer_allreduce_kernel<5><<<blocks, kPeerThreads, 0, st>>>(a); break;
    case 6: peer_allreduce_kernel<6><<<blocks, kPeerThreads, 0, st>>>(a); break;
    case 7: peer_allreduce_kernel<7><<<blocks, kPeerThreads, 0, st>>>(a); break;
    case 8: peer_allreduce_kernel<8><<<blocks, kPeerThreads, 0, st>>>(a); break;
    default: set_error("peer_allreduce: world=%d unsupported", world); return 1;
  }
  KP_LAUNCH_CHECK("peer_allreduce");
  return 0;
}
