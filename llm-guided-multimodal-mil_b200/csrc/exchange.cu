// exchange.cu — the data-parallel step's only exchange (train_ddp.py:79,346-348: DDP's gradient all-reduce followed by
// optimizer.step()) as ONE kernel over NVLink / NVSwitch peer memory: in-switch reduction + broadcast of the flat fp32
// gradient buffer (multimem.ld_reduce / multimem.st on a multicast mapping of symmetric memory), then the fused Adam /
// SGD update — no NCCL launch, no separate optimiser launch, ~2 barrier round trips of latency instead of a ring.
//
// The gradient buffers of all ranks are ONE symmetric allocation (same offset on every GPU; torch.distributed's symmetric
// memory supplies the mapping, the multicast pointer and the per-rank signal pads — plumbing).  Protocol per step:
//     barrier A   every rank's backward has written its local gradients
//     phase 1     rank r owns slice r: g = multimem.ld_reduce(slice r)   (the switch adds the W copies)
//                                      multimem.st(slice r, g)           (... and writes the sum into every copy)
//     barrier B   every slice is reduced and broadcast
//     phase 2     every rank: fused optimiser update from its (now identical) local copy
// Every element is reduced exactly once, by its owner, and the same bits are stored to every rank: replicas stay
// bit-identical (bench.py checks a parameter checksum across ranks every run).  The barriers are block-wise flag
// exchanges through the signal pads (block b of rank r <-> block b of every peer; release / acquire at system scope),
// so the grid must be co-resident: it is a few blocks only (the message is 1.6 MB).
#include <algorithm>

#include "common.cuh"

namespace milb200 {

constexpr int XCH_THREADS = 512;
constexpr int XCH_MAX_BLOCKS = 32;       // blocks that take part in the flag barriers (signal-pad slots: blocks x world)
constexpr int XCH_MAX_WORLD = 16;

__device__ __forceinline__ uint32_t cas_release_sys(uint32_t* addr, uint32_t cmp, uint32_t val) {
  uint32_t old;
  asm volatile("atom.global.release.sys.cas.b32 %0, [%1], %2, %3;" : "=r"(old) : "l"(addr), "r"(cmp), "r"(val) : "memory");
  return old;
}
__device__ __forceinline__ uint32_t cas_acquire_sys(uint32_t* addr, uint32_t cmp, uint32_t val) {
  uint32_t old;
  asm volatile("atom.global.acquire.sys.cas.b32 %0, [%1], %2, %3;" : "=r"(old) : "l"(addr), "r"(cmp), "r"(val) : "memory");
  return old;
}

// Block b of this rank meets block b of every peer.  Slot [b*W + src] of rank dst's pad is raised by src and lowered by
// dst; a raise spins until the previous use of the slot has been consumed, so the same slots serve every barrier.
__device__ __forceinline__ void peer_barrier(uint32_t* const* __restrict__ pads, int rank, int world, int slot0) {
  __syncthreads();
  if (threadIdx.x < world) {
    const int peer = threadIdx.x;
    uint32_t* put = pads[peer] + slot0 + blockIdx.x * world + rank;
    uint32_t* get = pads[rank] + slot0 + blockIdx.x * world + peer;
    while (cas_release_sys(put, 0u, 1u) != 0u) {}
    while (cas_acquire_sys(get, 1u, 0u) != 1u) {}
  }
  __syncthreads();
}

__device__ __forceinline__ float4 multimem_ld_reduce_add(const float* mc) {
  float4 v;
  asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(mc) : "memory");
  return v;
}
__device__ __forceinline__ void multimem_st(float* mc, const float4& v) {
  asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};"
               :: "l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// n4 = number of float4 of the (padded) buffer; slice of rank r = float4 [r*chunk4, (r+1)*chunk4)
__global__ void __launch_bounds__(XCH_THREADS)
k_allreduce_update(float* __restrict__ p, float* __restrict__ g_local, float* g_mc, uint32_t* const* __restrict__ pads,
                   const int rank, const int world, const int slot0, float* __restrict__ m, float* __restrict__ v,
                   const int64_t n, const int64_t chunk4, const int optimizer, const float lr, const float b1, const float b2,
                   const float eps, const float wd, const float gscale, const int step,
                   const int32_t* __restrict__ step_dev) {
  // replayable graphs: the step number lives in device memory.  The bias corrections are formed as milb200_adam_step
  // forms them, so the fused and the separate update agree bit for bit.
  const int s = (step_dev != nullptr && optimizer == 0) ? *step_dev : step;
  const float bc1 = optimizer != 0 ? 1.f : adam_bias_correction(b1, s);
  const float bc2 = optimizer != 0 ? 1.f : adam_bias_correction(b2, s);
  peer_barrier(pads, rank, world, slot0);
  {
    const int64_t lo = rank * chunk4, hi = min((n + 3) / 4, lo + chunk4);
    const int64_t stride = static_cast<int64_t>(gridDim.x) * XCH_THREADS;
    int64_t i = lo + static_cast<int64_t>(blockIdx.x) * XCH_THREADS + threadIdx.x;
    for (; i + 3 * stride < hi; i += 4 * stride) {        // four switch round trips in flight per thread
      float4 s[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) s[k] = multimem_ld_reduce_add(g_mc + 4 * (i + k * stride));
#pragma unroll
      for (int k = 0; k < 4; ++k) multimem_st(g_mc + 4 * (i + k * stride), s[k]);
    }
    for (; i < hi; i += stride) {
      const float4 s = multimem_ld_reduce_add(g_mc + 4 * i);
      multimem_st(g_mc + 4 * i, s);
    }
  }
  __threadfence_system();
  peer_barrier(pads, rank, world, slot0);
  if (optimizer < 0) return;       // exchange only: the caller runs its own (wide) optimiser kernel on the summed gradients
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * XCH_THREADS + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * XCH_THREADS) {
    const float pi = p[i];
    const float gi = fmaf(wd, pi, __ldcg(g_local + i) * gscale);
    if (optimizer == 1) {
      p[i] = pi - lr * gi;
    } else {
      const float mi = fmaf(b1, m[i], (1.f - b1) * gi);
      const float vi = fmaf(b2, v[i], (1.f - b2) * gi * gi);
      m[i] = mi;
      v[i] = vi;
      p[i] = pi - (lr / bc1) * (mi / (sqrtf(vi) / sqrtf(bc2) + eps));
    }
  }
}

// Large buffers (the 40 MB buffer of the aggregator trainer): the flag barrier as a one-block kernel on either side of a
// full-width reduce + broadcast kernel (a barrier inside that kernel would tie the grid to the signal-pad slots).
__global__ void __launch_bounds__(32) k_peer_barrier(uint32_t* const* __restrict__ pads, const int rank, const int world, const int slot0) {
  peer_barrier(pads, rank, world, slot0);
}
__global__ void __launch_bounds__(XCH_THREADS)
k_reduce_bcast(float* g_mc, const int rank, const int64_t n, const int64_t chunk4) {
  const int64_t lo = rank * chunk4, hi = min((n + 3) / 4, lo + chunk4);
  const int64_t stride = static_cast<int64_t>(gridDim.x) * XCH_THREADS;
  int64_t i = lo + static_cast<int64_t>(blockIdx.x) * XCH_THREADS + threadIdx.x;
  for (; i + 3 * stride < hi; i += 4 * stride) {
    float4 s[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) s[k] = multimem_ld_reduce_add(g_mc + 4 * (i + k * stride));
#pragma unroll
    for (int k = 0; k < 4; ++k) multimem_st(g_mc + 4 * (i + k * stride), s[k]);
  }
  for (; i < hi; i += stride) {
    const float4 s = multimem_ld_reduce_add(g_mc + 4 * i);
    multimem_st(g_mc + 4 * i, s);
  }
  __threadfence_system();
}

}  // namespace milb200

using namespace milb200;

extern "C" {

/* Replaces DDP's bucketed all-reduce + optimizer.step() (train_ddp.py:79,346-348) for one flat fp32 gradient buffer that
 * lives in symmetric memory: grad_local = this rank's mapping, grad_multicast = the multicast mapping of the same
 * allocation, signal_pads_dev = device array of `world` pointers to the ranks' uint32 signal pads (zero-initialised; at
 * least pad_slot0 + 32 * world entries).  n elements (the allocation must be padded to a multiple of 4 * world
 * elements).  optimizer: 0 Adam (exp_avg / exp_avg_sq updated), 1 SGD, -1 none (exchange only: large buffers, whose
 * update wants a full-width grid, call milb200_adam_step afterwards).  After the call every rank's gradient buffer holds
 * the SUM over ranks and its parameters have taken the step with grad_scale (= 1/world for DDP's average).  step_dev
 * (optional): the Adam step number in device memory, read by the kernel instead of `step` (replayable CUDA graphs).    */
int milb200_allreduce_update_symm(float* param, float* grad_local, void* grad_multicast, void* const* signal_pads_dev,
                                  int pad_slot0, int rank, int world, float* exp_avg, float* exp_avg_sq, int64_t n,
                                  int optimizer, float lr, float beta1, float beta2, float eps, float weight_decay,
                                  float grad_scale, int step, const int32_t* step_dev, void* stream) {
  MIL_CHECK_ARG(param && grad_local && grad_multicast && signal_pads_dev && n > 0, MILB200_EINVAL, "allreduce_update: null pointer");
  MIL_CHECK_ARG(world >= 2 && world <= XCH_MAX_WORLD && rank >= 0 && rank < world && pad_slot0 >= 0, MILB200_EINVAL,
                "allreduce_update: rank %d / world %d", rank, world);
  MIL_CHECK_ARG(optimizer != 0 || (exp_avg && exp_avg_sq && (step >= 1 || step_dev)), MILB200_EINVAL, "allreduce_update: Adam needs its state and step >= 1");
  MIL_CHECK_ARG(aligned16(grad_local) && aligned16(grad_multicast), MILB200_EALIGN, "allreduce_update: buffers must be 16-byte aligned");
  const int64_t n4 = (n + 3) / 4;
  const int64_t chunk4 = (n4 + world - 1) / world;
  if (optimizer < 0 && n > (1 << 20)) {
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    uint32_t* const* pads = reinterpret_cast<uint32_t* const*>(signal_pads_dev);
    k_peer_barrier<<<1, 32, 0, st>>>(pads, rank, world, pad_slot0);
    MIL_LAUNCH_CHECK();
    const int wide = static_cast<int>(std::min<int64_t>(2 * sm_count(), (chunk4 + XCH_THREADS - 1) / XCH_THREADS));
    k_reduce_bcast<<<std::max(wide, 1), XCH_THREADS, 0, st>>>(static_cast<float*>(grad_multicast), rank, n, chunk4);
    MIL_LAUNCH_CHECK();
    k_peer_barrier<<<1, 32, 0, st>>>(pads, rank, world, pad_slot0);
    MIL_LAUNCH_CHECK();
    return MILB200_OK;
  }
  int blocks = static_cast<int>(std::min<int64_t>(XCH_MAX_BLOCKS, std::max<int64_t>(1, (n + XCH_THREADS * 8 - 1) / (XCH_THREADS * 8))));
  k_allreduce_update<<<blocks, XCH_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      param, grad_local, static_cast<float*>(grad_multicast), reinterpret_cast<uint32_t* const*>(signal_pads_dev), rank, world,
      pad_slot0, exp_avg, exp_avg_sq, n, chunk4, optimizer, lr, beta1, beta2, eps, weight_decay, grad_scale, step,
      step_dev);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

}  // extern "C"
