// Device side of the resident feeder: the slide set lives in HBM as one [total_rows, L] store, and each training batch
// is sampled and packed there (reference: dataset.py:366-393, augmentation dataset.py:375-381).
//
// k_select_rows picks, per bag, the store rows the batch takes: all of the slide's rows, or a uniformly random k-subset
// of them in increasing order (what `sorted(random.sample(range(n), k))` gives, drawn from a Philox stream instead of
// Python's Mersenne Twister).  k_gather_rows then copies those rows back to back into the packed-CSR batch.
#include <algorithm>
#include <cstdint>

#include "common.cuh"

namespace milb200 {
namespace {

constexpr int kSelThreads = 1024;
constexpr int kSelWarps = kSelThreads / 32;

// 64-bit sampling key of one row: a pure function of (seed, epoch, rank, slide id, row), so a slide's subset does not
// depend on the batch it lands in, its position there or the batch size.
__device__ __forceinline__ uint64_t row_key(uint2 seed, uint32_t slide, uint32_t epoch, uint32_t rank, uint32_t row) {
  const uint4 r = philox4x32_10(make_uint4(row, slide, epoch, rank), seed);
  return (static_cast<uint64_t>(r.x) << 32) | r.y;
}

// Exclusive block scan of one uint32 per thread; returns the prefix and writes the block total to *total.
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* warp_tot, uint32_t* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) warp_tot[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    uint32_t w = lane < kSelWarps ? warp_tot[lane] : 0u, winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= o) winc += t;
    }
    if (lane < kSelWarps) warp_tot[lane] = winc - w;
    if (lane == 31) *total = winc;
  }
  __syncthreads();
  const uint32_t out = warp_tot[warp] + inc - v;
  __syncthreads();  // warp_tot is reused by the next call
  return out;
}

// One CTA per bag b: slide ids[b] with n = slide_start[id+1] - slide_start[id] rows keeps k = offsets[b+1] - offsets[b]
// of them; their store row numbers go to src_rows[offsets[b] ..).  For k < n the kept rows are the k smallest
// (key, row) pairs: a radix select over the 64-bit keys (eight 8-bit digits, keys regenerated in every pass, so the
// slide size is not bounded by shared memory) finds the k-th smallest key T, then an ordered compaction keeps every row
// with key < T and, of the rows with key == T, the ones with the lowest row numbers until k rows are kept.
__global__ void __launch_bounds__(kSelThreads) k_select_rows(const int64_t* __restrict__ slide_start,
                                                             const int32_t* __restrict__ ids,
                                                             const int32_t* __restrict__ offsets, uint2 seed,
                                                             uint32_t epoch, uint32_t rank,
                                                             int64_t* __restrict__ src_rows) {
  __shared__ uint32_t hist[256];
  __shared__ uint32_t warp_tot[kSelWarps];
  __shared__ uint32_t s_total;
  __shared__ uint32_t s_digit, s_below;
  const int b = blockIdx.x;
  const int32_t id = ids[b];
  const int64_t s0 = slide_start[id];
  const int64_t n64 = slide_start[id + 1] - s0;
  const int32_t o0 = offsets[b];
  const uint32_t k = static_cast<uint32_t>(offsets[b + 1] - o0);
  int64_t* __restrict__ dst = src_rows + o0;
  if (k == 0 || static_cast<int64_t>(k) > n64) return;  // outside the caller's contract: write nothing
  const uint32_t n = static_cast<uint32_t>(n64);
  if (k == n) {
    for (uint32_t i = threadIdx.x; i < n; i += kSelThreads) dst[i] = s0 + i;
    return;
  }
  const uint32_t slide = static_cast<uint32_t>(id);

  // radix select: after the pass at `shift`, `prefix` holds the top (64 - shift) bits of T and `want` the rank of T
  // among the keys that share them
  uint64_t prefix = 0;
  uint32_t want = k;
  for (int shift = 56; shift >= 0; shift -= 8) {
    const uint64_t hi_mask = shift == 56 ? 0ull : ~0ull << (shift + 8);
    for (int i = threadIdx.x; i < 256; i += kSelThreads) hist[i] = 0u;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < n; i += kSelThreads) {
      const uint64_t key = row_key(seed, slide, epoch, rank, i);
      if ((key & hi_mask) == prefix) atomicAdd(&hist[(key >> shift) & 0xffu], 1u);
    }
    __syncthreads();
    if (threadIdx.x < 32) {  // warp 0: the digit whose cumulative count reaches `want`
      const int lane = threadIdx.x;
      uint32_t c[8], sum = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        c[j] = hist[lane * 8 + j];
        sum += c[j];
      }
      uint32_t inc = sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
      }
      uint32_t run = inc - sum;
      if (run < want && want <= inc) {  // exactly one lane holds the crossing
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (run < want && want <= run + c[j]) {
            s_digit = lane * 8 + j;
            s_below = run;
          }
          run += c[j];
        }
      }
    }
    __syncthreads();
    prefix |= static_cast<uint64_t>(s_digit) << shift;
    want -= s_below;
    __syncthreads();  // s_digit / s_below / hist are rewritten by the next pass
  }
  const uint64_t T = prefix;
  const uint32_t need_eq = want;  // rows with key == T to keep; the rows with key < T number k - need_eq

  // ordered compaction over chunks of kSelThreads rows: one scan of (less-than, equal) counts packed in 16-bit halves
  uint32_t run_lt = 0, run_eq = 0;
  for (uint32_t base = 0; base < n; base += kSelThreads) {
    const uint32_t i = base + threadIdx.x;
    uint32_t lt = 0, eq = 0;
    if (i < n) {
      const uint64_t key = row_key(seed, slide, epoch, rank, i);
      lt = key < T;
      eq = key == T;
    }
    const uint32_t pre = block_exclusive_scan(lt | (eq << 16), warp_tot, &s_total);
    const uint32_t eq_before = run_eq + (pre >> 16);
    if (lt || (eq && eq_before < need_eq)) dst[run_lt + (pre & 0xffffu) + min(eq_before, need_eq)] = s0 + i;
    run_lt += s_total & 0xffffu;
    run_eq += s_total >> 16;
  }
}

constexpr int kGatherThreads = 256;
constexpr int kGatherUnroll = 4;

// dst[r] = store[src_rows[r]] for r < n_rows, one warp per row on a persistent grid; rows of `vecs` 16-byte vectors.
// Streaming loads and stores: the batch is read and written once and should not evict anything from L2.
__global__ void __launch_bounds__(kGatherThreads) k_gather_rows(const uint4* __restrict__ store,
                                                                const int64_t* __restrict__ src_rows, int64_t n_rows,
                                                                int vecs, uint4* __restrict__ dst) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = static_cast<int64_t>(gridDim.x) * (kGatherThreads / 32);
  for (int64_t r = static_cast<int64_t>(blockIdx.x) * (kGatherThreads / 32) + (threadIdx.x >> 5); r < n_rows; r += warps) {
    const uint4* __restrict__ s = store + __ldg(src_rows + r) * vecs;
    uint4* __restrict__ d = dst + r * vecs;
    int v = lane;
#pragma unroll 1
    for (; v + 32 * (kGatherUnroll - 1) < vecs; v += 32 * kGatherUnroll) {
      uint4 t[kGatherUnroll];
#pragma unroll
      for (int u = 0; u < kGatherUnroll; ++u) t[u] = ldg_stream(s + v + 32 * u);
#pragma unroll
      for (int u = 0; u < kGatherUnroll; ++u) __stcs(d + v + 32 * u, t[u]);
    }
#pragma unroll 1
    for (; v < vecs; v += 32) __stcs(d + v, ldg_stream(s + v));
  }
}

}  // namespace
}  // namespace milb200

using namespace milb200;

extern "C" {

int milb200_select_rows(const int64_t* slide_start, const int32_t* ids, const int32_t* offsets, int n_bags,
                        uint64_t seed, uint32_t epoch, uint32_t rank, int64_t* src_rows, void* stream) {
  MIL_CHECK_ARG(slide_start && ids && offsets && src_rows && n_bags >= 0, MILB200_EINVAL, "select_rows: bad arguments");
  if (n_bags == 0) return MILB200_OK;
  const uint2 key = make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
  k_select_rows<<<n_bags, kSelThreads, 0, static_cast<cudaStream_t>(stream)>>>(slide_start, ids, offsets, key, epoch,
                                                                                rank, src_rows);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_gather_rows(const void* store, const int64_t* src_rows, int64_t n_rows, int L, int dtype, void* dst,
                        void* stream) {
  MIL_CHECK_ARG(store && src_rows && dst && n_rows >= 0 && L >= 1, MILB200_EINVAL, "gather_rows: bad arguments");
  MIL_CHECK_ARG(dtype == MILB200_F32 || dtype == MILB200_BF16, MILB200_EUNSUPPORTED,
                "gather_rows: rows must be fp32 or bf16");
  const int64_t row_bytes = static_cast<int64_t>(L) * elem_size(dtype);
  MIL_CHECK_ARG(row_bytes % 16 == 0, MILB200_EUNSUPPORTED, "gather_rows: row of %lld bytes is not a multiple of 16",
                static_cast<long long>(row_bytes));
  MIL_CHECK_ARG(aligned16(store) && aligned16(dst), MILB200_EALIGN, "gather_rows: store and dst must be 16-byte aligned");
  if (n_rows == 0) return MILB200_OK;
  const int warps_per_block = kGatherThreads / 32;
  const int64_t blocks = std::min<int64_t>((n_rows + warps_per_block - 1) / warps_per_block,
                                           static_cast<int64_t>(sm_count()) * (2048 / kGatherThreads));
  k_gather_rows<<<static_cast<unsigned>(blocks), kGatherThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint4*>(store), src_rows, n_rows, static_cast<int>(row_bytes / 16), static_cast<uint4*>(dst));
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

}  // extern "C"
