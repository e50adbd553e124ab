// pool.cu — ragged segmented softmax + attention-weighted instance sum over CSR bag offsets,
// forward and backward (replaces F.softmax(A, dim=1) and torch.matmul(A, x), model/dim1/ABMIL.py:56-59,
// and their autograd).  Bandwidth-bound: X is streamed exactly once per pass with 128-bit loads.
//
// Forward = ONE persistent kernel: two CTAs per SM, each owning a contiguous slab of the packed rows and
// walking the bag pieces inside it.  For every piece it computes a local (max, sum, weighted accumulator)
// softmax partial; a bag that lies inside one slab is finished on the spot, a bag that spans slabs is
// finished by whichever CTA publishes its last piece (per-bag arrival counter), which folds the partials
// in piece order, so the result is deterministic.
#include <algorithm>
#include <cfloat>
#include <type_traits>

#include "common.cuh"

namespace milb200 {

constexpr int POOL_THREADS = 256;
constexpr int POOL_WARPS = POOL_THREADS / 32;
constexpr int POOL_BLK = 16;         // rows a warp owns at a time (one score per lane 0..15)
constexpr int POOL_MIN_SLAB = 256;   // rows per CTA at least (512 KB of bf16 x 1024)
constexpr int POOL_MAX_DOTS = 8;     // row dots per row of the row-dot forward (widest NC bucket)
constexpr size_t POOL_SMEM_LIMIT = 227 * 1024;  // dynamic + static shared memory of one CTA (sm_100)

template <typename T> __device__ __forceinline__ float exp_t(float x);
template <> __device__ __forceinline__ float exp_t<float>(float x) { return expf(x); }
template <> __device__ __forceinline__ float exp_t<__nv_bfloat16>(float x) { return __expf(x); }

// the VN floats of a staged dot vector that line up with 16-byte vector `vec` of a row, from shared memory; 0 past the
// row (vec >= V)
template <int VN>
__device__ __forceinline__ void dm_chunk(const float* dms, int vec, int V, float* d) {
#pragma unroll
  for (int k = 0; k < VN; k += 4) {
    const float4 q = vec < V ? *reinterpret_cast<const float4*>(dms + vec * VN + k) : make_float4(0.f, 0.f, 0.f, 0.f);
    d[k] = q.x; d[k + 1] = q.y; d[k + 2] = q.z; d[k + 3] = q.w;
  }
}

struct PiecePartial {  // published per (CTA, bag) piece
  float m, l;
  int argmax;  // index within the bag
  int pad;
};

// Persistent layout: CTA c owns the contiguous row slab [c*slab, (c+1)*slab) and walks the bag pieces inside it.
// Per piece: (1) block max/argmax of the piece's scores, (2) every warp streams 16-row blocks of the piece — lane j
// owns the 16-byte vectors j, j+32, ... of a row, two rows in flight — accumulating exp(s_i - max) * x_i in registers,
// (3) one shared-memory fold across the 8 warps.  A bag inside one slab is finished on the spot; a bag spanning
// slabs is finished by the CTA that publishes its last piece, folding the partials in piece order (deterministic).
//
// NC > 0 (row dots): the caller already knows what the upstream gradient is made of, so the pass also writes C dots per
// row, dots[i * C + c] = v_bc . x_i, on the rows it has in registers anyway; the backward then forms the score gradients
// without reading X again.  v_bc[l] = dv[b * dv_bag_stride + c * L + l] * (col_scale ? col_scale[b * L + l] : 1):
//   - the _rowdot form is C = 1 with dv = dM (stride L, no scale): dots[i] = dM_b . x_i;
//   - the _headdot form takes dv = a linear head's W [C, L] (stride 0) and col_scale = the head's dropout scale s_b, so
//     that dM_b . x_i = sum_c dz_bc dots[i * C + c] once the head's dz exists.
// NC is C rounded up to a bucket {1, 2, 4, 8}; vectors C..NC-1 are staged as zeros and their dots are not written.  The
// vectors are staged once per piece in shared memory next to `red`; one shared-memory read of a chunk serves both rows of
// the two-row loop.  Each dot is accumulated exactly as k_pool_bwd accumulates dM_b . x_i (j then k ascending, masked
// lanes included in the two-row loop, the same warp_sum), so the C = 1 gradients do not change by a bit.
template <typename T, int NV, int NC>
__device__ __forceinline__ void
pool_fwd_body(const T* __restrict__ X, const float* __restrict__ scores, const int32_t* __restrict__ offsets, int B,
              int64_t total_n, int L, int V, int64_t slab, float* __restrict__ M, T* __restrict__ M_lowp,
              int32_t* __restrict__ argmax_out, float* __restrict__ lse_out, float* __restrict__ ws_acc,
              PiecePartial* __restrict__ ws_ml, unsigned int* __restrict__ counters, int normalize,
              const float* __restrict__ dv, int64_t dv_bag_stride, const float* __restrict__ col_scale, int C,
              float* __restrict__ dots) {
  constexpr int VN = Vec16<T>::N;
  constexpr int ND = NC > 0 ? NC : 1;           // (array extent; no dot is formed when NC == 0)
  extern __shared__ __align__(16) float red[];  // [POOL_WARPS][L], then (NC > 0) the dot vectors [NC][L]
  float* dms = red + static_cast<int64_t>(POOL_WARPS) * L;
  __shared__ float wred_v[POOL_WARPS];
  __shared__ int wred_i[POOL_WARPS];
  __shared__ float piece_m, piece_l;
  __shared__ int piece_arg, is_last;

  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int64_t cta = blockIdx.x;
  const int64_t r0 = cta * slab;
  if (r0 >= total_n) return;
  const int64_t r1 = (r0 + slab < total_n) ? r0 + slab : total_n;
  const uint4* Xv = reinterpret_cast<const uint4*>(X);

  int b = find_bag(offsets, B, r0);
  while (b > 0 && __ldg(offsets + b - 1) == r0) --b;   // empty bags that sit exactly at the start of this slab
  for (; b < B; ++b) {
    const int64_t ob = __ldg(offsets + b), oe = __ldg(offsets + b + 1);
    const bool empty = oe == ob;
    if (ob >= r1 && !(empty && r1 == total_n)) break;  // (trailing empty bags belong to the last CTA)
    const int64_t s0 = ob > r0 ? ob : r0, s1 = oe < r1 ? oe : r1;
    const int nseg = static_cast<int>(s1 - s0);
    if (nseg <= 0) {
      // an empty bag has no rows, so no piece would ever write its outputs: the CTA whose slab contains its position does
      // (pooled vector 0, argmax -1, lse -inf; torch gives NaN for a softmax over nothing — the reference never builds one)
      if (empty && ob >= r0) {
        for (int c = t; c < L; c += POOL_THREADS) {
          M[static_cast<int64_t>(b) * L + c] = 0.f;
          if (M_lowp) M_lowp[static_cast<int64_t>(b) * L + c] = from_f32<T>(0.f);
        }
        if (t == 0) {
          if (argmax_out) argmax_out[b] = -1;
          if (lse_out) lse_out[b] = -INFINITY;
        }
      }
      continue;
    }
    // read after the barrier of (1); the previous piece ended with one
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      float* dst = dms + static_cast<int64_t>(c) * L;
      const float* src = dv + static_cast<int64_t>(b) * dv_bag_stride + static_cast<int64_t>(c) * L;
      if (c >= C) {
        for (int l = t; l < L; l += POOL_THREADS) dst[l] = 0.f;
      } else if (col_scale) {
        const float* cs = col_scale + static_cast<int64_t>(b) * L;
        for (int l = t; l < L; l += POOL_THREADS) dst[l] = __ldg(src + l) * __ldg(cs + l);
      } else {
        for (int l = t; l < L; l += POOL_THREADS) dst[l] = __ldg(src + l);  // (independent loads: the loop unrolls)
      }
    }

    // ---- (1) piece max and first argmax ----
    float pm = 0.f;
    if (scores) {
      float mv = -FLT_MAX;
      int mi = 0x7fffffff;
      for (int i = t; i < nseg; i += POOL_THREADS) {
        float v = __ldg(scores + s0 + i);
        if (v > mv) { mv = v; mi = i; }  // i ascends: the first maximum is kept
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        float ov = __shfl_xor_sync(0xffffffffu, mv, o);
        int oi = __shfl_xor_sync(0xffffffffu, mi, o);
        if (ov > mv || (ov == mv && oi < mi)) { mv = ov; mi = oi; }
      }
      if (lane == 0) { wred_v[warp] = mv; wred_i[warp] = mi; }
      __syncthreads();
      if (t == 0) {
        float bv = wred_v[0];
        int bi = wred_i[0];
        for (int w = 1; w < POOL_WARPS; ++w)
          if (wred_v[w] > bv || (wred_v[w] == bv && wred_i[w] < bi)) { bv = wred_v[w]; bi = wred_i[w]; }
        piece_m = bv;
        piece_arg = bi + static_cast<int>(s0 - ob);
      }
      __syncthreads();
      pm = piece_m;
    } else if (t == 0) {
      piece_m = 0.f;
      piece_arg = 0;
    }

    // ---- (2) stream the piece ----
    float acc[NV][VN];
#pragma unroll
    for (int j = 0; j < NV; ++j)
#pragma unroll
      for (int k = 0; k < VN; ++k) acc[j][k] = 0.f;
    float lsum = 0.f;
    const int nblk = (nseg + POOL_BLK - 1) / POOL_BLK;
    for (int blk = warp; blk < nblk; blk += POOL_WARPS) {
      const int64_t rb = s0 + static_cast<int64_t>(blk) * POOL_BLK;
      const int nr = (nseg - blk * POOL_BLK < POOL_BLK) ? nseg - blk * POOL_BLK : POOL_BLK;
      float e = 0.f;
      if (lane < nr) e = scores ? exp_t<T>(__ldg(scores + rb + lane) - pm) : 1.f;
      lsum += e;
      int i = 0;
      for (; i + 1 < nr; i += 2) {
        uint4 v0[NV], v1[NV];
#pragma unroll
        for (int j = 0; j < NV; ++j) {
          const int vec = lane + j * 32;
          v0[j] = (vec < V) ? ldg_stream(Xv + (rb + i) * V + vec) : make_uint4(0, 0, 0, 0);
          v1[j] = (vec < V) ? ldg_stream(Xv + (rb + i + 1) * V + vec) : make_uint4(0, 0, 0, 0);
        }
        const float w0 = __shfl_sync(0xffffffffu, e, i), w1 = __shfl_sync(0xffffffffu, e, i + 1);
        float g0[ND], g1[ND];
#pragma unroll
        for (int c = 0; c < ND; ++c) g0[c] = g1[c] = 0.f;
#pragma unroll
        for (int j = 0; j < NV; ++j) {
          if constexpr (NC <= 1) {
            // no dots, or one: the staged chunk is held across both rows, each row unpacked once into the same registers
            float f[VN], d[VN];
            if (NC == 1) dm_chunk<VN>(dms, lane + j * 32, V, d);  // one read serves both rows
            Vec16<T>::unpack(v0[j], f);
#pragma unroll
            for (int k = 0; k < VN; ++k) acc[j][k] = fmaf(w0, f[k], acc[j][k]);
            if (NC == 1)
#pragma unroll
              for (int k = 0; k < VN; ++k) g0[0] = fmaf(d[k], f[k], g0[0]);
            Vec16<T>::unpack(v1[j], f);
#pragma unroll
            for (int k = 0; k < VN; ++k) acc[j][k] = fmaf(w1, f[k], acc[j][k]);
            if (NC == 1)
#pragma unroll
              for (int k = 0; k < VN; ++k) g1[0] = fmaf(d[k], f[k], g1[0]);
          } else {
            // several: both rows unpacked once, the staged vectors streamed past them one chunk at a time (holding NC
            // chunks instead would cost NC * VN registers)
            float f0[VN], f1[VN];
            Vec16<T>::unpack(v0[j], f0);
#pragma unroll
            for (int k = 0; k < VN; ++k) acc[j][k] = fmaf(w0, f0[k], acc[j][k]);
            Vec16<T>::unpack(v1[j], f1);
#pragma unroll
            for (int k = 0; k < VN; ++k) acc[j][k] = fmaf(w1, f1[k], acc[j][k]);
#pragma unroll
            for (int c = 0; c < NC; ++c) {
              float d[VN];
              dm_chunk<VN>(dms + static_cast<int64_t>(c) * L, lane + j * 32, V, d);  // one read serves both rows
#pragma unroll
              for (int k = 0; k < VN; ++k) g0[c] = fmaf(d[k], f0[k], g0[c]);
#pragma unroll
              for (int k = 0; k < VN; ++k) g1[c] = fmaf(d[k], f1[k], g1[c]);
            }
          }
        }
        if constexpr (NC == 1) {  // (C == 1)
          g0[0] = warp_sum(g0[0]);
          g1[0] = warp_sum(g1[0]);
          if (lane == 0) { dots[rb + i] = g0[0]; dots[rb + i + 1] = g1[0]; }
        } else if constexpr (NC > 1) {
          float o0 = 0.f, o1 = 0.f;  // lane c writes dot c of both rows
#pragma unroll
          for (int c = 0; c < NC; ++c) {
            g0[c] = warp_sum(g0[c]);
            g1[c] = warp_sum(g1[c]);
            if (lane == c) { o0 = g0[c]; o1 = g1[c]; }
          }
          if (lane < C) { dots[(rb + i) * C + lane] = o0; dots[(rb + i + 1) * C + lane] = o1; }
        }
      }
      if (i < nr) {
        const float w0 = __shfl_sync(0xffffffffu, e, i);
        float g0[ND];
#pragma unroll
        for (int c = 0; c < ND; ++c) g0[c] = 0.f;
#pragma unroll
        for (int j = 0; j < NV; ++j) {
          const int vec = lane + j * 32;
          if (vec < V) {
            float f[VN];
            Vec16<T>::unpack(ldg_stream(Xv + (rb + i) * V + vec), f);
#pragma unroll
            for (int k = 0; k < VN; ++k) acc[j][k] = fmaf(w0, f[k], acc[j][k]);
#pragma unroll
            for (int c = 0; c < NC; ++c) {
              float d[VN];
              dm_chunk<VN>(dms + static_cast<int64_t>(c) * L, vec, V, d);
#pragma unroll
              for (int k = 0; k < VN; ++k) g0[c] = fmaf(d[k], f[k], g0[c]);
            }
          }
        }
        if constexpr (NC == 1) {
          g0[0] = warp_sum(g0[0]);
          if (lane == 0) dots[rb + i] = g0[0];
        } else if constexpr (NC > 1) {
          float o0 = 0.f;
#pragma unroll
          for (int c = 0; c < NC; ++c) {
            g0[c] = warp_sum(g0[c]);
            if (lane == c) o0 = g0[c];
          }
          if (lane < C) dots[(rb + i) * C + lane] = o0;
        }
      }
    }
    lsum = warp_sum(lsum);

    // ---- (3) fold the 8 warps in fixed order ----
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const int vec = lane + j * 32;
      if (vec < V) {
        float* dst = red + static_cast<int64_t>(warp) * L + vec * VN;
#pragma unroll
        for (int k = 0; k < VN; k += 4) *reinterpret_cast<float4*>(dst + k) = make_float4(acc[j][k], acc[j][k + 1], acc[j][k + 2], acc[j][k + 3]);
      }
    }
    if (lane == 0) wred_v[warp] = lsum;
    __syncthreads();
    for (int c = t; c < L; c += POOL_THREADS) {
      float a = red[c];
#pragma unroll
      for (int g = 1; g < POOL_WARPS; ++g) a += red[static_cast<int64_t>(g) * L + c];
      red[c] = a;
    }
    if (t == 0) {
      float l = 0.f;
      for (int w = 0; w < POOL_WARPS; ++w) l += wred_v[w];
      piece_l = l;
    }
    __syncthreads();

    const int64_t c_first = ob / slab, c_last = (oe - 1) / slab;
    const int pieces = static_cast<int>(c_last - c_first + 1);
    if (pieces == 1) {
      const float inv = normalize ? 1.f / piece_l : 1.f;
      for (int c = t; c < L; c += POOL_THREADS) {
        float mval = red[c] * inv;
        M[static_cast<int64_t>(b) * L + c] = mval;
        if (M_lowp) M_lowp[static_cast<int64_t>(b) * L + c] = from_f32<T>(mval);
      }
      if (t == 0) {
        if (argmax_out) argmax_out[b] = piece_arg;
        if (lse_out) lse_out[b] = piece_m + logf(piece_l);
      }
    } else {
      const int64_t slot = cta + b;  // unique per (CTA, bag) piece, consecutive along the row order
      for (int c = t; c < L; c += POOL_THREADS) ws_acc[slot * L + c] = red[c];
      if (t == 0) {
        PiecePartial pp;
        pp.m = piece_m; pp.l = piece_l; pp.argmax = piece_arg; pp.pad = 0;
        ws_ml[slot] = pp;
      }
      __threadfence();
      __syncthreads();
      if (t == 0) {
        unsigned int old = atomicAdd(counters + b, 1u);
        is_last = (old == static_cast<unsigned int>(pieces - 1));
      }
      __syncthreads();
      if (is_last) {
        __threadfence();
        const int64_t slot0 = c_first + b;
        float gm = -FLT_MAX;
        int garg = 0;
        for (int p = 0; p < pieces; ++p) {
          PiecePartial pp = ws_ml[slot0 + p];
          if (pp.m > gm) { gm = pp.m; garg = pp.argmax; }
        }
        float gl = 0.f;
        for (int p = 0; p < pieces; ++p) {
          PiecePartial pp = ws_ml[slot0 + p];
          gl += pp.l * exp_t<T>(pp.m - gm);
        }
        const float inv = normalize ? 1.f / gl : 1.f;
        for (int c = t; c < L; c += POOL_THREADS) {
          float a = 0.f;
          int p = 0;
          for (; p + 4 <= pieces; p += 4) {  // four independent loads in flight; the fold order stays p ascending
            float x0 = __ldcg(ws_acc + (slot0 + p) * L + c), x1 = __ldcg(ws_acc + (slot0 + p + 1) * L + c);
            float x2 = __ldcg(ws_acc + (slot0 + p + 2) * L + c), x3 = __ldcg(ws_acc + (slot0 + p + 3) * L + c);
            a = fmaf(exp_t<T>(ws_ml[slot0 + p].m - gm), x0, a);
            a = fmaf(exp_t<T>(ws_ml[slot0 + p + 1].m - gm), x1, a);
            a = fmaf(exp_t<T>(ws_ml[slot0 + p + 2].m - gm), x2, a);
            a = fmaf(exp_t<T>(ws_ml[slot0 + p + 3].m - gm), x3, a);
          }
          for (; p < pieces; ++p) a = fmaf(exp_t<T>(ws_ml[slot0 + p].m - gm), __ldcg(ws_acc + (slot0 + p) * L + c), a);
          float mval = a * inv;
          M[static_cast<int64_t>(b) * L + c] = mval;
          if (M_lowp) M_lowp[static_cast<int64_t>(b) * L + c] = from_f32<T>(mval);
        }
        if (t == 0) {
          if (argmax_out) argmax_out[b] = garg;
          if (lse_out) lse_out[b] = gm + logf(gl);
        }
      }
    }
    __syncthreads();  // smem (red, wred_*, piece_*) is reused by the next piece
  }
}

#define MIL_POOL_FWD_PARAMS                                                                                             \
  const T *__restrict__ X, const float *__restrict__ scores, const int32_t *__restrict__ offsets, int B,               \
      int64_t total_n, int L, int V, int64_t slab, float *__restrict__ M, T *__restrict__ M_lowp,                      \
      int32_t *__restrict__ argmax_out, float *__restrict__ lse_out, float *__restrict__ ws_acc,                       \
      PiecePartial *__restrict__ ws_ml, unsigned int *__restrict__ counters, int normalize
#define MIL_POOL_FWD_ARGS \
  X, scores, offsets, B, total_n, L, V, slab, M, M_lowp, argmax_out, lse_out, ws_acc, ws_ml, counters, normalize

template <typename T, int NV>
__global__ void __launch_bounds__(POOL_THREADS) k_pool_fwd(MIL_POOL_FWD_PARAMS) {
  pool_fwd_body<T, NV, 0>(MIL_POOL_FWD_ARGS, nullptr, 0, nullptr, 0, nullptr);
}

// The row dots cost registers (the staged chunk, two dots per vector).  Where the plain kernel runs two CTAs per SM
// (<= 128 registers: bf16 NV <= 6, fp32 NV <= 8) the one-dot kernel is held to two as well, so that the HBM-bound pass
// keeps its bytes in flight; the wider instantiations run one CTA per SM either way.  More dots per row keep two CTAs
// only where they fit in 128 registers without spilling (ptxas -v, CUDA 12.9); elsewhere they run one CTA per SM.
template <typename T, int NV, int NC>
constexpr int pool_fwd_rowdot_min_blocks() {
  constexpr bool two = sizeof(T) == 2 ? NV <= 6 : NV <= 8;
  constexpr bool fits = NC == 1 || (NC <= 4 && NV <= (sizeof(T) == 2 ? 4 : 6)) || (NC == 8 && NV <= (sizeof(T) == 2 ? 1 : 4));
  return two && fits ? 2 : 1;
}

template <typename T, int NV, int NC>
__global__ void __launch_bounds__(POOL_THREADS, pool_fwd_rowdot_min_blocks<T, NV, NC>())
k_pool_fwd_rowdot(MIL_POOL_FWD_PARAMS, const float* __restrict__ dv, int64_t dv_bag_stride,
                  const float* __restrict__ col_scale, int C, float* __restrict__ dots) {
  pool_fwd_body<T, NV, NC>(MIL_POOL_FWD_ARGS, dv, dv_bag_stride, col_scale, C, dots);
}
#undef MIL_POOL_FWD_PARAMS
#undef MIL_POOL_FWD_ARGS

// ---- backward ------------------------------------------------------------------------------------
// stats[b] = (lse_b, dM_b . M_b): softmax statistics are recomputed from the scores, not stored.
// SWEEP (row dots written by the row-dot forward): the same CTA then sweeps its bag and writes the score gradients and
// attention weights without reading X, from g_i = dM_b . x_i:
//   - dz == NULL (_rowdot): g_i = rowdot[i], and the expressions are k_pool_bwd's on the same floats;
//   - dz [B, C] (_headdot): g_i = sum_c dz[b, c] * rowdot[i * C + c], c ascending.
// A template flag, so that the statistics-only kernel keeps its registers (two 1024-thread CTAs per SM).
template <bool SWEEP>
__global__ void __launch_bounds__(1024)
k_pool_bwd_stats(const float* __restrict__ scores, const int32_t* __restrict__ offsets, int L,
                 const float* __restrict__ dM, const float* __restrict__ M, float2* __restrict__ stats,
                 const float* __restrict__ rowdot, float* __restrict__ dscores, float* __restrict__ attn,
                 const float* __restrict__ dz = nullptr, int C = 1) {
  __shared__ float red[32];
  __shared__ float bc;
  __shared__ float dzs[POOL_MAX_DOTS];
  __shared__ float2 bag_stats;
  const int b = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5, nt = blockDim.x, nw = blockDim.x >> 5;
  const int64_t ob = offsets[b], oe = offsets[b + 1];
  // the bag's scores stay in registers between the two passes (up to 8 per thread; longer bags re-read from L2)
  constexpr int KEEP = 8;
  float sc[KEEP];
  float mx = -FLT_MAX;
#pragma unroll
  for (int k = 0; k < KEEP; ++k) {
    const int64_t i = ob + t + static_cast<int64_t>(k) * nt;
    sc[k] = i < oe ? scores[i] : -FLT_MAX;
    mx = fmaxf(mx, sc[k]);
  }
  for (int64_t i = ob + t + static_cast<int64_t>(KEEP) * nt; i < oe; i += nt) mx = fmaxf(mx, scores[i]);
  mx = warp_max(mx);
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  if (t == 0) {
    float v = red[0];
    for (int w = 1; w < nw; ++w) v = fmaxf(v, red[w]);
    bc = v;
  }
  __syncthreads();
  mx = bc;
  float sum = 0.f;
#pragma unroll
  for (int k = 0; k < KEEP; ++k)
    if (ob + t + static_cast<int64_t>(k) * nt < oe) sum += expf(sc[k] - mx);
  for (int64_t i = ob + t + static_cast<int64_t>(KEEP) * nt; i < oe; i += nt) sum += expf(scores[i] - mx);
  sum = warp_sum(sum);
  __syncthreads();
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  float tot = 0.f;
  if (t == 0) {
    for (int w = 0; w < nw; ++w) tot += red[w];
  }
  float dot = 0.f;
  for (int c = t; c < L; c += nt) dot = fmaf(dM[static_cast<int64_t>(b) * L + c], M[static_cast<int64_t>(b) * L + c], dot);
  dot = warp_sum(dot);
  __syncthreads();
  if (lane == 0) red[warp] = dot;
  __syncthreads();
  if (t == 0) {
    float d = 0.f;
    for (int w = 0; w < nw; ++w) d += red[w];
    bag_stats = make_float2(oe > ob ? mx + logf(tot) : 0.f, d);
    stats[b] = bag_stats;
  }
  if (!SWEEP) return;
  if (dz && t < C) dzs[t] = dz[static_cast<int64_t>(b) * C + t];
  __syncthreads();
  const float lse = bag_stats.x, cdot = bag_stats.y;
  auto row_dot = [&](int64_t i) {
    if (!dz) return rowdot[i];
    float g = 0.f;
    for (int c = 0; c < C; ++c) g = fmaf(dzs[c], rowdot[i * C + c], g);
    return g;
  };
#pragma unroll
  for (int k = 0; k < KEEP; ++k) {
    const int64_t i = ob + t + static_cast<int64_t>(k) * nt;
    if (i < oe) {
      const float a = expf(sc[k] - lse);
      dscores[i] = a * (row_dot(i) - cdot);
      if (attn) attn[i] = a;
    }
  }
#pragma unroll 4
  for (int64_t i = ob + t + static_cast<int64_t>(KEEP) * nt; i < oe; i += nt) {
    const float a = expf(scores[i] - lse);
    dscores[i] = a * (row_dot(i) - cdot);
    if (attn) attn[i] = a;
  }
}

constexpr int BWD_ROWS_PER_WARP = 16;

template <typename T, int NV>
__global__ void __launch_bounds__(256)
k_pool_bwd(const T* __restrict__ X, const float* __restrict__ scores, const int32_t* __restrict__ offsets, int B,
           int64_t total_n, int L, int V, int64_t slab, const float* __restrict__ dM, const float2* __restrict__ stats,
           float* __restrict__ dscores, float* __restrict__ attn) {
  constexpr int VN = Vec16<T>::N;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // persistent: CTA c owns the row slab [c * slab, (c + 1) * slab); its warps take 16-row blocks round-robin and keep the
  // bag's dM slice in registers for as long as consecutive blocks stay inside one bag
  const int64_t slab_r0 = static_cast<int64_t>(blockIdx.x) * slab;
  const int64_t slab_r1 = (slab_r0 + slab < total_n) ? slab_r0 + slab : total_n;
  const uint4* Xv = reinterpret_cast<const uint4*>(X);
  int b = -1;
  int64_t bag_end = -1;
  float dm[NV][VN];
  float lse = 0.f, cdot = 0.f;
  auto load_bag = [&](int bag) {
    float2 st = __ldg(stats + bag);
    lse = st.x;
    cdot = st.y;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      int vec = lane + j * 32;
#pragma unroll
      for (int k = 0; k < VN; ++k) dm[j][k] = (vec < V) ? __ldg(dM + static_cast<int64_t>(bag) * L + vec * VN + k) : 0.f;
    }
  };
  for (int64_t r0 = slab_r0 + static_cast<int64_t>(warp) * BWD_ROWS_PER_WARP; r0 < slab_r1;
       r0 += static_cast<int64_t>(blockDim.x >> 5) * BWD_ROWS_PER_WARP) {
  const int64_t r1 = (r0 + BWD_ROWS_PER_WARP < slab_r1) ? r0 + BWD_ROWS_PER_WARP : slab_r1;
  if (b < 0 || r0 >= bag_end) {
    b = find_bag(offsets, B, r0);
    bag_end = __ldg(offsets + b + 1);
    load_bag(b);
  }

  int64_t i = r0;
  for (; i + 1 < r1; i += 2) {
    uint4 v0[NV], v1[NV];
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      int vec = lane + j * 32;
      v0[j] = (vec < V) ? ldg_stream(Xv + i * V + vec) : make_uint4(0, 0, 0, 0);
      v1[j] = (vec < V) ? ldg_stream(Xv + (i + 1) * V + vec) : make_uint4(0, 0, 0, 0);
    }
    float s0 = __ldg(scores + i), s1 = __ldg(scores + i + 1);
    // row i
    while (i >= bag_end) { ++b; bag_end = __ldg(offsets + b + 1); load_bag(b); }
    float g = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      float f[VN];
      Vec16<T>::unpack(v0[j], f);
#pragma unroll
      for (int k = 0; k < VN; ++k) g = fmaf(dm[j][k], f[k], g);
    }
    g = warp_sum(g);
    float a = expf(s0 - lse);
    if (lane == 0) {
      dscores[i] = a * (g - cdot);
      if (attn) attn[i] = a;
    }
    // row i+1
    while (i + 1 >= bag_end) { ++b; bag_end = __ldg(offsets + b + 1); load_bag(b); }
    g = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      float f[VN];
      Vec16<T>::unpack(v1[j], f);
#pragma unroll
      for (int k = 0; k < VN; ++k) g = fmaf(dm[j][k], f[k], g);
    }
    g = warp_sum(g);
    a = expf(s1 - lse);
    if (lane == 0) {
      dscores[i + 1] = a * (g - cdot);
      if (attn) attn[i + 1] = a;
    }
  }
  if (i < r1) {
    while (i >= bag_end) { ++b; bag_end = __ldg(offsets + b + 1); load_bag(b); }
    float g = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      int vec = lane + j * 32;
      if (vec < V) {
        float f[VN];
        Vec16<T>::unpack(ldg_stream(Xv + i * V + vec), f);
#pragma unroll
        for (int k = 0; k < VN; ++k) g = fmaf(dm[j][k], f[k], g);
      }
    }
    g = warp_sum(g);
    float a = expf(__ldg(scores + i) - lse);
    if (lane == 0) {
      dscores[i] = a * (g - cdot);
      if (attn) attn[i] = a;
    }
  }
  }  // 16-row blocks of this warp
}

// out[i, :] = (w ? w[i] : 1) * src[bag(i), :]   (dX of a plain sum pool; the pooling term of the gated dX)
template <typename T>
__global__ void __launch_bounds__(256)
k_bag_broadcast(const float* __restrict__ src, const float* __restrict__ w, const int32_t* __restrict__ offsets, int B,
                int64_t total_n, int L, T* __restrict__ out) {
  constexpr int VN = Vec16<T>::N;
  const int V = L / VN;
  const int64_t total = total_n * V;
  for (int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
       idx += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t row = idx / V;
    const int vec = static_cast<int>(idx % V);
    const int b = find_bag(offsets, B, row);
    const float a = w ? __ldg(w + row) : 1.f;
    float f[VN];
#pragma unroll
    for (int k = 0; k < VN; ++k) f[k] = a * __ldg(src + static_cast<int64_t>(b) * L + vec * VN + k);
    reinterpret_cast<uint4*>(out)[idx] = Vec16<T>::pack(f);
  }
}

// rows per CTA: persistent slabs, two CTAs per SM, never below POOL_MIN_SLAB rows
static int64_t pool_slab_rows(int64_t total_n) {
  int64_t ctas = static_cast<int64_t>(sm_count()) * 2;
  int64_t slab = (total_n + ctas - 1) / ctas;
  if (slab < POOL_MIN_SLAB) slab = POOL_MIN_SLAB;
  return (slab + POOL_BLK - 1) / POOL_BLK * POOL_BLK;
}

struct PoolWs {
  float* acc;
  PiecePartial* ml;
  unsigned int* counters;
  float2* stats;
  size_t bytes;
};
static PoolWs pool_ws(void* base, int64_t total_n, int B, int L) {
  const int64_t slab = pool_slab_rows(total_n);
  const int64_t slots = (total_n + slab - 1) / slab + B + 1;  // (CTA, bag) pieces: slot = cta + bag
  size_t off = 0;
  PoolWs w;
  char* p = static_cast<char*>(base);
  w.counters = reinterpret_cast<unsigned int*>(p + off);
  off = align_up(off + sizeof(unsigned int) * static_cast<size_t>(B), 256);
  w.stats = reinterpret_cast<float2*>(p + off);
  off = align_up(off + sizeof(float2) * static_cast<size_t>(B), 256);
  w.ml = reinterpret_cast<PiecePartial*>(p + off);
  off = align_up(off + sizeof(PiecePartial) * static_cast<size_t>(slots), 256);
  w.acc = reinterpret_cast<float*>(p + off);
  off = align_up(off + sizeof(float) * static_cast<size_t>(slots) * L, 256);
  w.bytes = off;
  return w;
}

// NC bucket of C row dots per row (0: no dots)
static int pool_dot_bucket(int C) { return C <= 0 ? 0 : C == 1 ? 1 : C == 2 ? 2 : C <= 4 ? 4 : 8; }

// per-warp accumulator rows, plus the staged dot vectors of the row-dot kernels
static size_t pool_fwd_smem_bytes(int L, int C) {
  return sizeof(float) * static_cast<size_t>(POOL_WARPS + pool_dot_bucket(C)) * L;
}

// dv != NULL selects the row-dot kernels: C dots per row, dots[i * C + c] = v_bc . x_i (see pool_fwd_body)
template <typename T>
static int pool_fwd_t(const T* X, const float* scores, const int32_t* offsets, int B, int64_t total_n, int L, float* M,
                      T* M_lowp, int32_t* argmax, float* lse, void* workspace, size_t ws_bytes, cudaStream_t st,
                      int normalize = 1, const float* dv = nullptr, int64_t dv_bag_stride = 0,
                      const float* col_scale = nullptr, int C = 0, float* dots = nullptr) {
  const int V = L * static_cast<int>(sizeof(T)) / 16;
  const int nv = (V + 31) / 32;
  MIL_CHECK_ARG(nv <= 16, MILB200_EUNSUPPORTED, "pool: row of %d bytes exceeds the 8 KB limit", L * (int)sizeof(T));
  if (!dv) C = 0;
  MIL_CHECK_ARG(C <= POOL_MAX_DOTS, MILB200_EUNSUPPORTED, "pool_fwd: %d row dots per row exceed the limit of %d", C,
                POOL_MAX_DOTS);
  // eight dots per row on a bf16 row of more than 6 vectors per lane do not fit in 255 registers without spilling
  MIL_CHECK_ARG(!(sizeof(T) == 2 && nv > 6 && C > 4), MILB200_EUNSUPPORTED,
                "pool_fwd: more than 4 row dots per row need a bf16 row of at most 1536 elements (L=%d)", L);
  const size_t smem = pool_fwd_smem_bytes(L, C);
  // the kernel's static shared memory (< 1 KB) counts against the same limits as the dynamic part
  MIL_CHECK_ARG(smem + 1024 <= POOL_SMEM_LIMIT, MILB200_EUNSUPPORTED,
                "pool_fwd: L=%d with %d row dots per row needs %zu bytes of shared memory (limit %zu)", L, C, smem + 1024,
                POOL_SMEM_LIMIT);
  PoolWs w = pool_ws(workspace, total_n, B, L);
  MIL_CHECK_ARG(workspace && ws_bytes >= w.bytes, MILB200_EWORKSPACE, "pool_fwd: workspace %zu < %zu", ws_bytes, w.bytes);
  MIL_CUDA(cudaMemsetAsync(w.counters, 0, sizeof(unsigned int) * static_cast<size_t>(B), st));
  const int64_t slab = pool_slab_rows(total_n);
  const int64_t ctas = (total_n + slab - 1) / slab;
  auto launch = [&](auto kern, auto... rowdot_args) -> int {
    if (smem + 1024 > 48 * 1024) MIL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<static_cast<unsigned>(ctas), POOL_THREADS, smem, st>>>(X, scores, offsets, B, total_n, L, V, slab, M, M_lowp,
                                                                 argmax, lse, w.acc, w.ml, w.counters, normalize,
                                                                 rowdot_args...);
    MIL_LAUNCH_CHECK();
    return MILB200_OK;
  };
  // (the same NV buckets as pool_bwd_t: a row's dot then has the same lane mapping in both kernels)
  auto launch_dots = [&](auto nc) -> int {
    constexpr int NC = decltype(nc)::value;
    if constexpr (sizeof(T) == 2 && NC > 4) {  // (refused above past NV = 6)
      if (nv <= 1) return launch(k_pool_fwd_rowdot<T, 1, NC>, dv, dv_bag_stride, col_scale, C, dots);
      if (nv == 2) return launch(k_pool_fwd_rowdot<T, 2, NC>, dv, dv_bag_stride, col_scale, C, dots);
      if (nv == 3) return launch(k_pool_fwd_rowdot<T, 3, NC>, dv, dv_bag_stride, col_scale, C, dots);
      if (nv == 4) return launch(k_pool_fwd_rowdot<T, 4, NC>, dv, dv_bag_stride, col_scale, C, dots);
      return launch(k_pool_fwd_rowdot<T, 6, NC>, dv, dv_bag_stride, col_scale, C, dots);
    } else {
      if (nv <= 1) return launch(k_pool_fwd_rowdot<T, 1, NC>, dv, dv_bag_stride, col_scale, C, dots);
      if (nv == 2) return launch(k_pool_fwd_rowdot<T, 2, NC>, dv, dv_bag_stride, col_scale, C, dots);
      if (nv == 3) return launch(k_pool_fwd_rowdot<T, 3, NC>, dv, dv_bag_stride, col_scale, C, dots);
      if (nv == 4) return launch(k_pool_fwd_rowdot<T, 4, NC>, dv, dv_bag_stride, col_scale, C, dots);
      if (nv <= 6) return launch(k_pool_fwd_rowdot<T, 6, NC>, dv, dv_bag_stride, col_scale, C, dots);
      if (nv <= 8) return launch(k_pool_fwd_rowdot<T, 8, NC>, dv, dv_bag_stride, col_scale, C, dots);
      return launch(k_pool_fwd_rowdot<T, 16, NC>, dv, dv_bag_stride, col_scale, C, dots);
    }
  };
  switch (pool_dot_bucket(C)) {
    case 1: return launch_dots(std::integral_constant<int, 1>());
    case 2: return launch_dots(std::integral_constant<int, 2>());
    case 4: return launch_dots(std::integral_constant<int, 4>());
    case 8: return launch_dots(std::integral_constant<int, 8>());
    default: break;
  }
  if (nv <= 1) return launch(k_pool_fwd<T, 1>);
  if (nv == 2) return launch(k_pool_fwd<T, 2>);
  if (nv == 3) return launch(k_pool_fwd<T, 3>);
  if (nv == 4) return launch(k_pool_fwd<T, 4>);
  if (nv <= 6) return launch(k_pool_fwd<T, 6>);
  if (nv <= 8) return launch(k_pool_fwd<T, 8>);
  return launch(k_pool_fwd<T, 16>);
}

template <typename T>
static int pool_bwd_t(const T* X, const float* scores, const int32_t* offsets, int B, int64_t total_n, int L,
                      const float* dM, const float* M, float* dscores, float* attn, void* workspace, size_t ws_bytes,
                      cudaStream_t st) {
  int V = L * static_cast<int>(sizeof(T)) / 16;
  int nv = (V + 31) / 32;
  MIL_CHECK_ARG(nv <= 16, MILB200_EUNSUPPORTED, "pool_bwd: row too long (L=%d)", L);
  PoolWs w = pool_ws(workspace, total_n, B, L);
  MIL_CHECK_ARG(workspace && ws_bytes >= w.bytes, MILB200_EWORKSPACE, "pool_bwd: workspace %zu < %zu", ws_bytes, w.bytes);
  k_pool_bwd_stats<false><<<B, 1024, 0, st>>>(scores, offsets, L, dM, M, w.stats, nullptr, nullptr, nullptr);
  MIL_LAUNCH_CHECK();
  // two CTAs per SM, each a contiguous slab of whole 128-row groups (8 warps x 16 rows)
  int64_t ctas = static_cast<int64_t>(sm_count()) * 2;
  int64_t slab = (total_n + ctas - 1) / ctas;
  slab = (slab + 8 * BWD_ROWS_PER_WARP - 1) / (8 * BWD_ROWS_PER_WARP) * (8 * BWD_ROWS_PER_WARP);
  unsigned blocks = static_cast<unsigned>((total_n + slab - 1) / slab);
#define MIL_POOL_BWD(NVV)                                                                                   \
  k_pool_bwd<T, NVV><<<blocks, 256, 0, st>>>(X, scores, offsets, B, total_n, L, V, slab, dM, w.stats, dscores, attn)
  if (nv <= 1) MIL_POOL_BWD(1);
  else if (nv == 2) MIL_POOL_BWD(2);
  else if (nv == 3) MIL_POOL_BWD(3);
  else if (nv == 4) MIL_POOL_BWD(4);
  else if (nv <= 6) MIL_POOL_BWD(6);
  else if (nv <= 8) MIL_POOL_BWD(8);
  else MIL_POOL_BWD(16);
#undef MIL_POOL_BWD
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

static int pool_check(const void* X, const float* scores, const int32_t* offsets, int B, int64_t total_n, int L, int dtype,
                      bool need_scores = true) {
  MIL_CHECK_ARG(X && (scores || !need_scores) && offsets, MILB200_EINVAL, "pool: null pointer");
  MIL_CHECK_ARG(B > 0 && total_n > 0 && L > 0, MILB200_EINVAL, "pool: B=%d total_n=%lld L=%d must be positive", B,
                (long long)total_n, L);
  MIL_CHECK_ARG(dtype == MILB200_F32 || dtype == MILB200_BF16, MILB200_EINVAL, "pool: bad dtype %d", dtype);
  MIL_CHECK_ARG((L * elem_size(dtype)) % 16 == 0, MILB200_EALIGN, "pool: row pitch %d bytes is not a multiple of 16",
                L * elem_size(dtype));
  MIL_CHECK_ARG(aligned16(X), MILB200_EALIGN, "pool: X must be 16-byte aligned");
  MIL_CHECK_ARG(total_n < (1ll << 31), MILB200_EINVAL, "pool: total_n exceeds int32 CSR offsets");
  return MILB200_OK;
}

static bool aligned_f32(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3u) == 0; }

}  // namespace milb200

using namespace milb200;

extern "C" {

size_t milb200_pool_workspace_bytes(int64_t total_n, int B, int L) {
  if (total_n <= 0 || B <= 0 || L <= 0) return 256;
  return pool_ws(nullptr, total_n, B, L).bytes;
}

int milb200_segment_softmax_pool_fwd(const void* X, const float* scores, const int32_t* offsets, int B,
                                     int64_t total_n, int L, int dtype, float* M, void* M_lowp, int32_t* argmax,
                                     float* lse, void* workspace, size_t ws_bytes, void* stream) {
  int rc = pool_check(X, scores, offsets, B, total_n, L, dtype);
  if (rc) return rc;
  MIL_CHECK_ARG(M != nullptr, MILB200_EINVAL, "pool_fwd: M is null");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == MILB200_BF16)
    return pool_fwd_t<__nv_bfloat16>((const __nv_bfloat16*)X, scores, offsets, B, total_n, L, M, (__nv_bfloat16*)M_lowp,
                                     argmax, lse, workspace, ws_bytes, st);
  return pool_fwd_t<float>((const float*)X, scores, offsets, B, total_n, L, M, (float*)M_lowp, argmax, lse, workspace,
                           ws_bytes, st);
}

int milb200_segment_softmax_pool_fwd_rowdot(const void* X, const float* scores, const int32_t* offsets, int B,
                                            int64_t total_n, int L, int dtype, const float* dM, float* M, void* M_lowp,
                                            int32_t* argmax, float* lse, float* rowdot, void* workspace, size_t ws_bytes,
                                            void* stream) {
  int rc = pool_check(X, scores, offsets, B, total_n, L, dtype);
  if (rc) return rc;
  MIL_CHECK_ARG(M && dM && rowdot, MILB200_EINVAL, "pool_fwd_rowdot: M, dM and rowdot must be non-null");
  MIL_CHECK_ARG(aligned_f32(dM) && aligned_f32(rowdot), MILB200_EALIGN, "pool_fwd_rowdot: dM and rowdot must be 4-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == MILB200_BF16)
    return pool_fwd_t<__nv_bfloat16>((const __nv_bfloat16*)X, scores, offsets, B, total_n, L, M, (__nv_bfloat16*)M_lowp,
                                     argmax, lse, workspace, ws_bytes, st, 1, dM, L, nullptr, 1, rowdot);
  return pool_fwd_t<float>((const float*)X, scores, offsets, B, total_n, L, M, (float*)M_lowp, argmax, lse, workspace,
                           ws_bytes, st, 1, dM, L, nullptr, 1, rowdot);
}

int milb200_segment_softmax_pool_fwd_headdot(const void* X, const float* scores, const int32_t* offsets, int B,
                                             int64_t total_n, int L, int dtype, const float* W, int C,
                                             const float* col_scale, float* M, void* M_lowp, int32_t* argmax, float* lse,
                                             float* hdot, void* workspace, size_t ws_bytes, void* stream) {
  int rc = pool_check(X, scores, offsets, B, total_n, L, dtype);
  if (rc) return rc;
  MIL_CHECK_ARG(M && W && hdot, MILB200_EINVAL, "pool_fwd_headdot: M, W and hdot must be non-null");
  MIL_CHECK_ARG(C >= 1, MILB200_EINVAL, "pool_fwd_headdot: C=%d must be positive", C);
  MIL_CHECK_ARG(aligned_f32(W) && aligned_f32(hdot) && aligned_f32(col_scale), MILB200_EALIGN,
                "pool_fwd_headdot: W, col_scale and hdot must be 4-byte aligned");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == MILB200_BF16)
    return pool_fwd_t<__nv_bfloat16>((const __nv_bfloat16*)X, scores, offsets, B, total_n, L, M, (__nv_bfloat16*)M_lowp,
                                     argmax, lse, workspace, ws_bytes, st, 1, W, 0, col_scale, C, hdot);
  return pool_fwd_t<float>((const float*)X, scores, offsets, B, total_n, L, M, (float*)M_lowp, argmax, lse, workspace,
                           ws_bytes, st, 1, W, 0, col_scale, C, hdot);
}

/* M[b] = sum_i x_i over CSR offsets (no softmax): the reference's dense-batch behaviour (ABMIL.py:56-59 with
 * B>1, where the softmax runs over a size-1 axis; SURVEY F2) and SwinUNETR_wMask's 3-crop pool. */
int milb200_segment_sum_fwd(const void* X, const int32_t* offsets, int B, int64_t total_n, int L, int dtype, float* M,
                            void* M_lowp, void* workspace, size_t ws_bytes, void* stream) {
  int rc = pool_check(X, nullptr, offsets, B, total_n, L, dtype, false);
  if (rc) return rc;
  MIL_CHECK_ARG(M != nullptr, MILB200_EINVAL, "segment_sum_fwd: M is null");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == MILB200_BF16)
    return pool_fwd_t<__nv_bfloat16>((const __nv_bfloat16*)X, nullptr, offsets, B, total_n, L, M, (__nv_bfloat16*)M_lowp,
                                     nullptr, nullptr, workspace, ws_bytes, st, 0);
  return pool_fwd_t<float>((const float*)X, nullptr, offsets, B, total_n, L, M, (float*)M_lowp, nullptr, nullptr, workspace,
                           ws_bytes, st, 0);
}

/* out[i, :] = (w ? w[i] : 1) * src[bag(i), :], src fp32 [B, L], out [total_n, L] in `dtype`. */
int milb200_bag_broadcast(const float* src, const float* w, const int32_t* offsets, int B, int64_t total_n, int L,
                          int dtype, void* out, void* stream) {
  MIL_CHECK_ARG(src && offsets && out && B > 0 && total_n > 0 && L > 0, MILB200_EINVAL, "bag_broadcast: bad arguments");
  MIL_CHECK_ARG((L * elem_size(dtype)) % 16 == 0 && aligned16(out), MILB200_EALIGN, "bag_broadcast: misaligned output");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int64_t total = total_n * (L * elem_size(dtype) / 16);
  unsigned blocks = static_cast<unsigned>(std::min<int64_t>((total + 255) / 256, static_cast<int64_t>(sm_count()) * 16));
  if (dtype == MILB200_BF16)
    k_bag_broadcast<__nv_bfloat16><<<blocks, 256, 0, st>>>(src, w, offsets, B, total_n, L, (__nv_bfloat16*)out);
  else
    k_bag_broadcast<float><<<blocks, 256, 0, st>>>(src, w, offsets, B, total_n, L, (float*)out);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_segment_softmax_pool_bwd(const void* X, const float* scores, const int32_t* offsets, int B,
                                     int64_t total_n, int L, int dtype, const float* dM, const float* M,
                                     float* dscores, float* attn, void* workspace, size_t ws_bytes, void* stream) {
  int rc = pool_check(X, scores, offsets, B, total_n, L, dtype);
  if (rc) return rc;
  MIL_CHECK_ARG(dM && M && dscores, MILB200_EINVAL, "pool_bwd: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == MILB200_BF16)
    return pool_bwd_t<__nv_bfloat16>((const __nv_bfloat16*)X, scores, offsets, B, total_n, L, dM, M, dscores, attn,
                                     workspace, ws_bytes, st);
  return pool_bwd_t<float>((const float*)X, scores, offsets, B, total_n, L, dM, M, dscores, attn, workspace, ws_bytes, st);
}

int milb200_segment_softmax_pool_bwd_rowdot(const float* scores, const int32_t* offsets, int B, int64_t total_n, int L,
                                            const float* dM, const float* M, const float* rowdot, float* dscores,
                                            float* attn, void* workspace, size_t ws_bytes, void* stream) {
  MIL_CHECK_ARG(scores && offsets && dM && M && rowdot && dscores, MILB200_EINVAL, "pool_bwd_rowdot: null pointer");
  MIL_CHECK_ARG(aligned_f32(rowdot) && aligned_f32(dscores) && aligned_f32(attn), MILB200_EALIGN,
                "pool_bwd_rowdot: rowdot, dscores and attn must be 4-byte aligned");
  MIL_CHECK_ARG(B > 0 && total_n > 0 && L > 0, MILB200_EINVAL, "pool_bwd_rowdot: B=%d total_n=%lld L=%d must be positive",
                B, (long long)total_n, L);
  MIL_CHECK_ARG(total_n < (1ll << 31), MILB200_EINVAL, "pool_bwd_rowdot: total_n exceeds int32 CSR offsets");
  PoolWs w = pool_ws(workspace, total_n, B, L);
  MIL_CHECK_ARG(workspace && ws_bytes >= w.bytes, MILB200_EWORKSPACE, "pool_bwd_rowdot: workspace %zu < %zu", ws_bytes,
                w.bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  k_pool_bwd_stats<true><<<B, 1024, 0, st>>>(scores, offsets, L, dM, M, w.stats, rowdot, dscores, attn);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_segment_softmax_pool_bwd_headdot(const float* scores, const int32_t* offsets, int B, int64_t total_n, int L,
                                             int C, const float* dz, const float* dM, const float* M, const float* hdot,
                                             float* dscores, float* attn, void* workspace, size_t ws_bytes, void* stream) {
  MIL_CHECK_ARG(scores && offsets && dz && dM && M && hdot && dscores, MILB200_EINVAL, "pool_bwd_headdot: null pointer");
  MIL_CHECK_ARG(C >= 1, MILB200_EINVAL, "pool_bwd_headdot: C=%d must be positive", C);
  MIL_CHECK_ARG(C <= POOL_MAX_DOTS, MILB200_EUNSUPPORTED, "pool_bwd_headdot: C=%d exceeds the limit of %d", C,
                POOL_MAX_DOTS);
  MIL_CHECK_ARG(aligned_f32(dz) && aligned_f32(hdot) && aligned_f32(dscores) && aligned_f32(attn), MILB200_EALIGN,
                "pool_bwd_headdot: dz, hdot, dscores and attn must be 4-byte aligned");
  MIL_CHECK_ARG(B > 0 && total_n > 0 && L > 0, MILB200_EINVAL, "pool_bwd_headdot: B=%d total_n=%lld L=%d must be positive",
                B, (long long)total_n, L);
  MIL_CHECK_ARG(total_n < (1ll << 31), MILB200_EINVAL, "pool_bwd_headdot: total_n exceeds int32 CSR offsets");
  PoolWs w = pool_ws(workspace, total_n, B, L);
  MIL_CHECK_ARG(workspace && ws_bytes >= w.bytes, MILB200_EWORKSPACE, "pool_bwd_headdot: workspace %zu < %zu", ws_bytes,
                w.bytes);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  k_pool_bwd_stats<true><<<B, 1024, 0, st>>>(scores, offsets, L, dM, M, w.stats, hdot, dscores, attn, dz, C);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

}  // extern "C"
