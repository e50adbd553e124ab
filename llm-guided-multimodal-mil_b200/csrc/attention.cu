// attention.cu — multi-head attention core of the SAM-style two-way transformer
// (model/sam/transformer.py:434-446): O = softmax(Q K^T / sqrt(c)) V per head, forward and backward.
//
// On this path one side is always a handful of text tokens (T = 1 or 10, <= 16) and the other side is the
// image bag (N up to ~2e4 instances), so there are two kernel families instead of a generic flash kernel:
//   "t2i"  few queries (tokens) over many keys (instances):   bandwidth-bound on the K,V reads; every warp owns
//          one head and a key range, keeps an online-softmax partial (m, l, acc) per query and the partials
//          are merged in a fixed order (deterministic).
//   "i2t"  many queries (instances) over few keys (tokens):   every warp owns one head and a query range,
//          the token-side K,V live in shared memory; softmax over <= 16 keys happens inside the warp.
// Layouts: Q [nq, H*c], K/V [nk, H*c], O [nq, H*c] row-major in `dtype`; lse [H, nq] fp32.
#include <algorithm>
#include <cfloat>

#include "simt_gemm.cuh"

namespace milb200 {

constexpr int ATT_MAXT = 16;     // the small side
__host__ __device__ __forceinline__ int64_t imin64(int64_t a, int64_t b) { return a < b ? a : b; }

template <typename T> __device__ __forceinline__ float att_exp(float x);
template <> __device__ __forceinline__ float att_exp<float>(float x) { return expf(x); }
template <> __device__ __forceinline__ float att_exp<__nv_bfloat16>(float x) { return __expf(x); }
template <typename T> __device__ __forceinline__ float att_log(float x);
template <> __device__ __forceinline__ float att_log<float>(float x) { return logf(x); }
template <> __device__ __forceinline__ float att_log<__nv_bfloat16>(float x) { return __logf(x); }

template <typename T>
__device__ __forceinline__ void load_row_slice(const T* p, int c, float* out);  // c contiguous elements -> fp32
template <>
__device__ __forceinline__ void load_row_slice<float>(const float* p, int c, float* out) {
  for (int d = 0; d < c; d += 4) {
    float4 v = *reinterpret_cast<const float4*>(p + d);
    out[d] = v.x; out[d + 1] = v.y; out[d + 2] = v.z; out[d + 3] = v.w;
  }
}
template <>
__device__ __forceinline__ void load_row_slice<__nv_bfloat16>(const __nv_bfloat16* p, int c, float* out) {
  for (int d = 0; d < c; d += 8) {
    uint4 v = *reinterpret_cast<const uint4*>(p + d);
    Vec16<__nv_bfloat16>::unpack(v, out + d);
  }
}

// =====================================================================================================
// t2i forward: nq <= 16 queries, nk keys.  grid = (key chunks, 1), block = H warps (one head per warp).
// partial record per (chunk, head, query): m, l, acc[c]
// =====================================================================================================
template <typename T, int C>
__global__ void __launch_bounds__(256)
k_t2i_fwd(const T* __restrict__ Q, const T* __restrict__ K, const T* __restrict__ V, int nq, int64_t nk, int H,
          int keys_per_cta, float* __restrict__ part_ml, float* __restrict__ part_acc) {
  extern __shared__ float sm[];  // q[H][nq][C] fp32 (pre-scaled by 1/sqrt(C)) | per-warp V tile [32][C + 1]
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5;
  const int HC = H * C;
  const float scale = rsqrtf(static_cast<float>(C));
  for (int i = threadIdx.x; i < nq * HC; i += blockDim.x) {
    int q = i / HC, col = i % HC;
    sm[(col / C * nq + q) * C + col % C] = to_f32<T>(Q[i]) * scale;
  }
  __syncthreads();
  if (h >= H) return;
  const float* qh = sm + static_cast<int64_t>(h) * nq * C;
  float* vs = sm + static_cast<int64_t>(H) * nq * C + static_cast<int64_t>(h) * 32 * (C + 1);
  const int64_t k0 = static_cast<int64_t>(blockIdx.x) * keys_per_cta;
  const int64_t k1 = imin64(nk, k0 + keys_per_cta);

  float m[ATT_MAXT], l[ATT_MAXT], acc[ATT_MAXT][C / 32];
#pragma unroll
  for (int i = 0; i < ATT_MAXT; ++i) {
    m[i] = -FLT_MAX; l[i] = 0.f;
#pragma unroll
    for (int u = 0; u < C / 32; ++u) acc[i][u] = 0.f;
  }
  for (int64_t t0 = k0; t0 < k1; t0 += 32) {
    const int64_t j = t0 + lane;
    const bool ok = j < k1;
    float kf[C];
    if (ok) load_row_slice<T>(K + j * HC + h * C, C, kf);
    else {
#pragma unroll
      for (int d = 0; d < C; ++d) kf[d] = 0.f;
    }
    float p[ATT_MAXT];
#pragma unroll
    for (int i = 0; i < ATT_MAXT; ++i) {
      if (i < nq) {
        float s = 0.f;
#pragma unroll
        for (int d = 0; d < C; d += 4) {
          float4 qv = *reinterpret_cast<const float4*>(qh + i * C + d);
          s = fmaf(qv.x, kf[d], s); s = fmaf(qv.y, kf[d + 1], s);
          s = fmaf(qv.z, kf[d + 2], s); s = fmaf(qv.w, kf[d + 3], s);
        }
        s = ok ? s : -FLT_MAX;
        float mt = warp_max(s);
        float mn = fmaxf(m[i], mt);
        float corr = att_exp<T>(m[i] - mn);
        m[i] = mn;
        float pi = ok ? att_exp<T>(s - mn) : 0.f;
        p[i] = pi;
        l[i] = l[i] * corr + pi;  // per-lane partial sum; reduced across lanes at the end
#pragma unroll
        for (int u = 0; u < C / 32; ++u) acc[i][u] *= corr;
      }
    }
    // acc_i[channel = lane + 32u] += sum_j p_ij V[j, channel]: every lane fetches ITS key's V row with 128-bit
    // loads and parks it in the warp's shared tile; the channel-major pass then reads it conflict-free
    {
      float vf[C];
      if (ok) load_row_slice<T>(V + j * HC + h * C, C, vf);
      else {
#pragma unroll
        for (int d = 0; d < C; ++d) vf[d] = 0.f;
      }
      __syncwarp();
#pragma unroll
      for (int d = 0; d < C; ++d) vs[lane * (C + 1) + d] = vf[d];
      __syncwarp();
    }
#pragma unroll 8
    for (int jj = 0; jj < 32; ++jj) {
      float vv[C / 32];
#pragma unroll
      for (int u = 0; u < C / 32; ++u) vv[u] = vs[jj * (C + 1) + lane + 32 * u];
#pragma unroll
      for (int i = 0; i < ATT_MAXT; ++i) {
        if (i < nq) {
          float pj = __shfl_sync(0xffffffffu, p[i], jj);
#pragma unroll
          for (int u = 0; u < C / 32; ++u) acc[i][u] = fmaf(pj, vv[u], acc[i][u]);
        }
      }
    }
  }
  // note: l[i] holds per-lane partial sums that were rescaled consistently (corr is warp-uniform)
#pragma unroll
  for (int i = 0; i < ATT_MAXT; ++i) {
    if (i < nq) {
      float lt = warp_sum(l[i]);
      int64_t rec = (static_cast<int64_t>(blockIdx.x) * H + h) * nq + i;
      if (lane == 0) { part_ml[rec * 2] = m[i]; part_ml[rec * 2 + 1] = lt; }
#pragma unroll
      for (int u = 0; u < C / 32; ++u) part_acc[rec * C + lane + 32 * u] = acc[i][u];
    }
  }
}

// merge the chunk partials: O[i, h*C + d], lse[h, i].  One warp per (query, head): lanes stride the chunks (fixed
// assignment, fixed fold order => deterministic), then the per-lane partials are folded across the warp.
template <typename T, int C>
__global__ void __launch_bounds__(32)
k_t2i_combine(const float* __restrict__ part_ml, const float* __restrict__ part_acc, int chunks, int nq, int H,
              T* __restrict__ O, float* __restrict__ lse) {
  const int i = blockIdx.x, h = blockIdx.y, lane = threadIdx.x;
  float gm = -FLT_MAX;
  for (int c = lane; c < chunks; c += 32) gm = fmaxf(gm, part_ml[((static_cast<int64_t>(c) * H + h) * nq + i) * 2]);
  gm = warp_max(gm);
  float gl = 0.f, a[C];
#pragma unroll
  for (int d = 0; d < C; ++d) a[d] = 0.f;
  for (int c = lane; c < chunks; c += 32) {
    const int64_t rec = (static_cast<int64_t>(c) * H + h) * nq + i;
    const float w = att_exp<T>(part_ml[rec * 2] - gm);
    gl = fmaf(part_ml[rec * 2 + 1], w, gl);
    const float4* pa = reinterpret_cast<const float4*>(part_acc + rec * C);
#pragma unroll
    for (int d = 0; d < C; d += 4) {
      const float4 v = pa[d / 4];
      a[d] = fmaf(v.x, w, a[d]); a[d + 1] = fmaf(v.y, w, a[d + 1]);
      a[d + 2] = fmaf(v.z, w, a[d + 2]); a[d + 3] = fmaf(v.w, w, a[d + 3]);
    }
  }
  gl = warp_sum(gl);
  float mine = 0.f;
#pragma unroll
  for (int d = 0; d < C; ++d) {
    const float t = warp_sum(a[d]);
    if ((d & 31) == lane) mine = t;   // C == 32: lane d keeps channel d
  }
  if (lane < C) O[static_cast<int64_t>(i) * H * C + h * C + lane] = from_f32<T>(mine / gl);
  if (lane == 0 && lse) lse[h * nq + i] = gm + att_log<T>(gl);
}

// =====================================================================================================
// t2i backward: lane = key.  dK, dV rows are complete per key; dQ partials per CTA -> fixed-order reduce.
// =====================================================================================================
template <typename T, int C>
__global__ void __launch_bounds__(256)
k_t2i_bwd(const T* __restrict__ Q, const T* __restrict__ K, const T* __restrict__ V, const T* __restrict__ O,
          const float* __restrict__ lse, const T* __restrict__ dO, int nq, int64_t nk, int H, int keys_per_cta,
          T* __restrict__ dK, T* __restrict__ dV, float* __restrict__ dq_part) {
  extern __shared__ float sm[];
  // q[H][nq][C] (scaled) | do[H][nq][C] | delta[H][nq] | lse[H][nq] | per-warp K tile [32][C + 1]
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5;
  const int HC = H * C;
  const float scale = rsqrtf(static_cast<float>(C));
  float* s_q = sm;
  float* s_do = s_q + H * nq * C;
  float* s_delta = s_do + H * nq * C;
  float* s_lse = s_delta + H * nq;
  float* ks = s_lse + H * nq + static_cast<int64_t>(h) * 32 * (C + 1);
  for (int i = threadIdx.x; i < nq * HC; i += blockDim.x) {
    int q = i / HC, col = i % HC;
    int dst = (col / C * nq + q) * C + col % C;
    s_q[dst] = to_f32<T>(Q[i]) * scale;
    s_do[dst] = to_f32<T>(dO[i]);
  }
  for (int i = threadIdx.x; i < H * nq; i += blockDim.x) {
    int hh = i / nq, q = i % nq;
    float dlt = 0.f;
    for (int d = 0; d < C; ++d)
      dlt = fmaf(to_f32<T>(dO[static_cast<int64_t>(q) * HC + hh * C + d]), to_f32<T>(O[static_cast<int64_t>(q) * HC + hh * C + d]), dlt);
    s_delta[i] = dlt;
    s_lse[i] = lse[i];
  }
  __syncthreads();
  if (h >= H) return;
  const float* qh = s_q + static_cast<int64_t>(h) * nq * C;
  const float* doh = s_do + static_cast<int64_t>(h) * nq * C;
  const int64_t k0 = static_cast<int64_t>(blockIdx.x) * keys_per_cta;
  const int64_t k1 = imin64(nk, k0 + keys_per_cta);
  float dq[ATT_MAXT][C / 32];
#pragma unroll
  for (int i = 0; i < ATT_MAXT; ++i)
#pragma unroll
    for (int u = 0; u < C / 32; ++u) dq[i][u] = 0.f;

  for (int64_t t0 = k0; t0 < k1; t0 += 32) {
    const int64_t j = t0 + lane;
    const bool ok = j < k1;
    float kf[C], vf[C], dkf[C], dvf[C];
    if (ok) {
      load_row_slice<T>(K + j * HC + h * C, C, kf);
      load_row_slice<T>(V + j * HC + h * C, C, vf);
    } else {
#pragma unroll
      for (int d = 0; d < C; ++d) kf[d] = vf[d] = 0.f;
    }
#pragma unroll
    for (int d = 0; d < C; ++d) dkf[d] = dvf[d] = 0.f;
    float ds[ATT_MAXT];
#pragma unroll
    for (int i = 0; i < ATT_MAXT; ++i) {
      ds[i] = 0.f;
      if (i < nq) {
        float s = 0.f, dp = 0.f;
#pragma unroll
        for (int d = 0; d < C; d += 4) {
          float4 qv = *reinterpret_cast<const float4*>(qh + i * C + d);
          float4 gv = *reinterpret_cast<const float4*>(doh + i * C + d);
          s = fmaf(qv.x, kf[d], s); s = fmaf(qv.y, kf[d + 1], s); s = fmaf(qv.z, kf[d + 2], s); s = fmaf(qv.w, kf[d + 3], s);
          dp = fmaf(gv.x, vf[d], dp); dp = fmaf(gv.y, vf[d + 1], dp); dp = fmaf(gv.z, vf[d + 2], dp); dp = fmaf(gv.w, vf[d + 3], dp);
        }
        float p = ok ? att_exp<T>(s - s_lse[h * nq + i]) : 0.f;
        float dsi = p * (dp - s_delta[h * nq + i]);
        ds[i] = dsi;
#pragma unroll
        for (int d = 0; d < C; d += 4) {
          float4 qv = *reinterpret_cast<const float4*>(qh + i * C + d);   // already scaled by 1/sqrt(C)
          float4 gv = *reinterpret_cast<const float4*>(doh + i * C + d);
          dkf[d] = fmaf(dsi, qv.x, dkf[d]); dkf[d + 1] = fmaf(dsi, qv.y, dkf[d + 1]);
          dkf[d + 2] = fmaf(dsi, qv.z, dkf[d + 2]); dkf[d + 3] = fmaf(dsi, qv.w, dkf[d + 3]);
          dvf[d] = fmaf(p, gv.x, dvf[d]); dvf[d + 1] = fmaf(p, gv.y, dvf[d + 1]);
          dvf[d + 2] = fmaf(p, gv.z, dvf[d + 2]); dvf[d + 3] = fmaf(p, gv.w, dvf[d + 3]);
        }
      }
    }
    if (ok) {
      T* dkr = dK + j * HC + h * C;
      T* dvr = dV + j * HC + h * C;
      constexpr int VN = Vec16<T>::N;
#pragma unroll
      for (int d = 0; d < C; d += VN) {
        *reinterpret_cast<uint4*>(dkr + d) = Vec16<T>::pack(dkf + d);
        *reinterpret_cast<uint4*>(dvr + d) = Vec16<T>::pack(dvf + d);
      }
    }
    // dQ_i[channel] += scale * sum_j ds_ij K[j, channel]  (K rows parked in the warp's shared tile; ds = 0 past the end)
    __syncwarp();
#pragma unroll
    for (int d = 0; d < C; ++d) ks[lane * (C + 1) + d] = kf[d];
    __syncwarp();
#pragma unroll 8
    for (int jj = 0; jj < 32; ++jj) {
      float kk[C / 32];
#pragma unroll
      for (int u = 0; u < C / 32; ++u) kk[u] = ks[jj * (C + 1) + lane + 32 * u];
#pragma unroll
      for (int i = 0; i < ATT_MAXT; ++i) {
        if (i < nq) {
          float dsj = __shfl_sync(0xffffffffu, ds[i], jj);
#pragma unroll
          for (int u = 0; u < C / 32; ++u) dq[i][u] = fmaf(dsj, kk[u], dq[i][u]);
        }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < ATT_MAXT; ++i) {
    if (i < nq) {
#pragma unroll
      for (int u = 0; u < C / 32; ++u)
        dq_part[(static_cast<int64_t>(blockIdx.x) * nq + i) * HC + h * C + lane + 32 * u] = dq[i][u] * scale;
    }
  }
}

// =====================================================================================================
// i2t forward: nk <= 16 keys (tokens) in shared memory, nq query rows; warp = (head, query range), lane = query.
// =====================================================================================================
template <typename T, int C>
__global__ void __launch_bounds__(256)
k_i2t_fwd(const T* __restrict__ Q, const T* __restrict__ K, const T* __restrict__ V, int64_t nq, int nk, int H,
          int rows_per_cta, T* __restrict__ O, float* __restrict__ lse) {
  extern __shared__ float sm[];  // k[H][nk][C] | v[H][nk][C]
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5;
  const int HC = H * C;
  const float scale = rsqrtf(static_cast<float>(C));
  float* s_k = sm;
  float* s_v = sm + H * nk * C;
  for (int i = threadIdx.x; i < nk * HC; i += blockDim.x) {
    int t = i / HC, col = i % HC;
    int dst = (col / C * nk + t) * C + col % C;
    s_k[dst] = to_f32<T>(K[i]) * scale;
    s_v[dst] = to_f32<T>(V[i]);
  }
  __syncthreads();
  if (h >= H) return;
  const float* kh = s_k + static_cast<int64_t>(h) * nk * C;
  const float* vh = s_v + static_cast<int64_t>(h) * nk * C;
  const int64_t r0 = static_cast<int64_t>(blockIdx.x) * rows_per_cta;
  const int64_t r1 = imin64(nq, r0 + rows_per_cta);
  for (int64_t t0 = r0; t0 < r1; t0 += 32) {
    const int64_t i = t0 + lane;
    if (i >= r1) continue;
    float qf[C];
    load_row_slice<T>(Q + i * HC + h * C, C, qf);
    float s[ATT_MAXT];
    float mx = -FLT_MAX;
#pragma unroll
    for (int t = 0; t < ATT_MAXT; ++t) {
      s[t] = -FLT_MAX;
      if (t < nk) {
        float a = 0.f;
#pragma unroll
        for (int d = 0; d < C; d += 4) {
          float4 kv = *reinterpret_cast<const float4*>(kh + t * C + d);
          a = fmaf(qf[d], kv.x, a); a = fmaf(qf[d + 1], kv.y, a); a = fmaf(qf[d + 2], kv.z, a); a = fmaf(qf[d + 3], kv.w, a);
        }
        s[t] = a;
        mx = fmaxf(mx, a);
      }
    }
    float sum = 0.f;
#pragma unroll
    for (int t = 0; t < ATT_MAXT; ++t) {
      if (t < nk) { s[t] = att_exp<T>(s[t] - mx); sum += s[t]; }
    }
    const float inv = 1.f / sum;
    float of[C];
#pragma unroll
    for (int d = 0; d < C; ++d) of[d] = 0.f;
#pragma unroll
    for (int t = 0; t < ATT_MAXT; ++t) {
      if (t < nk) {
        const float p = s[t] * inv;
#pragma unroll
        for (int d = 0; d < C; d += 4) {
          float4 vv = *reinterpret_cast<const float4*>(vh + t * C + d);
          of[d] = fmaf(p, vv.x, of[d]); of[d + 1] = fmaf(p, vv.y, of[d + 1]);
          of[d + 2] = fmaf(p, vv.z, of[d + 2]); of[d + 3] = fmaf(p, vv.w, of[d + 3]);
        }
      }
    }
    T* orow = O + i * HC + h * C;
    constexpr int VN = Vec16<T>::N;
#pragma unroll
    for (int d = 0; d < C; d += VN) *reinterpret_cast<uint4*>(orow + d) = Vec16<T>::pack(of + d);
    if (lse) lse[static_cast<int64_t>(h) * nq + i] = mx + att_log<T>(sum);
  }
}

// i2t backward: dQ rows complete per query; dK, dV (token side) are sums over all queries:
// per-warp register partials -> per-CTA shared reduction -> partial buffer [cta][2][nk][HC] -> fixed-order reduce.
template <typename T, int C>
__global__ void __launch_bounds__(256)
k_i2t_bwd(const T* __restrict__ Q, const T* __restrict__ K, const T* __restrict__ V, const float* __restrict__ lse,
          const T* __restrict__ dO, int64_t nq, int nk, int H, int rows_per_cta, T* __restrict__ dQ,
          float* __restrict__ dkv_part) {
  extern __shared__ float sm[];  // k[H][nk][C] (scaled) | v[H][nk][C] | per-warp Q tile, dO tile [32][C + 1] each
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5;
  const int HC = H * C;
  const float scale = rsqrtf(static_cast<float>(C));
  float* s_k = sm;
  float* s_v = sm + H * nk * C;
  for (int i = threadIdx.x; i < nk * HC; i += blockDim.x) {
    int t = i / HC, col = i % HC;
    int dst = (col / C * nk + t) * C + col % C;
    s_k[dst] = to_f32<T>(K[i]) * scale;
    s_v[dst] = to_f32<T>(V[i]);
  }
  __syncthreads();
  if (h >= H) return;
  const float* kh = s_k + static_cast<int64_t>(h) * nk * C;
  const float* vh = s_v + static_cast<int64_t>(h) * nk * C;
  float* qs = sm + 2 * static_cast<int64_t>(H) * nk * C + static_cast<int64_t>(h) * 2 * 32 * (C + 1);
  float* gs = qs + 32 * (C + 1);
  const int64_t r0 = static_cast<int64_t>(blockIdx.x) * rows_per_cta;
  const int64_t r1 = imin64(nq, r0 + rows_per_cta);
  float* out_dk = dkv_part + static_cast<int64_t>(blockIdx.x) * 2 * nk * HC;
  float* out_dv = out_dk + static_cast<int64_t>(nk) * HC;
  // token-side accumulators: lane = channel (c = lane + 32u), one slot per token
  float dkacc[ATT_MAXT][C / 32], dvacc[ATT_MAXT][C / 32];
#pragma unroll
  for (int t = 0; t < ATT_MAXT; ++t)
#pragma unroll
    for (int u = 0; u < C / 32; ++u) dkacc[t][u] = dvacc[t][u] = 0.f;

  for (int64_t t0 = r0; t0 < r1; t0 += 32) {
    const int64_t i = t0 + lane;
    const bool ok = i < r1;
    float qf[C], gf[C];
    if (ok) {
      load_row_slice<T>(Q + i * HC + h * C, C, qf);
      load_row_slice<T>(dO + i * HC + h * C, C, gf);
    } else {
#pragma unroll
      for (int d = 0; d < C; ++d) qf[d] = gf[d] = 0.f;
    }
    const float ls = ok ? lse[static_cast<int64_t>(h) * nq + i] : 0.f;
    float p[ATT_MAXT], dp[ATT_MAXT];
    float delta = 0.f;
#pragma unroll
    for (int t = 0; t < ATT_MAXT; ++t) {
      p[t] = 0.f; dp[t] = 0.f;
      if (t < nk) {
        float a = 0.f, b = 0.f;
#pragma unroll
        for (int d = 0; d < C; d += 4) {
          float4 kv = *reinterpret_cast<const float4*>(kh + t * C + d);
          float4 vv = *reinterpret_cast<const float4*>(vh + t * C + d);
          a = fmaf(qf[d], kv.x, a); a = fmaf(qf[d + 1], kv.y, a); a = fmaf(qf[d + 2], kv.z, a); a = fmaf(qf[d + 3], kv.w, a);
          b = fmaf(gf[d], vv.x, b); b = fmaf(gf[d + 1], vv.y, b); b = fmaf(gf[d + 2], vv.z, b); b = fmaf(gf[d + 3], vv.w, b);
        }
        p[t] = ok ? att_exp<T>(a - ls) : 0.f;
        dp[t] = b;
        delta = fmaf(p[t], b, delta);
      }
    }
    float dqf[C];
#pragma unroll
    for (int d = 0; d < C; ++d) dqf[d] = 0.f;
    float ds[ATT_MAXT];
#pragma unroll
    for (int t = 0; t < ATT_MAXT; ++t) {
      ds[t] = 0.f;
      if (t < nk) {
        ds[t] = p[t] * (dp[t] - delta);
#pragma unroll
        for (int d = 0; d < C; d += 4) {
          float4 kv = *reinterpret_cast<const float4*>(kh + t * C + d);  // already scaled
          dqf[d] = fmaf(ds[t], kv.x, dqf[d]); dqf[d + 1] = fmaf(ds[t], kv.y, dqf[d + 1]);
          dqf[d + 2] = fmaf(ds[t], kv.z, dqf[d + 2]); dqf[d + 3] = fmaf(ds[t], kv.w, dqf[d + 3]);
        }
      }
    }
    if (ok) {
      T* dqr = dQ + i * HC + h * C;
      constexpr int VN = Vec16<T>::N;
#pragma unroll
      for (int d = 0; d < C; d += VN) *reinterpret_cast<uint4*>(dqr + d) = Vec16<T>::pack(dqf + d);
    }
    // token-side sums over this tile's 32 queries: lane = channel, loop queries with shuffles of (ds, p); the Q and
    // dO rows each lane already holds are parked in the warp's shared tiles (rows past the end carry ds = p = 0)
    __syncwarp();
#pragma unroll
    for (int d = 0; d < C; ++d) { qs[lane * (C + 1) + d] = qf[d] * scale; gs[lane * (C + 1) + d] = gf[d]; }
    __syncwarp();
#pragma unroll 4
    for (int jj = 0; jj < 32; ++jj) {
      float qq[C / 32], gg[C / 32];
#pragma unroll
      for (int u = 0; u < C / 32; ++u) {
        qq[u] = qs[jj * (C + 1) + lane + 32 * u];
        gg[u] = gs[jj * (C + 1) + lane + 32 * u];
      }
#pragma unroll
      for (int t = 0; t < ATT_MAXT; ++t) {
        if (t < nk) {
          float dsj = __shfl_sync(0xffffffffu, ds[t], jj);
          float pj = __shfl_sync(0xffffffffu, p[t], jj);
#pragma unroll
          for (int u = 0; u < C / 32; ++u) {
            dkacc[t][u] = fmaf(dsj, qq[u], dkacc[t][u]);
            dvacc[t][u] = fmaf(pj, gg[u], dvacc[t][u]);
          }
        }
      }
    }
  }
#pragma unroll
  for (int t = 0; t < ATT_MAXT; ++t) {
    if (t < nk) {
#pragma unroll
      for (int u = 0; u < C / 32; ++u) {
        out_dk[static_cast<int64_t>(t) * HC + h * C + lane + 32 * u] = dkacc[t][u];
        out_dv[static_cast<int64_t>(t) * HC + h * C + lane + 32 * u] = dvacc[t][u];
      }
    }
  }
}

// part [parts][2n] -> (a[n], b[n])
template <typename T>
__global__ void k_reduce_cast2(const float* __restrict__ part, int parts, int64_t n, T* __restrict__ a, T* __restrict__ b) {
  int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= 2 * n) return;
  float acc = 0.f;
  for (int s = 0; s < parts; ++s) acc += part[static_cast<int64_t>(s) * 2 * n + i];
  if (i < n) a[i] = from_f32<T>(acc);
  else b[i - n] = from_f32<T>(acc);
}

template <typename T>
__global__ void k_reduce_cast(const float* __restrict__ part, int parts, int64_t n, T* __restrict__ out) {
  int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float a = 0.f;
  for (int s = 0; s < parts; ++s) a += part[static_cast<int64_t>(s) * n + i];
  out[i] = from_f32<T>(a);
}

struct AttPlan {
  bool t2i;         // few queries over many keys
  int ctas;         // CTAs along the big side
  int per_cta;      // rows of the big side per CTA
  size_t ws_bytes;  // partial buffers
};
// floats of the (max, sum) partials of the many-key forward, rounded up to 16 bytes: the accumulator partials that follow
// are read as float4 (an odd heads * nq would otherwise leave them 8 bytes off)
static size_t att_ml_floats(int64_t ctas, int heads, int64_t nq) {
  return (static_cast<size_t>(ctas) * heads * nq * 2 + 3) / 4 * 4;
}
static AttPlan att_plan(int64_t nq, int64_t nk, int heads, int c, int backward) {
  AttPlan p{};
  const int64_t HC = static_cast<int64_t>(heads) * c;
  p.t2i = (nk > ATT_MAXT);  // keys are the big side
  const int64_t big = p.t2i ? nk : nq;
  int64_t want = std::min<int64_t>((big + 63) / 64, static_cast<int64_t>(sm_count()) * 2);
  if (want < 1) want = 1;
  int64_t per = (big + want - 1) / want;
  per = (per + 31) / 32 * 32;
  p.per_cta = static_cast<int>(per);
  p.ctas = static_cast<int>((big + per - 1) / per);
  if (p.t2i) {
    if (!backward) p.ws_bytes = sizeof(float) * (att_ml_floats(p.ctas, heads, nq) + static_cast<size_t>(p.ctas) * heads * nq * c);
    else p.ws_bytes = sizeof(float) * static_cast<size_t>(p.ctas) * nq * HC;
  } else {
    p.ws_bytes = backward ? sizeof(float) * static_cast<size_t>(p.ctas) * 2 * nk * HC : 0;
  }
  p.ws_bytes += 256;
  return p;
}

template <typename T, int C>
static int attention_fwd_t(const T* Q, const T* K, const T* V, T* O, float* lse, int64_t nq, int64_t nk, int heads,
                           void* ws, size_t ws_bytes, cudaStream_t st) {
  AttPlan p = att_plan(nq, nk, heads, C, 0);
  const int HC = heads * C;
  if (p.t2i) {
   if constexpr (C != 32) {
    MIL_CHECK_ARG(false, MILB200_EUNSUPPORTED, "attention_fwd: many-key attention is built for head dim 32 only");
   } else {
    MIL_CHECK_ARG(ws && ws_bytes >= p.ws_bytes, MILB200_EWORKSPACE, "attention_fwd: workspace %zu < %zu", ws_bytes, p.ws_bytes);
    float* part_ml = static_cast<float*>(ws);
    float* part_acc = part_ml + att_ml_floats(p.ctas, heads, nq);
    size_t smem = sizeof(float) * (nq * HC + static_cast<size_t>(heads) * 32 * (C + 1));
    auto kern = k_t2i_fwd<T, C>;
    if (smem > 48 * 1024) MIL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<p.ctas, heads * 32, smem, st>>>(Q, K, V, static_cast<int>(nq), nk, heads, p.per_cta, part_ml, part_acc);
    MIL_LAUNCH_CHECK();
    k_t2i_combine<T, C><<<dim3(static_cast<unsigned>(nq), heads), 32, 0, st>>>(part_ml, part_acc, p.ctas,
                                                                               static_cast<int>(nq), heads, O, lse);
    MIL_LAUNCH_CHECK();
   }
  } else {
    size_t smem = sizeof(float) * 2 * nk * HC;
    auto kern = k_i2t_fwd<T, C>;
    if (smem > 48 * 1024) MIL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<p.ctas, heads * 32, smem, st>>>(Q, K, V, nq, static_cast<int>(nk), heads, p.per_cta, O, lse);
    MIL_LAUNCH_CHECK();
  }
  return MILB200_OK;
}

template <typename T, int C>
static int attention_bwd_t(const T* Q, const T* K, const T* V, const T* O, const float* lse, const T* dO, T* dQ, T* dK,
                           T* dV, int64_t nq, int64_t nk, int heads, void* ws, size_t ws_bytes, cudaStream_t st) {
  AttPlan p = att_plan(nq, nk, heads, C, 1);
  const int HC = heads * C;
  MIL_CHECK_ARG(ws && ws_bytes >= p.ws_bytes, MILB200_EWORKSPACE, "attention_bwd: workspace %zu < %zu", ws_bytes, p.ws_bytes);
  float* part = static_cast<float*>(ws);
  if (p.t2i) {
   if constexpr (C != 32) {
    MIL_CHECK_ARG(false, MILB200_EUNSUPPORTED, "attention_bwd: many-key attention is built for head dim 32 only");
   } else {
    size_t smem = sizeof(float) * (2 * nq * HC + 2 * heads * nq + static_cast<size_t>(heads) * 32 * (C + 1));
    auto kern = k_t2i_bwd<T, C>;
    if (smem > 48 * 1024) MIL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<p.ctas, heads * 32, smem, st>>>(Q, K, V, O, lse, dO, static_cast<int>(nq), nk, heads, p.per_cta, dK, dV, part);
    MIL_LAUNCH_CHECK();
    int64_t n = nq * HC;
    k_reduce_cast<T><<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(part, p.ctas, n, dQ);
    MIL_LAUNCH_CHECK();
   }
  } else {
    size_t smem = sizeof(float) * (2 * nk * HC + static_cast<size_t>(heads) * 2 * 32 * (C + 1));
    auto kern = k_i2t_bwd<T, C>;
    if (smem > 48 * 1024) MIL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<p.ctas, heads * 32, smem, st>>>(Q, K, V, lse, dO, nq, static_cast<int>(nk), heads, p.per_cta, dQ, part);
    MIL_LAUNCH_CHECK();
    // part is [cta][dK | dV][nk*HC]
    int64_t n = nk * HC;
    k_reduce_cast2<T><<<static_cast<unsigned>((2 * n + 255) / 256), 256, 0, st>>>(part, p.ctas, n, dK, dV);
    MIL_LAUNCH_CHECK();
  }
  return MILB200_OK;
}

static int att_check(const void* Q, const void* K, const void* V, int64_t nq, int64_t nk, int heads, int c, int dtype) {
  MIL_CHECK_ARG(Q && K && V, MILB200_EINVAL, "attention: null pointer");
  MIL_CHECK_ARG(nq > 0 && nk > 0 && heads > 0 && heads <= 8, MILB200_EINVAL, "attention: bad shape nq=%lld nk=%lld heads=%d",
                (long long)nq, (long long)nk, heads);
  MIL_CHECK_ARG(c == 32 || c == 64, MILB200_EUNSUPPORTED, "attention: head dim %d not built (32 or 64)", c);
  MIL_CHECK_ARG(std::min(nq, nk) <= ATT_MAXT, MILB200_EUNSUPPORTED,
                "attention: one side must have <= %d tokens (nq=%lld nk=%lld)", ATT_MAXT, (long long)nq, (long long)nk);
  MIL_CHECK_ARG(dtype == MILB200_F32 || dtype == MILB200_BF16, MILB200_EINVAL, "attention: bad dtype");
  MIL_CHECK_ARG(aligned16(Q) && aligned16(K) && aligned16(V), MILB200_EALIGN, "attention: pointers must be 16-byte aligned");
  return MILB200_OK;
}

}  // namespace milb200

using namespace milb200;

extern "C" {

size_t milb200_attention_workspace_bytes(int64_t nq, int64_t nk, int heads, int c, int backward) {
  if (nq <= 0 || nk <= 0 || heads <= 0) return 256;
  return att_plan(nq, nk, heads, c, backward).ws_bytes;
}

int milb200_attention_fwd(const void* Q, const void* K, const void* V, void* O, float* lse, int64_t nq, int64_t nk,
                          int heads, int c, int dtype, void* workspace, size_t ws_bytes, void* stream) {
  int rc = att_check(Q, K, V, nq, nk, heads, c, dtype);
  if (rc) return rc;
  MIL_CHECK_ARG(O && lse, MILB200_EINVAL, "attention_fwd: null output");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
#define MIL_ATT_FWD(TT, CC) \
  return attention_fwd_t<TT, CC>((const TT*)Q, (const TT*)K, (const TT*)V, (TT*)O, lse, nq, nk, heads, workspace, ws_bytes, st)
  if (dtype == MILB200_BF16) { if (c == 32) MIL_ATT_FWD(__nv_bfloat16, 32); else MIL_ATT_FWD(__nv_bfloat16, 64); }
  if (c == 32) MIL_ATT_FWD(float, 32); else MIL_ATT_FWD(float, 64);
#undef MIL_ATT_FWD
}

int milb200_attention_bwd(const void* Q, const void* K, const void* V, const void* O, const float* lse, const void* dO,
                          void* dQ, void* dK, void* dV, int64_t nq, int64_t nk, int heads, int c, int dtype,
                          void* workspace, size_t ws_bytes, void* stream) {
  int rc = att_check(Q, K, V, nq, nk, heads, c, dtype);
  if (rc) return rc;
  MIL_CHECK_ARG(O && lse && dO && dQ && dK && dV, MILB200_EINVAL, "attention_bwd: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
#define MIL_ATT_BWD(TT, CC)                                                                                        \
  return attention_bwd_t<TT, CC>((const TT*)Q, (const TT*)K, (const TT*)V, (const TT*)O, lse, (const TT*)dO, (TT*)dQ, \
                                 (TT*)dK, (TT*)dV, nq, nk, heads, workspace, ws_bytes, st)
  if (dtype == MILB200_BF16) { if (c == 32) MIL_ATT_BWD(__nv_bfloat16, 32); else MIL_ATT_BWD(__nv_bfloat16, 64); }
  if (c == 32) MIL_ATT_BWD(float, 32); else MIL_ATT_BWD(float, 64);
#undef MIL_ATT_BWD
}

}  // extern "C"
