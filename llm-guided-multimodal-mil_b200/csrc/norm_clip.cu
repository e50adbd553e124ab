// norm_clip.cu — LayerNorm (+ fused residual) forward/backward for the two-way transformer's norm1..4 /
// norm_final_attn (model/sam/transformer.py:288,295,300,307,118), the CLIP-style cosine logits
// (clip/model.py:354-368), CLIPloss_v1's logits + cross-entropy (utils.py:277-282) and the cosine
// embedding loss of train_ddp.py:102,326.  All latency/bandwidth-class kernels; fp32 math, `dtype` storage.
#include <algorithm>
#include <cfloat>

#include "simt_gemm.cuh"

namespace milb200 {

// ---------------------------------------------------------------------------------------------------
// LayerNorm: one warp per row, eps = 1e-5
// ---------------------------------------------------------------------------------------------------
constexpr int LN_MAX_PER_LANE = 32;  // n <= 1024

// Vector layout: lane owns the 16-byte vectors lane, lane + 32, ... of its row (n % VN == 0, rows 16-byte aligned).
template <typename T> struct LnCfg { static constexpr int VN = Vec16<T>::N; static constexpr int MAXV = 32 * LN_MAX_PER_LANE / (32 * VN); };

template <typename T>
__global__ void __launch_bounds__(256)
k_ln_fwd(const T* __restrict__ X, const T* __restrict__ R, const float* __restrict__ gamma, const float* __restrict__ beta,
         T* __restrict__ Y, float* __restrict__ mean, float* __restrict__ rstd, int64_t m, int n, int r_bcast) {
  constexpr int VN = LnCfg<T>::VN, MAXV = LnCfg<T>::MAXV;
  const int lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (row >= m) return;
  const int nvec = n / VN;
  const uint4* x = reinterpret_cast<const uint4*>(X + row * n);
  const uint4* r = R ? reinterpret_cast<const uint4*>(R + (r_bcast ? 0 : row * n)) : nullptr;   // r_bcast: one row for all
  float v[MAXV][VN];
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < MAXV; ++j) {
    const int vec = lane + 32 * j;
#pragma unroll
    for (int e = 0; e < VN; ++e) v[j][e] = 0.f;
    if (vec < nvec) {
      Vec16<T>::unpack(ldg_stream(x + vec), v[j]);
      if (r) {
        float f[VN];
        Vec16<T>::unpack(ldg_stream(r + vec), f);
#pragma unroll
        for (int e = 0; e < VN; ++e) v[j][e] += f[e];
      }
#pragma unroll
      for (int e = 0; e < VN; ++e) s += v[j][e];
    }
  }
  const float mu = warp_sum(s) / static_cast<float>(n);
  float q = 0.f;
#pragma unroll
  for (int j = 0; j < MAXV; ++j) {
    if (lane + 32 * j < nvec) {
#pragma unroll
      for (int e = 0; e < VN; ++e) { const float d = v[j][e] - mu; q = fmaf(d, d, q); }
    }
  }
  const float rs = rsqrtf(warp_sum(q) / static_cast<float>(n) + 1e-5f);
  uint4* y = reinterpret_cast<uint4*>(Y + row * n);
#pragma unroll
  for (int j = 0; j < MAXV; ++j) {
    const int vec = lane + 32 * j;
    if (vec < nvec) {
      float o[VN];
#pragma unroll
      for (int e = 0; e < VN; ++e) o[e] = (v[j][e] - mu) * rs * __ldg(gamma + vec * VN + e) + __ldg(beta + vec * VN + e);
      y[vec] = Vec16<T>::pack(o);
    }
  }
  if (lane == 0) { mean[row] = mu; rstd[row] = rs; }
}

// dXR = rstd * (g - mean(g) - xhat * mean(g * xhat)), g = dY * gamma;  per-CTA partial (dgamma, dbeta) -> part[cta][2][n]
template <typename T>
__global__ void __launch_bounds__(256)
k_ln_bwd(const T* __restrict__ X, const T* __restrict__ R, const float* __restrict__ gamma, const float* __restrict__ mean,
         const float* __restrict__ rstd, const T* __restrict__ dY, T* __restrict__ dXR, float* __restrict__ part, int64_t m,
         int n, int rows_per_cta, int r_bcast, float* __restrict__ dgamma, float* __restrict__ dbeta, int final_mode) {
  constexpr int VN = LnCfg<T>::VN, MAXV = LnCfg<T>::MAXV;
  extern __shared__ float sm[];  // [8 warps][2][n]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nvec = n / VN;
  float dg[MAXV][VN], db[MAXV][VN], gm[MAXV][VN];
#pragma unroll
  for (int j = 0; j < MAXV; ++j) {
    const int vec = lane + 32 * j;
#pragma unroll
    for (int e = 0; e < VN; ++e) {
      dg[j][e] = db[j][e] = 0.f;
      gm[j][e] = (vec < nvec) ? __ldg(gamma + vec * VN + e) : 0.f;
    }
  }
  const int64_t r0 = static_cast<int64_t>(blockIdx.x) * rows_per_cta;
  const int64_t r1 = (r0 + rows_per_cta < m) ? r0 + rows_per_cta : m;
  for (int64_t row = r0 + warp; row < r1; row += 8) {
    const float mu = mean[row], rs = rstd[row];
    const uint4* x = reinterpret_cast<const uint4*>(X + row * n);
    const uint4* r = R ? reinterpret_cast<const uint4*>(R + (r_bcast ? 0 : row * n)) : nullptr;
    const uint4* dy = reinterpret_cast<const uint4*>(dY + row * n);
    float xh[MAXV][VN], g[MAXV][VN];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int j = 0; j < MAXV; ++j) {
      const int vec = lane + 32 * j;
#pragma unroll
      for (int e = 0; e < VN; ++e) xh[j][e] = g[j][e] = 0.f;
      if (vec < nvec) {
        float xv[VN], dv[VN];
        Vec16<T>::unpack(ldg_stream(x + vec), xv);
        Vec16<T>::unpack(ldg_stream(dy + vec), dv);
        if (r) {
          float f[VN];
          Vec16<T>::unpack(ldg_stream(r + vec), f);
#pragma unroll
          for (int e = 0; e < VN; ++e) xv[e] += f[e];
        }
#pragma unroll
        for (int e = 0; e < VN; ++e) {
          xh[j][e] = (xv[e] - mu) * rs;
          g[j][e] = dv[e] * gm[j][e];
          s1 += g[j][e];
          s2 = fmaf(g[j][e], xh[j][e], s2);
          dg[j][e] = fmaf(dv[e], xh[j][e], dg[j][e]);
          db[j][e] += dv[e];
        }
      }
    }
    s1 = warp_sum(s1) / static_cast<float>(n);
    s2 = warp_sum(s2) / static_cast<float>(n);
    uint4* dx = reinterpret_cast<uint4*>(dXR + row * n);
#pragma unroll
    for (int j = 0; j < MAXV; ++j) {
      const int vec = lane + 32 * j;
      if (vec < nvec) {
        float o[VN];
#pragma unroll
        for (int e = 0; e < VN; ++e) o[e] = rs * (g[j][e] - s1 - xh[j][e] * s2);
        dx[vec] = Vec16<T>::pack(o);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < MAXV; ++j) {
    const int vec = lane + 32 * j;
    if (vec < nvec) {
#pragma unroll
      for (int e = 0; e < VN; ++e) {
        sm[(warp * 2) * n + vec * VN + e] = dg[j][e];
        sm[(warp * 2 + 1) * n + vec * VN + e] = db[j][e];
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * n; i += blockDim.x) {
    int which = i / n, c = i % n;
    float a = 0.f;
    for (int w = 0; w < 8; ++w) a += sm[(w * 2 + which) * n + c];
    if (final_mode) {      // a single CTA covers all rows (the <= 16-row token side): no partials, no reduce launch
      float* dst = which == 0 ? dgamma + c : dbeta + c;
      *dst = final_mode == 2 ? *dst + a : a;
    } else {
      part[static_cast<int64_t>(blockIdx.x) * 2 * n + i] = a;
    }
  }
}

// block = 32 columns x 8 part-lanes; the 8 lanes' sums are folded in fixed order
__global__ void __launch_bounds__(256)
k_ln_reduce(const float* __restrict__ part, int parts, int n, float* __restrict__ dgamma, float* __restrict__ dbeta,
            int accumulate) {
  __shared__ float red[8][33];
  const int c = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + c;
  float a = 0.f;
  if (i < 2 * n)
    for (int s = w; s < parts; s += 8) a += part[static_cast<int64_t>(s) * 2 * n + i];
  red[w][c] = a;
  __syncthreads();
  if (w == 0 && i < 2 * n) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][c];
    float* dst = (i < n) ? dgamma + i : dbeta + (i - n);
    *dst = accumulate ? *dst + t : t;
  }
}

// one row per warp up to 4 CTAs per SM; beyond that the CTAs walk more rows
static int ln_ctas(int64_t m) {
  int64_t c = std::min<int64_t>((m + 7) / 8, static_cast<int64_t>(sm_count()) * 4);
  return static_cast<int>(c < 1 ? 1 : c);
}

// ---------------------------------------------------------------------------------------------------
// CLIP cosine logits
// ---------------------------------------------------------------------------------------------------
constexpr int CLIP_MAX_D = 1024;  // k_clip_bwd_side: 4 columns per thread of 256

template <typename T>
__global__ void k_inv_norm(const T* __restrict__ A, int rows, int d, float* __restrict__ inv) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  float s = 0.f;
  for (int c = lane; c < d; c += 32) { float v = to_f32<T>(A[static_cast<int64_t>(row) * d + c]); s = fmaf(v, v, s); }
  s = warp_sum(s);
  if (lane == 0) inv[row] = rsqrtf(s);
}
// logits[i, j] = exp(ls) * (I_i . T_j) * inv_i[i] * inv_t[j]; one warp per (i, j)
template <typename T>
__global__ void k_clip_logits(const T* __restrict__ I, const T* __restrict__ Tt, const float* __restrict__ ls,
                              const float* __restrict__ inv_i, const float* __restrict__ inv_t, float* __restrict__ logits,
                              int bi, int bt, int d) {
  const int lane = threadIdx.x & 31;
  const int64_t pair = static_cast<int64_t>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (pair >= static_cast<int64_t>(bi) * bt) return;
  const int i = static_cast<int>(pair / bt), j = static_cast<int>(pair % bt);
  float s = 0.f;
  for (int c = lane; c < d; c += 32)
    s = fmaf(to_f32<T>(I[static_cast<int64_t>(i) * d + c]), to_f32<T>(Tt[static_cast<int64_t>(j) * d + c]), s);
  s = warp_sum(s);
  if (lane == 0) logits[pair] = expf(ls[0]) * s * inv_i[i] * inv_t[j];
}
// dA_i = (g - ahat (g . ahat)) * inv_a[i],  g = exp(ls) * sum_j G[i,j] bhat_j;   G = dli (+ dlt^T); `transpose`
// selects the text side (G^T).  One CTA per row.
template <typename T>
__global__ void __launch_bounds__(256)
k_clip_bwd_side(const T* __restrict__ A, const T* __restrict__ Bm, const float* __restrict__ ls,
                const float* __restrict__ inv_a, const float* __restrict__ inv_b, const float* __restrict__ dli,
                const float* __restrict__ dlt, int na, int nb, int d, int transpose, T* __restrict__ dA) {
  __shared__ float red[8];
  __shared__ float bc;
  const int i = blockIdx.x;
  const float sc = expf(ls[0]);
  const float ia = inv_a[i];
  float g[4] = {0.f, 0.f, 0.f, 0.f};  // d <= CLIP_MAX_D with 256 threads
  for (int j = 0; j < nb; ++j) {
    // image side: G[i, j] = dli[i, j] + dlt[j, i]   (dli is [bi, bt], dlt is [bt, bi])
    // text side (transpose): row i is a text row: G^T[i, j] = dli[j, i] + dlt[i, j]
    float gij = 0.f;
    if (!transpose) gij = (dli ? dli[static_cast<int64_t>(i) * nb + j] : 0.f) + (dlt ? dlt[static_cast<int64_t>(j) * na + i] : 0.f);
    else gij = (dli ? dli[static_cast<int64_t>(j) * na + i] : 0.f) + (dlt ? dlt[static_cast<int64_t>(i) * nb + j] : 0.f);
    const float w = sc * gij * inv_b[j];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      int c = threadIdx.x + 256 * u;
      if (c < d) g[u] = fmaf(w, to_f32<T>(Bm[static_cast<int64_t>(j) * d + c]), g[u]);
    }
  }
  float dot = 0.f;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    int c = threadIdx.x + 256 * u;
    if (c < d) dot = fmaf(g[u], to_f32<T>(A[static_cast<int64_t>(i) * d + c]) * ia, dot);
  }
  dot = warp_sum(dot);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = dot;
  __syncthreads();
  if (threadIdx.x == 0) { float a = 0.f; for (int w = 0; w < 8; ++w) a += red[w]; bc = a; }
  __syncthreads();
  dot = bc;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    int c = threadIdx.x + 256 * u;
    if (c < d) {
      float ah = to_f32<T>(A[static_cast<int64_t>(i) * d + c]) * ia;
      dA[static_cast<int64_t>(i) * d + c] = from_f32<T>((g[u] - ah * dot) * ia);
    }
  }
}
// dscale = sum_ij G[i,j] * logits[i,j]
__global__ void __launch_bounds__(256)
k_clip_dscale(const float* __restrict__ logits, const float* __restrict__ dli, const float* __restrict__ dlt, int bi, int bt,
              float* __restrict__ dscale) {
  __shared__ float red[8];
  float a = 0.f;
  for (int64_t p = threadIdx.x; p < static_cast<int64_t>(bi) * bt; p += 256) {
    int i = static_cast<int>(p / bt), j = static_cast<int>(p % bt);
    float g = (dli ? dli[p] : 0.f) + (dlt ? dlt[static_cast<int64_t>(j) * bi + i] : 0.f);
    a = fmaf(g, logits[p], a);
  }
  a = warp_sum(a);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = a;
  __syncthreads();
  if (threadIdx.x == 0) { float s = 0.f; for (int w = 0; w < 8; ++w) s += red[w]; dscale[0] = s; }
}

// ---------------------------------------------------------------------------------------------------
// CLIPloss_v1: logits[i][r][c] = out[r] . feat[c][i]; CE over r (dim 1) against the identity, mean over I*b
// ---------------------------------------------------------------------------------------------------
// one CTA per (i, c) column: logits column, its log-sum-exp, loss contribution
constexpr size_t CLIPLOSS_STATIC_SMEM = 8 * sizeof(float);  // red[8]
template <typename T>
__global__ void __launch_bounds__(256)
k_cliploss_cols(const T* __restrict__ out, const T* __restrict__ feat, float* __restrict__ logits, float* __restrict__ lse,
                float* __restrict__ loss_part, int b, int n_info, int d) {
  extern __shared__ float sm[];  // f[d] | col[b]
  float* f = sm;
  float* col = sm + d;
  __shared__ float red[CLIPLOSS_STATIC_SMEM / sizeof(float)];
  const int i = blockIdx.x / b, c = blockIdx.x % b;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int k = threadIdx.x; k < d; k += 256) f[k] = to_f32<T>(feat[(static_cast<int64_t>(c) * n_info + i) * d + k]);
  __syncthreads();
  for (int r = warp; r < b; r += 8) {
    float s = 0.f;
    for (int k = lane; k < d; k += 32) s = fmaf(to_f32<T>(out[static_cast<int64_t>(r) * d + k]), f[k], s);
    s = warp_sum(s);
    if (lane == 0) { col[r] = s; logits[(static_cast<int64_t>(i) * b + r) * b + c] = s; }
  }
  __syncthreads();
  float mx = -FLT_MAX;
  for (int r = threadIdx.x; r < b; r += 256) mx = fmaxf(mx, col[r]);
  mx = warp_max(mx);
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  mx = red[0];
  for (int w = 1; w < 8; ++w) mx = fmaxf(mx, red[w]);
  __syncthreads();
  float sum = 0.f;
  for (int r = threadIdx.x; r < b; r += 256) sum += expf(col[r] - mx);
  sum = warp_sum(sum);
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < 8; ++w) t += red[w];
    float l = mx + logf(t);
    lse[blockIdx.x] = l;
    loss_part[blockIdx.x] = l - col[c];  // -log_softmax at the diagonal element
  }
}
// dout[r, :] = (1/(I b)) sum_{i,c} (softmax_r(logits[i][:, c])[r] - [r == c]) feat[c][i][:]; one CTA per r; also the loss
template <typename T>
__global__ void __launch_bounds__(256)
k_cliploss_dout(const T* __restrict__ feat, const float* __restrict__ logits, const float* __restrict__ lse,
                const float* __restrict__ loss_part, float* __restrict__ loss, float* __restrict__ dout, int b, int n_info,
                int d) {
  const int r = blockIdx.x;
  const float inv = 1.f / (static_cast<float>(n_info) * static_cast<float>(b));
  float g[4] = {0.f, 0.f, 0.f, 0.f};
  for (int i = 0; i < n_info; ++i) {
    for (int c = 0; c < b; ++c) {
      float p = expf(logits[(static_cast<int64_t>(i) * b + r) * b + c] - lse[i * b + c]);
      float w = (p - (r == c ? 1.f : 0.f)) * inv;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        int k = threadIdx.x + 256 * u;
        if (k < d) g[u] = fmaf(w, to_f32<T>(feat[(static_cast<int64_t>(c) * n_info + i) * d + k]), g[u]);
      }
    }
  }
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    int k = threadIdx.x + 256 * u;
    if (k < d && dout) dout[static_cast<int64_t>(r) * d + k] = g[u];
  }
  if (r == 0) {
    __shared__ float red[8];
    float a = 0.f;
    for (int p = threadIdx.x; p < n_info * b; p += 256) a += loss_part[p];
    a = warp_sum(a);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = a;
    __syncthreads();
    if (threadIdx.x == 0) { float s = 0.f; for (int w = 0; w < 8; ++w) s += red[w]; loss[0] = s * inv; }
  }
}

// CosineEmbeddingLoss(a, b, target=+1) = mean_i (1 - cos_i), cos = a.b / sqrt((a.a + eps)(b.b + eps)), eps = 1e-12 (ATen Loss.cpp EPSILON)
template <typename T>
__global__ void __launch_bounds__(256)
k_cosine_loss(const T* __restrict__ A, const T* __restrict__ Bm, int n, int d, float* __restrict__ loss_rows,
              T* __restrict__ dA, T* __restrict__ dB) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= n) return;
  float ab = 0.f, aa = 0.f, bb = 0.f;
  for (int c = lane; c < d; c += 32) {
    float a = to_f32<T>(A[static_cast<int64_t>(row) * d + c]), b = to_f32<T>(Bm[static_cast<int64_t>(row) * d + c]);
    ab = fmaf(a, b, ab); aa = fmaf(a, a, aa); bb = fmaf(b, b, bb);
  }
  ab = warp_sum(ab); aa = warp_sum(aa) + 1e-12f; bb = warp_sum(bb) + 1e-12f;
  const float inv = rsqrtf(aa * bb);
  const float cs = ab * inv;
  if (lane == 0) loss_rows[row] = 1.f - cs;
  const float k = -1.f / static_cast<float>(n);  // d(mean(1 - cos))/dcos
  for (int c = lane; c < d; c += 32) {
    float a = to_f32<T>(A[static_cast<int64_t>(row) * d + c]), b = to_f32<T>(Bm[static_cast<int64_t>(row) * d + c]);
    if (dA) dA[static_cast<int64_t>(row) * d + c] = from_f32<T>(k * (b * inv - cs * a / aa));
    if (dB) dB[static_cast<int64_t>(row) * d + c] = from_f32<T>(k * (a * inv - cs * b / bb));
  }
}
__global__ void k_mean_small(const float* __restrict__ v, int n, float* __restrict__ out) {
  float a = 0.f;
  for (int i = threadIdx.x; i < n; i += 32) a += v[i];
  a = warp_sum(a);
  if (threadIdx.x == 0) out[0] = a / static_cast<float>(n);
}

}  // namespace milb200

using namespace milb200;

extern "C" {

size_t milb200_layernorm_workspace_bytes(int64_t m, int n) {
  if (m <= 0 || n <= 0) return 256;
  return sizeof(float) * static_cast<size_t>(ln_ctas(m)) * 2 * n + 256;
}

int milb200_layernorm_fwd(const void* X, const void* R, const float* gamma, const float* beta, void* Y, float* mean,
                          float* rstd, int64_t m, int n, int dtype, int r_broadcast, void* stream) {
  MIL_CHECK_ARG(X && gamma && beta && Y && mean && rstd, MILB200_EINVAL, "layernorm_fwd: null pointer");
  MIL_CHECK_ARG(m > 0 && n > 0 && n <= 32 * LN_MAX_PER_LANE, MILB200_EUNSUPPORTED, "layernorm_fwd: n=%d not in (0, %d]", n,
                32 * LN_MAX_PER_LANE);
  MIL_CHECK_ARG((n * elem_size(dtype)) % 16 == 0 && aligned16(X) && aligned16(Y) && (!R || aligned16(R)), MILB200_EALIGN,
                "layernorm_fwd: rows must be 16-byte aligned multiples of 16 bytes (n=%d)", n);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned blocks = static_cast<unsigned>((m + 7) / 8);
  if (dtype == MILB200_BF16)
    k_ln_fwd<__nv_bfloat16><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)X, (const __nv_bfloat16*)R, gamma, beta,
                                                    (__nv_bfloat16*)Y, mean, rstd, m, n, r_broadcast);
  else
    k_ln_fwd<float><<<blocks, 256, 0, st>>>((const float*)X, (const float*)R, gamma, beta, (float*)Y, mean, rstd, m, n,
                                            r_broadcast);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_layernorm_bwd(const void* X, const void* R, const float* gamma, const float* mean, const float* rstd,
                          const void* dY, void* dXR, float* dgamma, float* dbeta, int64_t m, int n, int dtype,
                          int accumulate, int r_broadcast, void* workspace, size_t ws_bytes, void* stream) {
  MIL_CHECK_ARG(X && gamma && mean && rstd && dY && dXR && dgamma && dbeta, MILB200_EINVAL, "layernorm_bwd: null pointer");
  MIL_CHECK_ARG(m > 0 && n > 0 && n <= 32 * LN_MAX_PER_LANE, MILB200_EUNSUPPORTED, "layernorm_bwd: n=%d unsupported", n);
  MIL_CHECK_ARG((n * elem_size(dtype)) % 16 == 0 && aligned16(X) && aligned16(dY) && aligned16(dXR) && (!R || aligned16(R)),
                MILB200_EALIGN, "layernorm_bwd: rows must be 16-byte aligned multiples of 16 bytes (n=%d)", n);
  size_t need = milb200_layernorm_workspace_bytes(m, n);
  MIL_CHECK_ARG(workspace && ws_bytes >= need, MILB200_EWORKSPACE, "layernorm_bwd: workspace %zu < %zu", ws_bytes, need);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int ctas = ln_ctas(m);
  const int rows_per_cta = static_cast<int>((m + ctas - 1) / ctas);
  float* part = static_cast<float*>(workspace);
  const int final_mode = ctas == 1 ? (accumulate ? 2 : 1) : 0;
  size_t smem = sizeof(float) * 8 * 2 * n;
  if (dtype == MILB200_BF16) {
    auto kern = k_ln_bwd<__nv_bfloat16>;
    if (smem > 48 * 1024) MIL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<ctas, 256, smem, st>>>((const __nv_bfloat16*)X, (const __nv_bfloat16*)R, gamma, mean, rstd,
                                  (const __nv_bfloat16*)dY, (__nv_bfloat16*)dXR, part, m, n, rows_per_cta, r_broadcast, dgamma,
                                  dbeta, final_mode);
  } else {
    auto kern = k_ln_bwd<float>;
    if (smem > 48 * 1024) MIL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<ctas, 256, smem, st>>>((const float*)X, (const float*)R, gamma, mean, rstd, (const float*)dY, (float*)dXR, part, m,
                                  n, rows_per_cta, r_broadcast, dgamma, dbeta, final_mode);
  }
  MIL_LAUNCH_CHECK();
  if (final_mode) return MILB200_OK;
  k_ln_reduce<<<(2 * n + 31) / 32, 256, 0, st>>>(part, ctas, n, dgamma, dbeta, accumulate);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_clip_logits_fwd(const void* I, const void* T, const float* logit_scale, float* logits, float* inv_norm_i,
                            float* inv_norm_t, int bi, int bt, int d, int dtype, void* stream) {
  MIL_CHECK_ARG(I && T && logit_scale && logits && inv_norm_i && inv_norm_t, MILB200_EINVAL, "clip_logits_fwd: null pointer");
  MIL_CHECK_ARG(bi > 0 && bt > 0 && d > 0, MILB200_EINVAL, "clip_logits_fwd: bad shape");
  // the backward keeps a row in four registers per thread of a 256-thread CTA: refuse here what it cannot take
  MIL_CHECK_ARG(d <= CLIP_MAX_D, MILB200_EUNSUPPORTED, "clip_logits_fwd: d=%d > %d unsupported", d, CLIP_MAX_D);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int64_t pairs = static_cast<int64_t>(bi) * bt;
  if (dtype == MILB200_BF16) {
    k_inv_norm<__nv_bfloat16><<<(bi + 7) / 8, 256, 0, st>>>((const __nv_bfloat16*)I, bi, d, inv_norm_i);
    k_inv_norm<__nv_bfloat16><<<(bt + 7) / 8, 256, 0, st>>>((const __nv_bfloat16*)T, bt, d, inv_norm_t);
    k_clip_logits<__nv_bfloat16><<<static_cast<unsigned>((pairs + 7) / 8), 256, 0, st>>>(
        (const __nv_bfloat16*)I, (const __nv_bfloat16*)T, logit_scale, inv_norm_i, inv_norm_t, logits, bi, bt, d);
  } else {
    k_inv_norm<float><<<(bi + 7) / 8, 256, 0, st>>>((const float*)I, bi, d, inv_norm_i);
    k_inv_norm<float><<<(bt + 7) / 8, 256, 0, st>>>((const float*)T, bt, d, inv_norm_t);
    k_clip_logits<float><<<static_cast<unsigned>((pairs + 7) / 8), 256, 0, st>>>((const float*)I, (const float*)T, logit_scale,
                                                                                 inv_norm_i, inv_norm_t, logits, bi, bt, d);
  }
  count_launch(2);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_clip_logits_bwd(const void* I, const void* T, const float* logit_scale, const float* logits,
                            const float* inv_norm_i, const float* inv_norm_t, const float* dlogits_per_image,
                            const float* dlogits_per_text, void* dI, void* dT, float* dscale, int bi, int bt, int d,
                            int dtype, void* stream) {
  MIL_CHECK_ARG(I && T && logit_scale && logits && inv_norm_i && inv_norm_t, MILB200_EINVAL, "clip_logits_bwd: null pointer");
  MIL_CHECK_ARG(dlogits_per_image || dlogits_per_text, MILB200_EINVAL, "clip_logits_bwd: no upstream gradient");
  MIL_CHECK_ARG(bi > 0 && bt > 0 && d > 0 && d <= CLIP_MAX_D, MILB200_EUNSUPPORTED, "clip_logits_bwd: d=%d unsupported", d);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == MILB200_BF16) {
    if (dI) k_clip_bwd_side<__nv_bfloat16><<<bi, 256, 0, st>>>((const __nv_bfloat16*)I, (const __nv_bfloat16*)T, logit_scale,
                                                               inv_norm_i, inv_norm_t, dlogits_per_image, dlogits_per_text,
                                                               bi, bt, d, 0, (__nv_bfloat16*)dI);
    if (dT) k_clip_bwd_side<__nv_bfloat16><<<bt, 256, 0, st>>>((const __nv_bfloat16*)T, (const __nv_bfloat16*)I, logit_scale,
                                                               inv_norm_t, inv_norm_i, dlogits_per_image, dlogits_per_text,
                                                               bt, bi, d, 1, (__nv_bfloat16*)dT);
  } else {
    if (dI) k_clip_bwd_side<float><<<bi, 256, 0, st>>>((const float*)I, (const float*)T, logit_scale, inv_norm_i, inv_norm_t,
                                                       dlogits_per_image, dlogits_per_text, bi, bt, d, 0, (float*)dI);
    if (dT) k_clip_bwd_side<float><<<bt, 256, 0, st>>>((const float*)T, (const float*)I, logit_scale, inv_norm_t, inv_norm_i,
                                                       dlogits_per_image, dlogits_per_text, bt, bi, d, 1, (float*)dT);
  }
  if (dscale) k_clip_dscale<<<1, 256, 0, st>>>(logits, dlogits_per_image, dlogits_per_text, bi, bt, dscale);
  const int launched = (dI ? 1 : 0) + (dT ? 1 : 0) + (dscale ? 1 : 0);
  if (launched == 0) return MILB200_OK;
  count_launch(launched - 1);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_cliploss_fwd_bwd(const void* out, const void* feat, float* logits, float* lse_ws, float* loss, float* dout,
                             int b, int n_info, int d, int dtype, void* stream) {
  MIL_CHECK_ARG(out && feat && logits && lse_ws && loss, MILB200_EINVAL, "cliploss: null pointer");
  MIL_CHECK_ARG(b > 0 && n_info > 0 && d > 0 && d <= 1024, MILB200_EUNSUPPORTED, "cliploss: bad shape b=%d I=%d d=%d", b, n_info, d);
  // k_cliploss_cols stages feat[c][i] and one logits column in dynamic shared memory, next to its static red[8]; the
  // two together must fit the 48 KB every launch gets without an opt-in
  const size_t smem = sizeof(float) * (static_cast<size_t>(d) + b);
  MIL_CHECK_ARG(smem + CLIPLOSS_STATIC_SMEM <= 48 * 1024, MILB200_EUNSUPPORTED,
                "cliploss: b + d = %d exceeds %d", b + d, static_cast<int>((48 * 1024 - CLIPLOSS_STATIC_SMEM) / sizeof(float)));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* lse = lse_ws;                 // [I*b]
  float* loss_part = lse_ws + n_info * b;  // [I*b]
  if (dtype == MILB200_BF16) {
    k_cliploss_cols<__nv_bfloat16><<<n_info * b, 256, smem, st>>>((const __nv_bfloat16*)out, (const __nv_bfloat16*)feat, logits,
                                                                  lse, loss_part, b, n_info, d);
    k_cliploss_dout<__nv_bfloat16><<<b, 256, 0, st>>>((const __nv_bfloat16*)feat, logits, lse, loss_part, loss, dout, b, n_info, d);
  } else {
    k_cliploss_cols<float><<<n_info * b, 256, smem, st>>>((const float*)out, (const float*)feat, logits, lse, loss_part, b,
                                                          n_info, d);
    k_cliploss_dout<float><<<b, 256, 0, st>>>((const float*)feat, logits, lse, loss_part, loss, dout, b, n_info, d);
  }
  count_launch(1);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_cosine_embedding_fwd_bwd(const void* a, const void* b, float* loss, float* loss_rows_ws, void* da, void* db,
                                     int n, int d, int dtype, void* stream) {
  MIL_CHECK_ARG(a && b && loss && loss_rows_ws && n > 0 && d > 0, MILB200_EINVAL, "cosine_embedding: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == MILB200_BF16)
    k_cosine_loss<__nv_bfloat16><<<(n + 7) / 8, 256, 0, st>>>((const __nv_bfloat16*)a, (const __nv_bfloat16*)b, n, d,
                                                              loss_rows_ws, (__nv_bfloat16*)da, (__nv_bfloat16*)db);
  else
    k_cosine_loss<float><<<(n + 7) / 8, 256, 0, st>>>((const float*)a, (const float*)b, n, d, loss_rows_ws, (float*)da, (float*)db);
  k_mean_small<<<1, 32, 0, st>>>(loss_rows_ws, n, loss);
  count_launch(1);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

}  // extern "C"
