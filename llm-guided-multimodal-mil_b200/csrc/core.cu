// core.cu — error plumbing, launch accounting, TMA descriptor factory and small glue kernels of
// libmilb200 (see include/milb200.h for the C ABI).
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "simt_gemm.cuh"
#include "tc_common.cuh"

namespace milb200 {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int sm_count() {
  static int cached = 0;
  if (cached == 0) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      cached = n;
    else
      cached = 148;
  }
  return cached;
}

bool gate_layout_interleaved(int L, int D, int dtype);

bool force_simt() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MILB200_FORCE_SIMT");
    v = (e && e[0] == '1') ? 1 : 0;
  }
  return v == 1;
}

// ---- TMA descriptor factory (driver entry point fetched through the runtime) -------------------
namespace tc {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encoder() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

static int make_tmap(CUtensorMap* out, CUtensorMapDataType dt, int esz, const void* base, uint64_t rows,
                     uint64_t cols, uint64_t ld, uint32_t box_rows, uint32_t box_cols, bool swizzle128 = true,
                     int small_swizzle = 0) {
  EncodeTiledFn enc = get_encoder();
  MIL_CHECK_ARG(enc != nullptr, MILB200_ECUDA, "cuTensorMapEncodeTiled entry point unavailable");
  MIL_CHECK_ARG(aligned16(base) && (ld * esz) % 16 == 0, MILB200_EALIGN,
                "TMA operand needs a 16-byte aligned base and row pitch (ld=%llu)", (unsigned long long)ld);
  MIL_CHECK_ARG(box_rows >= 1 && box_rows <= 256 && box_cols >= 1 && box_cols <= 256 &&
                    (!swizzle128 || box_cols * esz <= 128) && (box_cols * esz) % 16 == 0,
                MILB200_EINVAL, "bad TMA box");
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld * esz};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, dt, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B
                              : (small_swizzle == 32 ? CU_TENSOR_MAP_SWIZZLE_32B
                                                     : (small_swizzle == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE)),
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  MIL_CHECK_ARG(r == CUDA_SUCCESS, MILB200_ECUDA, "cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu ld=%llu box=%ux%u",
                (int)r, (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)ld, box_rows, box_cols);
  return MILB200_OK;
}
int make_tmap_bf16_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                      uint32_t box_rows, uint32_t box_cols) {
  return make_tmap(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, rows, cols, ld, box_rows, box_cols);
}
int make_tmap_bf16_2d_linear(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                             uint32_t box_rows, uint32_t box_cols) {
  return make_tmap(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, rows, cols, ld, box_rows, box_cols, false);
}
// boxes whose rows are 32 bytes (16 bf16), 32-byte swizzle: the two 16-byte halves of a row swap when bit 7 of the shared
// address is set (rows 4-7 of every 8) — lets 32 lanes write their rows with conflict-free 128-bit stores
int make_tmap_bf16_2d_sw32(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                           uint32_t box_rows) {
  return make_tmap(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, rows, cols, ld, box_rows, 16, false, 32);
}
// boxes whose rows are 64 bytes (32 bf16), 64-byte swizzle: 16-byte chunk index ^= bits 7-8 of the shared address
int make_tmap_bf16_2d_sw64(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                           uint32_t box_rows) {
  return make_tmap(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, rows, cols, ld, box_rows, 32, false, 64);
}
int make_tmap_f32_2d(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                     uint32_t box_rows, uint32_t box_cols) {
  return make_tmap(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base, rows, cols, ld, box_rows, box_cols);
}
int make_tmap_f32_2d_linear(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t ld,
                            uint32_t box_rows, uint32_t box_cols) {
  return make_tmap(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, base, rows, cols, ld, box_rows, box_cols, false);
}
}  // namespace tc

// ---- split-K reduction ---------------------------------------------------------------------------
__global__ void k_splitk_reduce(const float* __restrict__ part, int splits, int64_t n, float* __restrict__ out,
                                int accumulate) {
  int64_t i = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  if (i >= n) return;
  if (i + 4 <= n) {
    float4 a = accumulate ? *reinterpret_cast<const float4*>(out + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = 0; s < splits; ++s) {
      float4 p = *reinterpret_cast<const float4*>(part + static_cast<int64_t>(s) * n + i);
      a.x += p.x; a.y += p.y; a.z += p.z; a.w += p.w;
    }
    *reinterpret_cast<float4*>(out + i) = a;
  } else {
    for (; i < n; ++i) {
      float a = accumulate ? out[i] : 0.f;
      for (int s = 0; s < splits; ++s) a += part[static_cast<int64_t>(s) * n + i];
      out[i] = a;
    }
  }
}
int splitk_reduce(const float* part, int splits, int64_t n, float* out, int accumulate, cudaStream_t st) {
  // n is a multiple of 4 for every caller except tiny vectors; the tail loop handles the rest
  int64_t threads = (n + 3) / 4;
  k_splitk_reduce<<<static_cast<unsigned>((threads + 255) / 256), 256, 0, st>>>(part, splits, n, out, accumulate);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

// dWcat (natural [dWv; dWu] rows) = sum_s part[s] with part rows in the interleaved-halves order
__global__ void k_splitk_reduce_gate(const float* __restrict__ part, int splits, int D, int L, int dh,
                                     float* __restrict__ out) {
  int64_t i = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  const int64_t n = static_cast<int64_t>(2) * D * L;
  if (i >= n) return;
  const int r = static_cast<int>(i / L), c = static_cast<int>(i % L);
  const bool is_u = r >= D;
  const int d = is_u ? r - D : r;
  const int pr = (d / dh) * 2 * dh + (is_u ? dh : 0) + d % dh;
  const float* src = part + static_cast<int64_t>(pr) * L + c;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int s = 0; s < splits; ++s) {
    float4 p = *reinterpret_cast<const float4*>(src + static_cast<int64_t>(s) * n);
    a.x += p.x; a.y += p.y; a.z += p.z; a.w += p.w;
  }
  *reinterpret_cast<float4*>(out + i) = a;
}
// same for partials whose rows are in the saved activations' tile-64 order (unit d: V row 128 (d/64) + d%64, U 64 on)
__global__ void k_splitk_reduce_gate64(const float* __restrict__ part, int splits, int D, int L, float* __restrict__ out) {
  int64_t i = (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  const int64_t n = static_cast<int64_t>(2) * D * L;
  if (i >= n) return;
  const int r = static_cast<int>(i / L), c = static_cast<int>(i % L);
  const bool is_u = r >= D;
  const int d = is_u ? r - D : r;
  const int pr = 128 * (d / 64) + (is_u ? 64 : 0) + d % 64;
  const float* src = part + static_cast<int64_t>(pr) * L + c;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int s = 0; s < splits; ++s) {
    float4 p = *reinterpret_cast<const float4*>(src + static_cast<int64_t>(s) * n);
    a.x += p.x; a.y += p.y; a.z += p.z; a.w += p.w;
  }
  *reinterpret_cast<float4*>(out + i) = a;
}
int splitk_reduce_gate64(const float* part, int splits, int D, int L, float* out, cudaStream_t st) {
  int64_t threads = static_cast<int64_t>(2) * D * L / 4;
  k_splitk_reduce_gate64<<<static_cast<unsigned>((threads + 255) / 256), 256, 0, st>>>(part, splits, D, L, out);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int splitk_reduce_gate(const float* part, int splits, int D, int L, int dh, float* out, cudaStream_t st) {
  int64_t threads = static_cast<int64_t>(2) * D * L / 4;  // L % 8 == 0 on this path
  k_splitk_reduce_gate<<<static_cast<unsigned>((threads + 255) / 256), 256, 0, st>>>(part, splits, D, L, dh, out);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

// ---- elementwise glue ----------------------------------------------------------------------------
template <typename T>
__global__ void k_add(const T* __restrict__ a, const T* __restrict__ b, T* __restrict__ out, int64_t n, float alpha,
                      float beta) {
  int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  constexpr int V = Vec16<T>::N;
  int64_t nv = n / V;
  for (int64_t v = i; v < nv; v += stride) {
    uint4 ua = reinterpret_cast<const uint4*>(a)[v], ub = b ? reinterpret_cast<const uint4*>(b)[v] : make_uint4(0, 0, 0, 0);
    float fa[V], fb[V];
    Vec16<T>::unpack(ua, fa);
    Vec16<T>::unpack(ub, fb);
#pragma unroll
    for (int j = 0; j < V; ++j) fa[j] = alpha * fa[j] + beta * fb[j];
    reinterpret_cast<uint4*>(out)[v] = Vec16<T>::pack(fa);
  }
  for (int64_t e = nv * V + i; e < n; e += stride)
    out[e] = from_f32<T>(alpha * to_f32<T>(a[e]) + (b ? beta * to_f32<T>(b[e]) : 0.f));
}

template <typename T>
__global__ void k_sinusoid(T* __restrict__ pe, int64_t n_pos, int dim) {
  int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  int half = dim / 2;
  if (idx >= n_pos * half) return;
  int64_t p = idx / half;
  int i = static_cast<int>(idx % half);
  // aggregator.py:102-105 — div_term computed in fp32, then position * div_term in fp32
  float div = expf(static_cast<float>(2 * i) * (-(logf(10000.0f) / static_cast<float>(dim))));
  float ang = static_cast<float>(p) * div;
  pe[p * dim + 2 * i] = from_f32<T>(sinf(ang));
  pe[p * dim + 2 * i + 1] = from_f32<T>(cosf(ang));
}

// (C, T, HW) -> (T, C): tokens[t, c] = mean_hw fmap[c, t, hw]      (transformer.py:93)
template <typename T>
__global__ void k_ct_tokens_fwd(const T* __restrict__ fmap, T* __restrict__ tokens, int c, int t, int hw) {
  int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= c * t) return;
  int ti = idx / c, ci = idx % c;
  const T* src = fmap + (static_cast<int64_t>(ci) * t + ti) * hw;
  float s = 0.f;
  for (int k = 0; k < hw; ++k) s += to_f32<T>(src[k]);
  tokens[idx] = from_f32<T>(s / static_cast<float>(hw));
}
template <typename T>
__global__ void k_ct_tokens_bwd(const T* __restrict__ dtokens, T* __restrict__ dfmap, int c, int t, int hw) {
  int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  int64_t n = static_cast<int64_t>(c) * t * hw;
  if (idx >= n) return;
  int64_t ct = idx / hw;
  int ci = static_cast<int>(ct / t), ti = static_cast<int>(ct % t);
  dfmap[idx] = from_f32<T>(to_f32<T>(dtokens[static_cast<int64_t>(ti) * c + ci]) / static_cast<float>(hw));
}

// step_dev != nullptr: the step number is read from device memory (so that a CUDA graph that contains the optimiser
// can be replayed: the bias corrections must not be baked into the launch parameters); otherwise it is `step`
__global__ void k_adam(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                       float* __restrict__ v, int64_t n, float lr, float b1, float b2, float eps, float wd,
                       float gscale, int step, const int32_t* __restrict__ step_dev) {
  const int s = step_dev ? *step_dev : step;
  const float bc1 = adam_bias_correction(b1, s), bc2 = adam_bias_correction(b2, s);
  int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) {
    float pi = p[i];
    float gi = fmaf(wd, pi, g[i] * gscale);  // torch Adam: grad + weight_decay * param
    float mi = fmaf(b1, m[i], (1.f - b1) * gi);
    float vi = fmaf(b2, v[i], (1.f - b2) * gi * gi);
    m[i] = mi;
    v[i] = vi;
    float denom = sqrtf(vi) / sqrtf(bc2) + eps;  // torch: (sqrt(v)/sqrt(bias_correction2)) + eps
    p[i] = pi - (lr / bc1) * (mi / denom);
  }
}
__global__ void k_counter_inc(int32_t* c) { *c += 1; }

__global__ void k_sgd(float* __restrict__ p, const float* __restrict__ g, int64_t n, float lr, float wd, float gscale) {
  int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) {
    float pi = p[i];
    p[i] = pi - lr * fmaf(wd, pi, g[i] * gscale);  // torch SGD: d_p = grad + weight_decay * param
  }
}

// sigmoid + BCELoss(mean) fwd + bwd (n is tiny: B x num_classes)
__global__ void k_sigmoid_bce(const float* __restrict__ z, const float* __restrict__ target, float* __restrict__ prob,
                              float* __restrict__ loss, float* __restrict__ dz, int n) {
  __shared__ float red[32];
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    float p = sigmoid_precise(z[i]);
    float t = target[i];
    if (prob) prob[i] = p;
    float lp = fmaxf(logf(p), -100.f), l1p = fmaxf(log1pf(-p), -100.f);  // torch clamps the logs at -100
    acc -= t * lp + (1.f - t) * l1p;
    if (dz) dz[i] = (p - t) / static_cast<float>(n);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0 && loss) loss[0] = v / static_cast<float>(n);
  }
}

// dh > 0: interleaved-halves row order [V 0..dh-1 | U 0..dh-1 | V dh..2dh-1 | U dh..2dh-1] (tensor-core gate tiles);
// dh == 0: plain [V | U].
template <typename TS, typename TD>
__global__ void k_pack_gate(const TS* __restrict__ Wv, const TS* __restrict__ Wu, const TS* __restrict__ bv,
                            const TS* __restrict__ bu, int L, int D, TD* __restrict__ Wcat,
                            float* __restrict__ bcat, int dh) {
  int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  int64_t n = static_cast<int64_t>(2) * D * L;
  auto src_of = [&](int r, bool& is_u) {
    if (dh > 0) {
      int h = r / (2 * dh), w = r % (2 * dh);
      is_u = w >= dh;
      return h * dh + (w % dh);
    }
    is_u = r >= D;
    return is_u ? r - D : r;
  };
  if (i < n) {
    int r = static_cast<int>(i / L);
    int c = static_cast<int>(i % L);
    bool is_u;
    int d = src_of(r, is_u);
    float v = is_u ? to_f32<TS>(Wu[static_cast<int64_t>(d) * L + c]) : to_f32<TS>(Wv[static_cast<int64_t>(d) * L + c]);
    Wcat[i] = from_f32<TD>(v);
  }
  if (i < 2 * D && bcat) {
    bool is_u;
    int d = src_of(static_cast<int>(i), is_u);
    bcat[i] = is_u ? to_f32<TS>(bu[d]) : to_f32<TS>(bv[d]);
  }
}

template <typename T>
__global__ void k_transpose(const T* __restrict__ in, T* __restrict__ out, int rows, int cols) {
  __shared__ T tile[32][33];
  int x = blockIdx.x * 32 + threadIdx.x, y0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y)
    if (x < cols && y0 + j < rows) tile[j][threadIdx.x] = in[static_cast<int64_t>(y0 + j) * cols + x];
  __syncthreads();
  int ox = blockIdx.y * 32 + threadIdx.x, oy0 = blockIdx.x * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y)
    if (ox < rows && oy0 + j < cols) out[static_cast<int64_t>(oy0 + j) * rows + ox] = tile[threadIdx.x][j];
}
// out[cols, rows] = in[rows, cols]^T
int transpose2d(const void* in, void* out, int rows, int cols, int dtype, cudaStream_t st) {
  dim3 grid((cols + 31) / 32, (rows + 31) / 32), block(32, 8);
  if (dtype == MILB200_BF16)
    k_transpose<__nv_bfloat16><<<grid, block, 0, st>>>(static_cast<const __nv_bfloat16*>(in),
                                                       static_cast<__nv_bfloat16*>(out), rows, cols);
  else
    k_transpose<float><<<grid, block, 0, st>>>(static_cast<const float*>(in), static_cast<float*>(out), rows, cols);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

// One Philox call (128 random bits) serves EIGHT elements (16 bits each: keep-probability resolution 2^-16) and one
// 128-bit (bf16) / two 128-bit (fp32) loads and stores; counter = index of the 8-element group (+ offset).
template <typename T>
__global__ void k_dropout(const T* __restrict__ x, T* __restrict__ out, int64_t n, float p, float scale,
                          uint64_t seed, uint64_t offset) {
  int64_t grp = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t ngrp = (n + 7) / 8, stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  const uint2 key = make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
  const uint32_t thr = static_cast<uint32_t>(fminf(fmaxf(p, 0.f), 1.f) * 65536.f);   // drop when u16 < thr
  const bool vec = (reinterpret_cast<uintptr_t>(x) % 16 == 0) && (reinterpret_cast<uintptr_t>(out) % 16 == 0);
  for (; grp < ngrp; grp += stride) {
    const uint64_t c = static_cast<uint64_t>(grp) + offset;
    const uint4 r = philox4x32_10(make_uint4(static_cast<uint32_t>(c), static_cast<uint32_t>(c >> 32), 0u, 0u), key);
    const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
    const int64_t i0 = grp * 8;
    float f[8];
    if (vec && i0 + 8 <= n) {
      if (sizeof(T) == 2) {
        Vec16<__nv_bfloat16>::unpack(ldg_stream(reinterpret_cast<const uint4*>(x) + grp), f);
      } else {
        const float4 a = __ldg(reinterpret_cast<const float4*>(x) + 2 * grp), b4 = __ldg(reinterpret_cast<const float4*>(x) + 2 * grp + 1);
        f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w; f[4] = b4.x; f[5] = b4.y; f[6] = b4.z; f[7] = b4.w;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) f[j] = ((rr[j >> 1] >> (16 * (j & 1))) & 0xffffu) >= thr ? f[j] * scale : 0.f;
      if (sizeof(T) == 2) {
        reinterpret_cast<uint4*>(out)[grp] = Vec16<__nv_bfloat16>::pack(f);
      } else {
        reinterpret_cast<float4*>(out)[2 * grp] = make_float4(f[0], f[1], f[2], f[3]);
        reinterpret_cast<float4*>(out)[2 * grp + 1] = make_float4(f[4], f[5], f[6], f[7]);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int64_t i = i0 + j;
        if (i < n) {
          const bool keep = ((rr[j >> 1] >> (16 * (j & 1))) & 0xffffu) >= thr;
          out[i] = from_f32<T>(keep ? to_f32<T>(x[i]) * scale : 0.f);
        }
      }
    }
  }
}

template <typename TS, typename TD>
__global__ void k_cast(const TS* __restrict__ in, TD* __restrict__ out, int64_t n) {
  int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) out[i] = from_f32<TD>(to_f32<TS>(in[i]));
}

}  // namespace milb200

using namespace milb200;

extern "C" {

int milb200_version(void) { return MILB200_VERSION; }
const char* milb200_last_error(void) { return g_err; }
int64_t milb200_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int milb200_pack_gate_weights(const void* Wv, const void* Wu, const void* bv, const void* bu, int src_dtype,
                              int L, int D, void* Wcat, int dst_dtype, float* bcat, void* stream) {
  MIL_CHECK_ARG(Wv && Wu && Wcat && L > 0 && D > 0, MILB200_EINVAL, "pack_gate_weights: null pointer or bad shape");
  MIL_CHECK_ARG(bcat == nullptr || (bv && bu), MILB200_EINVAL, "pack_gate_weights: bcat requested without biases");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int64_t n = static_cast<int64_t>(2) * D * L;
  unsigned blocks = static_cast<unsigned>((n + 255) / 256);
  const int dh = gate_layout_interleaved(L, D, dst_dtype) ? D / 2 : 0;
  if (src_dtype == MILB200_F32 && dst_dtype == MILB200_F32)
    k_pack_gate<float, float><<<blocks, 256, 0, st>>>((const float*)Wv, (const float*)Wu, (const float*)bv,
                                                      (const float*)bu, L, D, (float*)Wcat, bcat, dh);
  else if (src_dtype == MILB200_F32 && dst_dtype == MILB200_BF16)
    k_pack_gate<float, __nv_bfloat16><<<blocks, 256, 0, st>>>((const float*)Wv, (const float*)Wu, (const float*)bv,
                                                              (const float*)bu, L, D, (__nv_bfloat16*)Wcat, bcat, dh);
  else if (src_dtype == MILB200_BF16 && dst_dtype == MILB200_BF16)
    k_pack_gate<__nv_bfloat16, __nv_bfloat16><<<blocks, 256, 0, st>>>(
        (const __nv_bfloat16*)Wv, (const __nv_bfloat16*)Wu, (const __nv_bfloat16*)bv, (const __nv_bfloat16*)bu, L, D,
        (__nv_bfloat16*)Wcat, bcat, dh);
  else
    MIL_CHECK_ARG(false, MILB200_EUNSUPPORTED, "pack_gate_weights: unsupported dtype pair %d -> %d", src_dtype, dst_dtype);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_cast(const void* in, int src_dtype, void* out, int dst_dtype, int64_t n, void* stream) {
  MIL_CHECK_ARG(in && out && n >= 0, MILB200_EINVAL, "cast: null pointer");
  if (n == 0) return MILB200_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned blocks = static_cast<unsigned>(std::min<int64_t>((n + 255) / 256, 148 * 16));
  if (src_dtype == MILB200_F32 && dst_dtype == MILB200_BF16)
    k_cast<float, __nv_bfloat16><<<blocks, 256, 0, st>>>((const float*)in, (__nv_bfloat16*)out, n);
  else if (src_dtype == MILB200_BF16 && dst_dtype == MILB200_F32)
    k_cast<__nv_bfloat16, float><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)in, (float*)out, n);
  else
    MIL_CHECK_ARG(false, MILB200_EUNSUPPORTED, "cast: unsupported dtype pair");
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

/* nn.Dropout(p) in train mode (ABMIL.py:49, aggregator.py:129): out = keep ? x/(1-p) : 0 with a Philox mask that
 * is a pure function of (seed, offset, element index); applying the same call to a gradient is the backward. */
int milb200_dropout(const void* x, void* out, int64_t n, float p, uint64_t seed, uint64_t offset, int dtype,
                    void* stream) {
  MIL_CHECK_ARG(x && out && n >= 0 && p >= 0.f && p < 1.f, MILB200_EINVAL, "dropout: bad arguments (p=%f)", p);
  if (n == 0) return MILB200_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned blocks = static_cast<unsigned>(std::min<int64_t>(((n + 7) / 8 + 255) / 256, static_cast<int64_t>(sm_count()) * 16));
  const float scale = 1.f / (1.f - p);
  if (dtype == MILB200_BF16)
    k_dropout<__nv_bfloat16><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)out, n, p, scale, seed, offset);
  else
    k_dropout<float><<<blocks, 256, 0, st>>>((const float*)x, (float*)out, n, p, scale, seed, offset);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_transpose(const void* in, void* out, int rows, int cols, int dtype, void* stream) {
  MIL_CHECK_ARG(in && out && rows > 0 && cols > 0, MILB200_EINVAL, "transpose: bad arguments");
  return transpose2d(in, out, rows, cols, dtype, static_cast<cudaStream_t>(stream));
}

int milb200_axpby(const void* a, const void* b, void* out, int64_t n, float alpha, float beta, int dtype, void* stream) {
  MIL_CHECK_ARG(a && out && n >= 0, MILB200_EINVAL, "axpby: null pointer");
  MIL_CHECK_ARG(aligned16(a) && aligned16(b) && aligned16(out), MILB200_EALIGN, "axpby: pointers must be 16-byte aligned");
  if (n == 0) return MILB200_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned blocks = static_cast<unsigned>(std::min<int64_t>((n / 4 + 255) / 256 + 1, 148 * 8));
  if (dtype == MILB200_BF16)
    k_add<__nv_bfloat16><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)a, (const __nv_bfloat16*)b, (__nv_bfloat16*)out, n,
                                                 alpha, beta);
  else
    k_add<float><<<blocks, 256, 0, st>>>((const float*)a, (const float*)b, (float*)out, n, alpha, beta);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_add(const void* a, const void* b, void* out, int64_t n, int dtype, void* stream) {
  MIL_CHECK_ARG(b, MILB200_EINVAL, "add: null pointer");
  return milb200_axpby(a, b, out, n, 1.f, 1.f, dtype, stream);
}

int milb200_sinusoid_pe(void* pe, int64_t n_pos, int dim, int dtype, void* stream) {
  MIL_CHECK_ARG(pe && n_pos > 0 && dim > 0 && dim % 2 == 0, MILB200_EINVAL, "sinusoid_pe: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int64_t n = n_pos * (dim / 2);
  unsigned blocks = static_cast<unsigned>((n + 255) / 256);
  if (dtype == MILB200_BF16)
    k_sinusoid<__nv_bfloat16><<<blocks, 256, 0, st>>>((__nv_bfloat16*)pe, n_pos, dim);
  else
    k_sinusoid<float><<<blocks, 256, 0, st>>>((float*)pe, n_pos, dim);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_ct_tokens_fwd(const void* fmap, void* tokens, int c, int t, int hw, int dtype, void* stream) {
  MIL_CHECK_ARG(fmap && tokens && c > 0 && t > 0 && hw > 0, MILB200_EINVAL, "ct_tokens_fwd: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned blocks = static_cast<unsigned>((c * t + 255) / 256);
  if (dtype == MILB200_BF16)
    k_ct_tokens_fwd<__nv_bfloat16><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)fmap, (__nv_bfloat16*)tokens, c, t, hw);
  else
    k_ct_tokens_fwd<float><<<blocks, 256, 0, st>>>((const float*)fmap, (float*)tokens, c, t, hw);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_ct_tokens_bwd(const void* dtokens, void* dfmap, int c, int t, int hw, int dtype, void* stream) {
  MIL_CHECK_ARG(dtokens && dfmap && c > 0 && t > 0 && hw > 0, MILB200_EINVAL, "ct_tokens_bwd: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int64_t n = static_cast<int64_t>(c) * t * hw;
  unsigned blocks = static_cast<unsigned>((n + 255) / 256);
  if (dtype == MILB200_BF16)
    k_ct_tokens_bwd<__nv_bfloat16><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)dtokens, (__nv_bfloat16*)dfmap, c, t, hw);
  else
    k_ct_tokens_bwd<float><<<blocks, 256, 0, st>>>((const float*)dtokens, (float*)dfmap, c, t, hw);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                      float beta1, float beta2, float eps, float weight_decay, float grad_scale, int step,
                      void* stream) {
  MIL_CHECK_ARG(param && grad && exp_avg && exp_avg_sq && n >= 0 && step >= 1, MILB200_EINVAL, "adam_step: bad arguments");
  if (n == 0) return MILB200_OK;
  unsigned blocks = static_cast<unsigned>(std::min<int64_t>((n + 255) / 256, 148 * 8));
  k_adam<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2,
                                                                eps, weight_decay, grad_scale, step, nullptr);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

void milb200_count_launches(int64_t n) { count_launch(static_cast<int>(n)); }

int milb200_step_counter_inc(int32_t* step_dev, void* stream) {
  MIL_CHECK_ARG(step_dev != nullptr, MILB200_EINVAL, "step_counter_inc: null pointer");
  k_counter_inc<<<1, 1, 0, static_cast<cudaStream_t>(stream)>>>(step_dev);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_adam_step_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                          float beta1, float beta2, float eps, float weight_decay, float grad_scale,
                          const int32_t* step_dev, void* stream) {
  MIL_CHECK_ARG(param && grad && exp_avg && exp_avg_sq && n >= 0 && step_dev, MILB200_EINVAL, "adam_step_dev: bad arguments");
  if (n == 0) return MILB200_OK;
  unsigned blocks = static_cast<unsigned>(std::min<int64_t>((n + 255) / 256, 148 * 8));
  k_adam<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2,
                                                                eps, weight_decay, grad_scale, 0, step_dev);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_sgd_step(float* param, const float* grad, int64_t n, float lr, float weight_decay, float grad_scale,
                     void* stream) {
  MIL_CHECK_ARG(param && grad && n >= 0, MILB200_EINVAL, "sgd_step: bad arguments");
  if (n == 0) return MILB200_OK;
  unsigned blocks = static_cast<unsigned>(std::min<int64_t>((n + 255) / 256, 148 * 8));
  k_sgd<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(param, grad, n, lr, weight_decay, grad_scale);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int milb200_sigmoid_bce_fwd_bwd(const float* z, const float* target, float* prob, float* loss, float* dz, int n,
                                void* stream) {
  MIL_CHECK_ARG(z && target && n > 0, MILB200_EINVAL, "sigmoid_bce: bad arguments");
  k_sigmoid_bce<<<1, 256, 0, static_cast<cudaStream_t>(stream)>>>(z, target, prob, loss, dz, n);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

}  // extern "C"
