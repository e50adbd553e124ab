// gate.cu — C-ABI entry points for the gated-attention score (ABMIL.py:52-54) forward/backward and for
// the dense linear layers (nn.Linear sites of aggregator.py / sam/transformer.py), dispatching between
// the tcgen05 kernels (bf16) and the FFMA kernels (fp32, or shapes the tensor-core tiles do not cover).
#include <algorithm>
#include <type_traits>

#include "simt_gemm.cuh"
#include "tc_gemm.cuh"

namespace milb200 {

bool force_simt();
// smallm.cu: weight-streaming kernels for m <= 16 rows (token side, heads)
bool smallm_ok(int64_t m, int n, int k, int dtype);
int smallm_fwd(const void* X, const void* add, const void* W, const float* bias, void* Y, int64_t m, int n, int k, int act,
               int dtype, cudaStream_t st);
int smallm_bwd(const void* X, const void* add, const void* W, const void* Y, const void* dY, void* dX, float* dW,
               float* dbias, int64_t m, int n, int k, int act, int dtype, int accumulate, float* ws, cudaStream_t st);
size_t smallm_ws_bytes(int64_t m, int k);
int splitk_reduce_gate(const float* part, int splits, int D, int L, int dh, float* out, cudaStream_t st);
int splitk_reduce_gate64(const float* part, int splits, int D, int L, float* out, cudaStream_t st);
int transpose2d(const void* in, void* out, int rows, int cols, int dtype, cudaStream_t st);

constexpr int64_t SIMT_ROW_CHUNK = 32768;

// ---- optional per-sub-kernel timing of gated_score_bwd (bench.py's roofline uses it) ------------
constexpr int PROF_MAX = 8;
static bool g_prof_on = false;
static cudaEvent_t g_prof_ev[PROF_MAX];
static int g_prof_n = 0;
static void prof_mark(cudaStream_t st) {
  if (!g_prof_on || g_prof_n >= PROF_MAX) return;
  if (!g_prof_ev[g_prof_n]) cudaEventCreate(&g_prof_ev[g_prof_n]);
  cudaEventRecord(g_prof_ev[g_prof_n++], st);
}  // bounds the fp32 pre-activation workspace of the FFMA path

// ---- FFMA-path gate kernels (one warp per instance) -------------------------------------------
__global__ void __launch_bounds__(256)
k_gate_fwd(const float* __restrict__ Z, const float* __restrict__ ww, const float* __restrict__ bw,
           float* __restrict__ scores, int64_t rows, int D) {
  const int lane = threadIdx.x & 31;
  const int64_t r = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  const float* z = Z + r * 2 * D;
  float p = 0.f;
  for (int d = lane; d < D; d += 32) p = fmaf(tanhf(z[d]) * sigmoid_precise(z[D + d]), __ldg(ww + d), p);
  p = warp_sum(p);
  if (lane == 0) scores[r] = p + __ldg(bw);
}

constexpr int GATE_MAX_DPL = 8;  // D <= 256 on the FFMA path

// in place: Z (pre-activations, bias included) -> dZ = [dVpre | dUpre]; the column sums leave as one record per CTA
// [dVpre D | dUpre D | ds*V*U D | sum ds] that k_gate_bwd_fold adds up in CTA order (deterministic, no atomics)
__global__ void __launch_bounds__(256)
k_gate_bwd(const float* Zin, float* Z, const float* __restrict__ ww, const float* __restrict__ dscores, int64_t rows, int D,
           float* __restrict__ rec) {     // Zin == Z: in place; Zin = the pre-activations the forward saved otherwise
  __shared__ float red[8][3 * 32 * GATE_MAX_DPL + 1];
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = static_cast<int64_t>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  const int64_t nwarps = static_cast<int64_t>(gridDim.x) * 8;
  float sv[GATE_MAX_DPL], su[GATE_MAX_DPL], sw[GATE_MAX_DPL];
#pragma unroll
  for (int j = 0; j < GATE_MAX_DPL; ++j) sv[j] = su[j] = sw[j] = 0.f;
  float sds = 0.f;
  for (int64_t r = warp0; r < rows; r += nwarps) {
    float* z = Z + r * 2 * D;
    const float* zi = Zin + r * 2 * D;
    const float ds = __ldg(dscores + r);
    sds += ds;
#pragma unroll
    for (int j = 0; j < GATE_MAX_DPL; ++j) {
      int d = lane + j * 32;
      if (d < D) {
        float V = tanhf(zi[d]), U = sigmoid_precise(zi[D + d]);
        float g = ds * __ldg(ww + d);
        float dv = g * U * (1.f - V * V), du = g * V * U * (1.f - U);
        z[d] = dv;
        z[D + d] = du;
        sv[j] += dv;
        su[j] += du;
        sw[j] += ds * V * U;
      }
    }
  }
  const int wib = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < GATE_MAX_DPL; ++j) {
    int d = lane + j * 32;
    if (d < D) {
      red[wib][d] = sv[j];
      red[wib][D + d] = su[j];
      red[wib][2 * D + d] = sw[j];
    }
  }
  if (lane == 0) red[wib][3 * D] = sds;   // every lane read the same ds values: sds is already the warp's total
  __syncthreads();
  const int rl = 3 * D + 1;
  for (int c = threadIdx.x; c < rl; c += blockDim.x) {
    float a = 0.f;
#pragma unroll
    for (int w8 = 0; w8 < 8; ++w8) a += red[w8][c];
    rec[static_cast<int64_t>(blockIdx.x) * rl + c] = a;
  }
}

__global__ void __launch_bounds__(256)
k_gate_bwd_fold(const float* __restrict__ rec, int nrec, int D, float* __restrict__ dbcat, float* __restrict__ dww,
                float* __restrict__ dbw, int accumulate) {
  // 32 columns x 8 record slices per CTA (coalesced 128-byte rows of the records); slices folded in fixed order
  __shared__ float red[8][33];
  const int rl = 3 * D + 1;
  const int cx = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + cx;
  float a = 0.f;
  if (c < rl)
    for (int b = sl; b < nrec; b += 8) a += rec[static_cast<int64_t>(b) * rl + c];
  red[sl][cx] = a;
  __syncthreads();
  if (sl == 0 && c < rl) {
    float t = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) t += red[k][cx];
    float* o = c < 2 * D ? dbcat + c : (c < 3 * D ? dww + (c - 2 * D) : dbw);
    *o = accumulate ? *o + t : t;
  }
}

// records: [ncta][8 epilogue warps e = half*4 + q][stride]; column d of each kind was produced by the warps whose
// half == (d % (D/2)) / (D/4); the sum(ds) slot by the half-0 warps.
__global__ void k_colsum_finalize(const float* __restrict__ ws, int nrec, int stride, float* __restrict__ dbcat,
                                  float* __restrict__ dww, float* __restrict__ dbw, int D) {
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c > 3 * D) return;
  const int half = (c < 3 * D) ? ((c % D) % (D / 2)) / (D / 4) : 0;
  float a = 0.f;
  for (int r = 0; r < nrec; r += 8)
    for (int q = 0; q < 4; ++q) a += ws[static_cast<int64_t>(r + half * 4 + q) * stride + c];
  if (c < 2 * D) dbcat[c] = a;
  else if (c < 3 * D) dww[c - 2 * D] = a;
  else dbw[0] = a;
}

// ---- dZ from SAVED gate activations (tensor-core path, forward ran with gate_act != NULL) -------------------
// VU [n, 384] bf16 in the forward's tile-64 column order (unit d: V at 128 (d/64) + d%64, U 64 further; tc_gemm.cu).
// dZ [n, 384] bf16 in the weight rows' packed order [V 0..95 | U 0..95 | V 96..191 | U 96..191] (what the dX GEMM and the
// split-K dW GEMM of the recompute path consume) = [ds w U (1 - V^2) | ds w V U (1 - U)].  Elementwise and HBM-bound: 768 B read + 768 B written
// per instance, instead of re-running the X . Wcat^T GEMM.  Block = 16 row groups x 24 (V vector, U vector) pairs;
// column sums (-> dbcat, dww, dbw) are kept in registers, folded in fixed order and written one record per block.
constexpr int DZS_THREADS = 192;
constexpr int DZS_PAIRS = 24;
constexpr int DZS_RG = DZS_THREADS / DZS_PAIRS;  // 8
constexpr int DZS_UNR = 4;                       // rows in flight per thread (8 x 16-byte loads)
__global__ void __launch_bounds__(DZS_THREADS, 4)
k_gate_dz_saved(const __nv_bfloat16* __restrict__ VU, const float* __restrict__ ww, const float* __restrict__ dscores,
                int64_t n, int64_t rows_per_block, __nv_bfloat16* __restrict__ dZ, float* __restrict__ rec_ws, int stride) {
  constexpr int D = tc::GATE_D, DH = D / 2;
  __shared__ float red[DZS_RG][DZS_PAIRS][25];
  __shared__ float red_ds[DZS_RG];
  const int t = threadIdx.x, p = t % DZS_PAIRS, rg = t / DZS_PAIRS;
  const int d0 = p * 8;                                   // natural gate index of the first of this thread's 8 units
  const int srcV = 128 * (d0 / 64) + d0 % 64;             // where the forward saved them (tile-64 order)
  const int srcU = srcV + 64;
  const int colV = (d0 / DH) * (2 * DH) + d0 % DH;        // where dZ wants them (weight-row packed order)
  const int colU = colV + DH;
  float w[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) w[e] = __ldg(ww + d0 + e);
  float sdv[8], sdu[8], svu[8], sds = 0.f;
#pragma unroll
  for (int e = 0; e < 8; ++e) sdv[e] = sdu[e] = svu[e] = 0.f;
  const int64_t r0 = static_cast<int64_t>(blockIdx.x) * rows_per_block;
  const int64_t r1 = (r0 + rows_per_block < n) ? r0 + rows_per_block : n;
  auto body = [&](const uint4& qv, const uint4& qu, float ds, int64_t r) {
    float V[8], U[8], dv[8], du[8];
    Vec16<__nv_bfloat16>::unpack(qv, V);
    Vec16<__nv_bfloat16>::unpack(qu, U);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float gu = ds * w[e] * U[e];
      dv[e] = gu * (1.f - V[e] * V[e]);
      du[e] = gu * V[e] * (1.f - U[e]);
      sdv[e] += dv[e];
      sdu[e] += du[e];
      svu[e] = fmaf(ds * V[e], U[e], svu[e]);
    }
    *reinterpret_cast<uint4*>(dZ + r * (2 * D) + colV) = Vec16<__nv_bfloat16>::pack(dv);
    *reinterpret_cast<uint4*>(dZ + r * (2 * D) + colU) = Vec16<__nv_bfloat16>::pack(du);
  };
  int64_t r = r0 + rg;
  for (; r + (DZS_UNR - 1) * DZS_RG < r1; r += DZS_UNR * DZS_RG) {
    uint4 qv[DZS_UNR], qu[DZS_UNR];
    float dsv[DZS_UNR];
#pragma unroll
    for (int u = 0; u < DZS_UNR; ++u) {
      qv[u] = ldg_stream(VU + (r + u * DZS_RG) * (2 * D) + srcV);
      qu[u] = ldg_stream(VU + (r + u * DZS_RG) * (2 * D) + srcU);
      dsv[u] = __ldg(dscores + r + u * DZS_RG);
    }
#pragma unroll
    for (int u = 0; u < DZS_UNR; ++u) {
      if (p == 0) sds += dsv[u];
      body(qv[u], qu[u], dsv[u], r + u * DZS_RG);
    }
  }
  for (; r < r1; r += DZS_RG) {
    const uint4 qv0 = ldg_stream(VU + r * (2 * D) + srcV), qu0 = ldg_stream(VU + r * (2 * D) + srcU);
    const float ds0 = __ldg(dscores + r);
    if (p == 0) sds += ds0;
    body(qv0, qu0, ds0, r);
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) { red[rg][p][e] = sdv[e]; red[rg][p][8 + e] = sdu[e]; red[rg][p][16 + e] = svu[e]; }
  if (p == 0) red_ds[rg] = sds;
  __syncthreads();
  float* rec = rec_ws + static_cast<int64_t>(blockIdx.x) * stride;
  for (int i = t; i < 3 * D; i += DZS_THREADS) {  // record: dVpre[192] | dUpre[192] | ds*V*U[192] | sum ds (natural order)
    const int k = i / D, d = i % D;
    const int pp = d / 8, e = d % 8;
    float a = 0.f;
#pragma unroll
    for (int g = 0; g < DZS_RG; ++g) a += red[g][pp][k * 8 + e];
    rec[i] = a;
  }
  if (t == 0) {
    float a = 0.f;
    for (int g = 0; g < DZS_RG; ++g) a += red_ds[g];
    rec[3 * D] = a;
  }
}
// fold the per-block records in block order
// records of the fused dW kernel: [split][m-tile t][dVpre 64 | dUpre 64 | ds*V*U 64 | sum ds], unit d = 64 t + j
__global__ void k_colsum_finalize_tn(const float* __restrict__ ws, int splits, int rec, float* __restrict__ dbcat,
                                     float* __restrict__ dww, float* __restrict__ dbw, int D) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c > 3 * D) return;
  const int k = c < 3 * D ? c / D : 0, d = c < 3 * D ? c % D : 0;
  const int off = c < 3 * D ? (d / 64) * rec + k * 64 + d % 64 : 192;
  float a = 0.f;
  for (int s = 0; s < splits; ++s) a += ws[static_cast<int64_t>(s) * (D / 64) * rec + off];
  if (c < 2 * D) dbcat[c] = a;
  else if (c < 3 * D) dww[c - 2 * D] = a;
  else dbw[0] = a;
}

// block = 32 columns x 8 record-lanes; the 8 lanes' sums are folded in fixed order
__global__ void __launch_bounds__(256)
k_colsum_finalize_flat(const float* __restrict__ ws, int nrec, int stride, float* __restrict__ dbcat,
                       float* __restrict__ dww, float* __restrict__ dbw, int D) {
  __shared__ float red[8][33];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int c = blockIdx.x * 32 + lane;
  float a = 0.f;
  if (c <= 3 * D)
    for (int r = w; r < nrec; r += 8) a += ws[static_cast<int64_t>(r) * stride + c];
  red[w][lane] = a;
  __syncthreads();
  if (w != 0 || c > 3 * D) return;
  float t = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) t += red[k][lane];
  if (c < 2 * D) dbcat[c] = t;
  else if (c < 3 * D) dww[c - 2 * D] = t;
  else dbw[0] = t;
}

// dYpre = dY * act'(Y)   (Y is the activation OUTPUT)
template <typename T>
__global__ void k_act_bwd(const T* __restrict__ Y, const T* __restrict__ dY, T* __restrict__ out, int64_t n, int act) {
  int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (; i < n; i += stride) {
    float y = to_f32<T>(Y[i]), g = to_f32<T>(dY[i]);
    if (act == MILB200_ACT_TANH) g *= (1.f - y * y);
    else if (act == MILB200_ACT_RELU) g = y > 0.f ? g : 0.f;
    else if (act == MILB200_ACT_SIGMOID) g *= y * (1.f - y);
    out[i] = from_f32<T>(g);
  }
}

// same with fp32 Y / dY and a bf16 result (the tensor-core operand of the mixed-precision linear's backward)
__global__ void k_act_bwd_f32_bf16(const float* __restrict__ Y, const float* __restrict__ dY, __nv_bfloat16* __restrict__ out,
                                   int64_t n4, int act) {
  int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (; i < n4; i += stride) {
    float4 g = reinterpret_cast<const float4*>(dY)[i];
    if (act != MILB200_ACT_NONE) {
      const float4 y = reinterpret_cast<const float4*>(Y)[i];
      if (act == MILB200_ACT_TANH) { g.x *= 1.f - y.x * y.x; g.y *= 1.f - y.y * y.y; g.z *= 1.f - y.z * y.z; g.w *= 1.f - y.w * y.w; }
      else if (act == MILB200_ACT_RELU) { g.x = y.x > 0.f ? g.x : 0.f; g.y = y.y > 0.f ? g.y : 0.f; g.z = y.z > 0.f ? g.z : 0.f; g.w = y.w > 0.f ? g.w : 0.f; }
      else { g.x *= y.x * (1.f - y.x); g.y *= y.y * (1.f - y.y); g.z *= y.z * (1.f - y.z); g.w *= y.w * (1.f - y.w); }
    }
    reinterpret_cast<uint2*>(out)[i] = make_uint2(pack_bf16(g.x, g.y), pack_bf16(g.z, g.w));
  }
}

// out[c] (+)= sum_r A[r, c]
template <typename T>
__global__ void __launch_bounds__(256)
k_colsum(const T* __restrict__ A, int64_t rows, int cols, float* __restrict__ out, int rows_per_block) {
  const int64_t r0 = static_cast<int64_t>(blockIdx.x) * rows_per_block;
  const int64_t r1 = (r0 + rows_per_block < rows) ? r0 + rows_per_block : rows;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) {
    float a = 0.f;
    for (int64_t r = r0; r < r1; ++r) a += to_f32<T>(A[r * cols + c]);
    atomicAdd(out + c, a);
  }
}

// Deterministic variant (what the library uses): one CTA owns ONE 16-byte vector column over ALL rows, so there is no
// cross-CTA reduction and no atomics; threads stride the rows with four independent loads in flight, then fold through
// a fixed shuffle tree and a fixed-order pass over the warps' partials.  `accumulate` is applied by the single writer
// (no memset node in front).  The operand is the tensor the previous kernel just wrote (L2-resident), so the half-used
// 32-byte sectors of the 16-byte-wide stripes cost L2 bandwidth, not HBM.
template <typename T>
__global__ void __launch_bounds__(1024)
k_colsum_det(const T* __restrict__ A, int64_t rows, int cols, float* __restrict__ out, int accumulate) {
  constexpr int VN = Vec16<T>::N;
  __shared__ float red[32][VN];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int nvec = cols / VN;
  const uint4* base = reinterpret_cast<const uint4*>(A) + blockIdx.x;
  float acc[VN];
#pragma unroll
  for (int e = 0; e < VN; ++e) acc[e] = 0.f;
  const int64_t step = blockDim.x;
  int64_t r = threadIdx.x;
  for (; r + 3 * step < rows; r += 4 * step) {
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = ldg_stream(base + (r + u * step) * nvec);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float f[VN];
      Vec16<T>::unpack(v[u], f);
#pragma unroll
      for (int e = 0; e < VN; ++e) acc[e] += f[e];
    }
  }
  for (; r < rows; r += step) {
    float f[VN];
    Vec16<T>::unpack(ldg_stream(base + r * nvec), f);
#pragma unroll
    for (int e = 0; e < VN; ++e) acc[e] += f[e];
  }
#pragma unroll
  for (int e = 0; e < VN; ++e) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], o);
  }
  if (lane == 0) {
#pragma unroll
    for (int e = 0; e < VN; ++e) red[warp][e] = acc[e];
  }
  __syncthreads();
  if (threadIdx.x < VN) {
    float a = 0.f;
    for (int w = 0; w < nwarp; ++w) a += red[w][threadIdx.x];
    float* o = out + static_cast<int64_t>(blockIdx.x) * VN + threadIdx.x;
    *o = accumulate ? *o + a : a;
  }
}

// out[c] = (accumulate ? out[c] : 0) + sum_r A[r, c]
template <typename T>
static int colsum_launch(const T* A, int64_t rows, int cols, float* out, int accumulate, cudaStream_t st) {
  constexpr int VN = Vec16<T>::N;
  if (cols % VN == 0 && aligned16(A)) {
    int threads = static_cast<int>(std::min<int64_t>(1024, ((rows + 31) / 32) * 32));
    k_colsum_det<T><<<static_cast<unsigned>(cols / VN), threads, 0, st>>>(A, rows, cols, out, accumulate);
  } else {   // odd widths (no caller on the shipped path): the atomic kernels
    if (!accumulate) MIL_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * cols, st));
    int rpb = 128;
    k_colsum<T><<<static_cast<unsigned>((rows + rpb - 1) / rpb), 256, 0, st>>>(A, rows, cols, out, rpb);
  }
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

static size_t simt_splits(int64_t K) {
  int64_t s = K / 512;
  if (s < 1) s = 1;
  if (s > 64) s = 64;
  return static_cast<size_t>(s);
}

static bool tc_gate_ok(int L, int D, int dtype) {
  // L % 16: the input-gradient GEMM dX = dZ Wcat (N = L) runs on the tensor-core kernel, which takes N in steps of 16
  return dtype == MILB200_BF16 && D == tc::GATE_D && L >= 64 && L % 16 == 0 && !force_simt();
}
// The tensor-core gate kernels want the packed weight rows in interleaved-halves order (see tc_gemm.cu);
// milb200_pack_gate_weights asks here so that packer and consumer always agree.
bool gate_layout_interleaved(int L, int D, int dtype) { return tc_gate_ok(L, D, dtype); }

// ---- 3xTF32: the fp32 path on the tensor cores -----------------------------------------------------
// The reference computes in fp32 (no AMP anywhere in train_ddp.py); kind::tf32 MMAs over hi/lo operand splits give
// fp32-grade products (see k_gemm_kmajor, KIND 1).  hi = the nearest tf32 value of x, lo = the nearest tf32 value of
// x - hi: both are exact tf32 operands whether the tensor core truncates or rounds its inputs, the residual is 2^-22 |x|
// with either sign (a truncating split biases every product the same way and showed up as 1.1e-5 on single scores).
constexpr int TF32_CK = 512;   // k (= instance rows) per batch of the split-K dWcat product
constexpr int64_t TF32_MIN_ROWS = 4096;   // below this the row-tile-persistent GEMM leaves most SMs idle and the splits /
                                          // transposes cost more than the FFMA kernels (measured: 1 000 rows 2.2 vs 1.8 ms)

static bool tf32x3_enabled() {           // MILB200_TF32X3=0 keeps the FFMA kernels (read per call: tests flip it)
  const char* e = getenv("MILB200_TF32X3");
  return !(e && e[0] == '0');
}
// gate GEMMs in fp32: Z = X Wcat^T needs K = L, dWcat needs Mb = 2D (multiple of 128), N = L
static bool tf32_gate_ok(int L, int D, int dtype, int64_t rows = TF32_MIN_ROWS) {
  return rows >= TF32_MIN_ROWS && dtype == MILB200_F32 && tf32x3_enabled() && !force_simt() && (2 * D) % 128 == 0 && L % 16 == 0 && L >= 32 &&
         tc::gemm_tf32x3_supported(128, 2 * D, L);
}

__device__ __forceinline__ float tf32_rn(float x) {   // nearest tf32 value (ties away), returned as fp32
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}

__global__ void __launch_bounds__(256)
k_tf32_split(const float4* __restrict__ in, float4* __restrict__ hi, float4* __restrict__ lo, int64_t n4) {
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n4;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float4 x = __ldg(in + i);
    const float4 h = make_float4(tf32_rn(x.x), tf32_rn(x.y), tf32_rn(x.z), tf32_rn(x.w));
    hi[i] = h;
    lo[i] = make_float4(tf32_rn(x.x - h.x), tf32_rn(x.y - h.y), tf32_rn(x.z - h.z), tf32_rn(x.w - h.w));
  }
}
static int tf32_split(const float* in, float* hi, float* lo, int64_t n, cudaStream_t st) {   // n % 4 == 0
  const int64_t n4 = n / 4;
  unsigned blocks = static_cast<unsigned>(std::min<int64_t>((n4 + 255) / 256, static_cast<int64_t>(sm_count()) * 16));
  k_tf32_split<<<blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(in), reinterpret_cast<float4*>(hi),
                                       reinterpret_cast<float4*>(lo), n4);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

// in [rows, cols] -> hi/lo [batches][cols][TF32_CK] with row r at (batch r / CK, k = r % CK); rows past the end are zero:
// the K-major operands of the batched dWcat product (contraction over the instance rows)
__global__ void __launch_bounds__(256)
k_tf32_transpose_split(const float* __restrict__ in, int64_t rows, int cols, float* __restrict__ hi, float* __restrict__ lo) {
  __shared__ float t[32][33];
  const int64_t r0 = static_cast<int64_t>(blockIdx.y) * 32;
  const int c0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int64_t r = r0 + ty + 8 * j;
    const int c = c0 + tx;
    t[ty + 8 * j][tx] = (r < rows && c < cols) ? __ldg(in + r * cols + c) : 0.f;
  }
  __syncthreads();
  const int64_t batch = r0 / TF32_CK;
  const int k0 = static_cast<int>(r0 % TF32_CK);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = c0 + ty + 8 * j;
    if (c < cols) {
      const float x = t[tx][ty + 8 * j];
      const float h = tf32_rn(x);
      const int64_t o = (batch * cols + c) * TF32_CK + k0 + tx;
      hi[o] = h;
      lo[o] = tf32_rn(x - h);
    }
  }
}
static int tf32_transpose_split(const float* in, int64_t rows, int cols, float* hi, float* lo, cudaStream_t st) {
  const int64_t rows_pad = (rows + TF32_CK - 1) / TF32_CK * TF32_CK;
  dim3 grid(static_cast<unsigned>((cols + 31) / 32), static_cast<unsigned>(rows_pad / 32));
  k_tf32_transpose_split<<<grid, 256, 0, st>>>(in, rows, cols, hi, lo);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

// ---- workspace layouts ---------------------------------------------------------------------------
struct GateWs {
  // tensor-core path
  size_t dz, colsum, part, wT;
  // FFMA path
  size_t z, spart, rec;
  // 3xTF32 path (fp32 operands): hi/lo splits of Wcat and of the row chunk, transposed splits for dWcat, partials
  size_t whi, wlo, xhi, xlo, dzt_hi, dzt_lo, xt_hi, xt_lo, tpart;
  size_t total;
};
static GateWs gate_ws(int64_t total_n, int L, int D, int dtype, int backward) {
  GateWs w{};
  size_t off = 0;
  auto take = [&](size_t bytes) {
    size_t o = align_up(off, 256);
    off = o + bytes;
    return o;
  };
  if (tc_gate_ok(L, D, dtype)) {
    if (backward) {
      w.dz = take(static_cast<size_t>(total_n) * 2 * D * 2);
      w.colsum = take(sizeof(float) * tc::CS_STRIDE * static_cast<size_t>(tc::gated_dz_max_records()));
      w.part = take(sizeof(float) * static_cast<size_t>(tc::gemm_tn_max_splits(2 * D, L)) * 2 * D * L);
      w.wT = take(static_cast<size_t>(2) * D * L * 2);
    }
  } else {
    int64_t rows = std::min<int64_t>(total_n, SIMT_ROW_CHUNK);
    w.z = take(sizeof(float) * static_cast<size_t>(rows) * 2 * D);
    if (backward) {
      w.spart = take(sizeof(float) * simt_splits(rows) * 2 * D * L);
      w.rec = take(sizeof(float) * static_cast<size_t>(sm_count()) * 4 * (3 * D + 1));
    }
    if (tf32_gate_ok(L, D, dtype, total_n)) {
      const size_t rows_pad = static_cast<size_t>((rows + TF32_CK - 1) / TF32_CK * TF32_CK);
      w.whi = take(sizeof(float) * 2 * D * L);
      w.wlo = take(sizeof(float) * 2 * D * L);
      w.xhi = take(sizeof(float) * static_cast<size_t>(rows) * L);
      w.xlo = take(sizeof(float) * static_cast<size_t>(rows) * L);
      if (backward) {
        w.dzt_hi = take(sizeof(float) * rows_pad * 2 * D);
        w.dzt_lo = take(sizeof(float) * rows_pad * 2 * D);
        w.xt_hi = take(sizeof(float) * rows_pad * L);
        w.xt_lo = take(sizeof(float) * rows_pad * L);
        w.tpart = take(sizeof(float) * (rows_pad / TF32_CK) * 2 * D * L);
      }
    }
  }
  w.total = align_up(off, 256) + 256;
  return w;
}

template <typename T>
static int gate_fwd_simt(const T* X, const T* Wcat, const float* bcat, const float* ww, const float* bw, float* scores,
                         int64_t total_n, int L, int D, char* ws, const GateWs& w, cudaStream_t st) {
  float* Z = reinterpret_cast<float*>(ws + w.z);
  for (int64_t r0 = 0; r0 < total_n; r0 += SIMT_ROW_CHUNK) {
    int64_t rows = std::min<int64_t>(SIMT_ROW_CHUNK, total_n - r0);
    simt::EpiStore<float> ep{Z, 2 * D, bcat, MILB200_ACT_NONE, nullptr, nullptr, nullptr, 0, 0};
    int rc = simt::launch<T, T, true, true>(X + r0 * L, L, Wcat, L, rows, 2 * D, L, 1, ep, st);
    if (rc) return rc;
    k_gate_fwd<<<static_cast<unsigned>((rows + 7) / 8), 256, 0, st>>>(Z, ww, bw, scores + r0, rows, D);
    MIL_LAUNCH_CHECK();
  }
  return MILB200_OK;
}

template <typename T>
static int gate_bwd_simt(const T* X, const T* Wcat, const float* bcat, const float* ww, const float* dscores,
                         const float* attn, const float* dM, const int32_t* offsets, int B, int64_t total_n, int L,
                         int D, float* dWcat, float* dbcat, float* dww, float* dbw, T* dX, char* ws, const GateWs& w,
                         cudaStream_t st) {
  MIL_CHECK_ARG(D <= 32 * GATE_MAX_DPL, MILB200_EUNSUPPORTED, "gated_score_bwd (FFMA path): D=%d > %d", D, 32 * GATE_MAX_DPL);
  float* Z = reinterpret_cast<float*>(ws + w.z);
  float* part = reinterpret_cast<float*>(ws + w.spart);
  float* rec = reinterpret_cast<float*>(ws + w.rec);
  int chunk = 0;
  for (int64_t r0 = 0; r0 < total_n; r0 += SIMT_ROW_CHUNK, ++chunk) {
    int64_t rows = std::min<int64_t>(SIMT_ROW_CHUNK, total_n - r0);
    simt::EpiStore<float> ep{Z, 2 * D, bcat, MILB200_ACT_NONE, nullptr, nullptr, nullptr, 0, 0};
    int rc = simt::launch<T, T, true, true>(X + r0 * L, L, Wcat, L, rows, 2 * D, L, 1, ep, st);
    if (rc) return rc;
    unsigned blocks = static_cast<unsigned>(std::min<int64_t>((rows + 7) / 8, sm_count() * 4));
    k_gate_bwd<<<blocks, 256, 0, st>>>(Z, Z, ww, dscores + r0, rows, D, rec);
    MIL_LAUNCH_CHECK();
    k_gate_bwd_fold<<<(3 * D + 1 + 31) / 32, 256, 0, st>>>(rec, static_cast<int>(blocks), D, dbcat, dww, dbw, chunk > 0);
    MIL_LAUNCH_CHECK();
    // dWcat[j, l] (+)= sum_i dZ[i, j] X[i, l]
    int splits = static_cast<int>(simt_splits(rows));
    simt::EpiPartial pe{part, 2 * D, L};
    rc = simt::launch<float, T, false, false>(Z, 2 * D, X + r0 * L, L, 2 * D, L, rows, splits, pe, st);
    if (rc) return rc;
    rc = splitk_reduce(part, splits, static_cast<int64_t>(2) * D * L, dWcat, chunk > 0, st);
    if (rc) return rc;
    if (dX) {
      // dX[i, l] = sum_j dZ[i, j] Wcat[j, l]  (+ attn_i * dM[bag(i), l])
      simt::EpiStore<T> ex{dX + r0 * L, L, nullptr, MILB200_ACT_NONE, attn, dM, offsets, B, r0};
      rc = simt::launch<float, T, true, false>(Z, 2 * D, Wcat, L, rows, L, 2 * D, 1, ex, st);
      if (rc) return rc;
    }
  }
  return MILB200_OK;
}

// fp32 operands on the tensor cores (3xTF32): same sequence as the FFMA path with the GEMMs replaced
static int gate_fwd_tf32(const float* X, const float* Wcat, const float* bcat, const float* ww, const float* bw, float* scores,
                         float* zsave, int64_t total_n, int L, int D, char* ws, const GateWs& w, cudaStream_t st) {
  float* Zws = reinterpret_cast<float*>(ws + w.z);
  float* whi = reinterpret_cast<float*>(ws + w.whi);
  float* wlo = reinterpret_cast<float*>(ws + w.wlo);
  float* xhi = reinterpret_cast<float*>(ws + w.xhi);
  float* xlo = reinterpret_cast<float*>(ws + w.xlo);
  int rc = tf32_split(Wcat, whi, wlo, static_cast<int64_t>(2) * D * L, st);
  if (rc) return rc;
  for (int64_t r0 = 0; r0 < total_n; r0 += SIMT_ROW_CHUNK) {
    int64_t rows = std::min<int64_t>(SIMT_ROW_CHUNK, total_n - r0);
    rc = tf32_split(X + r0 * L, xhi, xlo, rows * L, st);
    if (rc) return rc;
    float* Z = zsave ? zsave + r0 * 2 * D : Zws;       // saved pre-activations (bias included): the backward skips this GEMM
    rc = tc::gemm_store_tf32x3(xhi, xlo, rows, L, L, whi, wlo, 2 * D, L, bcat, MILB200_ACT_NONE, Z, 2 * D, st);
    if (rc) return rc;
    k_gate_fwd<<<static_cast<unsigned>((rows + 7) / 8), 256, 0, st>>>(Z, ww, bw, scores + r0, rows, D);
    MIL_LAUNCH_CHECK();
  }
  return MILB200_OK;
}

static int gate_bwd_tf32(const float* X, const float* Wcat, const float* bcat, const float* ww, const float* dscores,
                         const float* zsaved, const float* attn, const float* dM, const int32_t* offsets, int B, int64_t total_n, int L,
                         int D, float* dWcat, float* dbcat, float* dww, float* dbw, float* dX, char* ws, const GateWs& w,
                         cudaStream_t st) {
  MIL_CHECK_ARG(D <= 32 * GATE_MAX_DPL, MILB200_EUNSUPPORTED, "gated_score_bwd (3xTF32 path): D=%d > %d", D, 32 * GATE_MAX_DPL);
  float* Z = reinterpret_cast<float*>(ws + w.z);
  float* rec = reinterpret_cast<float*>(ws + w.rec);
  float* whi = reinterpret_cast<float*>(ws + w.whi);
  float* wlo = reinterpret_cast<float*>(ws + w.wlo);
  float* xhi = reinterpret_cast<float*>(ws + w.xhi);
  float* xlo = reinterpret_cast<float*>(ws + w.xlo);
  float* dzt_hi = reinterpret_cast<float*>(ws + w.dzt_hi);
  float* dzt_lo = reinterpret_cast<float*>(ws + w.dzt_lo);
  float* xt_hi = reinterpret_cast<float*>(ws + w.xt_hi);
  float* xt_lo = reinterpret_cast<float*>(ws + w.xt_lo);
  float* part = reinterpret_cast<float*>(ws + w.tpart);
  int rc = MILB200_OK;
  if (!zsaved) {
    rc = tf32_split(Wcat, whi, wlo, static_cast<int64_t>(2) * D * L, st);
    if (rc) return rc;
  }
  int chunk = 0;
  for (int64_t r0 = 0; r0 < total_n; r0 += SIMT_ROW_CHUNK, ++chunk) {
    int64_t rows = std::min<int64_t>(SIMT_ROW_CHUNK, total_n - r0);
    if (!zsaved) {       // nothing saved: recompute the pre-activations of the chunk
      rc = tf32_split(X + r0 * L, xhi, xlo, rows * L, st);
      if (rc) return rc;
      rc = tc::gemm_store_tf32x3(xhi, xlo, rows, L, L, whi, wlo, 2 * D, L, bcat, MILB200_ACT_NONE, Z, 2 * D, st);
      if (rc) return rc;
    }
    unsigned blocks = static_cast<unsigned>(std::min<int64_t>((rows + 7) / 8, sm_count() * 4));
    k_gate_bwd<<<blocks, 256, 0, st>>>(zsaved ? zsaved + r0 * 2 * D : Z, Z, ww, dscores + r0, rows, D, rec);   // -> dZ
    MIL_LAUNCH_CHECK();
    k_gate_bwd_fold<<<(3 * D + 1 + 31) / 32, 256, 0, st>>>(rec, static_cast<int>(blocks), D, dbcat, dww, dbw, chunk > 0);
    MIL_LAUNCH_CHECK();
    // dWcat[j, l] (+)= sum_i dZ[i, j] X[i, l]: K-major operands = the transposes, split-K over batches of TF32_CK rows
    const int batches = static_cast<int>((rows + TF32_CK - 1) / TF32_CK);
    rc = tf32_transpose_split(Z, rows, 2 * D, dzt_hi, dzt_lo, st);
    if (rc) return rc;
    rc = tf32_transpose_split(X + r0 * L, rows, L, xt_hi, xt_lo, st);
    if (rc) return rc;
    rc = tc::gemm_batched_tf32x3(dzt_hi, dzt_lo, batches, 2 * D, TF32_CK, xt_hi, xt_lo, L, part, st);
    if (rc) return rc;
    rc = splitk_reduce(part, batches, static_cast<int64_t>(2) * D * L, dWcat, chunk > 0, st);
    if (rc) return rc;
    if (dX) {
      // dX[i, l] = sum_j dZ[i, j] Wcat[j, l]  (+ attn_i * dM[bag(i), l], in the epilogue): A = dZ (K = 2D), B = Wcat^T as one
      // zero-padded 512-column batch (2D <= 512); dZ's splits reuse the X-split buffers (X's are not needed any more)
      if (2 * D <= TF32_CK && 2 * D <= L) {
        rc = tf32_transpose_split(Wcat, 2 * D, L, xt_hi, xt_lo, st);        // [L][512]; the dW product above is done with xt_*
        if (rc) return rc;
        rc = tf32_split(Z, xhi, xlo, rows * 2 * D, st);
        if (rc) return rc;
        rc = tc::gemm_store_tf32x3(xhi, xlo, rows, 2 * D, 2 * D, xt_hi, xt_lo, L, TF32_CK, nullptr, MILB200_ACT_NONE,
                                   dX + r0 * L, L, st, attn, dM, offsets, B, r0);
        if (rc) return rc;
      } else {
        simt::EpiStore<float> ex{dX + r0 * L, L, nullptr, MILB200_ACT_NONE, attn, dM, offsets, B, r0};
        rc = simt::launch<float, float, true, false>(Z, 2 * D, Wcat, L, rows, L, 2 * D, 1, ex, st);
        if (rc) return rc;
      }
    }
  }
  return MILB200_OK;
}

// ---- linear workspace ------------------------------------------------------------------------------
struct LinWs {
  size_t xin, dypre, wT, part, smallm;
  // 3xTF32 path (fp32 operands, m >= TF32_MIN_ROWS): hi/lo splits of X and W; backward: transposed splits of dYpre and X and the
  // batched partials (dW), splits of dYpre and of W^T padded to 512 columns (dX)
  size_t t_xhi, t_xlo, t_whi, t_wlo, t_dyt_hi, t_dyt_lo, t_xt_hi, t_xt_lo, t_part, t_dyhi, t_dylo, t_wt_hi, t_wt_lo;
  size_t total;
};
static bool tf32_linear_ok(int64_t m, int n, int k, int dtype) {
  return dtype == MILB200_F32 && tf32x3_enabled() && !force_simt() && m >= TF32_MIN_ROWS && tc::gemm_tf32x3_supported(m, n, k);
}
static bool tf32_linear_dw_ok(int64_t m, int n, int k, int dtype) {   // dW[n, k] = dYpre^T X: Mb = n, N = k
  return tf32_linear_ok(m, n, k, dtype) && n % 128 == 0 && k % 16 == 0;
}
static bool tf32_linear_dx_ok(int64_t m, int n, int k, int dtype) {   // dX[m, k] = dYpre W: K = n (one 512-column batch of W^T)
  return tf32_linear_ok(m, n, k, dtype) && n <= TF32_CK && tc::gemm_tf32x3_supported(m, k, n);
}
static bool tc_linear_ok(int64_t m, int n, int k, int dtype) {
  return dtype == MILB200_BF16 && !force_simt() && tc::gemm_store_supported(m, n, k);
}
static bool tc_linear_bwd_ok(int64_t m, int n, int k, int dtype) {
  // dX = dYpre[m,n] . Wt[k,n]^T needs the reduction dim n >= 64; dW = dYpre^T X needs both >= 64
  return dtype == MILB200_BF16 && !force_simt() && tc::gemm_store_supported(m, k, n) && tc::gemm_tn_supported(n, k);
}
static LinWs linear_ws(int64_t m, int n, int k, int dtype, int backward, int has_add) {
  LinWs w{};
  size_t off = 0;
  const size_t e = elem_size(dtype);
  auto take = [&](size_t bytes) {
    size_t o = align_up(off, 256);
    off = o + bytes;
    return o;
  };
  if (has_add) w.xin = take(static_cast<size_t>(m) * k * e);
  if (backward) {
    w.dypre = take(static_cast<size_t>(m) * n * e);
    w.wT = take(static_cast<size_t>(n) * k * e);
    size_t splits = tc_linear_bwd_ok(m, n, k, dtype) ? static_cast<size_t>(tc::gemm_tn_max_splits(n, k)) : simt_splits(m);
    w.part = take(sizeof(float) * splits * n * k);
    if (smallm_ok(m, n, k, dtype)) w.smallm = take(smallm_ws_bytes(m, k));
  }
  if (tf32_linear_ok(m, n, k, dtype)) {
    const size_t f = sizeof(float);
    const size_t m_pad = static_cast<size_t>((m + TF32_CK - 1) / TF32_CK * TF32_CK);
    w.t_xhi = take(f * m * k);
    w.t_xlo = take(f * m * k);
    w.t_whi = take(f * n * k);
    w.t_wlo = take(f * n * k);
    if (backward) {
      if (tf32_linear_dw_ok(m, n, k, dtype)) {
        w.t_dyt_hi = take(f * m_pad * n);
        w.t_dyt_lo = take(f * m_pad * n);
        w.t_xt_hi = take(f * m_pad * k);
        w.t_xt_lo = take(f * m_pad * k);
        w.t_part = take(f * (m_pad / TF32_CK) * n * k);
      }
      if (tf32_linear_dx_ok(m, n, k, dtype)) {
        w.t_dyhi = take(f * m * n);
        w.t_dylo = take(f * m * n);
        w.t_wt_hi = take(f * static_cast<size_t>(k) * TF32_CK);
        w.t_wt_lo = take(f * static_cast<size_t>(k) * TF32_CK);
      }
    }
  }
  w.total = align_up(off, 256) + 256;
  return w;
}

}  // namespace milb200

using namespace milb200;

extern "C" {

int milb200_add(const void* a, const void* b, void* out, int64_t n, int dtype, void* stream);

/* Developer/bench hook: when enabled, the tensor-core path of milb200_gated_score_bwd records CUDA events
 * between its sub-kernels (dz recompute | dW split-K GEMM | split-K reduce | dX GEMM);
 * milb200_profile_read synchronises on the last event and returns the interval durations in ms. */
int milb200_colsum(const void* A, int64_t rows, int cols, float* out, int dtype, int accumulate, void* stream) {
  MIL_CHECK_ARG(A && out && rows > 0 && cols > 0, MILB200_EINVAL, "colsum: bad arguments");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (dtype == MILB200_BF16)
    return colsum_launch<__nv_bfloat16>(static_cast<const __nv_bfloat16*>(A), rows, cols, out, accumulate, st);
  return colsum_launch<float>(static_cast<const float*>(A), rows, cols, out, accumulate, st);
}

int milb200_debug_trace(void* dev_u64x16) { return tc::debug_set_trace(dev_u64x16); }
void milb200_profile_enable(int on) { g_prof_on = on != 0; g_prof_n = 0; }
int milb200_profile_read(float* ms, int max_intervals) {
  int n = g_prof_n - 1;
  if (n <= 0 || !ms) return 0;
  if (n > max_intervals) n = max_intervals;
  cudaEventSynchronize(g_prof_ev[g_prof_n - 1]);
  for (int i = 0; i < n; ++i) cudaEventElapsedTime(ms + i, g_prof_ev[i], g_prof_ev[i + 1]);
  return n;
}

size_t milb200_gated_score_workspace_bytes(int64_t total_n, int L, int D, int dtype, int backward) {
  if (total_n <= 0 || L <= 0 || D <= 0) return 256;
  return gate_ws(total_n, L, D, dtype, backward).total;
}

int milb200_gated_score_saves_activations(int L, int D, int dtype) {
  return (tc_gate_ok(L, D, dtype) || tf32_gate_ok(L, D, dtype)) ? 1 : 0;
}

int milb200_gated_score_fwd(const void* X, const void* Wcat, const float* bcat, const float* ww, const float* bw,
                            float* scores, void* gate_act, int64_t total_n, int L, int D, int dtype, void* workspace,
                            size_t ws_bytes, void* stream) {
  MIL_CHECK_ARG(X && Wcat && bcat && ww && bw && scores, MILB200_EINVAL, "gated_score_fwd: null pointer");
  MIL_CHECK_ARG(total_n > 0 && L > 0 && D > 0, MILB200_EINVAL, "gated_score_fwd: total_n=%lld L=%d D=%d must be positive",
                (long long)total_n, L, D);
  MIL_CHECK_ARG(dtype == MILB200_F32 || dtype == MILB200_BF16, MILB200_EINVAL, "gated_score_fwd: bad dtype %d", dtype);
  MIL_CHECK_ARG(aligned16(X) && aligned16(Wcat) && (L * elem_size(dtype)) % 16 == 0, MILB200_EALIGN,
                "gated_score_fwd: X/Wcat must be 16-byte aligned with a 16-byte multiple row pitch");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (tc_gate_ok(L, D, dtype)) {
    MIL_CHECK_ARG(gate_act == nullptr || aligned16(gate_act), MILB200_EALIGN, "gated_score_fwd: gate_act must be 16-byte aligned");
    return tc::gated_score(X, total_n, L, Wcat, bcat, ww, bw, scores, gate_act, st);
  }
  // FFMA path: nothing is saved (its backward recomputes the pre-activations chunk by chunk)
  GateWs w = gate_ws(total_n, L, D, dtype, 0);
  MIL_CHECK_ARG(workspace && ws_bytes >= w.total, MILB200_EWORKSPACE, "gated_score_fwd: workspace %zu < %zu", ws_bytes, w.total);
  char* ws = static_cast<char*>(workspace);
  if (dtype == MILB200_BF16)
    return gate_fwd_simt<__nv_bfloat16>((const __nv_bfloat16*)X, (const __nv_bfloat16*)Wcat, bcat, ww, bw, scores, total_n,
                                        L, D, ws, w, st);
  if (tf32_gate_ok(L, D, dtype, total_n))
    return gate_fwd_tf32((const float*)X, (const float*)Wcat, bcat, ww, bw, scores, static_cast<float*>(gate_act), total_n, L,
                         D, ws, w, st);
  return gate_fwd_simt<float>((const float*)X, (const float*)Wcat, bcat, ww, bw, scores, total_n, L, D, ws, w, st);
}

int milb200_gated_score_bwd(const void* X, const void* Wcat, const float* bcat, const float* ww, const float* bw,
                            const float* dscores, const void* gate_act, const float* attn, const float* dM,
                            const int32_t* offsets, int B,
                            int64_t total_n, int L, int D, int dtype, float* dWcat, float* dbcat, float* dww, float* dbw,
                            void* dX, void* workspace, size_t ws_bytes, void* stream) {
  (void)bw;
  MIL_CHECK_ARG(X && Wcat && bcat && ww && dscores && dWcat && dbcat && dww && dbw, MILB200_EINVAL,
                "gated_score_bwd: null pointer");
  MIL_CHECK_ARG(total_n > 0 && L > 0 && D > 0, MILB200_EINVAL, "gated_score_bwd: bad shape");
  MIL_CHECK_ARG(dtype == MILB200_F32 || dtype == MILB200_BF16, MILB200_EINVAL, "gated_score_bwd: bad dtype %d", dtype);
  MIL_CHECK_ARG(attn == nullptr || (dM && offsets && B > 0), MILB200_EINVAL,
                "gated_score_bwd: attn given without dM/offsets");
  MIL_CHECK_ARG(aligned16(X) && aligned16(Wcat) && (L * elem_size(dtype)) % 16 == 0, MILB200_EALIGN,
                "gated_score_bwd: X/Wcat must be 16-byte aligned with a 16-byte multiple row pitch");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  GateWs w = gate_ws(total_n, L, D, dtype, 1);
  MIL_CHECK_ARG(workspace && ws_bytes >= w.total, MILB200_EWORKSPACE, "gated_score_bwd: workspace %zu < %zu", ws_bytes, w.total);
  char* ws = static_cast<char*>(workspace);
  if (tc_gate_ok(L, D, dtype)) {
    void* dZ = ws + w.dz;
    float* colsum = reinterpret_cast<float*>(ws + w.colsum);
    float* part = reinterpret_cast<float*>(ws + w.part);
    int nrec = 0, splits = 0;
    g_prof_n = 0;
    prof_mark(st);
    int rc;
    if (gate_act && !dX) {
      // saved V,U and no input gradient wanted: dZ is never materialised — the dW GEMM builds its A operand from V,U
      MIL_CHECK_ARG(aligned16(gate_act), MILB200_EALIGN, "gated_score_bwd: gate_act must be 16-byte aligned");
      rc = tc::gemm_tn_gate(gate_act, dscores, ww, X, L, total_n, L, part, &splits, colsum, st);
      if (rc) return rc;
      prof_mark(st);
      k_colsum_finalize_tn<<<(3 * D + 1 + 255) / 256, 256, 0, st>>>(colsum, splits, tc::gemm_tn_gate_record_floats(), dbcat,
                                                                    dww, dbw, D);
      MIL_LAUNCH_CHECK();
      rc = splitk_reduce_gate64(part, splits, D, L, dWcat, st);
      if (rc) return rc;
      prof_mark(st);
      return MILB200_OK;
    }
    if (gate_act) {
      // saved V,U: dZ is an elementwise pass (1.5 KB of traffic per instance instead of the recompute GEMM)
      MIL_CHECK_ARG(aligned16(gate_act), MILB200_EALIGN, "gated_score_bwd: gate_act must be 16-byte aligned");
      int64_t blocks = std::min<int64_t>((total_n + 63) / 64, static_cast<int64_t>(sm_count()) * 4);
      int64_t rpb = (total_n + blocks - 1) / blocks;
      rpb = (rpb + DZS_RG - 1) / DZS_RG * DZS_RG;
      nrec = static_cast<int>((total_n + rpb - 1) / rpb);
      k_gate_dz_saved<<<nrec, DZS_THREADS, 0, st>>>((const __nv_bfloat16*)gate_act, ww, dscores, total_n, rpb,
                                                    (__nv_bfloat16*)dZ, colsum, tc::CS_STRIDE);
      MIL_LAUNCH_CHECK();
      k_colsum_finalize_flat<<<(3 * D + 1 + 31) / 32, 256, 0, st>>>(colsum, nrec, tc::CS_STRIDE, dbcat, dww, dbw, D);
      MIL_LAUNCH_CHECK();
    } else {
      rc = tc::gated_dz(X, total_n, L, Wcat, bcat, ww, dscores, dZ, colsum, &nrec, st);
      if (rc) return rc;
      k_colsum_finalize<<<(3 * D + 1 + 255) / 256, 256, 0, st>>>(colsum, nrec, tc::CS_STRIDE, dbcat, dww, dbw, D);
      MIL_LAUNCH_CHECK();
    }
    prof_mark(st);
    rc = tc::gemm_tn_splitk(dZ, 2 * D, X, L, total_n, 2 * D, L, part, &splits, st);
    if (rc) return rc;
    prof_mark(st);
    rc = splitk_reduce_gate(part, splits, D, L, D / 2, dWcat, st);
    if (rc) return rc;
    prof_mark(st);
    if (dX) {
      void* wT = ws + w.wT;  // [L, 2D]: the K-contiguous B operand of dX = dZ . Wcat
      rc = transpose2d(Wcat, wT, 2 * D, L, MILB200_BF16, st);
      if (rc) return rc;
      rc = tc::gemm_store(dZ, total_n, 2 * D, 2 * D, wT, L, 2 * D, nullptr, MILB200_ACT_NONE, dX, MILB200_BF16, L, attn, dM,
                          offsets, B, st);
      if (rc) return rc;
      prof_mark(st);
    }
    return MILB200_OK;
  }
  if (dtype == MILB200_BF16)
    return gate_bwd_simt<__nv_bfloat16>((const __nv_bfloat16*)X, (const __nv_bfloat16*)Wcat, bcat, ww, dscores, attn, dM,
                                        offsets, B, total_n, L, D, dWcat, dbcat, dww, dbw, (__nv_bfloat16*)dX, ws, w, st);
  if (tf32_gate_ok(L, D, dtype, total_n))
    return gate_bwd_tf32((const float*)X, (const float*)Wcat, bcat, ww, dscores, static_cast<const float*>(gate_act), attn, dM,
                         offsets, B, total_n, L, D,
                         dWcat, dbcat, dww, dbw, (float*)dX, ws, w, st);
  return gate_bwd_simt<float>((const float*)X, (const float*)Wcat, bcat, ww, dscores, attn, dM, offsets, B, total_n, L, D,
                              dWcat, dbcat, dww, dbw, (float*)dX, ws, w, st);
}

// The mirrored single-pass backward was removed (DESIGN §5c): callers take the two-call backward.
int milb200_gated_pool_bwd_supported(int /*L*/, int /*D*/, int /*dtype*/) { return 0; }

// ---- dense linear ------------------------------------------------------------------------------------
size_t milb200_linear_workspace_bytes(int64_t m, int n, int k, int dtype, int backward) {
  if (m <= 0 || n <= 0 || k <= 0) return 256;
  return linear_ws(m, n, k, dtype, backward, 1).total;
}

static int linear_check(const void* X, const void* W, int64_t m, int n, int k, int dtype) {
  MIL_CHECK_ARG(X && W, MILB200_EINVAL, "linear: null pointer");
  MIL_CHECK_ARG(m > 0 && n > 0 && k > 0, MILB200_EINVAL, "linear: m=%lld n=%d k=%d must be positive", (long long)m, n, k);
  MIL_CHECK_ARG(dtype == MILB200_F32 || dtype == MILB200_BF16, MILB200_EINVAL, "linear: bad dtype %d", dtype);
  return MILB200_OK;
}

}  // extern "C"
template <typename T>
static int linear_fwd_simt(const T* X, const T* W, const float* bias, T* Y, int64_t m, int n, int k, int act,
                           cudaStream_t st) {
  simt::EpiStore<T> ep{Y, n, bias, act, nullptr, nullptr, nullptr, 0, 0};
  return simt::launch<T, T, true, true>(X, k, W, k, m, n, k, 1, ep, st);
}

extern "C" {
int milb200_linear_fwd(const void* X, const void* add, const void* W, const float* bias, void* Y, int64_t m, int n,
                       int k, int act, int dtype, void* workspace, size_t ws_bytes, void* stream) {
  int rc = linear_check(X, W, m, n, k, dtype);
  if (rc) return rc;
  MIL_CHECK_ARG(Y != nullptr, MILB200_EINVAL, "linear_fwd: Y is null");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (smallm_ok(m, n, k, dtype) && aligned16(X) && aligned16(W) && (!add || aligned16(add)))
    return smallm_fwd(X, add, W, bias, Y, m, n, k, act, dtype, st);
  const void* xin = X;
  if (add) {
    LinWs w = linear_ws(m, n, k, dtype, 0, 1);
    MIL_CHECK_ARG(workspace && ws_bytes >= w.total, MILB200_EWORKSPACE, "linear_fwd: workspace %zu < %zu", ws_bytes, w.total);
    void* tmp = static_cast<char*>(workspace) + w.xin;
    rc = milb200_add(X, add, tmp, m * k, dtype, stream);
    if (rc) return rc;
    xin = tmp;
  }
  if (tc_linear_ok(m, n, k, dtype) && aligned16(xin) && aligned16(W) && aligned16(Y))
    return tc::gemm_store(xin, m, k, k, W, n, k, bias, act, Y, MILB200_BF16, n, nullptr, nullptr, nullptr, 0, st);
  if (tf32_linear_ok(m, n, k, dtype) && aligned16(xin) && aligned16(W) && aligned16(Y)) {
    // fp32 operands on the tensor cores (3xTF32)
    LinWs w = linear_ws(m, n, k, dtype, 0, add != nullptr);
    MIL_CHECK_ARG(workspace && ws_bytes >= w.total, MILB200_EWORKSPACE, "linear_fwd: workspace %zu < %zu", ws_bytes, w.total);
    char* ws = static_cast<char*>(workspace);
    float* xhi = reinterpret_cast<float*>(ws + w.t_xhi);
    float* xlo = reinterpret_cast<float*>(ws + w.t_xlo);
    float* whi = reinterpret_cast<float*>(ws + w.t_whi);
    float* wlo = reinterpret_cast<float*>(ws + w.t_wlo);
    rc = tf32_split(static_cast<const float*>(xin), xhi, xlo, m * k, st);
    if (rc) return rc;
    rc = tf32_split(static_cast<const float*>(W), whi, wlo, static_cast<int64_t>(n) * k, st);
    if (rc) return rc;
    return tc::gemm_store_tf32x3(xhi, xlo, m, k, k, whi, wlo, n, k, bias, act, static_cast<float*>(Y), n, st);
  }
  if (dtype == MILB200_BF16)
    return linear_fwd_simt<__nv_bfloat16>((const __nv_bfloat16*)xin, (const __nv_bfloat16*)W, bias, (__nv_bfloat16*)Y, m,
                                          n, k, act, st);
  return linear_fwd_simt<float>((const float*)xin, (const float*)W, bias, (float*)Y, m, n, k, act, st);
}

}  // extern "C"
template <typename T>
static int linear_bwd_t(const T* Xin, const T* W, const T* Y, const T* dY, T* dX, float* dW, float* dbias, int64_t m,
                        int n, int k, int act, int dtype, int accumulate, char* ws, const LinWs& w, cudaStream_t st) {
  const T* dypre = dY;
  if (act != MILB200_ACT_NONE) {
    MIL_CHECK_ARG(Y != nullptr, MILB200_EINVAL, "linear_bwd: the forward output Y is required for act=%d", act);
    T* tmp = reinterpret_cast<T*>(ws + w.dypre);
    int64_t tot = m * n;
    unsigned blocks = static_cast<unsigned>(std::min<int64_t>((tot + 255) / 256, sm_count() * 8));
    k_act_bwd<T><<<blocks, 256, 0, st>>>(Y, dY, tmp, tot, act);
    MIL_LAUNCH_CHECK();
    dypre = tmp;
  }
  if (dbias) {
    int rcs = colsum_launch<T>(dypre, m, n, dbias, accumulate, st);
    if (rcs) return rcs;
  }
  float* part = reinterpret_cast<float*>(ws + w.part);
  const bool use_tc = tc_linear_bwd_ok(m, n, k, dtype) && aligned16(dypre) && aligned16(Xin) && aligned16(W);
  int rc;
  if constexpr (std::is_same<T, float>::value) {
    // fp32 operands on the tensor cores (3xTF32): dW through the transposed splits (split-K over batches of rows), dX with
    // W^T as one zero-padded 512-column batch
    const bool dw_tc = dW && tf32_linear_dw_ok(m, n, k, dtype) && aligned16(dypre) && aligned16(Xin);
    const bool dx_tc = dX && tf32_linear_dx_ok(m, n, k, dtype) && aligned16(dypre) && aligned16(W) && aligned16(dX);
    if (dw_tc) {
      float* dyt_hi = reinterpret_cast<float*>(ws + w.t_dyt_hi);
      float* dyt_lo = reinterpret_cast<float*>(ws + w.t_dyt_lo);
      float* xt_hi = reinterpret_cast<float*>(ws + w.t_xt_hi);
      float* xt_lo = reinterpret_cast<float*>(ws + w.t_xt_lo);
      float* tpart = reinterpret_cast<float*>(ws + w.t_part);
      const int batches = static_cast<int>((m + TF32_CK - 1) / TF32_CK);
      rc = tf32_transpose_split(dypre, m, n, dyt_hi, dyt_lo, st);
      if (rc) return rc;
      rc = tf32_transpose_split(Xin, m, k, xt_hi, xt_lo, st);
      if (rc) return rc;
      rc = tc::gemm_batched_tf32x3(dyt_hi, dyt_lo, batches, n, TF32_CK, xt_hi, xt_lo, k, tpart, st);
      if (rc) return rc;
      rc = splitk_reduce(tpart, batches, static_cast<int64_t>(n) * k, dW, accumulate, st);
      if (rc) return rc;
      dW = nullptr;
    }
    if (dx_tc) {
      float* dyhi = reinterpret_cast<float*>(ws + w.t_dyhi);
      float* dylo = reinterpret_cast<float*>(ws + w.t_dylo);
      float* wt_hi = reinterpret_cast<float*>(ws + w.t_wt_hi);
      float* wt_lo = reinterpret_cast<float*>(ws + w.t_wt_lo);
      rc = tf32_split(dypre, dyhi, dylo, m * n, st);
      if (rc) return rc;
      rc = tf32_transpose_split(W, n, k, wt_hi, wt_lo, st);     // W [n, k] -> [k][512], columns >= n zero
      if (rc) return rc;
      // K = n: the operands' rows are n (dYpre, ld n) and 512 (W^T, ld 512) floats long; TMA zero-fills dYpre past n
      rc = tc::gemm_store_tf32x3(dyhi, dylo, m, n, n, wt_hi, wt_lo, k, TF32_CK, nullptr, MILB200_ACT_NONE, dX, k, st);
      if (rc) return rc;
      dX = nullptr;
    }
  }
  if (dW) {
    int splits = 0;
    if (use_tc) {
      rc = tc::gemm_tn_splitk(dypre, n, Xin, k, m, n, k, part, &splits, st);
    } else {
      splits = static_cast<int>(simt_splits(m));
      simt::EpiPartial pe{part, n, k};
      rc = simt::launch<T, T, false, false>(dypre, n, Xin, k, n, k, m, splits, pe, st);
    }
    if (rc) return rc;
    rc = splitk_reduce(part, splits, static_cast<int64_t>(n) * k, dW, accumulate, st);
    if (rc) return rc;
  }
  if (dX) {
    if (use_tc) {
      T* wT = reinterpret_cast<T*>(ws + w.wT);  // [k, n]
      rc = transpose2d(W, wT, n, k, dtype, st);
      if (rc) return rc;
      rc = tc::gemm_store(dypre, m, n, n, wT, k, n, nullptr, MILB200_ACT_NONE, dX, MILB200_BF16, k, nullptr, nullptr,
                          nullptr, 0, st);
    } else {
      simt::EpiStore<T> ex{dX, k, nullptr, MILB200_ACT_NONE, nullptr, nullptr, nullptr, 0, 0};
      rc = simt::launch<T, T, true, false>(dypre, n, W, k, m, k, n, 1, ex, st);
    }
    if (rc) return rc;
  }
  return MILB200_OK;
}

extern "C" {
int milb200_linear_bwd(const void* X, const void* add, const void* W, const void* Y, const void* dY, void* dX,
                       float* dW, float* dbias, int64_t m, int n, int k, int act, int dtype, int accumulate,
                       void* workspace, size_t ws_bytes, void* stream) {
  int rc = linear_check(X, W, m, n, k, dtype);
  if (rc) return rc;
  MIL_CHECK_ARG(dY != nullptr, MILB200_EINVAL, "linear_bwd: dY is null");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (smallm_ok(m, n, k, dtype) && aligned16(X) && aligned16(W) && (!add || aligned16(add)) && aligned16(dW)) {
    MIL_CHECK_ARG(act == MILB200_ACT_NONE || Y != nullptr, MILB200_EINVAL, "linear_bwd: the forward output Y is required for act=%d", act);
    MIL_CHECK_ARG(dW != nullptr || dbias == nullptr, MILB200_EINVAL, "linear_bwd: dbias without dW");
    LinWs ws_ = linear_ws(m, n, k, dtype, 1, add != nullptr);
    MIL_CHECK_ARG(workspace && ws_bytes >= ws_.total, MILB200_EWORKSPACE, "linear_bwd: workspace %zu < %zu", ws_bytes, ws_.total);
    return smallm_bwd(X, add, W, Y, dY, dX, dW, dbias, m, n, k, act, dtype, accumulate,
                      reinterpret_cast<float*>(static_cast<char*>(workspace) + ws_.smallm), st);
  }
  LinWs w = linear_ws(m, n, k, dtype, 1, add != nullptr);
  MIL_CHECK_ARG(workspace && ws_bytes >= w.total, MILB200_EWORKSPACE, "linear_bwd: workspace %zu < %zu", ws_bytes, w.total);
  char* ws = static_cast<char*>(workspace);
  const void* xin = X;
  if (add && dW) {
    void* tmp = ws + w.xin;
    rc = milb200_add(X, add, tmp, m * k, dtype, stream);
    if (rc) return rc;
    xin = tmp;
  }
  if (dtype == MILB200_BF16)
    return linear_bwd_t<__nv_bfloat16>((const __nv_bfloat16*)xin, (const __nv_bfloat16*)W, (const __nv_bfloat16*)Y,
                                       (const __nv_bfloat16*)dY, (__nv_bfloat16*)dX, dW, dbias, m, n, k, act, dtype,
                                       accumulate, ws, w, st);
  return linear_bwd_t<float>((const float*)xin, (const float*)W, (const float*)Y, (const float*)dY, (float*)dX, dW, dbias,
                             m, n, k, act, dtype, accumulate, ws, w, st);
}


/* Mixed-precision linear for the head of the fusion path's key stream (fc_pathology, aggregator.py:141): X [m, k] and
 * W [n, k] bf16 on the tensor cores, Y [m, n] fp32 — downstream the key stream stays fp32, so the bf16 storage of the patch
 * features is the only reduced-precision step.  Backward: dY fp32 -> bf16 operand (one elementwise pass), dW / dbias fp32,
 * dX bf16 (may be NULL).  Workspace: milb200_linear_workspace_bytes(m, n, k, MILB200_BF16, 1).                            */
int milb200_linear_f32out_fwd(const void* X, const void* W, const float* bias, float* Y, int64_t m, int n, int k, int act,
                              void* stream) {
  int rc = linear_check(X, W, m, n, k, MILB200_BF16);
  if (rc) return rc;
  MIL_CHECK_ARG(Y != nullptr, MILB200_EINVAL, "linear_f32out_fwd: Y is null");
  MIL_CHECK_ARG(tc::gemm_store_supported(m, n, k) && aligned16(X) && aligned16(W) && aligned16(Y), MILB200_EUNSUPPORTED,
                "linear_f32out_fwd: shape m=%lld n=%d k=%d is outside the tensor-core kernel (n %% 16, k >= 64, k %% 8)",
                (long long)m, n, k);
  return tc::gemm_store(X, m, k, k, W, n, k, bias, act, Y, MILB200_F32, n, nullptr, nullptr, nullptr, 0,
                        static_cast<cudaStream_t>(stream));
}

int milb200_linear_f32out_bwd(const void* X, const void* W, const float* Y, const float* dY, void* dX, float* dW, float* dbias,
                              int64_t m, int n, int k, int act, int accumulate, void* workspace, size_t ws_bytes,
                              void* stream) {
  int rc = linear_check(X, W, m, n, k, MILB200_BF16);
  if (rc) return rc;
  MIL_CHECK_ARG(dY != nullptr && (act == MILB200_ACT_NONE || Y != nullptr), MILB200_EINVAL, "linear_f32out_bwd: null pointer");
  MIL_CHECK_ARG(tc::gemm_store_supported(m, k, n) && tc::gemm_tn_supported(n, k) && (static_cast<int64_t>(m) * n) % 4 == 0,
                MILB200_EUNSUPPORTED, "linear_f32out_bwd: shape m=%lld n=%d k=%d is outside the tensor-core kernels",
                (long long)m, n, k);
  LinWs w = linear_ws(m, n, k, MILB200_BF16, 1, 0);
  MIL_CHECK_ARG(workspace && ws_bytes >= w.total, MILB200_EWORKSPACE, "linear_f32out_bwd: workspace %zu < %zu", ws_bytes, w.total);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  char* ws = static_cast<char*>(workspace);
  __nv_bfloat16* dypre = reinterpret_cast<__nv_bfloat16*>(ws + w.dypre);
  const int64_t n4 = m * n / 4;
  const unsigned blocks = static_cast<unsigned>(std::min<int64_t>((n4 + 255) / 256, sm_count() * 8));
  k_act_bwd_f32_bf16<<<blocks, 256, 0, st>>>(Y, dY, dypre, n4, act);
  MIL_LAUNCH_CHECK();
  if (dbias && (rc = colsum_launch<__nv_bfloat16>(dypre, m, n, dbias, accumulate, st))) return rc;
  if (dW) {
    int splits = 0;
    float* part = reinterpret_cast<float*>(ws + w.part);
    if ((rc = tc::gemm_tn_splitk(dypre, n, X, k, m, n, k, part, &splits, st))) return rc;
    if ((rc = splitk_reduce(part, splits, static_cast<int64_t>(n) * k, dW, accumulate, st))) return rc;
  }
  if (dX) {
    void* wT = ws + w.wT;
    if ((rc = transpose2d(W, wT, n, k, MILB200_BF16, st))) return rc;
    if ((rc = tc::gemm_store(dypre, m, n, n, wT, k, n, nullptr, MILB200_ACT_NONE, dX, MILB200_BF16, k, nullptr, nullptr, nullptr,
                             0, st)))
      return rc;
  }
  return MILB200_OK;
}

}  // extern "C"
