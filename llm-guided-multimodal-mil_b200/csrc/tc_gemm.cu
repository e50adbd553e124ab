// tc_gemm.cu — hand-written sm_100a tensor-core GEMMs: TMA (cp.async.bulk.tensor, 128-byte swizzle)
// feeds shared-memory stages, ONE thread issues tcgen05.mma with the fp32 accumulators in TMEM, four
// epilogue warps read them back with tcgen05.ld and apply the fused epilogue.
//
//   k_gemm_kmajor<BN, Epi>   D[128 x BN] tiles of A[M,K] . B[N,K]^T  (both K-contiguous); persistent,
//                            warp-specialised: warp0 = TMA producer, warp1 = MMA issuer, warp2 = TMEM
//                            allocator, warps 4-7 = epilogue.  Epilogues:
//                              EpiStore   bias + activation (+ rank-1 pooling term) -> bf16/fp32 store
//                                         (nn.Linear sites: aggregator.py:44,47,66; transformer.py:430-448)
//                              EpiDz      gated-attention backward: recompute V,U, emit dZ + column sums
//   k_gemm_kmajor_2sm<BN, Epi>  the same on CTA pairs (tcgen05 cta_group::2: one M = 256 MMA, the weight tile
//                            split between the two CTAs).  Epilogue:
//                              EpiScoreT  gated-attention score (ABMIL.py:52-54), writes 4 B per instance
//                                         (+ optionally the gate activations V,U for the backward)
//   k_gemm_tn                split-K  D[128 x 512] = sum_k A[k, m] B[k, n]  (both operands MN-major):
//                            dW = dZ^T X of the gate / linear backward.
#include <cstdlib>

#include "tc_common.cuh"
#include "tc_gemm.cuh"

namespace milb200 {
namespace tc {

// developer hook (milb200_debug_trace): CTA 0 stamps clock64() at its phase boundaries into a caller buffer
__device__ unsigned long long* g_trace = nullptr;
__device__ __forceinline__ void trace(int slot) {
  if (g_trace != nullptr && blockIdx.x == 0) g_trace[slot] = static_cast<unsigned long long>(clock64());
}

constexpr int BM = 128;      // rows per tile = TMEM lanes
constexpr int BK = 64;       // bf16 per 128-byte swizzle span
constexpr int UMMA_K = 16;
constexpr int EPI_WARP0 = 4;                 // warps 0-3: TMA producer, MMA issuer, TMEM allocator, spare
constexpr int EPI_WARPS = 8;                 // two warps per TMEM lane quarter, each takes half of the columns
constexpr int NUM_THREADS = (EPI_WARP0 + EPI_WARPS) * 32;
constexpr int GATE_DH = GATE_D / 2;          // gate tiles: [V half | U half] = 192 accumulator columns
constexpr int GATE_BN = 2 * GATE_DH;

template <int BN>
struct TileCfg {
  static constexpr int UMMA_N = (BN <= 256) ? BN : BN / 2;
  static constexpr int N_MMA = BN / UMMA_N;
  static constexpr int ACC_STAGES = (2 * BN <= 512) ? 2 : 1;
  static constexpr int TMEM_COLS = (BN * ACC_STAGES <= 128) ? 128 : ((BN * ACC_STAGES <= 256) ? 256 : 512);
  static constexpr int A_BYTES = BM * BK * 2;
  static constexpr int B_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static_assert(UMMA_N % 16 == 0 && UMMA_N <= 256, "invalid UMMA N");
  static_assert((UMMA_N * 128) % 1024 == 0, "B boxes must start on a swizzle-atom boundary");
};

constexpr int BAR_BYTES = 256;
constexpr int SMEM_BUDGET = 232448;  // 227 KB opt-in maximum per CTA

// shared-memory image: [stages][barriers 256 B][epilogue staging (TMA-store source)][epilogue floats]
template <int BN, class Epi>
__host__ __device__ constexpr int epi_bytes() { return Epi::STAGING_BYTES + static_cast<int>(sizeof(float)) * Epi::SMEM_FLOATS; }
template <int BN, class Epi>
__host__ __device__ constexpr int kmajor_stages() {
  int s = (SMEM_BUDGET - 1024 - BAR_BYTES - epi_bytes<BN, Epi>()) / TileCfg<BN>::STAGE_BYTES;
  return s > 8 ? 8 : s;
}
template <int BN, class Epi>
constexpr size_t kmajor_smem_bytes() {
  return 1024 + static_cast<size_t>(kmajor_stages<BN, Epi>()) * TileCfg<BN>::STAGE_BYTES + BAR_BYTES +
         epi_bytes<BN, Epi>();
}

// sub-CTA barrier for the two epilogue warps that share a TMEM lane quarter
__device__ __forceinline__ void quarter_sync(int q) {
  asm volatile("bar.sync %0, 64;" ::"r"(q + 1) : "memory");
}

// ---------------------------------------------------------------------------------------------
// epilogues.  tile<BN>(...) is called by each of the 8 epilogue warps: `q` = TMEM lane quarter (rows
// 32q..32q+31 of the tile), `half` = which half of the tile's columns this warp owns, `nt`/`n_tiles`
// = position in the row tile's sweep over N, `iter` = per-CTA row-tile counter.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float apply_act(float v, int act) {
  if (act == MILB200_ACT_TANH) return tanh_fast(v);
  if (act == MILB200_ACT_RELU) return fmaxf(v, 0.f);
  if (act == MILB200_ACT_SIGMOID) return sigmoid_fast(v);
  return v;
}

struct EpiCtx {
  int64_t row, M;
  int n0, N, nt, n_tiles, q, half, lane;
  int64_t iter;
};

struct EpiStore {
  struct Params {
    void* out;
    int out_bf16;
    int64_t ldo;
    const float* bias;
    int act;
    const float* attn;
    const float* dM;
    const int32_t* offsets;
    int nbags;
    int tma_out;        // bf16 output through staged TMA stores ([32 x 32] boxes, 64-byte swizzle)
    int bias_n;         // = N (length of bias)
    CUtensorMap tmO;
    int64_t row0 = 0;   // global row of the A operand's first row (row chunks of a longer batch: attn / bag lookups)
  };
  static constexpr int BIAS_CACHE = 1024;       // bias[N] lives in shared memory for N <= 1024 (a global load per
  static constexpr int SMEM_FLOATS = BIAS_CACHE;  // 32-column chunk put ~700 cycles of L2 latency on every chunk)
  // one [32 rows x 32 cols] bf16 box per warp: a lane's 16-byte pieces of its own row would otherwise leave as 32
  // partial-sector writes per store instruction (the epilogue of a 128 x 256 tile took 5.6 us of a 10 us kernel)
  static constexpr int BOX_BYTES = 32 * 32 * 2;
  static constexpr int STAGING_BYTES = EPI_WARPS * BOX_BYTES;
  __device__ static void prologue(const Params& p, float* esm, int tid) {
    if (p.bias && p.bias_n <= BIAS_CACHE)
      for (int i = tid; i < p.bias_n; i += NUM_THREADS) esm[i] = __ldg(p.bias + i);
  }
  __device__ EpiStore() {}
  template <int BN>
  __device__ __forceinline__ void tile(const Params& p, float* esm, uint8_t* staging, uint32_t tacc, const EpiCtx& cx) {
    const int64_t row = cx.row;
    const bool bias_smem = p.bias != nullptr && p.bias_n <= BIAS_CACHE;
    uint8_t* box = staging + (cx.half * 4 + cx.q) * BOX_BYTES;
    const uint32_t my_row = smem_u32(box) + static_cast<uint32_t>(cx.lane) * 64u;
    const uint32_t sw = (my_row >> 7) & 3u;
    const int n0 = cx.n0, N = cx.N;
    const bool row_ok = row < cx.M;
    float a = 0.f;
    const float* dmrow = nullptr;
    if (p.attn && row_ok) {
      a = __ldg(p.attn + p.row0 + row);
      dmrow = p.dM + static_cast<int64_t>(find_bag(p.offsets, p.nbags, p.row0 + row)) * p.ldo;
    }
    const bool bias_vec = p.bias != nullptr && (reinterpret_cast<uintptr_t>(p.bias) & 15u) == 0;
#pragma unroll 1
    for (int c = cx.half * (BN / 2); c < (cx.half + 1) * (BN / 2); c += 32) {
      if (n0 + c >= N) break;  // warp-uniform
      uint32_t r[32];
      tmem_ld32(tacc + c, r);
      tmem_ld_wait();
      if (!p.tma_out && !row_ok) continue;   // staged stores: every lane takes part, the TMA store clips rows >= M
      const int nvalid = (N - (n0 + c)) < 32 ? (N - (n0 + c)) : 32;  // multiple of 8 (N % 8 == 0)
      float v[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
      // bias: eight independent 128-bit loads (all lanes read the same addresses: one broadcast transaction each)
      if (bias_smem) {
        const float4* b4 = reinterpret_cast<const float4*>(esm + n0 + c);   // broadcast reads
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          if (j < nvalid) {
            const float4 t = b4[j / 4];
            v[j] += t.x; v[j + 1] += t.y; v[j + 2] += t.z; v[j + 3] += t.w;
          }
        }
      } else if (bias_vec) {
        const float4* b4 = reinterpret_cast<const float4*>(p.bias + n0 + c);
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          if (j < nvalid) {
            const float4 t = __ldg(b4 + j / 4);
            v[j] += t.x; v[j + 1] += t.y; v[j + 2] += t.z; v[j + 3] += t.w;
          }
        }
      } else if (p.bias) {
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (j < nvalid) v[j] += __ldg(p.bias + n0 + c + j);
      }
      if (p.act == MILB200_ACT_TANH) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = tanh_fast(v[j]);
      } else if (p.act == MILB200_ACT_RELU) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
      } else if (p.act == MILB200_ACT_SIGMOID) {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = sigmoid_fast(v[j]);
      }
      if (dmrow) {  // rank-1 pooling term of the gated pool's dX: + attn[row] * dM[bag(row), n]
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (j < nvalid) v[j] = fmaf(a, __ldg(dmrow + n0 + c + j), v[j]);
      }
      if (p.tma_out) {
        if (cx.lane == 0) tma_store_wait_read<0>();   // the previous chunk's box has been read out
        __syncwarp();
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint4 pk = Vec16<__nv_bfloat16>::pack(v + 8 * k);
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(my_row + ((static_cast<uint32_t>(k) ^ sw) << 4)),
                       "r"(pk.x), "r"(pk.y), "r"(pk.z), "r"(pk.w)
                       : "memory");
        }
        fence_proxy_async();
        __syncwarp();
        if (cx.lane == 0) {
          tma_store_2d(&p.tmO, box, n0 + c, static_cast<int32_t>(row));   // lane 0 holds the first row of the quarter
          tma_store_commit();
        }
      } else if (p.out_bf16) {
        __nv_bfloat16* o = static_cast<__nv_bfloat16*>(p.out) + row * p.ldo + n0 + c;
#pragma unroll
        for (int j = 0; j < 32; j += 8)
          if (j < nvalid) *reinterpret_cast<uint4*>(o + j) = Vec16<__nv_bfloat16>::pack(v + j);
      } else {
        float* o = static_cast<float*>(p.out) + row * p.ldo + n0 + c;
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          if (j < nvalid) *reinterpret_cast<float4*>(o + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
      }
    }
  }
  __device__ void finish(const Params& p, int, int lane) {
    if (p.tma_out && lane == 0) tma_store_wait<0>();   // all boxes are globally visible before the kernel ends
  }
};

// Gate tiles.  The packed weight rows (and bcat) are ordered [V 0..95 | U 0..95 | V 96..191 | U 96..191], so
// N tile h = 0/1 holds the matching (V, U) pairs of gate units d = 96h .. 96h+95 in its 192 columns and the
// accumulator is double-buffered in TMEM (2 x 192 columns): the epilogue of one half overlaps the MMAs of
// the next.  Warp (q, half) owns pairs [48 half, 48 half + 48) of rows [32q, 32q+32).
constexpr int GATE_PW = GATE_DH / 2;  // pairs per warp per tile = 48

// SAVE: additionally write the gate activations V = tanh(.), U = sigmoid(.) as bf16 [M, 384] so that the backward can
// form dZ without re-running this GEMM.  Column order of the saved matrix ("tile-64 order"): gate unit d lives at
// V -> 128 (d / 64) + d % 64, U -> 128 (d / 64) + 64 + d % 64, i.e. every 128-column tile of the dW GEMM's A operand
// holds 64 matching (V, U) pairs.  Six [32 rows x 16 cols] TMA-store boxes per warp per half tile.
template <bool SAVE>
struct EpiScoreT {
  struct Params {
    const float* bcat;  // [384] packed order
    const float* ww;    // [192] natural order
    const float* bw;    // [1]
    float* scores;
    CUtensorMap tmS;    // SAVE: gate activations [M, 384] bf16; box [32 rows x 48 cols]
  };
  // bias[384] | w[192] | partial[2 parities][4 (h, half)][128 rows]
  static constexpr int SMEM_FLOATS = 3 * GATE_D + 2 * 4 * BM;
  // staging: ONE [32 x 16] V sub-box + ONE U sub-box per warp (2 KB), recycled for each of the three 16-unit chunks of a
  // half tile.  The main loop is bound by operand supply, so shared memory is better spent on a fifth pipeline stage
  // than on epilogue staging (the epilogue warps wait for the accumulator most of the time anyway).
  static constexpr int SUB_BYTES = 32 * 16 * 2;
  static constexpr int STAGING_BYTES = SAVE ? EPI_WARPS * 2 * SUB_BYTES : 0;
  __device__ static void prologue(const Params& p, float* esm, int tid) {
    for (int i = tid; i < 2 * GATE_D; i += NUM_THREADS) esm[i] = __ldg(p.bcat + i);
    for (int i = tid; i < GATE_D; i += NUM_THREADS) esm[2 * GATE_D + i] = __ldg(p.ww + i);
  }
  __device__ EpiScoreT() {}
  template <int BN>
  __device__ __forceinline__ void tile(const Params& p, float* esm, uint8_t* staging, uint32_t tacc, const EpiCtx& cx) {
    static_assert(BN == GATE_BN, "score epilogue expects the [V half | U half] 192-column tile");
    const int h = cx.nt;
    const float* bV = esm + h * GATE_BN + cx.half * GATE_PW;
    const float* bU = bV + GATE_DH;
    const float* wv = esm + 2 * GATE_D + h * GATE_DH + cx.half * GATE_PW;
    uint8_t* rowV = nullptr;
    uint8_t* rowU = nullptr;
    uint8_t* boxV = nullptr;
    if (SAVE) {
      // per warp: one V sub-box | one U sub-box, each a [32 rows][16 bf16] image (1 KB) in the 32-byte-swizzled layout
      // of the store's tensor map: the 16-byte halves of rows 4-7 (mod 8) are swapped, so that a quarter-warp's eight
      // 128-bit stores (row pitch 32 B) hit all 32 banks instead of 16 of them twice
      boxV = staging + (cx.half * 4 + cx.q) * 2 * SUB_BYTES;
      rowV = boxV + cx.lane * 32;
      rowU = rowV + SUB_BYTES;
    }
    float part = 0.f;
#pragma unroll
    for (int c = 0; c < GATE_PW; c += 16) {
      uint32_t v[16], u[16];
      tmem_ld16(tacc + cx.half * GATE_PW + c, v);
      tmem_ld16(tacc + GATE_DH + cx.half * GATE_PW + c, u);
      tmem_ld_wait();
      float fv[16], fu[16];
#pragma unroll
      for (int j = 0; j < 16; j += 4) {
        float4 bv = *reinterpret_cast<const float4*>(bV + c + j);
        float4 bu = *reinterpret_cast<const float4*>(bU + c + j);
        float4 w = *reinterpret_cast<const float4*>(wv + c + j);
        fv[j] = tanh_fast(__uint_as_float(v[j]) + bv.x); fu[j] = sigmoid_fast(__uint_as_float(u[j]) + bu.x);
        fv[j + 1] = tanh_fast(__uint_as_float(v[j + 1]) + bv.y); fu[j + 1] = sigmoid_fast(__uint_as_float(u[j + 1]) + bu.y);
        fv[j + 2] = tanh_fast(__uint_as_float(v[j + 2]) + bv.z); fu[j + 2] = sigmoid_fast(__uint_as_float(u[j + 2]) + bu.z);
        fv[j + 3] = tanh_fast(__uint_as_float(v[j + 3]) + bv.w); fu[j + 3] = sigmoid_fast(__uint_as_float(u[j + 3]) + bu.w);
        part = fmaf(fv[j] * fu[j], w.x, part);
        part = fmaf(fv[j + 1] * fu[j + 1], w.y, part);
        part = fmaf(fv[j + 2] * fu[j + 2], w.z, part);
        part = fmaf(fv[j + 3] * fu[j + 3], w.w, part);
      }
      if (SAVE) {
        if (cx.lane == 0) tma_store_wait_read<0>();  // the previous chunk's sub-boxes have been read out
        __syncwarp();
        const int sw = (cx.lane & 4) << 2;   // 16 for rows 4-7 (mod 8), else 0
        *reinterpret_cast<uint4*>(rowV + sw) = Vec16<__nv_bfloat16>::pack(fv);
        *reinterpret_cast<uint4*>(rowV + (sw ^ 16)) = Vec16<__nv_bfloat16>::pack(fv + 8);
        *reinterpret_cast<uint4*>(rowU + sw) = Vec16<__nv_bfloat16>::pack(fu);
        *reinterpret_cast<uint4*>(rowU + (sw ^ 16)) = Vec16<__nv_bfloat16>::pack(fu + 8);
        fence_proxy_async();
        __syncwarp();
        if (cx.lane == 0) {
          const int32_t r0 = static_cast<int32_t>(cx.row);  // lane 0 holds the first row of this warp's quarter
          const int d0 = h * GATE_DH + cx.half * GATE_PW + c;  // first gate unit of the chunk (multiple of 16)
          const int colv = 128 * (d0 / 64) + d0 % 64;
          tma_store_2d(&p.tmS, boxV, colv, r0);
          tma_store_2d(&p.tmS, boxV + SUB_BYTES, colv + 64, r0);
          tma_store_commit();
        }
      }
    }
    // the four (h, half) partial sums of a row meet in shared memory; parity double-buffering keeps the next
    // row tile's writes away from this row tile's reads
    float* ps = esm + 3 * GATE_D + static_cast<int>(cx.iter & 1) * 4 * BM;
    const int r = cx.q * 32 + cx.lane;
    ps[(h * 2 + cx.half) * BM + r] = part;
    if (h == cx.n_tiles - 1) {
      quarter_sync(cx.q);
      if (cx.half == 0) {
        const float sc = ((ps[r] + ps[BM + r]) + (ps[2 * BM + r] + ps[3 * BM + r])) + __ldg(p.bw);
        if (cx.row < cx.M) p.scores[cx.row] = sc;
      }
    }
  }
  __device__ void finish(const Params&, int, int lane) {
    if (SAVE && lane == 0) tma_store_wait<0>();  // all boxes are globally visible before the kernel ends
  }
};

// sum over the 32 lanes of a warp of 16 per-lane columns; lanes 2c and 2c+1 both return column c's total
__device__ __forceinline__ float colsum16(float* v, int lane) {
  bool hi = lane & 16;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    float send = hi ? v[j] : v[j + 8], keep = hi ? v[j + 8] : v[j];
    v[j] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
  hi = lane & 8;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float send = hi ? v[j] : v[j + 4], keep = hi ? v[j + 4] : v[j];
    v[j] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
  hi = lane & 4;
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    float send = hi ? v[j] : v[j + 2], keep = hi ? v[j + 2] : v[j];
    v[j] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
  }
  hi = lane & 2;
  {
    float send = hi ? v[0] : v[1], keep = hi ? v[1] : v[0];
    v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
  }
  return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 1);
}

struct EpiDz {
  struct Params {
    const float* bcat;  // packed order
    const float* ww;
    const float* dscores;
    CUtensorMap tmZ;    // dZ [M, 384] bf16, packed column order (same as the weight rows); box [32 rows x 48 cols]
    float* colsum_ws;   // [gridDim.x * EPI_WARPS][CS_STRIDE], natural order: dVpre[192] | dUpre[192] | ds*V*U[192] | sum ds
  };
  static constexpr int SMEM_FLOATS = 3 * GATE_D;
  static constexpr int BOX_BYTES = 32 * GATE_PW * 2;              // one [32 rows x 48 bf16] TMA-store box
  static constexpr int STAGING_BYTES = EPI_WARPS * 2 * BOX_BYTES;  // per warp: dVpre box | dUpre box
  __device__ static void prologue(const Params& p, float* esm, int tid) {
    for (int i = tid; i < 2 * GATE_D; i += NUM_THREADS) esm[i] = __ldg(p.bcat + i);
    for (int i = tid; i < GATE_D; i += NUM_THREADS) esm[2 * GATE_D + i] = __ldg(p.ww + i);
  }
  static constexpr int NCH = GATE_PW / 16;  // 16-pair chunks per warp per tile = 3
  float colacc[2][3][NCH];                  // [h][dVpre, dUpre, ds*V*U][chunk]; column (lane>>1) of each chunk
  float ds_acc;
  __device__ EpiDz() {
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int c = 0; c < NCH; ++c) colacc[h][k][c] = 0.f;
    ds_acc = 0.f;
  }
  template <int H>
  __device__ __forceinline__ void half_tile(const Params& p, float* esm, uint8_t* staging, uint32_t tacc,
                                            const EpiCtx& cx) {
    const bool row_ok = cx.row < cx.M;
    const float ds = row_ok ? __ldg(p.dscores + cx.row) : 0.f;
    // this warp's staging boxes: thread (lane) owns row `lane` of each [32 x 48] box (96 B per row)
    uint8_t* boxV = staging + (cx.half * 4 + cx.q) * 2 * BOX_BYTES;
    uint8_t* boxU = boxV + BOX_BYTES;
    if (cx.lane == 0) tma_store_wait_read<0>();  // the previous half tile's boxes have been read out
    __syncwarp();
    if (H == 0 && cx.half == 0) ds_acc += ds;
    const int pbase = cx.half * GATE_PW;  // first pair of this warp inside the tile
    const float* bV = esm + H * GATE_BN + pbase;
    const float* bU = bV + GATE_DH;
    const float* wv = esm + 2 * GATE_D + H * GATE_DH + pbase;
    uint8_t* rowV = boxV + cx.lane * (GATE_PW * 2);
    uint8_t* rowU = boxU + cx.lane * (GATE_PW * 2);
#pragma unroll
    for (int ci = 0; ci < NCH; ++ci) {
      const int c = ci * 16;
      uint32_t v[16], u[16];
      tmem_ld16(tacc + pbase + c, v);
      tmem_ld16(tacc + GATE_DH + pbase + c, u);
      tmem_ld_wait();
      float dv[16], du[16], vu[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        float V = tanh_fast(__uint_as_float(v[j]) + bV[c + j]);
        float U = sigmoid_fast(__uint_as_float(u[j]) + bU[c + j]);
        float g = ds * wv[c + j];
        float gu = g * U;
        dv[j] = gu * (1.f - V * V);
        du[j] = gu * V * (1.f - U);
        vu[j] = ds * V * U;
      }
      *reinterpret_cast<uint4*>(rowV + c * 2) = Vec16<__nv_bfloat16>::pack(dv);
      *reinterpret_cast<uint4*>(rowV + c * 2 + 16) = Vec16<__nv_bfloat16>::pack(dv + 8);
      *reinterpret_cast<uint4*>(rowU + c * 2) = Vec16<__nv_bfloat16>::pack(du);
      *reinterpret_cast<uint4*>(rowU + c * 2 + 16) = Vec16<__nv_bfloat16>::pack(du + 8);
      colacc[H][0][ci] += colsum16(dv, cx.lane);
      colacc[H][1][ci] += colsum16(du, cx.lane);
      colacc[H][2][ci] += colsum16(vu, cx.lane);
    }
    // hand the two boxes to the TMA engine: rows beyond M are clipped by the tensor map
    fence_proxy_async();
    __syncwarp();
    if (cx.lane == 0) {
      const int32_t r0 = static_cast<int32_t>(cx.row);  // lane 0 holds the first row of this warp's quarter
      tma_store_2d(&p.tmZ, boxV, H * GATE_BN + pbase, r0);
      tma_store_2d(&p.tmZ, boxU, H * GATE_BN + GATE_DH + pbase, r0);
      tma_store_commit();
    }
  }
  template <int BN>
  __device__ __forceinline__ void tile(const Params& p, float* esm, uint8_t* staging, uint32_t tacc,
                                       const EpiCtx& cx) {
    static_assert(BN == GATE_BN, "dz epilogue expects the [V half | U half] 192-column tile");
    if (cx.nt == 0) half_tile<0>(p, esm, staging, tacc, cx);
    else half_tile<1>(p, esm, staging, tacc, cx);
  }
  __device__ void finish(const Params& p, int e, int lane) {
    if (lane == 0) tma_store_wait<0>();  // all dZ boxes are globally visible before the kernel ends
    const int half = e / 4;
    float* rec = p.colsum_ws + (static_cast<int64_t>(blockIdx.x) * EPI_WARPS + e) * CS_STRIDE;
    if ((lane & 1) == 0) {
#pragma unroll
      for (int h = 0; h < 2; ++h)
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
          for (int c = 0; c < NCH; ++c)
            rec[k * GATE_D + h * GATE_DH + half * GATE_PW + c * 16 + (lane >> 1)] = colacc[h][k][c];
    }
    float s = warp_sum(ds_acc);
    if (lane == 0) rec[3 * GATE_D] = s;
  }
};

// ---------------------------------------------------------------------------------------------
// K-major persistent GEMM.  A CTA owns row tiles mt = blockIdx.x, blockIdx.x + gridDim.x, ... and sweeps
// the N tiles of each (the A tile's second pass comes from L2).
// ---------------------------------------------------------------------------------------------
// KIND 1 = "3xTF32": fp32 operands pre-split into hi (tf32-exact) and lo (= x - hi) arrays; the k loop runs three times
// (hi.lo, lo.hi, hi.hi — the lo.lo term is below fp32 rounding) into the same accumulator with kind::tf32 MMAs, which
// gives fp32-grade products (error ~2^-21 per term) at a sixth of the bf16 rate instead of the FFMA path's fortieth.
// The shared-memory image is byte-for-byte the bf16 one (128-byte swizzle rows = 32 floats, 32 bytes of K per MMA).
// batch_mtiles > 0: batched mode for split-K products — m-tile mt belongs to batch mt / batch_mtiles and reads the B rows
// [batch * N, batch * N + N) (A = [batches * M_b, K], B = [batches * N, K], out = [batches * M_b, N] partials).
template <int BN, class Epi, int KIND = 0>
__global__ void __launch_bounds__(NUM_THREADS, 1)
k_gemm_kmajor(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, int64_t M, int N, int K,
              uint32_t b_box_bytes, const __grid_constant__ typename Epi::Params ep,
              const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2, int batch_mtiles) {
  constexpr int BKE = KIND ? 32 : BK;          // elements per 128-byte swizzle row
  constexpr int PHASES = KIND ? 3 : 1;
  using Cfg = TileCfg<BN>;
  constexpr int STAGES = kmajor_stages<BN, Epi>();
  static_assert(STAGES >= 3, "pipeline too shallow");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stage_base = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* full_bar = bars;                   // [STAGES]
  uint64_t* empty_bar = bars + STAGES;         // [STAGES]
  uint64_t* tfull_bar = bars + 2 * STAGES;     // [2]
  uint64_t* tempty_bar = bars + 2 * STAGES + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);
  uint8_t* staging = smem + STAGES * Cfg::STAGE_BYTES + BAR_BYTES;
  float* esm = reinterpret_cast<float*>(staging + Epi::STAGING_BYTES);
  static_assert((2 * STAGES + 4) * 8 + 8 <= BAR_BYTES, "barrier block overflow");
  static_assert(Epi::STAGING_BYTES % 128 == 0, "TMA-store staging must stay 128-byte aligned");

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t m_tiles = (M + BM - 1) / BM;
  const int n_tiles = (N + BN - 1) / BN;
  const int num_kb = (K + BKE - 1) / BKE;
  const int num_it = num_kb * PHASES;
  if (threadIdx.x == 0) trace(0);

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    if (KIND) {
      prefetch_tmap(&tmA2);
      prefetch_tmap(&tmB2);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar + s, 1);
      mbar_init(empty_bar + s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar + a, 1);
      mbar_init(tempty_bar + a, EPI_WARPS * 32);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  Epi::prologue(ep, esm, threadIdx.x);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) trace(1);

  if (warp == 0) {
    // ===== TMA producer =====
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      const uint32_t stage_tx = Cfg::A_BYTES + Cfg::N_MMA * b_box_bytes;
      for (int64_t mt = blockIdx.x; mt < m_tiles; mt += gridDim.x) {
        const int b_row0 = batch_mtiles > 0 ? static_cast<int>(mt / batch_mtiles) * N : 0;
        for (int nt = 0; nt < n_tiles; ++nt) {
          for (int ki = 0; ki < num_it; ++ki) {
            const int kb = KIND ? ki % num_kb : ki;
            const int phase = KIND ? ki / num_kb : 0;
            // small terms first (hi.lo, lo.hi, then hi.hi): the accumulator rounds toward zero on every MMA, so adding
            // 2 x K/8 tiny terms to an already large accumulator costs ~1e-5 (measured); into a still small one, nothing
            const CUtensorMap* mA = (KIND && phase == 1) ? &tmA2 : &tmA;
            const CUtensorMap* mB = (KIND && phase == 0) ? &tmB2 : &tmB;
            mbar_wait(empty_bar + s, ph ^ 1);
            uint8_t* sa = stage_base + s * Cfg::STAGE_BYTES;
            uint8_t* sb = sa + Cfg::A_BYTES;
            mbar_arrive_expect_tx(full_bar + s, stage_tx);
            // the A tile is read n_tiles times back to back: keep it in L2 until the last sweep
            tma_load_2d(sa, mA, full_bar + s, kb * BKE, static_cast<int32_t>(mt * BM),
                        (!KIND && nt == n_tiles - 1) ? kEvictFirst : kEvictNormal);
#pragma unroll
            for (int j = 0; j < Cfg::N_MMA; ++j)
              tma_load_2d(sb + j * Cfg::UMMA_N * 128, mB, full_bar + s, kb * BKE, b_row0 + nt * BN + j * Cfg::UMMA_N,
                          batch_mtiles > 0 ? kEvictNormal : kEvictLast);
            if (ki == 0 && nt == 0 && mt == blockIdx.x) trace(2);
            if (ki == num_it - 1 && nt == 0 && mt == blockIdx.x) trace(3);
            if (++s == STAGES) { s = 0; ph ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: the whole warp walks the loop (so addresses stay in uniform registers); one elected
    // lane issues tcgen05.mma / tcgen05.commit =====
    constexpr uint32_t idesc = KIND ? umma_idesc_tf32(BM, Cfg::UMMA_N, 0, 0) : umma_idesc_bf16(BM, Cfg::UMMA_N, 0, 0);
    const uint64_t desc0 = umma_desc_sw128(smem_u32(stage_base), 16, 1024);
    const uint32_t d_hi = static_cast<uint32_t>(desc0 >> 32);
    const uint32_t a_lo0 = static_cast<uint32_t>(desc0);
    const uint32_t b_lo0 = a_lo0 + (Cfg::A_BYTES >> 4);
    int s = 0;
    uint32_t ph = 0;
    int64_t it = 0;
    for (int64_t mt = blockIdx.x; mt < m_tiles; mt += gridDim.x) {
      for (int nt = 0; nt < n_tiles; ++nt, ++it) {
        const int acc = static_cast<int>(it % Cfg::ACC_STAGES);
        const uint32_t acc_ph = static_cast<uint32_t>((it / Cfg::ACC_STAGES) & 1);
        mbar_wait(tempty_bar + acc, acc_ph ^ 1);
        tc_fence_after();
        const uint32_t tacc = tmem_base + acc * BN;
        for (int kb = 0; kb < num_it; ++kb) {
          mbar_wait(full_bar + s, ph);
          tc_fence_after();
          if (it == 0 && lane == 0) { if (kb == 0) trace(4); if (kb == num_it - 1) trace(5); }
          if (elect_one()) {
            const uint32_t so = static_cast<uint32_t>(s) * (Cfg::STAGE_BYTES >> 4);
#pragma unroll
            for (int k = 0; k < BK / UMMA_K; ++k) {      // four MMAs of 32 bytes of K each (16 bf16 or 8 tf32)
#pragma unroll
              for (int j = 0; j < Cfg::N_MMA; ++j) {
                if (KIND)
                  umma_tf32_lohi(tacc + j * Cfg::UMMA_N, a_lo0 + so + k * (UMMA_K * 2 >> 4), d_hi,
                                 b_lo0 + so + ((j * Cfg::UMMA_N * 128) >> 4) + k * (UMMA_K * 2 >> 4), d_hi, idesc,
                                 (kb | k) != 0 ? 1u : 0u);
                else
                  umma_bf16_lohi(tacc + j * Cfg::UMMA_N, a_lo0 + so + k * (UMMA_K * 2 >> 4), d_hi,
                                 b_lo0 + so + ((j * Cfg::UMMA_N * 128) >> 4) + k * (UMMA_K * 2 >> 4), d_hi, idesc,
                                 (kb | k) != 0 ? 1u : 0u);
              }
            }
            tc_commit(empty_bar + s);  // frees the smem stage once these MMAs have read it
            if (kb == num_it - 1) tc_commit(tfull_bar + acc);  // accumulator complete -> epilogue
          }
          __syncwarp();
          if (++s == STAGES) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp >= EPI_WARP0) {
    // ===== epilogue warps: warp e may touch TMEM lanes [32 (e%4), 32 (e%4) + 32) =====
    const int e = warp - EPI_WARP0;
    Epi epi;
    EpiCtx cx;
    cx.M = M; cx.N = N; cx.n_tiles = n_tiles; cx.q = e & 3; cx.half = e >> 2; cx.lane = lane;
    int64_t it = 0;
    cx.iter = 0;
    for (int64_t mt = blockIdx.x; mt < m_tiles; mt += gridDim.x, ++cx.iter) {
      cx.row = mt * BM + cx.q * 32 + lane;
      for (int nt = 0; nt < n_tiles; ++nt, ++it) {
        const int acc = static_cast<int>(it % Cfg::ACC_STAGES);
        const uint32_t acc_ph = static_cast<uint32_t>((it / Cfg::ACC_STAGES) & 1);
        mbar_wait(tfull_bar + acc, acc_ph);
        tc_fence_after();
        if (it == 0 && e == 0 && lane == 0) trace(6);
        const uint32_t tacc = tmem_base + acc * BN + (static_cast<uint32_t>(cx.q * 32) << 16);
        cx.nt = nt;
        cx.n0 = nt * BN;
        epi.template tile<BN>(ep, esm, staging, tacc, cx);
        tc_fence_before();
        mbar_arrive(tempty_bar + acc);
        if (it == 0 && e == 0 && lane == 0) trace(7);
      }
    }
    epi.finish(ep, e, lane);
  }

  tc_fence_before();
  __syncthreads();
  if (threadIdx.x == 0) trace(8);
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
    if (lane == 0) trace(9);
  }
}

// ---------------------------------------------------------------------------------------------
// CTA-pair variant (tcgen05 cta_group::2): the two CTAs of a cluster own two adjacent 128-row tiles and share every B
// (weight) tile — each loads HALF of it and the pair's MMA (M = 256, issued by the even CTA) reads both halves.  Per CTA
// that halves the weight traffic from L2 (the main loop of the 1-SM kernel is bound by operand supply, not by the tensor
// pipe) and shrinks a stage from 40 KB to 28 KB, i.e. more stages in flight.  Barriers: both CTAs' TMA loads credit the
// leader's full barrier; the leader's MMA commits multicast to both CTAs' empty / accumulator-full barriers; both CTAs'
// epilogue warps arrive on the leader's accumulator-empty barrier.
// ---------------------------------------------------------------------------------------------
template <int BN, class Epi>
__host__ __device__ constexpr int kmajor2_stage_bytes() { return TileCfg<BN>::A_BYTES + TileCfg<BN>::B_BYTES / 2; }
template <int BN, class Epi>
__host__ __device__ constexpr int kmajor2_stages() {
  int s = (SMEM_BUDGET - 1024 - BAR_BYTES - epi_bytes<BN, Epi>()) / kmajor2_stage_bytes<BN, Epi>();
  return s > 8 ? 8 : s;
}
template <int BN, class Epi>
constexpr size_t kmajor2_smem_bytes() {
  return 1024 + static_cast<size_t>(kmajor2_stages<BN, Epi>()) * kmajor2_stage_bytes<BN, Epi>() + BAR_BYTES + epi_bytes<BN, Epi>();
}

template <int BN, class Epi>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(NUM_THREADS, 1)
k_gemm_kmajor_2sm(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, int64_t M, int N, int K,
                  const __grid_constant__ typename Epi::Params ep) {
  using Cfg = TileCfg<BN>;
  static_assert(Cfg::N_MMA == 1 && BN % 32 == 0, "pair kernel: one UMMA per k step, B split in two 8-row-aligned halves");
  constexpr int STAGES = kmajor2_stages<BN, Epi>();
  constexpr int STAGE_BYTES = kmajor2_stage_bytes<BN, Epi>();
  static_assert(STAGES >= 3 && STAGE_BYTES % 1024 == 0, "pair kernel pipeline");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* stage_base = smem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* full_bar = bars;                   // [STAGES]  (the leader's are the ones in use)
  uint64_t* empty_bar = bars + STAGES;         // [STAGES]  per CTA
  uint64_t* tfull_bar = bars + 2 * STAGES;     // [2]       per CTA
  uint64_t* tempty_bar = bars + 2 * STAGES + 2;  // [2]     leader's
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);
  uint8_t* staging = smem + STAGES * STAGE_BYTES + BAR_BYTES;
  float* esm = reinterpret_cast<float*>(staging + Epi::STAGING_BYTES);
  static_assert((2 * STAGES + 4) * 8 + 8 <= BAR_BYTES, "barrier block overflow");

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int64_t m_tiles = (M + BM - 1) / BM;
  const int64_t p_tiles = (m_tiles + 1) / 2;                 // pairs of row tiles
  const int64_t pair0 = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;
  const int n_tiles = (N + BN - 1) / BN;
  const int num_kb = (K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar + s, 1);
      mbar_init(empty_bar + s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar + a, 1);
      mbar_init(tempty_bar + a, 2 * EPI_WARPS);     // one arrival per epilogue warp of BOTH CTAs
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_2sm(tmem_slot, Cfg::TMEM_COLS);
  Epi::prologue(ep, esm, threadIdx.x);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                                          // the peer's barriers exist before anything signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer (both CTAs): my A tile, my half of the B tile =====
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int64_t pt = pair0; pt < p_tiles; pt += n_pairs) {
        const int64_t mt = 2 * pt + rank;
        for (int nt = 0; nt < n_tiles; ++nt) {
          for (int kb = 0; kb < num_kb; ++kb) {
            mbar_wait(empty_bar + s, ph ^ 1);
            uint8_t* sa = stage_base + s * STAGE_BYTES;
            uint8_t* sb = sa + Cfg::A_BYTES;
            if (rank == 0) mbar_arrive_expect_tx(full_bar + s, 2 * STAGE_BYTES);   // both CTAs' bytes land on my barrier
            // the A tile is read n_tiles times back to back: keep it in L2 until the last sweep
            tma_load_2d_2sm(sa, &tmA, full_bar + s, kb * BK, static_cast<int32_t>(mt * BM),
                            nt == n_tiles - 1 ? kEvictFirst : kEvictNormal);
            tma_load_2d_2sm(sb, &tmB, full_bar + s, kb * BK, nt * BN + static_cast<int>(rank) * (BN / 2), kEvictLast);
            if (++s == STAGES) { s = 0; ph ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: the leader CTA only =====
    if (rank == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(2 * BM, BN, 0, 0);
      const uint64_t desc0 = umma_desc_sw128(smem_u32(stage_base), 16, 1024);
      const uint32_t d_hi = static_cast<uint32_t>(desc0 >> 32);
      const uint32_t a_lo0 = static_cast<uint32_t>(desc0);
      const uint32_t b_lo0 = a_lo0 + (Cfg::A_BYTES >> 4);
      int s = 0;
      uint32_t ph = 0;
      int64_t it = 0;
      for (int64_t pt = pair0; pt < p_tiles; pt += n_pairs) {
        for (int nt = 0; nt < n_tiles; ++nt, ++it) {
          const int acc = static_cast<int>(it % Cfg::ACC_STAGES);
          const uint32_t acc_ph = static_cast<uint32_t>((it / Cfg::ACC_STAGES) & 1);
          mbar_wait(tempty_bar + acc, acc_ph ^ 1);
          tc_fence_after();
          const uint32_t tacc = tmem_base + acc * BN;
          for (int kb = 0; kb < num_kb; ++kb) {
            mbar_wait(full_bar + s, ph);
            tc_fence_after();
            if (elect_one()) {
              const uint32_t so = static_cast<uint32_t>(s) * (STAGE_BYTES >> 4);
#pragma unroll
              for (int k = 0; k < BK / UMMA_K; ++k)
                umma_bf16_lohi_2sm(tacc, a_lo0 + so + k * (UMMA_K * 2 >> 4), d_hi, b_lo0 + so + k * (UMMA_K * 2 >> 4), d_hi,
                                   idesc, (kb | k) != 0 ? 1u : 0u);
              tc_commit_2sm(empty_bar + s);                              // frees the stage in BOTH CTAs
              if (kb == num_kb - 1) tc_commit_2sm(tfull_bar + acc);      // accumulators complete in BOTH CTAs
            }
            __syncwarp();
            if (++s == STAGES) { s = 0; ph ^= 1; }
          }
        }
      }
    }
  } else if (warp >= EPI_WARP0) {
    // ===== epilogue warps (both CTAs): my 128 rows of the pair's accumulator live in MY tensor memory =====
    const int e = warp - EPI_WARP0;
    Epi epi;
    EpiCtx cx;
    cx.M = M; cx.N = N; cx.n_tiles = n_tiles; cx.q = e & 3; cx.half = e >> 2; cx.lane = lane;
    int64_t it = 0;
    cx.iter = 0;
    for (int64_t pt = pair0; pt < p_tiles; pt += n_pairs, ++cx.iter) {
      const int64_t mt = 2 * pt + rank;
      cx.row = mt * BM + cx.q * 32 + lane;
      for (int nt = 0; nt < n_tiles; ++nt, ++it) {
        const int acc = static_cast<int>(it % Cfg::ACC_STAGES);
        const uint32_t acc_ph = static_cast<uint32_t>((it / Cfg::ACC_STAGES) & 1);
        mbar_wait(tfull_bar + acc, acc_ph);
        tc_fence_after();
        const uint32_t tacc = tmem_base + acc * BN + (static_cast<uint32_t>(cx.q * 32) << 16);
        cx.nt = nt;
        cx.n0 = nt * BN;
        epi.template tile<BN>(ep, esm, staging, tacc, cx);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(tempty_bar + acc);
      }
    }
    epi.finish(ep, e, lane);
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                     // neither CTA leaves (or frees tensor memory) while the pair is still working
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, Cfg::TMEM_COLS);
  }
}

template <int BN, class Epi>
static int launch_kmajor_2sm(const void* A, int64_t M, int K, int64_t lda, const void* B, int N, int64_t ldb,
                             typename Epi::Params ep, cudaStream_t st) {
  CUtensorMap tmA, tmB;
  int rc = make_tmap_bf16_2d(&tmA, A, static_cast<uint64_t>(M), static_cast<uint64_t>(K), static_cast<uint64_t>(lda), BM);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tmB, B, static_cast<uint64_t>(N), static_cast<uint64_t>(K), static_cast<uint64_t>(ldb), BN / 2);
  if (rc) return rc;
  auto kern = k_gemm_kmajor_2sm<BN, Epi>;
  constexpr size_t smem = kmajor2_smem_bytes<BN, Epi>();
  static_assert(smem <= 232448, "shared memory budget exceeded");
  MIL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const int64_t p_tiles = ((M + BM - 1) / BM + 1) / 2;
  const int pairs = static_cast<int>(p_tiles < sm_count() / 2 ? p_tiles : sm_count() / 2);
  kern<<<2 * pairs, NUM_THREADS, smem, st>>>(tmA, tmB, M, N, K, ep);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

int debug_set_trace(void* dev_ptr) {
  unsigned long long* p = static_cast<unsigned long long*>(dev_ptr);
  MIL_CUDA(cudaMemcpyToSymbol(g_trace, &p, sizeof(p)));
  return MILB200_OK;
}

template <int BN, class Epi>
static int launch_kmajor(const void* A, int64_t M, int K, int64_t lda, const void* B, int N, int64_t ldb,
                         typename Epi::Params ep, int* grid_out, cudaStream_t st) {
  using Cfg = TileCfg<BN>;
  CUtensorMap tmA, tmB;
  int rc = make_tmap_bf16_2d(&tmA, A, static_cast<uint64_t>(M), static_cast<uint64_t>(K), static_cast<uint64_t>(lda), BM);
  if (rc) return rc;
  const uint32_t box_rows = static_cast<uint32_t>(N < Cfg::UMMA_N ? N : Cfg::UMMA_N);
  rc = make_tmap_bf16_2d(&tmB, B, static_cast<uint64_t>(N), static_cast<uint64_t>(K), static_cast<uint64_t>(ldb), box_rows);
  if (rc) return rc;
  auto kern = k_gemm_kmajor<BN, Epi>;
  constexpr size_t smem = kmajor_smem_bytes<BN, Epi>();
  static_assert(smem <= 232448, "shared memory budget exceeded");
  MIL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const int64_t m_tiles = (M + BM - 1) / BM;
  const int grid = static_cast<int>(m_tiles < sm_count() ? m_tiles : sm_count());
  if (grid_out) *grid_out = grid;
  kern<<<grid, NUM_THREADS, smem, st>>>(tmA, tmB, M, N, K, box_rows * 128u, ep, tmA, tmB, 0);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

// 3xTF32 launch: fp32 operands given as (hi, lo) pairs (see tf32_split); fp32 output through EpiStore
static int launch_kmajor_tf32x3(const float* Ahi, const float* Alo, int64_t M, int K, int64_t lda, const float* Bhi,
                                const float* Blo, int N, int64_t ldb, int64_t b_rows, EpiStore::Params ep, int batch_mtiles,
                                cudaStream_t st) {
  constexpr int BN = 256;
  using Cfg = TileCfg<BN>;
  CUtensorMap tmA, tmA2, tmB, tmB2;
  int rc = make_tmap_f32_2d(&tmA, Ahi, static_cast<uint64_t>(M), static_cast<uint64_t>(K), static_cast<uint64_t>(lda), BM);
  if (rc) return rc;
  rc = make_tmap_f32_2d(&tmA2, Alo, static_cast<uint64_t>(M), static_cast<uint64_t>(K), static_cast<uint64_t>(lda), BM);
  if (rc) return rc;
  const uint32_t box_rows = static_cast<uint32_t>(N < Cfg::UMMA_N ? N : Cfg::UMMA_N);
  rc = make_tmap_f32_2d(&tmB, Bhi, static_cast<uint64_t>(b_rows), static_cast<uint64_t>(K), static_cast<uint64_t>(ldb), box_rows);
  if (rc) return rc;
  rc = make_tmap_f32_2d(&tmB2, Blo, static_cast<uint64_t>(b_rows), static_cast<uint64_t>(K), static_cast<uint64_t>(ldb), box_rows);
  if (rc) return rc;
  auto kern = k_gemm_kmajor<BN, EpiStore, 1>;
  constexpr size_t smem = kmajor_smem_bytes<BN, EpiStore>();
  MIL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  const int64_t m_tiles = (M + BM - 1) / BM;
  const int grid = static_cast<int>(m_tiles < sm_count() ? m_tiles : sm_count());
  kern<<<grid, NUM_THREADS, smem, st>>>(tmA, tmB, M, N, K, box_rows * 128u, ep, tmA2, tmB2, batch_mtiles);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

bool gemm_tf32x3_supported(int64_t M, int N, int K) { return M >= 1 && N >= 16 && N % 16 == 0 && K >= 32 && K % 4 == 0; }

// out[M, N] fp32 = act(A[M, K] . B[N, K]^T + bias), A = Ahi + Alo, B = Bhi + Blo (fp32 arrays from tf32_split)
int gemm_store_tf32x3(const float* Ahi, const float* Alo, int64_t M, int K, int64_t lda, const float* Bhi, const float* Blo,
                      int N, int64_t ldb, const float* bias, int act, float* out, int64_t ldo, cudaStream_t st,
                      const float* attn, const float* dM, const int32_t* offsets, int nbags, int64_t row0) {
  MIL_CHECK_ARG(gemm_tf32x3_supported(M, N, K), MILB200_EUNSUPPORTED, "tc gemm_store_tf32x3: unsupported shape M=%lld N=%d K=%d",
                (long long)M, N, K);
  MIL_CHECK_ARG(aligned16(out) && (ldo * 4) % 16 == 0, MILB200_EALIGN, "tc gemm_store_tf32x3: output must be 16-byte aligned");
  EpiStore::Params ep{out, 0, ldo, bias, act, attn, dM, offsets, nbags, 0, N, {}};
  ep.row0 = row0;
  return launch_kmajor_tf32x3(Ahi, Alo, M, K, lda, Bhi, Blo, N, ldb, N, ep, 0, st);
}

// Batched split-K form: part[b * Mb + m, n] = sum_k A[b * Mb + m, k] * B[b * N + n, k] for b < batches (Mb % 128 == 0)
int gemm_batched_tf32x3(const float* Ahi, const float* Alo, int batches, int Mb, int K, const float* Bhi, const float* Blo,
                        int N, float* part, cudaStream_t st) {
  MIL_CHECK_ARG(Mb % BM == 0 && gemm_tf32x3_supported(static_cast<int64_t>(batches) * Mb, N, K), MILB200_EUNSUPPORTED,
                "tc gemm_batched_tf32x3: unsupported shape Mb=%d N=%d K=%d", Mb, N, K);
  EpiStore::Params ep{part, 0, N, nullptr, MILB200_ACT_NONE, nullptr, nullptr, nullptr, 0, 0, N, {}};
  return launch_kmajor_tf32x3(Ahi, Alo, static_cast<int64_t>(batches) * Mb, K, K, Bhi, Blo, N, K,
                              static_cast<int64_t>(batches) * N, ep, Mb / BM, st);
}

bool gemm_store_supported(int64_t M, int N, int K) { return M >= 1 && N >= 16 && N % 16 == 0 && K >= 64 && K % 8 == 0; }

int gemm_store(const void* A, int64_t M, int K, int64_t lda, const void* W, int N, int64_t ldw, const float* bias,
               int act, void* out, int out_dtype, int64_t ldo, const float* attn, const float* dM,
               const int32_t* offsets, int nbags, cudaStream_t st) {
  MIL_CHECK_ARG(gemm_store_supported(M, N, K), MILB200_EUNSUPPORTED, "tc gemm_store: unsupported shape M=%lld N=%d K=%d",
                (long long)M, N, K);
  MIL_CHECK_ARG(aligned16(out) && (ldo * (out_dtype == MILB200_BF16 ? 2 : 4)) % 16 == 0, MILB200_EALIGN,
                "tc gemm_store: output must be 16-byte aligned");
  EpiStore::Params ep{out, out_dtype == MILB200_BF16 ? 1 : 0, ldo, bias, act, attn, dM, offsets, nbags, 0, N, {}};
  if (out_dtype == MILB200_BF16 && M >= 32) {
    int rc0 = make_tmap_bf16_2d_sw64(&ep.tmO, out, static_cast<uint64_t>(M), static_cast<uint64_t>(N), static_cast<uint64_t>(ldo), 32);
    if (rc0) return rc0;
    ep.tma_out = 1;
  }
  if (N <= 128) return launch_kmajor<128, EpiStore>(A, M, K, lda, W, N, ldw, ep, nullptr, st);
  return launch_kmajor<256, EpiStore>(A, M, K, lda, W, N, ldw, ep, nullptr, st);
}

int gated_score(const void* X, int64_t n, int L, const void* Wcat, const float* bcat, const float* ww,
                const float* bw, float* scores, void* gate_act, cudaStream_t st) {
  if (gate_act) {
    EpiScoreT<true>::Params ep;
    ep.bcat = bcat; ep.ww = ww; ep.bw = bw; ep.scores = scores;
    int rc0 = make_tmap_bf16_2d_sw32(&ep.tmS, gate_act, static_cast<uint64_t>(n), 2 * GATE_D, 2 * GATE_D, 32);
    if (rc0) return rc0;
    return launch_kmajor_2sm<GATE_BN, EpiScoreT<true>>(X, n, L, L, Wcat, 2 * GATE_D, L, ep, st);
  }
  EpiScoreT<false>::Params ep;
  ep.bcat = bcat; ep.ww = ww; ep.bw = bw; ep.scores = scores;
  return launch_kmajor_2sm<GATE_BN, EpiScoreT<false>>(X, n, L, L, Wcat, 2 * GATE_D, L, ep, st);
}

int gated_dz_max_records() { return sm_count() * EPI_WARPS; }

int gated_dz(const void* X, int64_t n, int L, const void* Wcat, const float* bcat, const float* ww,
             const float* dscores, void* dZ, float* colsum_ws, int* nrec, cudaStream_t st) {
  EpiDz::Params ep;
  ep.bcat = bcat; ep.ww = ww; ep.dscores = dscores; ep.colsum_ws = colsum_ws;
  int rc0 = make_tmap_bf16_2d_linear(&ep.tmZ, dZ, static_cast<uint64_t>(n), 2 * GATE_D, 2 * GATE_D, 32, GATE_PW);
  if (rc0) return rc0;
  int grid = 0;
  int rc = launch_kmajor<GATE_BN, EpiDz>(X, n, L, L, Wcat, 2 * GATE_D, L, ep, &grid, st);
  if (nrec) *nrec = grid * EPI_WARPS;
  return rc;
}

// ---------------------------------------------------------------------------------------------
// split-K "TN" GEMM: D[mo, no] = sum_k A[k, mo] * B[k, no]
// ---------------------------------------------------------------------------------------------
constexpr int TN_BK = 32;                 // k rows per stage
constexpr int TN_BNO = 512;               // output columns per CTA = all 512 TMEM columns
constexpr int TN_BOX_BYTES = TN_BK * 128; // one [32 x 64] bf16 box
constexpr int TN_A_BYTES = 2 * TN_BOX_BYTES;
constexpr int TN_B_BYTES = (TN_BNO / 64) * TN_BOX_BYTES;
constexpr int TN_STAGE_BYTES = TN_A_BYTES + TN_B_BYTES;
constexpr int TN_STAGES = 5;
constexpr size_t TN_SMEM = 1024 + static_cast<size_t>(TN_STAGES) * TN_STAGE_BYTES + BAR_BYTES;
static_assert(TN_SMEM <= 232448, "TN smem budget");

__global__ void __launch_bounds__(NUM_THREADS, 1)
k_gemm_tn(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, int64_t Kr, int Mo, int No,
          int m_tiles, int n_tiles, int kb_per_split, float* __restrict__ part) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + TN_STAGES * TN_STAGE_BYTES);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + TN_STAGES;
  uint64_t* tfull_bar = bars + 2 * TN_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * TN_STAGES + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tile = blockIdx.x % (m_tiles * n_tiles);
  const int split = blockIdx.x / (m_tiles * n_tiles);
  const int mt = tile / n_tiles, nt = tile % n_tiles;
  const int64_t total_kb = (Kr + TN_BK - 1) / TN_BK;
  const int64_t kb0 = static_cast<int64_t>(split) * kb_per_split;
  int64_t kb1 = kb0 + kb_per_split;
  if (kb1 > total_kb) kb1 = total_kb;
  const int nkb = kb1 > kb0 ? static_cast<int>(kb1 - kb0) : 0;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < TN_STAGES; ++s) {
      mbar_init(full_bar + s, 1);
      mbar_init(empty_bar + s, 1);
    }
    mbar_init(tfull_bar, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      int s = 0;
      uint32_t ph = 0;
      for (int i = 0; i < nkb; ++i) {
        mbar_wait(empty_bar + s, ph ^ 1);
        uint8_t* sa = smem + s * TN_STAGE_BYTES;
        uint8_t* sb = sa + TN_A_BYTES;
        const int32_t krow = static_cast<int32_t>((kb0 + i) * TN_BK);
        mbar_arrive_expect_tx(full_bar + s, TN_STAGE_BYTES);
#pragma unroll
        for (int j = 0; j < 2; ++j)
          tma_load_2d(sa + j * TN_BOX_BYTES, &tmA, full_bar + s, mt * BM + j * 64, krow, kEvictNormal);
#pragma unroll
        for (int j = 0; j < TN_BNO / 64; ++j)
          tma_load_2d(sb + j * TN_BOX_BYTES, &tmB, full_bar + s, nt * TN_BNO + j * 64, krow, kEvictNormal);
        if (++s == TN_STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    if (nkb > 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(BM, 256, 1, 1);
      // MN-major, 128-byte swizzle: 8 k-rows x 128 B per atom; next 8 k-rows at SBO = 1024 B, next 64 m/n
      // elements at LBO = one box
      const uint64_t desc0 = umma_desc_sw128(smem_u32(smem), TN_BOX_BYTES, 1024);
      const uint32_t d_hi = static_cast<uint32_t>(desc0 >> 32);
      const uint32_t a_lo0 = static_cast<uint32_t>(desc0);
      const uint32_t b_lo0 = a_lo0 + (TN_A_BYTES >> 4);
      int s = 0;
      uint32_t ph = 0;
      for (int i = 0; i < nkb; ++i) {
        mbar_wait(full_bar + s, ph);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t so = static_cast<uint32_t>(s) * (TN_STAGE_BYTES >> 4);
#pragma unroll
          for (int k = 0; k < TN_BK / UMMA_K; ++k) {
#pragma unroll
            for (int h = 0; h < TN_BNO / 256; ++h)
              umma_bf16_lohi(tmem_base + h * 256, a_lo0 + so + k * (2048 >> 4), d_hi,
                             b_lo0 + so + ((h * 4 * TN_BOX_BYTES) >> 4) + k * (2048 >> 4), d_hi, idesc,
                             (i | k) != 0 ? 1u : 0u);
          }
          tc_commit(empty_bar + s);
          if (i == nkb - 1) tc_commit(tfull_bar);
        }
        __syncwarp();
        if (++s == TN_STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp >= EPI_WARP0) {
    const int q = (warp - EPI_WARP0) & 3, half = (warp - EPI_WARP0) >> 2;
    const int m = mt * BM + q * 32 + lane;
    float* prow = part + (static_cast<int64_t>(split) * Mo + m) * No + nt * TN_BNO;
    if (nkb > 0) {
      mbar_wait(tfull_bar, 0);
      tc_fence_after();
    }
    const uint32_t tacc = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
#pragma unroll 1
    for (int c = half * (TN_BNO / 2); c < (half + 1) * (TN_BNO / 2); c += 32) {
      if (nt * TN_BNO + c >= No) break;
      uint32_t r[32];
      if (nkb > 0) {
        tmem_ld32(tacc + c, r);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) r[j] = 0u;
      }
      if (m < Mo) {
        const int nvalid = (No - (nt * TN_BNO + c)) < 32 ? (No - (nt * TN_BNO + c)) : 32;
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          if (j < nvalid)
            *reinterpret_cast<float4*>(prow + c + j) =
                make_float4(__uint_as_float(r[j]), __uint_as_float(r[j + 1]), __uint_as_float(r[j + 2]),
                            __uint_as_float(r[j + 3]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------
// Fused gate backward: dWcat = dZ^T X with the A operand dZ = ds * [w U (1 - V^2) | w V U (1 - U)] built ON THE FLY from
// the V,U the forward saved (tile-64 column order, see EpiScoreT) — dZ never touches HBM (saves 1.5 KB of traffic per
// instance and a kernel).  Same split-K skeleton as k_gemm_tn.  Per stage the TMA producer lands the RAW operands: the
// [32 x 64] V box and U box of the m-tile exactly where the A tile lives (same 128-byte-swizzled MN-major image),
// 32 ds values, and the X boxes.  The 8 epilogue warps then turn V,U into dV,dU IN PLACE (thread (r, pc) owns k-row r
// and the 16-byte chunk pc of both boxes), fence the async proxy and release the stage to the MMA warp.  (Fetching
// V,U with ordinary loads instead serialises: the proxy fence drains the thread's outstanding global loads.)
// Column sums (-> dbcat, dww, dbw) ride along in registers; CTAs of n-tile 0 publish them per (split, m-tile).
// Warps: 0 X producer, 1 MMA issuer, 2 TMEM allocator, 3 raw V,U / ds producer, 4.. transform and accumulator epilogue.
// A variant that also ran the pooling backward inside this kernel was built, measured and removed (DESIGN §5c).
// ---------------------------------------------------------------------------------------------
constexpr int TNG_MT = 2 * GATE_D / BM;   // 3 m-tiles of 128 columns = 64 (V, U) pairs each
constexpr int TNG_REC = 200;              // record: dVpre[64] | dUpre[64] | ds*V*U[64] | sum ds | pad
constexpr int TNG_ASTAGES = 8;            // A ring (8 KB per stage): raw V,U land and are transformed well ahead of the MMA
constexpr int TNG_BSTAGES = 4;            // B ring (32 KB per stage)
constexpr int TNG_BAR_BYTES = 384;        // a multiple of 128: keeps ds_s 128-byte aligned
constexpr int TNG_XW = 8;                 // transform warps: two groups of four alternate over the stages (measured: three
                                          // groups at 111 registers 0.470 ms, two groups at 96 with the stage ring of 8 0.447 ms)
constexpr int TNG_DS_SLOTS = 32;          // ds ring (stages): refilled eight stages at a time, ahead of the A ring
constexpr int TNG_DS_CHUNK = 8;
constexpr int TNG_THREADS = (EPI_WARP0 + TNG_XW) * 32;
constexpr int TNG_RED_BYTES = static_cast<int>(sizeof(float)) * TNG_XW * 8 * 25;      // 9600: keeps ds_s 128-byte aligned
constexpr size_t TNG_SMEM = 1024 + static_cast<size_t>(TNG_ASTAGES) * TN_A_BYTES + static_cast<size_t>(TNG_BSTAGES) * TN_B_BYTES +
                            TNG_BAR_BYTES + TNG_RED_BYTES + TNG_DS_SLOTS * TN_BK * sizeof(float);
static_assert(TNG_SMEM <= 232448 && TNG_RED_BYTES % 128 == 0, "fused dW kernel smem budget");

__global__ void __launch_bounds__(TNG_THREADS, 1)
k_gemm_tn_gate(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const float* __restrict__ ds, const float* __restrict__ ww, int64_t Kr, int No, int n_tiles,
               int kb_per_split, float* __restrict__ part, float* __restrict__ rec_ws) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* a_ring = smem;                                          // [TNG_ASTAGES][V box | U box]
  uint8_t* b_ring = smem + TNG_ASTAGES * TN_A_BYTES;               // [TNG_BSTAGES][8 X boxes]
  uint64_t* bars = reinterpret_cast<uint64_t*>(b_ring + TNG_BSTAGES * TN_B_BYTES);
  uint64_t* araw_bar = bars;                                       // raw V,U + ds landed
  uint64_t* afull_bar = bars + TNG_ASTAGES;                        // transformed: the MMA may read the A stage
  uint64_t* aempty_bar = bars + 2 * TNG_ASTAGES;                   // MMA done with the A stage
  uint64_t* bfull_bar = bars + 3 * TNG_ASTAGES;
  uint64_t* bempty_bar = bars + 3 * TNG_ASTAGES + TNG_BSTAGES;
  uint64_t* tfull_bar = bars + 3 * TNG_ASTAGES + 2 * TNG_BSTAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tfull_bar + 1);
  static_assert((3 * TNG_ASTAGES + 2 * TNG_BSTAGES + 1) * 8 + 4 <= TNG_BAR_BYTES, "barrier block overflow");
  float* red = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + TNG_BAR_BYTES);  // [8 warps][8 pc][25]
  float* ds_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(red) + TNG_RED_BYTES);   // [TNG_DS_SLOTS][32]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int Mo = 2 * GATE_D;
  const int tile = blockIdx.x % (TNG_MT * n_tiles);
  const int split = blockIdx.x / (TNG_MT * n_tiles);
  const int mt = tile / n_tiles, nt = tile % n_tiles;
  const int64_t total_kb = (Kr + TN_BK - 1) / TN_BK;
  const int64_t kb0 = static_cast<int64_t>(split) * kb_per_split;
  int64_t kb1 = kb0 + kb_per_split;
  if (kb1 > total_kb) kb1 = total_kb;
  const int nkb = kb1 > kb0 ? static_cast<int>(kb1 - kb0) : 0;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < TNG_ASTAGES; ++s) {
      mbar_init(araw_bar + s, 1);
      mbar_init(afull_bar + s, 4);               // one arrival per warp of the group that transforms the stage
      mbar_init(aempty_bar + s, 1);
    }
    for (int s = 0; s < TNG_BSTAGES; ++s) {
      mbar_init(bfull_bar + s, 1);
      mbar_init(bempty_bar + s, 1);
    }
    mbar_init(tfull_bar, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== X (B operand) producer =====
    if (lane == 0) {
      for (int i = 0; i < nkb; ++i) {
        const int s = i % TNG_BSTAGES;
        mbar_wait(bempty_bar + s, static_cast<uint32_t>((i / TNG_BSTAGES) & 1) ^ 1);
        uint8_t* sb = b_ring + s * TN_B_BYTES;
        const int32_t krow = static_cast<int32_t>((kb0 + i) * TN_BK);
        mbar_arrive_expect_tx(bfull_bar + s, TN_B_BYTES);
#pragma unroll
        for (int j = 0; j < TN_BNO / 64; ++j)
          tma_load_2d(sb + j * TN_BOX_BYTES, &tmB, bfull_bar + s, nt * TN_BNO + j * 64, krow, kEvictNormal);
      }
    }
  } else if (warp == 3) {
    // ===== raw V,U / ds producer: runs up to TNG_ASTAGES stages ahead of the MMA =====
    // ds goes through the warp's registers into a 32-stage ring, eight stages per refill (one L2 round trip amortised
    // over eight stages); the next chunk's loads are in flight while the current eight stages are issued.
    float nx[8];
    bool have_next = false;
    auto fetch = [&](int ii, float* v) {                 // 8 ds values of this lane for the chunk that starts at stage ii
      const int nst = (nkb - ii) < TNG_DS_CHUNK ? (nkb - ii) : TNG_DS_CHUNK;
      const int64_t r = (kb0 + ii) * TN_BK + lane * 8;
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = 0.f;
      if (lane < nst * 4) {
        if (r + 7 < Kr) {
          const float4 a = __ldg(reinterpret_cast<const float4*>(ds + r));
          const float4 b = __ldg(reinterpret_cast<const float4*>(ds + r + 4));
          v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
          v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
        } else {
#pragma unroll
          for (int e = 0; e < 8; ++e)
            if (r + e < Kr) v[e] = __ldg(ds + r + e);
        }
      }
    };
    for (int i = 0; i < nkb; ++i) {
      if ((i & (TNG_DS_CHUNK - 1)) == 0) {
        float v[8];
        if (have_next) {
#pragma unroll
          for (int e = 0; e < 8; ++e) v[e] = nx[e];
        } else {
          fetch(i, v);
        }
        float* dst = ds_s + (i % TNG_DS_SLOTS) * TN_BK + lane * 8;
        *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(dst + 4) = make_float4(v[4], v[5], v[6], v[7]);
        __syncwarp();
        have_next = i + TNG_DS_CHUNK < nkb;
        if (have_next) fetch(i + TNG_DS_CHUNK, nx);     // in flight while the next eight stages are issued
      }
      if (lane == 0) {
        const int s = i % TNG_ASTAGES;
        mbar_wait(aempty_bar + s, static_cast<uint32_t>((i / TNG_ASTAGES) & 1) ^ 1);
        uint8_t* sa = a_ring + s * TN_A_BYTES;
        const int32_t krow = static_cast<int32_t>((kb0 + i) * TN_BK);
        mbar_arrive_expect_tx(araw_bar + s, TN_A_BYTES);   // (release: the ring refill above is visible to the waiters)
        tma_load_2d(sa, &tmA, araw_bar + s, Mo / TNG_MT * mt, krow, kEvictFirst);                       // V box
        tma_load_2d(sa + TN_BOX_BYTES, &tmA, araw_bar + s, Mo / TNG_MT * mt + 64, krow, kEvictFirst);   // U box
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    if (nkb > 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(BM, 256, 1, 1);
      const uint64_t desc0 = umma_desc_sw128(smem_u32(smem), TN_BOX_BYTES, 1024);
      const uint32_t d_hi = static_cast<uint32_t>(desc0 >> 32);
      const uint32_t a_lo0 = static_cast<uint32_t>(desc0);
      const uint32_t b_lo0 = a_lo0 + ((TNG_ASTAGES * TN_A_BYTES) >> 4);
      for (int i = 0; i < nkb; ++i) {
        const int sa = i % TNG_ASTAGES, sb = i % TNG_BSTAGES;
        mbar_wait(afull_bar + sa, static_cast<uint32_t>((i / TNG_ASTAGES) & 1));
        mbar_wait(bfull_bar + sb, static_cast<uint32_t>((i / TNG_BSTAGES) & 1));
        tc_fence_after();
        if (elect_one()) {
          const uint32_t ao = a_lo0 + static_cast<uint32_t>(sa) * (TN_A_BYTES >> 4);
          const uint32_t bo = b_lo0 + static_cast<uint32_t>(sb) * (TN_B_BYTES >> 4);
#pragma unroll
          for (int k = 0; k < TN_BK / UMMA_K; ++k) {
#pragma unroll
            for (int h = 0; h < TN_BNO / 256; ++h)
              umma_bf16_lohi(tmem_base + h * 256, ao + k * (2048 >> 4), d_hi,
                             bo + ((h * 4 * TN_BOX_BYTES) >> 4) + k * (2048 >> 4), d_hi, idesc, (i | k) != 0 ? 1u : 0u);
          }
          tc_commit(aempty_bar + sa);
          tc_commit(bempty_bar + sb);
          if (i == nkb - 1) tc_commit(tfull_bar);
        }
        __syncwarp();
      }
    }
  } else if (warp >= EPI_WARP0) {
    // ===== in-place V,U -> dV,dU transform (main loop), then the accumulator epilogue =====
    // TNG_XW / 4 groups of four warps rotate over the stages, so that many stages are in transformation at any time and the
    // latency of the proxy fence overlaps with the other groups' work.  Thread (r, pc) of a group owns k-rows r, r + 16.
    const int tid = threadIdx.x - EPI_WARP0 * 32;
    const int grp = tid >> 7, tg = tid & 127;
    const int r = tg >> 3, pc = tg & 7;
    const int d0 = 64 * mt + 8 * pc;                                    // first of this thread's 8 gate units
    const uint32_t a_off0 = static_cast<uint32_t>((r >> 3) * 1024 + (r & 7) * 128 + ((pc ^ (r & 7)) << 4));
    const uint32_t a_off1 = a_off0 + 2 * 1024;                          // k-row r + 16: same swizzle phase, two atoms on
    float w[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) w[e] = __ldg(ww + d0 + e);
    float sdv[8], sdu[8], svu[8], sds = 0.f;
#pragma unroll
    for (int e = 0; e < 8; ++e) sdv[e] = sdu[e] = svu[e] = 0.f;
    for (int i = grp; i < nkb; i += TNG_XW / 4) {
      const int s = i % TNG_ASTAGES;
      mbar_wait(araw_bar + s, static_cast<uint32_t>((i / TNG_ASTAGES) & 1));
      uint8_t* sa = a_ring + s * TN_A_BYTES;
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const uint32_t a_off = hh ? a_off1 : a_off0;
        uint4* pv = reinterpret_cast<uint4*>(sa + a_off);
        uint4* pu = reinterpret_cast<uint4*>(sa + TN_BOX_BYTES + a_off);
        const float dsi = ds_s[(i % TNG_DS_SLOTS) * TN_BK + r + 16 * hh];
        float V[8], U[8], dv[8], du[8];
        Vec16<__nv_bfloat16>::unpack(*pv, V);
        Vec16<__nv_bfloat16>::unpack(*pu, U);
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float gu = dsi * w[e] * U[e];
          dv[e] = gu * (1.f - V[e] * V[e]);
          du[e] = gu * V[e] * (1.f - U[e]);
          sdv[e] += dv[e];
          sdu[e] += du[e];
          svu[e] = fmaf(dsi * V[e], U[e], svu[e]);
        }
        if (pc == 0) sds += dsi;
        *pv = Vec16<__nv_bfloat16>::pack(dv);
        *pu = Vec16<__nv_bfloat16>::pack(du);
      }
      fence_proxy_async();                          // my generic-proxy writes -> visible to the MMA's async proxy
      __syncwarp();
      if (lane == 0) mbar_arrive(afull_bar + s);
    }
    // column sums: fold the 4 k-rows a warp holds per pc with shuffles, then the 8 warps through shared memory
    if (nt == 0) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        sdv[e] += __shfl_xor_sync(0xffffffffu, sdv[e], 8);  sdv[e] += __shfl_xor_sync(0xffffffffu, sdv[e], 16);
        sdu[e] += __shfl_xor_sync(0xffffffffu, sdu[e], 8);  sdu[e] += __shfl_xor_sync(0xffffffffu, sdu[e], 16);
        svu[e] += __shfl_xor_sync(0xffffffffu, svu[e], 8);  svu[e] += __shfl_xor_sync(0xffffffffu, svu[e], 16);
      }
      sds += __shfl_xor_sync(0xffffffffu, sds, 8);
      sds += __shfl_xor_sync(0xffffffffu, sds, 16);
      const int ew = warp - EPI_WARP0;
      if (lane < 8) {
        float* dst = red + (ew * 8 + lane) * 25;
#pragma unroll
        for (int e = 0; e < 8; ++e) { dst[e] = sdv[e]; dst[8 + e] = sdu[e]; dst[16 + e] = svu[e]; }
        dst[24] = sds;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(TNG_XW * 32) : "memory");
      float* rec = rec_ws + (static_cast<int64_t>(split) * TNG_MT + mt) * TNG_REC;
      if (tid < 192) {
        const int k = tid / 64, j = tid % 64;
        float a = 0.f;
#pragma unroll
        for (int q = 0; q < TNG_XW; ++q) a += red[(q * 8 + j / 8) * 25 + k * 8 + j % 8];
        rec[tid] = a;
      } else if (tid == 192) {
        float a = 0.f;
#pragma unroll
        for (int q = 0; q < TNG_XW; ++q) a += red[(q * 8) * 25 + 24];
        rec[192] = a;
      }
    }
    const int q = (warp - EPI_WARP0) & 3, third = (warp - EPI_WARP0) >> 2;
    const int m = mt * BM + q * 32 + lane;
    float* prow = part + (static_cast<int64_t>(split) * Mo + m) * No + nt * TN_BNO;
    if (nkb > 0) {
      mbar_wait(tfull_bar, 0);
      tc_fence_after();
    }
    const uint32_t tacc = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
#pragma unroll 1
    for (int c = third * 32; c < TN_BNO; c += 32 * (TNG_XW / 4)) {     // the warps of a lane quarter interleave chunks
      if (nt * TN_BNO + c >= No) break;
      uint32_t rr[32];
      if (nkb > 0) {
        tmem_ld32(tacc + c, rr);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) rr[j] = 0u;
      }
      const int nvalid = (No - (nt * TN_BNO + c)) < 32 ? (No - (nt * TN_BNO + c)) : 32;
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        if (j < nvalid)
          *reinterpret_cast<float4*>(prow + c + j) =
              make_float4(__uint_as_float(rr[j]), __uint_as_float(rr[j + 1]), __uint_as_float(rr[j + 2]),
                          __uint_as_float(rr[j + 3]));
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}


int gemm_tn_gate_max_records() { return sm_count(); }  // splits * 3 m-tiles <= resident CTAs
int gemm_tn_gate_record_floats() { return TNG_REC; }

// part[s][384 (tile-64 order)][No] partial dWcat; rec_ws[splits * 3][TNG_REC] column-sum records
int gemm_tn_gate(const void* VU, const float* ds, const float* ww, const void* X, int64_t ldx, int64_t Kr, int No,
                 float* part, int* splits_out, float* rec_ws, cudaStream_t st) {
  constexpr int Mo = 2 * GATE_D;
  MIL_CHECK_ARG(gemm_tn_supported(Mo, No), MILB200_EUNSUPPORTED, "tc gemm_tn_gate: unsupported No=%d", No);
  MIL_CHECK_ARG((reinterpret_cast<uintptr_t>(ds) & 15) == 0, MILB200_EALIGN, "tc gemm_tn_gate: ds must be 16-byte aligned");
  CUtensorMap tmA, tmB;
  int rc = make_tmap_bf16_2d(&tmA, VU, static_cast<uint64_t>(Kr), Mo, Mo, TN_BK);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tmB, X, static_cast<uint64_t>(Kr), static_cast<uint64_t>(No), static_cast<uint64_t>(ldx), TN_BK);
  if (rc) return rc;
  const int n_tiles = (No + TN_BNO - 1) / TN_BNO;
  const int64_t total_kb = (Kr + TN_BK - 1) / TN_BK;
  int splits = gemm_tn_max_splits(Mo, No);
  if (splits > total_kb) splits = static_cast<int>(total_kb);
  if (splits < 1) splits = 1;
  const int kb_per_split = static_cast<int>((total_kb + splits - 1) / splits);
  splits = static_cast<int>((total_kb + kb_per_split - 1) / kb_per_split);
  if (splits_out) *splits_out = splits;
  MIL_CUDA(cudaFuncSetAttribute(k_gemm_tn_gate, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(TNG_SMEM)));
  k_gemm_tn_gate<<<TNG_MT * n_tiles * splits, TNG_THREADS, TNG_SMEM, st>>>(tmA, tmB, ds, ww, Kr, No, n_tiles, kb_per_split,
                                                                           part, rec_ws);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

bool gemm_tn_supported(int Mo, int No) { return Mo >= 64 && Mo % 8 == 0 && No >= 64 && No % 8 == 0; }

int gemm_tn_max_splits(int Mo, int No) {
  int tiles = ((Mo + BM - 1) / BM) * ((No + TN_BNO - 1) / TN_BNO);
  int s = sm_count() / tiles;
  return s < 1 ? 1 : s;
}

int gemm_tn_splitk(const void* A, int64_t lda, const void* B, int64_t ldb, int64_t Kr, int Mo, int No, float* part,
                   int* splits_out, cudaStream_t st) {
  MIL_CHECK_ARG(gemm_tn_supported(Mo, No), MILB200_EUNSUPPORTED, "tc gemm_tn: unsupported shape Mo=%d No=%d", Mo, No);
  CUtensorMap tmA, tmB;
  int rc = make_tmap_bf16_2d(&tmA, A, static_cast<uint64_t>(Kr), static_cast<uint64_t>(Mo), static_cast<uint64_t>(lda), TN_BK);
  if (rc) return rc;
  rc = make_tmap_bf16_2d(&tmB, B, static_cast<uint64_t>(Kr), static_cast<uint64_t>(No), static_cast<uint64_t>(ldb), TN_BK);
  if (rc) return rc;
  const int m_tiles = (Mo + BM - 1) / BM, n_tiles = (No + TN_BNO - 1) / TN_BNO;
  const int64_t total_kb = (Kr + TN_BK - 1) / TN_BK;
  int splits = gemm_tn_max_splits(Mo, No);
  if (splits > total_kb) splits = static_cast<int>(total_kb);
  if (splits < 1) splits = 1;
  const int kb_per_split = static_cast<int>((total_kb + splits - 1) / splits);
  splits = static_cast<int>((total_kb + kb_per_split - 1) / kb_per_split);
  if (splits_out) *splits_out = splits;
  MIL_CUDA(cudaFuncSetAttribute(k_gemm_tn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(TN_SMEM)));
  k_gemm_tn<<<m_tiles * n_tiles * splits, NUM_THREADS, TN_SMEM, st>>>(tmA, tmB, Kr, Mo, No, m_tiles, n_tiles,
                                                                      kb_per_split, part);
  MIL_LAUNCH_CHECK();
  return MILB200_OK;
}

}  // namespace tc
}  // namespace milb200
