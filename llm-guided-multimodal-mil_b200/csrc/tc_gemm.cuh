// tc_gemm.cuh — host entry points of the tcgen05/TMEM/TMA GEMM kernels (bf16 operands, fp32 accumulate).
#pragma once

#include "common.cuh"

namespace milb200 {
namespace tc {

constexpr int GATE_D = 192;           // gate width the fused kernels are built for (ABMIL default D)
constexpr int CS_STRIDE = 592;        // per-warp column-sum record: 384 dZ cols + 192 (V*U) cols + sum(ds) + pad

// Y[m, n] = act(A[m, :] . W[n, :] + bias[n]) (+ attn[m] * dM[bag(m), n]);  A [M,K] and W [N,K] are bf16,
// K-contiguous.  out_dtype selects bf16 or fp32 output (ldo elements per row).
int gemm_store(const void* A, int64_t M, int K, int64_t lda, const void* W, int N, int64_t ldw, const float* bias,
               int act, void* out, int out_dtype, int64_t ldo, const float* attn, const float* dM,
               const int32_t* offsets, int nbags, cudaStream_t st);
bool gemm_store_supported(int64_t M, int N, int K);

// s[i] = sum_d tanh(x_i.Wv_d + bv_d) * sigmoid(x_i.Wu_d + bu_d) * ww_d + bw     (D = 192)
// gate_act (optional): bf16 [n, 384] gate activations V|U in the packed column order, saved for the backward.
int gated_score(const void* X, int64_t n, int L, const void* Wcat, const float* bcat, const float* ww,
                const float* bw, float* scores, void* gate_act, cudaStream_t st);

// Recompute V,U and emit dZ[n, 384] = [dL/dVpre | dL/dUpre] (bf16) for upstream dscores; per-warp column sums
// (-> dbcat, dww, dbw) are written to colsum_ws[nrec][CS_STRIDE]; *nrec receives the record count.
int gated_dz(const void* X, int64_t n, int L, const void* Wcat, const float* bcat, const float* ww,
             const float* dscores, void* dZ, float* colsum_ws, int* nrec, cudaStream_t st);
int gated_dz_max_records();

// part[s][mo][no] = sum over the k rows of split s of A[k, mo] * B[k, no]   (A [Kr, Mo], B [Kr, No] bf16,
// both row-major => both operands MN-major for the tensor core).  *splits receives the split count.
int gemm_tn_splitk(const void* A, int64_t lda, const void* B, int64_t ldb, int64_t Kr, int Mo, int No, float* part,
                   int* splits, cudaStream_t st);
int gemm_tn_max_splits(int Mo, int No);
// Gate backward without materialising dZ: dWcat partials from the saved V,U (tile-64 column order), ds and ww; see
// k_gemm_tn_gate.  part rows are in tile-64 order; rec_ws receives splits*3 column-sum records of record_floats().
// ds fp32[Kr] must be 16-byte aligned.
int gemm_tn_gate(const void* VU, const float* ds, const float* ww, const void* X, int64_t ldx, int64_t Kr, int No,
                 float* part, int* splits, float* rec_ws, cudaStream_t st);
int gemm_tn_gate_max_records();
int gemm_tn_gate_record_floats();
// 3xTF32 tensor-core products for fp32 operands (kind::tf32 MMAs over hi/lo splits, fp32-grade results); operands are
// (hi, lo) pairs of fp32 arrays with 16-byte aligned rows.
bool gemm_tf32x3_supported(int64_t M, int N, int K);
int gemm_store_tf32x3(const float* Ahi, const float* Alo, int64_t M, int K, int64_t lda, const float* Bhi, const float* Blo,
                      int N, int64_t ldb, const float* bias, int act, float* out, int64_t ldo, cudaStream_t st,
                      const float* attn = nullptr, const float* dM = nullptr, const int32_t* offsets = nullptr, int nbags = 0,
                      int64_t row0 = 0);     // attn != NULL: + attn[row0 + i] * dM[bag(row0 + i), :] (pooling term of the gate's dX)
int gemm_batched_tf32x3(const float* Ahi, const float* Alo, int batches, int Mb, int K, const float* Bhi, const float* Blo,
                        int N, float* part, cudaStream_t st);
int debug_set_trace(void* dev_ptr);
bool gemm_tn_supported(int Mo, int No);

}  // namespace tc
}  // namespace milb200
