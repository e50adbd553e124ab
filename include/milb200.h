/* milb200.h — C ABI of the B200 (sm_100a) MIL-aggregator kernel library (libmilb200.so).
 *
 * The reference (KyleKWKim/LLM-guided-Multimodal-MIL) is pure Python: its "operator API" for this
 * path is torch.nn.Linear / torch.softmax / torch.matmul / nn.LayerNorm called from nn.Modules
 * (SURVEY.md §1, §8b).  There is no FFI upstream; each entry point below names the reference lines
 * whose eager-PyTorch ops it replaces.  The Python host (package mil_b200) binds these with ctypes and
 * wraps them in torch.autograd.Functions behind the reference's nn.Module interfaces.
 *
 * Conventions (all entry points)
 *   - plain C: raw device pointers, sizes, a cudaStream_t passed as void*; no torch types.
 *   - the caller allocates every output and the workspace (query sizes with *_workspace_bytes);
 *     kernels never malloc/free and never synchronise; all work is enqueued on `stream`.
 *   - return 0 on success, a negative MILB200_E* code otherwise; milb200_last_error() gives the text
 *     (thread-local).  Nothing is launched when an argument check fails.
 *   - matrices are row-major and densely packed unless a leading dimension is given.
 *   - dtype: MILB200_F32 (SIMT fp32 kernels, <=1e-5 parity) or MILB200_BF16 (tcgen05/TMEM/TMA kernels,
 *     fp32 accumulate).  Scores, statistics and all gradients of parameters are fp32.
 *   - ragged bags: packed rows X[total_n, L] + CSR offsets[B+1] (int32, offsets[0]=0, non-decreasing,
 *     offsets[B]=total_n; every bag non-empty).
 */
#ifndef MILB200_H_
#define MILB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MILB200_VERSION 200

enum { MILB200_F32 = 0, MILB200_BF16 = 1 };

enum {
  MILB200_OK = 0,
  MILB200_EINVAL = -1,      /* bad shape / null pointer / unsupported size */
  MILB200_EALIGN = -2,      /* pointer or row pitch not 16-byte aligned */
  MILB200_EWORKSPACE = -3,  /* workspace too small */
  MILB200_ECUDA = -4,       /* CUDA runtime / launch error */
  MILB200_EUNSUPPORTED = -5 /* dtype/shape combination not built */
};

enum { MILB200_ACT_NONE = 0, MILB200_ACT_TANH = 1, MILB200_ACT_RELU = 2, MILB200_ACT_SIGMOID = 3 };

int milb200_version(void);
const char* milb200_last_error(void);
/* Number of kernels this library has launched in the calling process (bench.py's gpu_launches).  A host that replays a
 * captured CUDA graph of library launches itself reports the graph's kernel count with milb200_count_launches. */
int64_t milb200_launch_count(void);
void milb200_count_launches(int64_t n);

/* ---- gated-attention scores -------------------------------------------------------------------
 * Replaces ABMIL.forward's attention_V / attention_U / attention_weights chain
 * (model/dim1/ABMIL.py:52-54): s_i = (tanh(x_i Wv^T + bv) * sigmoid(x_i Wu^T + bu)) . ww + bw.
 * Packed gate weights: Wcat[2D, L] rows [0,D) = attention_V.0.weight, rows [D,2D) = attention_U.0.weight
 * (dtype of X); bcat[2D] fp32; ww[D] fp32 (attention_weights.weight row); bw[1] fp32 on device.       */
int milb200_pack_gate_weights(const void* Wv, const void* Wu, const void* bv, const void* bu,
                              int src_dtype, int L, int D, void* Wcat, int dst_dtype, float* bcat,
                              void* stream);

size_t milb200_gated_score_workspace_bytes(int64_t total_n, int L, int D, int dtype, int backward);

/* gate_act (optional, may be NULL): receives what the backward needs of the gate, [total_n, 2D] in X's dtype — bf16: the
 * activations V = tanh(.), U = sigmoid(.) (column order of Wcat's packed rows); fp32 (3xTF32 tensor-core path): the
 * pre-activations X Wcat^T + bcat.  Only the tensor-core paths write it (milb200_gated_score_saves_activations() == 1);
 * passing it to milb200_gated_score_bwd replaces the recompute GEMM by an elementwise pass (bf16: +0.77 KB/instance of
 * memory for -35 % of the backward time at L = 1024).  fp32 inputs run on the tensor cores as three kind::tf32 MMAs
 * over hi/lo operand splits ("3xTF32", fp32-grade results: <= 1e-5 of the float64 oracle); MILB200_TF32X3=0 in the
 * environment, D % 64 != 0 or L % 16 != 0 select the FFMA kernels.  bf16 runs on the tensor cores for D = 192, L >= 64,
 * L % 16 == 0 (the input-gradient GEMM takes N = L in steps of 16) and on the FFMA kernels otherwise.  The FFMA
 * backward takes D <= 256.                                                                                             */
int milb200_gated_score_saves_activations(int L, int D, int dtype);
int milb200_gated_score_fwd(const void* X, const void* Wcat, const float* bcat, const float* ww,
                            const float* bw, float* scores, void* gate_act, int64_t total_n, int L, int D,
                            int dtype, void* workspace, size_t ws_bytes, void* stream);

/* Backward of the line above (autograd of ABMIL.py:52-54).  dscores[total_n] is dL/ds.
 * gate_act == NULL: recomputes V,U from X (nothing but s is kept from forward); otherwise uses the activations
 * the forward saved.  Outputs (fp32, overwritten):
 * dWcat[2D,L], dbcat[2D], dww[D], dbw[1].  If dX != NULL it receives
 *   dX_i = attn_i * dM[bag(i)] + dVpre_i Wv + dUpre_i Wu      (dtype of X)
 * where attn/dM/offsets describe the pooling term (pass attn=NULL to get the GEMM term only).       */
int milb200_gated_score_bwd(const void* X, const void* Wcat, const float* bcat, const float* ww,
                            const float* bw, const float* dscores, const void* gate_act, const float* attn,
                            const float* dM, const int32_t* offsets, int B, int64_t total_n, int L,
                            int D, int dtype, float* dWcat, float* dbcat, float* dww, float* dbw,
                            void* dX, void* workspace, size_t ws_bytes, void* stream);

/* Bench hook: with profiling enabled the bf16 path of milb200_gated_score_bwd records CUDA events between its
 * sub-kernels (dZ pass: recompute GEMM or elementwise | dW split-K GEMM | split-K reduce | optional dX GEMM); profile_read waits for the
 * last one and returns up to max_intervals durations in milliseconds (return value = count).              */
void milb200_profile_enable(int on);
/* Developer hook: CTA 0 of the K-major tensor-core GEMM stamps clock64() at its phase boundaries into dev_u64x16
 * (16 x uint64 on the device; NULL switches it off): 0 entry, 1 prologue done, 2/3 first/last TMA stage issued,
 * 4/5 first/last stage landed, 6 accumulator ready, 7 epilogue done, 8 all warps done, 9 TMEM released.        */
int milb200_debug_trace(void* dev_u64x16);
int milb200_profile_read(float* ms, int max_intervals);

/* ---- ragged segmented softmax + attention-weighted instance sum ---------------------------------
 * Replaces F.softmax(A, dim=1) and torch.matmul(A, x) (model/dim1/ABMIL.py:56-59), one launch for a
 * whole CSR batch: M[b] = sum_i softmax_b(s)_i x_i.  Outputs: M[B,L] fp32; M_lowp[B,L] in X's dtype
 * (may be NULL); argmax[B] int32 = index *within the bag* of the largest score, first index on ties
 * (may be NULL); lse[B] fp32 = log sum exp of the bag's scores (may be NULL).                       */
size_t milb200_pool_workspace_bytes(int64_t total_n, int B, int L);

int milb200_segment_softmax_pool_fwd(const void* X, const float* scores, const int32_t* offsets, int B,
                                     int64_t total_n, int L, int dtype, float* M, void* M_lowp,
                                     int32_t* argmax, float* lse, void* workspace, size_t ws_bytes,
                                     void* stream);

/* Backward of the pooling w.r.t. the scores (and the attention weights needed for dX):
 *   attn_i = softmax_b(s)_i (recomputed from s),  dscores_i = attn_i * (dM_b . x_i - dM_b . M_b).
 * dM, M are [B,L] fp32.  attn (fp32[total_n]) may be NULL.                                          */
int milb200_segment_softmax_pool_bwd(const void* X, const float* scores, const int32_t* offsets, int B,
                                     int64_t total_n, int L, int dtype, const float* dM, const float* M,
                                     float* dscores, float* attn, void* workspace, size_t ws_bytes,
                                     void* stream);

/* The same pair for a caller that knows dM before the forward runs (a training step whose loss gradient does not depend
 * on M): the forward also writes rowdot[i] = dM_b . x_i (fp32[total_n]) from the rows it streams anyway, and the
 * backward forms dscores and attn from rowdot without reading X.  M, M_lowp, argmax and lse equal those of
 * milb200_segment_softmax_pool_fwd, and dscores and attn equal those of milb200_segment_softmax_pool_bwd, bit for bit.
 * dM, M are [B,L] fp32.  dM, rowdot, dscores and attn must be 4-byte aligned; attn may be NULL.
 * Workspace of both: milb200_pool_workspace_bytes.                                                      */
int milb200_segment_softmax_pool_fwd_rowdot(const void* X, const float* scores, const int32_t* offsets, int B,
                                            int64_t total_n, int L, int dtype, const float* dM, float* M, void* M_lowp,
                                            int32_t* argmax, float* lse, float* rowdot, void* workspace, size_t ws_bytes,
                                            void* stream);
int milb200_segment_softmax_pool_bwd_rowdot(const float* scores, const int32_t* offsets, int B, int64_t total_n, int L,
                                            const float* dM, const float* M, const float* rowdot, float* dscores,
                                            float* attn, void* workspace, size_t ws_bytes, void* stream);

/* ---- dense linear layers ------------------------------------------------------------------------
 * Y[m,n] = act(X[m,k] W[n,k]^T + bias[n])  — nn.Linear (+Tanh/ReLU) as used by fc_pathology,
 * fc_CI2CT/fc_CI2Pth (model/aggregator.py:44,47,66), q/k/v/out projections
 * (model/sam/transformer.py:430-432,448) and MLPBlock (model/sam/common.py:26).
 * X, W, Y share `dtype`; bias fp32 (may be NULL).  If `add` != NULL the input is (X + add) — the
 * `keys + key_pe` / `queries + query_pe` sums of transformer.py:291-292,303-304 (the sum is staged in
 * the workspace, so query milb200_linear_workspace_bytes for the forward too).                      */
size_t milb200_linear_workspace_bytes(int64_t m, int n, int k, int dtype, int backward);

int milb200_linear_fwd(const void* X, const void* add, const void* W, const float* bias, void* Y,
                       int64_t m, int n, int k, int act, int dtype, void* workspace, size_t ws_bytes,
                       void* stream);

/* Backward: given dY (dtype) and the forward OUTPUT Y (for the activation derivative; unused for
 * ACT_NONE), computes dX[m,k] (dtype, may be NULL), dW[n,k] fp32, dbias[n] fp32 (may be NULL).
 * If accumulate != 0, dW/dbias are added to instead of overwritten.                                 */
int milb200_linear_bwd(const void* X, const void* add, const void* W, const void* Y, const void* dY,
                       void* dX, float* dW, float* dbias, int64_t m, int n, int k, int act, int dtype,
                       int accumulate, void* workspace, size_t ws_bytes, void* stream);

/* Mixed-precision variant for the head of the fusion path's key stream (fc_pathology, model/aggregator.py:141): X, W bf16
 * on the tensor cores, Y fp32; backward takes fp32 dY (and the fp32 output Y), returns dW / dbias fp32 and dX bf16 (may be
 * NULL).  Tensor-core shapes only (n % 16 == 0, k >= 64, k % 8 == 0; the backward also needs n >= 64 and k % 16 == 0,
 * since its dX GEMM has N = k and K = n).  Workspace (backward only):
 * milb200_linear_workspace_bytes(m, n, k, MILB200_BF16, 1).                                                          */
int milb200_linear_f32out_fwd(const void* X, const void* W, const float* bias, float* Y, int64_t m, int n, int k, int act,
                              void* stream);
int milb200_linear_f32out_bwd(const void* X, const void* W, const float* Y, const float* dY, void* dX, float* dW,
                              float* dbias, int64_t m, int n, int k, int act, int accumulate, void* workspace,
                              size_t ws_bytes, void* stream);

/* ---- LayerNorm over the last dim (nn.LayerNorm, eps 1e-5; transformer.py:288,295,300,307,118) ----
 * Y = LN(X + R) * gamma + beta, R optional residual (may be NULL).  mean/rstd[m] fp32 are saved.
 * r_broadcast != 0: R is ONE row [n] added to every row of X — with a single text token the image->token attention of
 * transformer.py:302-307 degenerates to softmax over one key (weights exactly 1, SURVEY F10), so its output is the
 * same row for every instance; the gradient of that row is the column sum of dXR (milb200_colsum).      */
int milb200_layernorm_fwd(const void* X, const void* R, const float* gamma, const float* beta, void* Y,
                          float* mean, float* rstd, int64_t m, int n, int dtype, int r_broadcast, void* stream);
/* dXR = dL/d(X+R) (same for both addends); dgamma/dbeta fp32[n] overwritten (or added to).          */
int milb200_layernorm_bwd(const void* X, const void* R, const float* gamma, const float* mean,
                          const float* rstd, const void* dY, void* dXR, float* dgamma, float* dbeta,
                          int64_t m, int n, int dtype, int accumulate, int r_broadcast, void* workspace,
                          size_t ws_bytes, void* stream);
/* out[c] (+)= sum_r A[r, c] (fp32 out): bias gradients and the gradient of a broadcast residual row.        */
int milb200_colsum(const void* A, int64_t rows, int cols, float* out, int dtype, int accumulate, void* stream);
size_t milb200_layernorm_workspace_bytes(int64_t m, int n);

/* ---- multi-head attention core (transformer.py:434-446): O = softmax(Q K^T / sqrt(c)) V per head ---
 * Q[nq, H*c], K[nk, H*c], V[nk, H*c], O[nq, H*c] (dtype); lse[H, nq] fp32 saved for backward.
 * One of nq / nk is small (text tokens, <= 16) on this path; both orientations are covered.          */
size_t milb200_attention_workspace_bytes(int64_t nq, int64_t nk, int heads, int c, int backward);
int milb200_attention_fwd(const void* Q, const void* K, const void* V, void* O, float* lse, int64_t nq,
                          int64_t nk, int heads, int c, int dtype, void* workspace, size_t ws_bytes,
                          void* stream);
int milb200_attention_bwd(const void* Q, const void* K, const void* V, const void* O, const float* lse,
                          const void* dO, void* dQ, void* dK, void* dV, int64_t nq, int64_t nk, int heads,
                          int c, int dtype, void* workspace, size_t ws_bytes, void* stream);

/* ---- CLIP-style logits and small losses -----------------------------------------------------------
 * clip/model.py:359-365: logits_per_image = exp(logit_scale) * norm(I) norm(T)^T  ([bi,bt] fp32).
 * d <= 1024, the backward's limit: a wider d is refused here, before anything is launched.           */
int milb200_clip_logits_fwd(const void* I, const void* T, const float* logit_scale, float* logits,
                            float* inv_norm_i, float* inv_norm_t, int bi, int bt, int d, int dtype,
                            void* stream);
/* Backward: upstream gradients of logits_per_image ([bi,bt]) and/or logits_per_text ([bt,bi]) — either may be
 * NULL.  dI/dT in `dtype` (may be NULL), dscale[1] = d/d logit_scale (may be NULL).  One kernel per requested
 * output; omitted outputs are not written.                                                               */
int milb200_clip_logits_bwd(const void* I, const void* T, const float* logit_scale, const float* logits,
                            const float* inv_norm_i, const float* inv_norm_t, const float* dlogits_per_image,
                            const float* dlogits_per_text, void* dI, void* dT, float* dscale, int bi, int bt,
                            int d, int dtype, void* stream);
/* utils.py:277-282 (CLIPloss_v1): logits[i] = out @ feat[:,i,:]^T ([I,b,b]), CE over dim 1 against the
 * identity, mean over I*b.  out[b,d] (dtype), feat[b,I,d] (dtype, frozen).  logits fp32 [I,b,b];
 * lse_ws fp32 [2*I*b] scratch; loss[1]; dout[b,d] fp32 (may be NULL).  d <= 1024 and b + d <= 12280 (the
 * feature row and one logits column share 48 KB of shared memory); larger shapes are refused.             */
int milb200_cliploss_fwd_bwd(const void* out, const void* feat, float* logits, float* lse_ws, float* loss,
                             float* dout, int b, int n_info, int d, int dtype, void* stream);
/* nn.CosineEmbeddingLoss(a, b, target=+1) (train_ddp.py:102,326): loss[1] = mean_i(1 - cos(a_i, b_i)) and its
 * gradients da, db ([n,d] in dtype, may be NULL).  loss_rows_ws fp32 [n] scratch.                          */
int milb200_cosine_embedding_fwd_bwd(const void* a, const void* b, float* loss, float* loss_rows_ws, void* da,
                                     void* db, int n, int d, int dtype, void* stream);
/* sigmoid + BCELoss(mean) of aggregator.py:200 / train_ddp.py:99,319: prob = sigmoid(z),
 * loss = mean BCE(prob, target) with torch's -100 clamp of both logs, dz = (prob - target)/numel.
 * z,target,prob,dz fp32[n]; prob, loss and dz may each be NULL.
 * dz is the derivative of mean BCE(sigmoid(z), target) for every z.  torch's fp32 autograd through sigmoid + BCELoss
 * agrees only for -27.6 < z < 16.6: where the fp32 prob rounds to 1 (z >= 16.6) it gives 0, because p(1-p) = 0,
 * and for z <= -27.6 it scales the gradient by p(1-p)/1e-12 (its clamp of the BCE denominator).                  */
int milb200_sigmoid_bce_fwd_bwd(const float* z, const float* target, float* prob, float* loss, float* dz,
                                int n, void* stream);

/* M[b] = sum_i x_i over CSR offsets, no softmax: what the reference computes when ABMIL.forward is handed a
 * dense batch B>1 (softmax over the size-1 K axis, model/dim1/ABMIL.py:48,56-59) and in SwinUNETR_wMask's
 * 3-crop pool (model/dim3/swinUNETR_wMask.py:60-67).  Workspace: milb200_pool_workspace_bytes.            */
int milb200_segment_sum_fwd(const void* X, const int32_t* offsets, int B, int64_t total_n, int L, int dtype,
                            float* M, void* M_lowp, void* workspace, size_t ws_bytes, void* stream);
/* out[i,:] = (w ? w[i] : 1) * src[bag(i),:]  (src fp32 [B,L], out [total_n,L] in dtype): backward of the
 * sum pool, and the a_i * dM term of the gated pool's dX.                                                */
int milb200_bag_broadcast(const float* src, const float* w, const int32_t* offsets, int B, int64_t total_n,
                          int L, int dtype, void* out, void* stream);

/* ---- elementwise glue -----------------------------------------------------------------------------*/
/* nn.Dropout(p) in train mode (ABMIL.py:49; aggregator.py:129): out = keep ? x/(1-p) : 0.  The Philox4x32-10
 * mask is a pure function of (seed, offset, element index): the same call on a gradient is the backward,
 * nothing is stored.  It cannot reproduce torch's own mask bit for bit (SURVEY F11).                       */
int milb200_dropout(const void* x, void* out, int64_t n, float p, uint64_t seed, uint64_t offset, int dtype,
                    void* stream);
/* dtype conversion fp32 <-> bf16 and a 2-D transpose out[cols,rows] = in[rows,cols]^T (weight repacking).  */
int milb200_cast(const void* in, int src_dtype, void* out, int dst_dtype, int64_t n, void* stream);
int milb200_transpose(const void* in, void* out, int rows, int cols, int dtype, void* stream);
/* out = a + b (broadcast none); any of the three dtypes per `dtype`. (keys + key_pe, residual adds)   */
int milb200_add(const void* a, const void* b, void* out, int64_t n, int dtype, void* stream);
/* out = alpha * a + beta * b (b may be NULL: out = alpha * a) — (x_CT + x_pathology) / 2 of
 * model/aggregator_clip.py:94 and gradient scaling.                                                  */
int milb200_axpby(const void* a, const void* b, void* out, int64_t n, float alpha, float beta, int dtype,
                  void* stream);
/* on-device sinusoidal table pe[n_pos, dim] (model/aggregator.py:99-106), written in `dtype`.         */
int milb200_sinusoid_pe(void* pe, int64_t n_pos, int dim, int dtype, void* stream);
/* (B,C,T,H*W) -> (T,C) mean over the trailing axis then transpose (transformer.py:93), fwd and bwd.    */
int milb200_ct_tokens_fwd(const void* fmap, void* tokens, int c, int t, int hw, int dtype, void* stream);
int milb200_ct_tokens_bwd(const void* dtokens, void* dfmap, int c, int t, int hw, int dtype, void* stream);

/* ---- static operator programs ("tapes") ------------------------------------------------------------------
 * The cross-modal fusion path (model/sam/transformer.py:58-120,278-309 as called by model/aggregator.py:160,168) is
 * ~130 launches forward / ~370 backward per bag; driven op by op from the host language it is launch-bound.  A tape
 * is that forward written down once as ops over numbered tensor slots; milb200_tape_forward runs it in ONE call and
 * keeps every activation in `arena`; milb200_tape_backward runs the reverse program (reverse-mode accumulation over
 * the slots, parameter gradients accumulated into one flat fp32 buffer).
 *   slots   [rows, cols] matrices in `dtype`; external = 1: the caller supplies the pointer (program inputs, and
 *           outputs it wants written in place, e.g. straight into the packed multi-modal bag of aggregator.py:173)
 *   params  ranges of two flat buffers with identical element offsets: w_compute (weights in `dtype`) and p_f32
 *           (fp32: biases, LayerNorm gamma/beta); gradients go to g_f32 (fp32, same offsets; cleared by the call)
 *   ops     LINEAR    out = act((in0 [+ in1]) W^T + b)      p0 = W [out.cols, in0.cols], p1 = bias or -1, a0 = act
 *           ATTENTION out = softmax(Q K^T / sqrt(c)) V      in0/in1/in2 = Q/K/V (distinct slots), a0 = heads
 *           LAYERNORM out = LN(in0 [+ in1]) * gamma + beta  p0 = gamma, p1 = beta (eps 1e-5)
 *           ADD       out = in0 + in1                       (a sum several ops share, e.g. keys + key_pe)
 *           JOIN      out = rows of in0 followed by rows of in1 (in0 is written in place: its producer's output IS the
 *                     head of out; in1 is copied)           assembling the key stream / the token rows of all segments
 *           HEADDIAG_U out[r*H + h, :] = sum_c in0[r, h*32 + c] W[h*32 + c, :]      p0 = W [256, 512] (fp32 slots)
 *           HEADDIAG_O out[r, h*32 + c] = in0[r*H + h, :] . W[h*32 + c, :] + b      p0 = W [256, 512], p1 = b [256]
 *           T2I_POOL  token -> image attention of transformer.py:290-295 with the key/value projections folded into
 *                     the token side: in0 = keys, in1 = position table, in2 = U (HEADDIAG_U of the projected queries
 *                     with k_proj.weight); out[(seg, t, h), :] = sum_n softmax_n(scale (keys + pe) . U) keys[n]
 *                     a0 = 1: keys are addressed in the packed-bag layout (segment out_start), 0: key-stream layout
 *                     (the position table in1 is always fp32)
 *           LN_SEG    out = LN(in0 + in1[segment]) * gamma + beta — image -> token attention with ONE token per
 *                     segment (softmax over one key = 1: the attention output is one row per segment, SURVEY F10)
 *                     a0 bit 0: write the rows at out_start (the packed bag of aggregator.py:173)
 *           TOK_SCATTER out = in1 with the token rows in0 [n_segs*T, 512] (fp32) written at tok_row, IN PLACE: out and in1
 *                     must be external slots at the same address (value and gradient) — the x_CT2CI / x_Pth2CI rows of
 *                     the packed bag, filled once the final token -> image attention has produced them
 * Slots may be forced to fp32 inside a bf16 program (external bit 1): the text-token side (<= 16 rows) always runs in
 * fp32 with the fp32 master weights; an op's arithmetic dtype is that of its in0.  Two mixed ops exist for bf16 programs
 * whose key stream is kept in fp32: LINEAR with a bf16 input and an fp32 result (milb200_linear_f32out_*), and LN_SEG
 * with an fp32 input and a bf16 result (the last layer writes the bf16 packed bag).  The segment ops read the segment
 * table handed to milb200_tape_forward/backward (host memory; NULL when the program has no segment ops).
 * Backward: seed_ptrs[s] != NULL gives dL/d(slot s) for program outputs (copied into the slot's gradient buffer
 * ext_grad_ptrs[s] unless the two pointers are equal: a caller-owned buffer may be seeded in place); ext_grad_ptrs[s] !=
 * NULL asks for the gradient of external input s (written there); internal slots' gradients live in the workspace.  */
enum { MILB200_OP_LINEAR = 1, MILB200_OP_ATTENTION = 2, MILB200_OP_LAYERNORM = 3, MILB200_OP_ADD = 4,
       MILB200_OP_JOIN = 5, MILB200_OP_HEADDIAG_U = 6, MILB200_OP_HEADDIAG_O = 7, MILB200_OP_T2I_POOL = 8,
       MILB200_OP_LN_SEG = 9, MILB200_OP_TOK_SCATTER = 10 };
enum { MILB200_SLOT_EXTERNAL = 1, MILB200_SLOT_F32 = 2 };
#define MILB200_MAX_SEGMENTS 16
typedef struct milb200_tape_op {
  int32_t kind, in0, in1, in2, out, p0, p1, a0;
  int32_t lane; /* 0 or 1: ops of different lanes may run concurrently (two streams / parallel graph branches); the
                   executor orders every cross-lane use of a slot, slot gradient or parameter gradient */
} milb200_tape_op;
typedef struct milb200_tape_slot {
  int64_t rows;
  int32_t cols, external; /* external: MILB200_SLOT_* flags */
} milb200_tape_slot;
typedef struct milb200_tape_param {
  int64_t offset; /* elements from the start of the flat buffers; multiple of 8 */
  int32_t rows, cols;
} milb200_tape_param;
/* One image-side bag of the fusion path: `len` rows starting at row k_start of the key stream (JOIN output); the same
 * rows start at out_start in the packed multi-modal bag, the segment's text-token rows at tok_row.                  */
typedef struct milb200_segment {
  int32_t k_start, len, out_start, tok_row;
} milb200_segment;
typedef struct milb200_segments {
  const milb200_segment* seg; /* host memory, n_segs entries */
  int32_t n_segs;
  int32_t tokens; /* T: text tokens per segment */
} milb200_segments;
size_t milb200_tape_arena_bytes(const milb200_tape_op* ops, int n_ops, const milb200_tape_slot* slots, int n_slots,
                                int dtype, const milb200_segments* segs);
size_t milb200_tape_workspace_bytes(const milb200_tape_op* ops, int n_ops, const milb200_tape_slot* slots, int n_slots,
                                    int dtype, int backward, const milb200_segments* segs);
int milb200_tape_forward(const milb200_tape_op* ops, int n_ops, const milb200_tape_slot* slots, int n_slots,
                         const milb200_tape_param* params, int n_params, void* const* ext_ptrs, const void* w_compute,
                         const float* p_f32, void* arena, size_t arena_bytes, void* workspace, size_t ws_bytes,
                         int dtype, const milb200_segments* segs, void* stream);
int milb200_tape_backward(const milb200_tape_op* ops, int n_ops, const milb200_tape_slot* slots, int n_slots,
                          const milb200_tape_param* params, int n_params, void* const* ext_ptrs,
                          void* const* ext_grad_ptrs, const void* const* seed_ptrs, const void* w_compute,
                          const float* p_f32, float* g_f32, const void* arena, size_t arena_bytes, void* workspace,
                          size_t ws_bytes, int dtype, const milb200_segments* segs, void* stream);

/* ---- single-pass backward of the gated pool: removed ------------------------------------------------------------
 * The mirrored single-pass backward (the pooling backward inside the dWcat tensor-core kernel) was slower than the
 * two-call backward once the pooling backward's row dots moved into the pool forward, and was removed (DESIGN §5c).
 * Always returns 0: callers take the two-call backward, milb200_segment_softmax_pool_bwd (or its _rowdot form) followed
 * by milb200_gated_score_bwd.                                                                                      */
int milb200_gated_pool_bwd_supported(int L, int D, int dtype);

/* ---- optimiser (train_ddp.py:111-118): fused Adam over one flat fp32 buffer -----------------------
 * g is first scaled by grad_scale (1/world after the NCCL sum = DDP's average).                      */
int milb200_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                      float lr, float beta1, float beta2, float eps, float weight_decay,
                      float grad_scale, int step, void* stream);
/* The same update with the step number in device memory: lets a captured CUDA graph of the whole training step be
 * replayed.  Both entry points form the bias corrections 1 - beta^step on the device in one way, so a counter at s
 * gives the bit-identical result of milb200_adam_step(step = s).  milb200_step_counter_inc adds 1 to the counter (one-thread kernel).   */
int milb200_adam_step_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float lr,
                          float beta1, float beta2, float eps, float weight_decay, float grad_scale,
                          const int32_t* step_dev, void* stream);
int milb200_step_counter_inc(int32_t* step_dev, void* stream);
/* torch.optim.SGD(lr, weight_decay) as the learnable-prompt configuration builds it (train_ddp.py:103-108; no
 * momentum): p -= lr * (grad_scale * g + weight_decay * p).                                          */
int milb200_sgd_step(float* param, const float* grad, int64_t n, float lr, float weight_decay, float grad_scale,
                     void* stream);

/* ---- gradient exchange + optimiser as ONE kernel over NVLink / NVSwitch peer memory -------------------------------
 * Replaces DDP's bucketed NCCL all-reduce + optimizer.step() (train_ddp.py:79,346-348) for one flat fp32 gradient buffer
 * that lives in symmetric memory (the same allocation mapped on every rank of the node; the host side obtains the
 * mappings from torch.distributed's symmetric memory): grad_local = this rank's mapping, grad_multicast = the multicast
 * mapping, signal_pads_dev = device array of `world` pointers to the ranks' zero-initialised uint32 signal pads (at least
 * pad_slot0 + 32 * world entries each).  Slice r of the buffer is reduced in the switch (multimem.ld_reduce) and
 * broadcast (multimem.st) by rank r, between two flag barriers; then every rank applies the fused optimiser update
 * (optimizer 0: Adam, 1: SGD, -1: none — exchange only, for large buffers whose update wants a full-width grid: call
 * milb200_adam_step afterwards) with grad_scale (1/world = DDP's average).  On return the gradient buffer holds the SUM over
 * ranks — bit-identical on every rank.  The allocation must be padded to a multiple of 4 * world elements.  step_dev
 * (optional, device int32): the Adam step number is read from device memory instead of `step` — a training step that is
 * replayed as a CUDA graph keeps its counter there (milb200_step_counter_inc).                                          */
int milb200_allreduce_update_symm(float* param, float* grad_local, void* grad_multicast, void* const* signal_pads_dev,
                                  int pad_slot0, int rank, int world, float* exp_avg, float* exp_avg_sq, int64_t n,
                                  int optimizer, float lr, float beta1, float beta2, float eps, float weight_decay,
                                  float grad_scale, int step, const int32_t* step_dev, void* stream);

/* ---- feeder, host side (dataset.py:366-393) ---------------------------------------------------------
 * Gathers the per-slide feature matrices of one step (what `np.load(<patient>.npy)` returns: [rows_b, L] row-major
 * HOST memory, fp32/fp64/fp16/bf16) into the packed-CSR batch the kernels read: rows back to back in `dst` (normally
 * pinned host memory, fp32 or bf16 with round-to-nearest-even) plus offsets[n_bags+1].  Replaces the reference's
 * zero-padding to 15 592 rows (dataset.py:383-390) and its per-sample `.float()`; `keep_rows[b]` (optional, strictly
 * increasing, keep_counts[b] entries) is the augmentation subset `sorted(random.sample(range(n), k))` of
 * dataset.py:375-381.  bag_pitch_bytes (optional) gives the byte stride between rows of each source matrix.
 * n_threads <= 0 uses every hardware thread.  No CUDA calls; usable without a GPU.                               */
enum { MILB200_HOST_F32 = 0, MILB200_HOST_BF16 = 1, MILB200_HOST_F16 = 2, MILB200_HOST_F64 = 3 };
int milb200_pack_bags_offsets(const int64_t* bag_rows, const int64_t* keep_counts, int n_bags, int32_t* offsets,
                              int64_t* total_rows);
int milb200_pack_bags_host(const void* const* bag_ptrs, const int64_t* bag_rows, const int64_t* bag_pitch_bytes,
                           const int32_t* const* keep_rows, const int64_t* keep_counts, int n_bags, int L,
                           int src_dtype, void* dst, int dst_dtype, int64_t dst_capacity_rows, int32_t* offsets,
                           int n_threads);

#ifdef __cplusplus
}
#endif
#endif /* MILB200_H_ */
