/* vqa_b200.h -- C ABI of the B200 (sm_100a) fusion / co-attention kernels.
 *
 * This is the drop-in boundary of the repository: plain pointers and sizes, no torch types.
 * The Python modules in vqa_attention_networks_b200/ (same class names / constructors / forward
 * signatures as klory/vqa-attention-networks' mfb.py, mhb_coAtt.py, hieCoAtten.py, modules.py)
 * bind these entry points with ctypes; INTEGRATION.md shows the binding a maintainer of the
 * reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer on the CUDA device that is current on the calling thread;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, nothing synchronises;
 *   - nothing is allocated inside: outputs / workspaces are caller-owned;
 *   - return value: 0 = OK, < 0 = argument error (VQA_B200_E*), > 0 = cudaError_t of the failing call;
 *     vqa_b200_last_error() returns a thread-local message for the last non-zero status;
 *   - dropout: every entry point that applies a dropout mask takes a host `seed` and an optional DEVICE pointer
 *     `seed_dev` (NULL = unused).  The mask is a counter hash of (seed', row, column) with seed' = seed when
 *     seed_dev == NULL, else mix(seed + 0x9E3779B9 * *seed_dev): a launch captured in a CUDA graph keeps its host
 *     seed for ever, so the per-step variation comes from a device counter that the graph itself increments
 *     (the low 32 bits of the training step count);
 *   - re-entrant: no mutable global state apart from per-device read-only caches (SM count).
 *   - matrices are row-major with a leading dimension in ELEMENTS; bf16 = __nv_bfloat16.
 *
 * Each entry point cites the reference code it replaces (file:line in klory/vqa-attention-networks).
 */
#ifndef VQA_B200_H_
#define VQA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VQA_B200_ABI_VERSION 2

#define VQA_B200_EINVAL (-1)   /* bad shape / null pointer                                  */
#define VQA_B200_EALIGN (-2)   /* pointer or leading dimension violates a 16-byte alignment */
#define VQA_B200_EDRIVER (-3)  /* cuTensorMapEncodeTiled unavailable or failed              */

/* operand layout of a GEMM operand X(rows, k) */
#define VQA_B200_K_MAJOR 0     /* memory [rows, K], K contiguous   */
#define VQA_B200_MN_MAJOR 1    /* memory [K, rows], rows contiguous */

#define VQA_B200_F32 0
#define VQA_B200_BF16 1

int vqa_b200_abi_version(void);
const char* vqa_b200_last_error(void);

/* ---------------------------------------------------------------------------------------------
 * vqa_b200_gemm -- tcgen05/TMEM GEMM  C[m,n] = epi( sum_k A(m,k) * B(n,k) ), bf16 in, fp32 accumulate.
 * Replaces every dense contraction on the path: nn.Linear (mhb_coAtt.py:94,124-125,136-137;
 * hieCoAtten.py:25,30-31,35-36), the 1x1 nn.Conv2d layers (mhb_coAtt.py:81,111; mfb.py:76,78,109,111)
 * and their autograd dgrad / wgrad (via the MN-major operand layouts).
 *   epilogue (accumulate == 0):  out = acc * row_scale[m / rows_per_group] + bias[n]; relu optional;
 *                                optional dot_out[m / rows_per_group] += sum_n out * dot_with[m,n];
 *                                stored as c_dtype.
 *   accumulate == 1:             C (fp32) += acc with atomics; K is split over k_split CTAs
 *                                (k_split == 0 -> chosen from the SM count).  bias/row_scale/relu unused.
 */
int vqa_b200_gemm(const void* A, int a_layout, int64_t lda,
                  const void* B, int b_layout, int64_t ldb,
                  void* C, int c_dtype, int64_t ldc,
                  int M, int N, int K,
                  const float* bias, const float* row_scale, int rows_per_group, int relu,
                  int accumulate, int k_split,
                  const void* dot_with, int64_t ld_dot, float* dot_out,
                  void* stream);

/* ---------------------------------------------------------------------------------------------
 * vqa_b200_mfb_fused -- the MFB block in one kernel (mhb_coAtt.py:97-106, mfb.py:95-104; with
 * rows_per_group == 1 also mhb_coAtt.py:125-131,137-143):
 *   acc[m, c]  = sum_k X[m,k] * W[c,k] + bias[c]            (image projection, c = 5*o + j)
 *   keep[m, c] = acc * dropout_mask(seed, m, c) / (1 - p)   (optional copy for backward, keep_dtype bf16/fp32)
 *   z[m, o]    = sum_{j<5} keep[m, 5o+j] * Q[m / rows_per_group, 5o+j]
 *   y[m, o]    = sign(z) * sqrt|z|                          (stored, y_dtype)
 *   ssq[g]    += sum |z|  over the rows of group g          (== ||y_g||^2, for F.normalize)
 * The [M, 5*o] product never reaches HBM unless `keep` is requested (training).
 * seg_cols (0 = N): columns per L2-norm segment.  Two MFB blocks that share their input (img_proj2 / img_proj3 on the
 * same pooled image vector, mhb_coAtt.py:125,137) run as ONE launch over the row-concatenated weights (N = 10000,
 * seg_cols = 5000): ssq is then [groups, N / seg_cols] and y [M, N/5] holds the blocks side by side.
 * extra (optional, fp32 [groups, N], ld = ldq) multiplies the product as well, and prod (optional, fp32 [M, N]) receives
 * the dropped-out product keep * Q * extra itself: MHB's cascade (mhb_coAtt.py:193-205) is block 1 with `prod`, then
 * block 2 with extra = block 1's prod -- the high-order coupling happens inside the epilogue, before the k-pool.
 * Requirements: N % 20 == 0, K % 8 == 0, seg_cols % 40 == 0, ssq zero-initialised by the caller.
 */
int vqa_b200_mfb_fused(const void* X, int64_t ldx, const void* W, int64_t ldw, const float* bias,
                       const float* Q, int64_t ldq, int rows_per_group,
                       void* Y, int y_dtype, int64_t ldy, float* ssq, void* keep, int keep_dtype,
                       int M, int N, int K, int seg_cols, const float* extra, float* prod, float drop_p, uint32_t seed,
                       const uint32_t* seed_dev, void* stream);

/* Materialise the dropout mask vqa_b200_mfb_fused uses (pre-scaled by 1/(1-p)); test hook so the
 * oracle can be run with the identical mask.  mask: fp32 [M, N]. */
int vqa_b200_dropout_mask(float* mask, int M, int N, float drop_p, uint32_t seed, const uint32_t* seed_dev,
                          void* stream);

/* ---------------------------------------------------------------------------------------------
 * Packing: fp32 -> bf16 with an arbitrary 3-D source stride (s0,s1,s2) and destination pitch (t0,t1; 0 =
 * contiguous [d0,d1,d2]).  Padded pitches keep TMA's 16-byte stride rule when an inner extent (L=196, T=26) is odd.
 * Replaces the permute/unsqueeze views in front of the 1x1 convs (mhb_coAtt.py:77-78,97).
 * split3: error-compensated fp32 path -- writes the bf16 hi/lo split of a [R, C] fp32 matrix three
 * times along the contraction axis so that one bf16 GEMM over 3K reproduces an fp32 GEMM to ~1e-5:
 *   role 0 (A side): [hi | hi | lo],  role 1 (B side): [hi | lo | hi].
 *   concat_rows == 0: dst [R, 3C] (K-major operand);  concat_rows == 1: dst [3R, C] (MN-major operand);
 *   per batch entry (src/dst batch strides in elements, ldd = dst row pitch).
 */
int vqa_b200_pack_bf16(const float* src, void* dst, int64_t d0, int64_t d1, int64_t d2,
                       int64_t s0, int64_t s1, int64_t s2, int64_t t0, int64_t t1, void* stream);
int vqa_b200_split3_bf16(const float* src, int64_t lds, int64_t src_bstride, void* dst, int64_t ldd,
                         int64_t dst_bstride, int64_t batch, int64_t R, int64_t C, int role,
                         int concat_rows, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Attention logits: logits[m, g] = sum_j H[m, j] * W2[g, j] + b2[g]   (the Ah -> G 1x1 conv,
 * mhb_coAtt.py:83,113; mfb.py:81,114; also fc_Whv / fc_Whq of hieCoAtten.py:40,47 with G == 1).
 * H is bf16 or fp32 [M, J]; optional per-row scale row_scale[m / rows_per_group] applied to H.
 * Backward: dH[m, j] = (H[m,j] > 0 or !relu_mask) * sum_g dlogits[m,g] * W2[g,j] (* out_scale[m/rpg]),
 *           dW2[g, j] += sum_m dlogits[m,g] * H[m,j],  db2[g] += sum_m dlogits[m,g],
 *           dbias_h[j] += sum_m dH_unscaled[m, j]   (bias gradient of the layer that produced H)
 */
int vqa_b200_attn_logits_fwd(const void* H, int h_dtype, int64_t ldh, const float* W2, const float* b2,
                             float* logits, int M, int J, int G, void* stream);
int vqa_b200_attn_logits_bwd(const void* H, int h_dtype, int64_t ldh, const float* W2, const float* dlogits,
                             void* dH, int dh_dtype, int64_t lddh, const float* out_scale, int rows_per_group,
                             int relu_mask, float* dW2, float* db2, float* dbias_h,
                             int M, int J, int G, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Softmax over the region / token axis + multi-glimpse weighted pooling in one pass over the
 * features (mhb_coAtt.py:84-91,114-121; mfb.py:82-89,116-123; hieCoAtten.py:40-43,47-50):
 *   att[n, g, l]   = softmax_l(logits[n, l, g])        (degenerate != 0: att == 1, mfb.py:84,118)
 *   pooled[n, g*D + d] = sum_l att[n,g,l] * X[n,l,d]   (glimpse-major concat)
 * X is bf16 or fp32 [N, L, D] contiguous; logits fp32 [N, L, G]; att fp32 [N, G, L]; pooled fp32.
 * Backward: dlogits[n,l,g] (fp32) and optionally dX[n,l,d] (fp32; += when accumulate_dx != 0);
 * datt_extra (optional, [N,G,L]) is an additional gradient flowing directly into att.
 * One kernel: every (sample, column chunk) CTA adds its part of datt = dP . X into the dlogits buffer, and the CTA that
 * completes a sample (ticket in done[n]; `done` is N uint32 of scratch, zeroed here together with dlogits -- by a single
 * memset when done == dlogits + N*G*L) applies the softmax Jacobian in place.
 */
int vqa_b200_softmax_pool_fwd(const void* X, int x_dtype, const float* logits, float* att, float* pooled,
                              int N, int L, int D, int G, int degenerate, void* stream);
int vqa_b200_softmax_pool_bwd(const void* X, int x_dtype, const float* att, const float* dpooled,
                              const float* datt_extra, float* dlogits, uint32_t* done, float* dX,
                              int N, int L, int D, int G, int degenerate, int accumulate_dx, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Backward of the MFB block's elementwise tail (signed sqrt + per-group L2 normalise + k-pool +
 * Hadamard), mhb_coAtt.py:100-108 in reverse:
 *   given g = d(loss)/d(y_hat) * inv[grp]  ([M, No], bf16/fp32), y, inv[grp] = 1/max(||y_g||,eps),
 *   t[grp] = sum y*g:   dy = g - y * inv^2 * t;  dz = dy / (2|y|) (0 where y == 0);
 *   dI[m, c]  = dz[m, c/5] * Q[grp, c] * mask(m, c) / (1-p)          -> bf16 or fp32 [M, N] (wgrad operand)
 *   dQ[grp,c] = sum_{m in grp} dz[m, c/5] * keep[m, c]                (keep = saved (acc+bias)*mask, ld = N)
 *   dbias[c] += sum_m dz[m, c/5] * Q[grp, c] * mask / (1-p)           (atomic; zero-initialise)
 * seg_cols (0 = N) as in vqa_b200_mfb_fused: inv and t are then [groups, N / seg_cols].
 * Cascade (rows_per_group == 1 only): with u[m,c] = dz[m,c/5] + dprod_in[m,c] (dprod_in: optional gradient arriving at the
 * block's dropped-out product from the NEXT block) and Qe = Q * extra (extra optional):
 *   dI = u * Qe * mask/(1-p);   dQ = (sum u * keep) * extra;   dExtra (optional) = (sum u * keep) * Q.
 */
int vqa_b200_mfb_bwd(const void* G, int g_dtype, int64_t ldg, const void* Y, int y_dtype, int64_t ldy,
                     const float* inv, const float* t, const float* Q, int64_t ldq, const void* keep,
                     int keep_dtype, void* dI, int di_dtype, float* dQ, float* dbias, int rows_per_group,
                     int M, int N, int seg_cols, const float* extra, const float* dprod_in, float* dExtra,
                     float drop_p, uint32_t seed, const uint32_t* seed_dev, void* stream);

/* First half of F.normalize's backward for the vector MFB blocks (mhb_coAtt.py:133,145 in reverse):
 *   g[m,o] = d[m,o] * inv[m / rows_per_group];   t[grp] += sum_o y[m,o] * g[m,o]   (zero-initialise t) */
int vqa_b200_norm_bwd_prep(const float* d, int64_t ldd, const void* Y, int y_dtype, int64_t ldy,
                           const float* inv, float* g, int64_t ldg, float* t, int rows_per_group,
                           int M, int No, void* stream);

/* y_hat[m, o] = y[m, o] * inv[m / rows_per_group], inv = 1 / max(sqrt(ssq), 1e-12)   (F.normalize,
 * mhb_coAtt.py:107,133,145).  vqa_b200_inv_norm fills inv from ssq. */
int vqa_b200_inv_norm(const float* ssq, float* inv, int n, void* stream);
int vqa_b200_scale_rows(const void* Y, int y_dtype, int64_t ldy, const float* inv, int rows_per_group,
                        float* out, int64_t ldo, int M, int No, void* stream);

/* Small reductions / elementwise steps of the backward pass.
 *   group_dot: t[m / rows_per_group] += sum_o A[m,o] * B[m,o]         (zero-initialise t)
 *   colsum   : out[j] += sum_m X[m,j]                                 (bias gradients)
 *   relu_bwd : out[m,j] = (H[m,j] > 0 ? D[m,j] : 0) * scale[m / rows_per_group] (scale optional);
 *              dbias[j] += the unscaled masked value                  (autograd of F.relu + conv bias) */
int vqa_b200_group_dot(const void* A, int a_dtype, int64_t lda, const void* B, int b_dtype, int64_t ldb,
                       float* t, int rows_per_group, int M, int No, void* stream);
int vqa_b200_colsum(const void* X, int x_dtype, int64_t ldx, float* out, int M, int J, void* stream);
int vqa_b200_relu_bwd(const void* D, int d_dtype, int64_t ldd, const void* H, int h_dtype, int64_t ldh,
                      void* out, int o_dtype, int64_t ldo, const float* scale, int rows_per_group,
                      float* dbias, int M, int J, void* stream);

/* ---------------------------------------------------------------------------------------------
 * vqa_b200_gemm_batched -- the same tcgen05 kernel over `batch` independent problems (rank-3 TMA maps),
 * used for hieCoAtten's per-sample products (hieCoAtten.py:32 affinity Cq Cv^T, :38 que_^T C, :45 img_^T C^T,
 * and their autograd) and modules.py's Attention_2 (modules.py:91,94):
 *   C[b,m,n] = dropout( act( sum_k A_b(m,k) B_b(n,k) + bias[n] + add[b,m,n] ) )      act: 0 none, 1 ReLU, 2 tanh
 * Strides are in elements; C / add share ldc and c_bstride.  batch == 1 with bstride 0 is a plain GEMM with
 * the extended epilogue (e.g. img_emb + ReLU + always-on dropout, hieCoAtten.py:25-26).
 * accumulate != 0: C (fp32) += product (atomics), epilogue options unused.
 */
int vqa_b200_gemm_batched(const void* A, int a_layout, int64_t lda, int64_t a_bstride,
                          const void* B, int b_layout, int64_t ldb, int64_t b_bstride,
                          void* C, int c_dtype, int64_t ldc, int64_t c_bstride,
                          int batch, int M, int N, int K, const float* bias, int act,
                          const void* add, int add_dtype, float drop_p, uint32_t seed, const uint32_t* seed_dev,
                          int accumulate, void* stream);

/* Elementwise steps of hieCoAtten.py:25-50 and modules.py:26-33,103-109.
 *   act_fwd : out = dropout(act(x + add + bias[col])), fp32, act 0 none / 1 ReLU / 2 tanh / 3 sigmoid; the mask is
 *             the counter hash of (row, col, seed) (same function as the GEMM epilogues).
 *   act_bwd : dpre = dout * mask/(1-p) * act'(.) with act' recovered from the saved OUTPUT h (relu: h > 0;
 *             tanh: 1 - (h (1-p))^2 on kept elements); dbias[col] += dpre (optional).
 *   row_softmax_{fwd,bwd}: softmax over the last axis of a [rows, cols] fp32 matrix (modules.py:90).
 *   gate_{fwd,bwd}: o = tanh(a) * sigmoid(b) (modules.py:105-108) and its backward. */
int vqa_b200_act_fwd(const float* x, const float* add, const float* bias, float* out, int64_t rows, int cols,
                     int act, float drop_p, uint32_t seed, const uint32_t* seed_dev, void* stream);
int vqa_b200_act_bwd(const void* D, int d_dtype, int64_t ldd, const void* H, int h_dtype, int64_t ldh,
                     void* out, int o_dtype, int64_t ldo, float* dbias, int M, int J, int act, float drop_p,
                     uint32_t seed, const uint32_t* seed_dev, void* stream);
int vqa_b200_row_softmax_fwd(const float* x, float* y, int64_t rows, int cols, void* stream);
int vqa_b200_row_softmax_bwd(const float* y, const float* dy, float* dx, int64_t rows, int cols, void* stream);
int vqa_b200_gate_fwd(const float* a, const float* b, float* o, int64_t n, void* stream);
int vqa_b200_gate_bwd(const float* a, const float* b, const float* d_o, float* da, float* db, int64_t n, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Question-encoder recurrence (the stage that feeds the question attention; SURVEY.md 8f rank 2).
 * Replaces the cuDNN/ATen recurrence behind `self.lstm(...)` at mhb_coAtt.py:72-74 (single layer, zero
 * initial state, gate order i,f,g,o as torch.nn.LSTM) for the reference's shape regime: S sequence steps
 * over Bt <= 32 rows (the reference feeds the [T, N, E] permutation to a batch_first LSTM, so S = N = 256
 * and Bt = T = 26).  One cooperative persistent kernel per direction: H/8 CTAs, W_hh resident in registers
 * as mma fragments, per-CTA step flags instead of a kernel launch per step.
 *   lstm_fwd: gates [S,Bt,4H] fp32 holds x W_ih^T + b_ih + b_hh on entry (tcgen05 GEMM, vqa_b200_gemm);
 *             out[t] = h_t (fp32 [S,Bt,H]); hb (bf16 [S+1,Bt,H]) is the step-to-step exchange buffer: on entry
 *             hb[0] = 0 (h_{-1}) and every other element = the bf16 bit pattern 0xFFFF ("not written yet"; consumers
 *             poll the data itself, there are no flags); on exit hb[t+1] = bf16(h_t);
 *             c_all != NULL (training): gates is overwritten with the activated gates, c_all[t] = c_t.
 *   lstm_bwd: dout[t] = dL/dh_t; writes dg[t] = dL/d(pre-activation gates) (bf16 [S,Bt,4H], pre-filled with
 *             0xFFFF by the caller: it is the exchange buffer of the backward recurrence); the weight / input
 *             gradients are GEMMs over dg (vqa_b200_gemm).  dout element (t, b, j) is read at dout[t*dout_st + b*dout_sb + j]
 *             (the gradient arrives in the caller's [Bt, S, H] order: no transposing copy); whh is the bf16 recurrent
 *             weight, w_layout 1 = W_hh itself [4H, H] (the parameter's layout), 0 = a transposed copy [H, 4H].
 *   drop_p > 0: the dropout the reference applies to the LSTM's output (`self.dropout_l(lstm_o)`, mhb_coAtt.py:74,
 *             mfb.py:70) is fused: lstm_fwd stores out[t] = h_t * mask / (1 - p) (hb and the recurrence keep the clean h_t)
 *             and lstm_bwd multiplies dout by the same mask, regenerated from (seed, seed_dev) as in vqa_b200_mfb_fused;
 *             mask element (t * Bt + b, j) = vqa_b200_dropout_mask's element of the [S * Bt, H] matrix.
 * H in {128,256,512,1024}; time-major layouts.  vqa_b200_lstm_supported reports whether (Bt, H) is inside that regime. */
int vqa_b200_lstm_supported(int Bt, int H);
int vqa_b200_lstm_fwd(float* gates, const void* whh, float* out, void* hb, float* c_all,
                      int S, int Bt, int H, float drop_p, uint32_t seed, const uint32_t* seed_dev, void* stream);
int vqa_b200_lstm_bwd(const float* gates, const float* c_all, const float* dout, int64_t dout_st, int64_t dout_sb,
                      const void* whh, int w_layout, void* dg, int S, int Bt, int H,
                      float drop_p, uint32_t seed, const uint32_t* seed_dev, void* stream);

/* Wide-batch regime of the same recurrence (mfb.py:68-70: MFB's question encoder is a proper batch_first LSTM, S = T = 26
 * steps over Bt = N = 64..512 rows).  Per step the recurrent product is a tcgen05 GEMM (vqa_b200_gemm, accumulate == 1)
 * onto the x-projection that `gates` already holds, followed by ONE elementwise pass:
 *   lstm_cell_fwd: gates [Bt,4H] fp32 = x_t W_ih^T + b + h_{t-1} W_hh^T on entry (planes i,f,g,o as torch.nn.LSTM);
 *                  c_out = f c_prev + i g (c_prev NULL = zero initial state), h = o tanh(c_out) stored fp32 at
 *                  out[b * ld_out + j] (any row pitch: the caller's [Bt, S, H] result is written in place) and bf16 at
 *                  hb_next [Bt,H] (the A operand of the next step's GEMM and of the dW_hh wgrad); save_gates != 0
 *                  (training): gates is overwritten with the activated gates.
 *   lstm_cell_bwd: step t of the reverse sweep.  dout[b * ld_dout + j] = dL/dh_t from above; dh [Bt,H] fp32 = the
 *                  recurrent part (accumulated by the GEMM dg_{t+1} W_hh of the previous call; zero at t = S-1) and is
 *                  RESET to zero for this step's GEMM; dc [Bt,H] fp32 carries dL/dc across steps (zero at t = S-1);
 *                  writes dg [Bt,4H] bf16 = dL/d(pre-activation gates), the operand of the dh, dW_ih, dW_hh, dx GEMMs.
 *   row0 = t * Bt (the step's first row of the time-major [S * Bt, H] matrix) indexes the fused output dropout
 *   (drop_p, seed, seed_dev as in lstm_fwd / lstm_bwd): applied to `out` in the forward, to `dout` in the backward.
 * H % 4 == 0; fp32 pointers 16-byte aligned, bf16 pointers 8-byte aligned. */
int vqa_b200_lstm_cell_fwd(float* gates, const float* c_prev, float* c_out, float* out, int64_t ld_out,
                           void* hb_next, int Bt, int H, int save_gates,
                           int64_t row0, float drop_p, uint32_t seed, const uint32_t* seed_dev, void* stream);
int vqa_b200_lstm_cell_bwd(const float* gates, const float* c_prev, const float* c_t, const float* dout,
                           int64_t ld_dout, float* dh, float* dc, void* dg, int Bt, int H,
                           int64_t row0, float drop_p, uint32_t seed, const uint32_t* seed_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Fused multi-tensor Adam step (SURVEY.md 8f rank 1: the optimizer right behind the block; replaces the
 * torch.optim.Adam update of solver.py:30,91-94 -- same arithmetic as ATen's fused kernel: no amsgrad, no weight
 * decay).  For tensor i (fp32, numel[i] elements):
 *   m = m + (g - m)(1 - beta1);  v = beta2 v + (1 - beta2) g^2;
 *   p = p - (lr / (1 - beta1^step)) * m / (sqrt(v) / sqrt(1 - beta2^step) + eps)
 * and, when params_bf16 != NULL and params_bf16[i] != NULL, the bf16 copy of the new p is written as well (the
 * K-major / MN-major GEMM operand of the next step).  The pointer tables are HOST arrays of n_tensors DEVICE pointers;
 * tensors are processed 32 per launch.  step is the 1-based count of this update. */
int vqa_b200_adam_step(int n_tensors, void* const* params, const void* const* grads, void* const* exp_avg,
                       void* const* exp_avg_sq, void* const* params_bf16, const int64_t* numel, double lr,
                       double beta1, double beta2, double eps, int64_t step, void* stream);
/* The same update with the step count read from DEVICE memory (int64, 1-based, already incremented for this update):
 * the form a CUDA graph of the whole train step captures -- the graph increments the counter itself, so every replay
 * applies the bias corrections of its own step (solver.py:91-94 inside torch.cuda.graph). */
int vqa_b200_adam_step_dev(int n_tensors, void* const* params, const void* const* grads, void* const* exp_avg,
                           void* const* exp_avg_sq, void* const* params_bf16, const int64_t* numel, double lr,
                           double beta1, double beta2, double eps, const int64_t* step_dev, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Classifier tail of the eval / inference path (SURVEY.md 8f rank 3): F.log_softmax over the answer axis
 * (mhb_coAtt.py:149-151) and the prediction `softmax(logits).max(1)[1]` of the val loop (solver.py:148-149) in one
 * kernel over the classifier GEMM's logits: logp[m,:] = logits[m,:] - logsumexp (may alias logits; NULL = not wanted),
 * pred[m] = argmax (int64, lowest index on ties, as torch), pred_logp[m] = its log-probability.  fp32, ld in elements. */
int vqa_b200_logsoftmax_argmax(const float* logits, int64_t ldl, float* logp, int64_t ldo, int64_t* pred,
                               float* pred_logp, int M, int N, void* stream);

/* Training loss of the reference's solver in one pass per direction (solver.py:26-29,77-92: nn.KLDivLoss(), i.e.
 * reduction 'mean' = sum over ALL M * N elements / (M * N), on log_softmax(logits, 1) -- mhb_coAtt.py:149-151 -- against
 * the soft answers of utils.py:250-265; SURVEY.md 8f rank 1 "optimizer + loss step"):
 *   fwd: loss[0] += sum_{m,n} (xlogy(t, t) - t * (x - lse_m)) / (M * N)   (loss zeroed by the caller; atomics);
 *        lse[m] = log sum_n exp(x[m,n]), tsum[m] = sum_n t[m,n] are left for the backward.
 *   bwd: dlogits[m,n] = gout[0] * (exp(x[m,n] - lse[m]) * tsum[m] - t[m,n]) / (M * N)   (gout NULL = 1).
 * fp32, row pitches in elements. */
int vqa_b200_kldiv_logsoftmax_fwd(const float* logits, int64_t ldl, const float* target, int64_t ldt,
                                  float* loss, float* lse, float* tsum, int M, int N, void* stream);
int vqa_b200_kldiv_logsoftmax_bwd(const float* logits, int64_t ldl, const float* target, int64_t ldt,
                                  const float* lse, const float* tsum, const float* gout, float* dlogits,
                                  int64_t ldd, int M, int N, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Debug builds only (-DVQA_B200_DEBUG; `VQA_B200_DEBUG=1 python -m vqa_attention_networks_b200.build`): hooks that write
 * PROCESS-GLOBAL state and instrumented kernels.  They are not part of the drop-in boundary: a release library neither
 * exports them nor carries the cycle counters they read, and is free of mutable global state.
 *   set_mn_desc : override the MN-major shared-memory descriptor strides of every later GEMM (descriptor sweeps);
 *   set_counters: device buffer of 16 uint64 that vqa_b200_gemm fills with pipeline wait-cycle counters of CTA 0/1;
 *   set_lstm    : device buffer of 16 uint64 per CTA for the recurrence kernels' per-phase cycle counters + experiment
 *                 switches (bits 0..7 of `mode`: 2 skips the MMAs, for timing only; bits 16..31 = the number of CTAs the
 *                 buffer holds, 0 = CTA 0 only; tools/lstm_phase_probe.py). */
#ifdef VQA_B200_DEBUG
void vqa_b200_debug_set_mn_desc(uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t kadv_bytes);
void vqa_b200_debug_set_counters(void* device_u64x16);
void vqa_b200_debug_set_lstm(void* device_u64x16, int mode);
#endif

#ifdef __cplusplus
}
#endif
#endif /* VQA_B200_H_ */
