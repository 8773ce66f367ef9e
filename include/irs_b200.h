/*
 * irs_b200.h -- C ABI of libirs_b200.so: the B200 (sm_100a) kernels behind the IRN hot path of
 * JackShDr/InfluentialRS.  This is the drop-in boundary (SURVEY.md section 8b): plain pointers and
 * sizes, no torch types.  The reference has no FFI of its own (it is pure PyTorch), so each entry
 * point cites the reference Python call site whose arithmetic it replaces (paths relative to the
 * reference tree); INTEGRATION.md shows the ctypes binding a reference maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; tensors are row-major and
 *     contiguous; ids are int64_t (torch.LongTensor, data_provider.py:575); data are float (fp32).
 *   - item ids are 1-based, 0 = PAD; score column j <-> item id j + item_base (item_base = 1 for
 *     `project`, model/influentialRS.py:83,422).
 *   - all functions are asynchronous on `stream` (a cudaStream_t passed as void*), never allocate,
 *     never synchronise; scratch memory is passed in by the caller and sized with the matching
 *     *_workspace_bytes() query.
 *   - return value: 0 = OK; > 0 = cudaError_t of the failing launch; < 0 = IRS_E_* argument error.
 *     irs_error_string() explains either.  There is no CPU fallback anywhere.
 */
#ifndef IRS_B200_H_
#define IRS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IRS_B200_ABI_VERSION 1

#define IRS_E_BADARG   (-1)   /* null pointer / non-positive size                       */
#define IRS_E_SHAPE    (-2)   /* shape outside what the kernel supports (message says)  */
#define IRS_E_WORKSPACE (-3)  /* workspace too small                                    */
#define IRS_E_OVERFLOW (-4)   /* candidate buffer overflow (mass ties at the threshold) */

int irs_abi_version(void);
const char* irs_error_string(int code);
/* Number of kernel launches issued through this library since the last reset (bench.py's
 * gpu_launches claim is read from here). */
long long irs_launch_count(void);
void irs_launch_count_reset(void);

/* ---- a1 : item embedding gather + sqrt(d) scale + positional encoding -------------------------
 * out[r,:] = table[ids[r],:] * scale + pe[r % L,:]      (two separately rounded fp32 ops)
 * replaces  self.item_embedder(seq) * math.sqrt(d) + self.pos_embedder(seq)
 *           model/influentialRS.py:174-175, model/uRS.py:55, model/layers.py:31-32
 * rows = B*L.  pe may be NULL (no positional term). */
int irs_embed_gather_fwd(const int64_t* ids, const float* table, const float* pe, float scale,
                         float* out, int64_t rows, int L, int d, int64_t table_rows, void* stream);

/* ---- backward of a1 : scatter-add into the embedding table ------------------------------------
 * d_table[ids[r],:] += d_out[r,:] * scale   for ids[r] != pad_id      (d_table is NOT zeroed here)
 * replaces  autograd of nn.Embedding(padding_idx=0) under loss.backward()
 *           model/influentialRS.py:111,307  (ATen embedding_dense_backward) */
int irs_embed_scatter_add_bwd(const int64_t* ids, const float* d_out, float scale, float* d_table,
                              int64_t rows, int d, int64_t table_rows, int64_t pad_id, void* stream);

/* ---- a2 : personalised impressionability factor --------------------------------------------------
 * r_u[b] = w . user_table[users[b],:] + c[0]      (c may be NULL)
 * replaces  self.user_mask_layer(self.user_embedder(user))    model/influentialRS.py:56-61,76,180
 * user_table [n_user,du] fp32, w [du] = user_mask_layer.weight, c [1] = user_mask_layer.bias. */
int irs_pif_fwd(const int64_t* users, const float* user_table, const float* w, const float* c, float* r_u,
                int B, int du, int64_t n_user, void* stream);

/* ---- a3+a4 : self-attention with the Personalized Impressionability Mask built in-kernel ------
 * Scores s[i,j] = (q_i . k_j)/sqrt(dh) + M[b,i,j];  out_i = softmax_j(s) V.
 *   mode IRS_MASK_PIM    : M = (j == L-1) ? w_obj*r_u[b] : (j <= i ? w_h : -inf),  -inf if ids[b,j]==0
 *                          model/influentialRS.py:139-151 (keyword branch) + :171,189-193
 *   mode IRS_MASK_CAUSAL_PAD : M = (j <= i ? 0 : -inf), -inf if ids[b,j]==0        model/uRS.py:47-61
 *   mode IRS_MASK_CAUSAL : M = (j <= i ? 0 : -inf), ids ignored (may be NULL)      model/sas.py:168-177
 * q/k/v point at element [b=0, l=0, head 0, 0]; position l of batch b is at  + (b*L + l)*ld_x,
 * head h at + h*dh (this is the layout nn.MultiheadAttention's packed in_proj produces).
 * Only query rows [q_row0, q_row0+n_q) are computed; out is [B, n_q, H*dh]; lse (optional,
 * [B,H,n_q]) receives log-sum-exp of the masked scores for the backward pass.
 * A query row whose keys are all masked yields NaN, as torch's softmax does.
 * p_drop > 0 (training): attention-probability dropout, out_i = sum_j softmax(s)_ij m_ij V_j with m_ij in {0, 1/(1-p)}
 * a counter-based function of (seed, b*H+h, i, j) -- what nn.MultiheadAttention(dropout=p) does in train mode
 * (model/influentialRS.py:67-74); irs_pim_attn_bwd regenerates the same mask from the same (p_drop, seed).
 * Windows of up to IRS_ATTN_MAX_L positions: every attention entry point returns IRS_E_SHAPE above it.  The whole
 * head's K and V stay in shared memory while that layout fits 227 KB (L <= 582 for dh = 32, <= 346 for dh = 64);
 * longer windows run the key-blocked kernel of irs_pim_attn_fwd_blocked, with the same results up to rounding. */
#define IRS_ATTN_MAX_L      2048
#define IRS_MASK_PIM        0
#define IRS_MASK_CAUSAL_PAD 1
#define IRS_MASK_CAUSAL     2
int irs_pim_attn_fwd(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                     const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                     float* out, float* lse, int B, int L, int H, int dh, int q_row0, int n_q,
                     float p_drop, unsigned long long seed, void* stream);
/* Key-blocked fp32 forward with the same contract (dropout mask included, bit for bit), for 1 <= L <= 2048 and
 * 1 <= dh <= 256; shared memory holds one 64-key block at a time, so it does not depend on L.  Online softmax:
 * results equal irs_pim_attn_fwd's up to fp32 rounding.  irs_pim_attn_fwd calls it when its own layout exceeds
 * 227 KB; it is exported for tests and benchmarks. */
int irs_pim_attn_fwd_blocked(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                             const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                             float* out, float* lse, int B, int L, int H, int dh, int q_row0, int n_q,
                             float p_drop, unsigned long long seed, void* stream);

/* Tensor-core (tcgen05) forward with the same contract, for dh in {16,32,48,64} and 1 <= L <= 2048
 * (irs_pim_attn_tc_supported); bf16 hi/lo split MMAs with fp32 accumulation, ~1e-5 relative.  No dropout.
 * lse (optional, [B,H,n_q]) as for irs_pim_attn_fwd: the training forward (dropout 0) runs here and hands lse to
 * irs_pim_attn_bwd.  L <= 223 runs the kernel that keeps the head's K and V^T in shared memory, as before;
 * longer windows run irs_pim_attn_fwd_tc_blocked. */
int irs_pim_attn_tc_supported(int L, int dh);
int irs_pim_attn_fwd_tc(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                        const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                        float* out, float* lse, int B, int L, int H, int dh, int q_row0, int n_q,
                        int* error_flag, void* stream);
/* Key-blocked tcgen05 forward, same contract and shapes as irs_pim_attn_fwd_tc (any 1 <= L <= 2048).  One CTA per
 * (batch, head, 128-row query tile); K and V stream through shared memory in blocks of 128 keys, so shared memory
 * and tensor memory (256 columns) do not depend on L.  Two passes per tile: the row max of the masked scores, then
 * P = exp2(s - max) and O += P V.  The PIM objective key L-1 is an exact fp32 term of every row.  q/k/v rows and
 * out must be 16-byte aligned. */
int irs_pim_attn_fwd_tc_blocked(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                                const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                                float* out, float* lse, int B, int L, int H, int dh, int q_row0, int n_q,
                                int* error_flag, void* stream);

/* Persistent tcgen05 forward for full windows of 129..223 positions with 32-wide heads
 * (irs_pim_attn_img_supported), the BASELINE cfg3/cfg5 decoder shape.  Its input is the q/k/v projection in
 * "operand image" form: per (batch, head) one contiguous block (irs_qkv_images_bytes / (B*H) bytes) holding
 * q (pre-scaled by log2(e)/sqrt(dh)), k and v as bf16 hi/lo halves in the shared-memory layout the MMAs
 * consume (csrc/qkv_image.cuh), so that staging a head is one bulk copy.  The images are produced either by
 * irs_qkv_to_images from the fp32 packed projection, or directly by irs_decoder_chain_tc (qkv_images).
 * The image buffer must be zero-initialised once by the caller (padding rows/columns are never written);
 * after that it can be reused for any call with the same (B, L, H).
 * n_q must be L (out [B, L, H*32]) or 1 (only row q_row0, out [B, 1, H*32]). */
int irs_pim_attn_img_supported(int L, int dh);
size_t irs_qkv_images_bytes(int B, int L, int H, int dh);
int irs_qkv_to_images(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                      void* images, int B, int L, int H, int dh, int mode, void* stream);
int irs_pim_attn_fwd_img(const void* images, const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                         float* out, int B, int L, int H, int dh, int q_row0, int n_q,
                         int* error_flag, void* stream);

/* backward of the above (all rows).  d_q/d_k/d_v are written (not accumulated) with the same
 * leading dimensions as q/k/v;  d_r_u[b] += w_obj * sum_{h,i} dS[b,h,i,L-1]   (PIM mode only; the
 * caller zeroes d_r_u once per step and every layer accumulates into it).  Windows whose q, k, v and dO do not
 * fit 227 KB of shared memory (L > 286 for dh = 32, > 171 for dh = 64) run irs_pim_attn_bwd_blocked. */
int irs_pim_attn_bwd(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                     const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                     const float* out, const float* lse, const float* d_out,
                     float* d_q, float* d_k, float* d_v, float* d_r_u,
                     int B, int L, int H, int dh, float p_drop, unsigned long long seed, void* stream);
/* Key-blocked fp32 backward, same contract (1 <= L <= 2048, 1 <= dh <= 256, shared memory independent of L): one
 * kernel per 32-row query tile gives dQ and the objective's d_r_u, one per 32-key tile gives dK and dV. */
int irs_pim_attn_bwd_blocked(const float* q, const float* k, const float* v, int64_t ld_q, int64_t ld_k, int64_t ld_v,
                             const int64_t* ids, const float* r_u, float w_h, float w_obj, int mode,
                             const float* out, const float* lse, const float* d_out,
                             float* d_q, float* d_k, float* d_v, float* d_r_u,
                             int B, int L, int H, int dh, float p_drop, unsigned long long seed, void* stream);

/* ---- a4 : fused (bias +) residual + LayerNorm, optionally followed by "+ const, LayerNorm" ----
 * t = x + y (+ y_bias);  o = LN(t; g1,b1,eps);  if g2: o = LN(o + c2; g2,b2,eps)
 * replaces norm1(x + sa) and norm2(x + cross_attn) of nn.TransformerDecoderLayer as configured at
 * model/influentialRS.py:67-74; the cross-attention over the all-zero memory (:172-173) is the
 * constant vector c2 = W_o b_v + b_o.  y/y_bias/c2/g2/b2 may be NULL. */
int irs_residual_layernorm(const float* x, const float* y, const float* y_bias,
                           const float* g1, const float* b1, const float* c2, const float* g2, const float* b2,
                           float eps, float* out, int64_t rows, int d, void* stream);

/* ---- a4 on the tensor cores : decoder-body linear layers with fused epilogues ------------------
 * C[R,Nout] = epi(A[R,K] W[Nout,K]^T), fp32 in HBM, bf16 hi/lo split + 3 tcgen05.mma per K step
 * (fp32-faithful to ~1e-5 relative), K <= 256, Nout <= 256, lda/ldc/K multiples of 4, 16-byte aligned.
 * `prepared` = W re-tiled once by irs_linear_prepare_weights (irs_linear_prepared_bytes bytes).
 *   epilogue 0: acc + bias            self_attn.in_proj           (nn.MultiheadAttention in_proj)
 *   epilogue 1: relu(acc + bias)      linear1 + activation        (model/influentialRS.py:67-74)
 *   epilogue 2: LN(resid + acc + bias; g1,b1,eps) and, if g2, LN(. + c2; g2,b2,eps)
 *                                     out_proj + norm1 (+ zero-memory cross-attention constant + norm2),
 *                                     linear2 + norm3
 * error_flag: device int, set non-zero if the kernel's pipeline watchdog fires (never in normal use). */
size_t irs_linear_prepared_bytes(int Nout, int K);
int irs_linear_prepare_weights(const float* W, int Nout, int K, void* prepared, void* stream);
int irs_linear_tc(const float* A, int64_t lda, const void* prepared, const float* bias, int epilogue,
                  const float* resid, int64_t ldr, const float* g1, const float* b1,
                  const float* c2, const float* g2, const float* b2, float eps,
                  float* C, int64_t ldc, int64_t R, int K, int Nout, int* error_flag, void* stream);

/* ---- a4 fused : everything between two attention kernels of a post-norm decoder layer ---------
 * One persistent tcgen05 kernel per layer (d = 128, ffn = 256; irs_decoder_chain_supported):
 *   y   = LN2( LN1(x + attn Wo^T + bo; g1,b1) + c2; g2,b2 )     out_proj, norm1, zero-memory cross-attention
 *                                                               constant (c2 = Wo' b_v' + bo'), norm2
 *   x'  = LN3( y + relu(y W1^T + bf1) W2^T + bf2; g3,b3 )       linear1, relu, linear2, norm3
 *   qkv'= x' Win^T + bin                                        in_proj of the NEXT layer
 * Same arithmetic as three irs_linear_tc calls + the next in_proj; the activations never leave the SM
 * in between.  `prepared` = the four matrices re-tiled once, in consumption order, by
 * irs_decoder_chain_prepare_weights (Win NULL <=> no in_proj; irs_decoder_chain_prepared_bytes bytes).
 * attn, x, x_out [R,128]: contiguous rows, 32-byte aligned; x_out may alias x.
 * qkv' goes either to qkv_out [R,384] (fp32 rows) or to qkv_images (the operand images of
 * irs_pim_attn_fwd_img for windows of L positions, R = B*L, 4 heads of 32; buffer zero-initialised once by
 * the caller) -- at most one of the two; with both NULL the in_proj is skipped.
 * replaces nn.TransformerDecoderLayer.forward minus self-attention, model/influentialRS.py:67-74,189-193
 *          (+ MultiheadAttention in_proj of the following layer), model/uRS.py:62-66. */
int irs_decoder_chain_supported(int d, int ffn);
size_t irs_decoder_chain_prepared_bytes(int d, int ffn, int with_in_proj);
int irs_decoder_chain_prepare_weights(const float* Wo, const float* W1, const float* W2, const float* Win,
                                      int d, int ffn, void* prepared, void* stream);
int irs_decoder_chain_tc(const float* attn, const float* x, const void* prepared,
                         const float* bo, const float* g1, const float* b1, const float* c2,
                         const float* g2, const float* b2, const float* bf1, const float* bf2,
                         const float* g3, const float* b3, const float* bin,
                         float eps1, float eps2, float eps3,
                         float* x_out, float* qkv_out, void* qkv_images, int L, int mask_mode,
                         int64_t R, int d, int ffn, int* error_flag, void* stream);
/* First layer: qkv = x Win^T + bin straight into operand images (same kernel, in_proj stage only).
 * `prepared_with_in_proj` is ANY chain stream prepared with this Win (its in_proj units are used). */
int irs_in_proj_images_tc(const float* x, const void* prepared_with_in_proj, const float* bin,
                          void* qkv_images, int L, int mask_mode, int64_t R, int d,
                          int* error_flag, void* stream);

/* ---- window / history exclusion lists ---------------------------------------------------------
 * Sorts each row of excl_ids [M, Lx] (0 = ignore) ascending into int32 columns (id - item_base),
 * dropping pads and ids outside [item_base, item_base+N) (an id held twice is listed twice).  out_sorted is [M, Lx]
 * int32, out_count [M] int32.  Lx <= 2048.
 * replaces the boolean outer compares of  model/influentialRS.py:423-427, :312-323, utils.py:8-12 */
int irs_sort_exclusions(const int64_t* excl_ids, int M, int Lx, int64_t item_base, int64_t N,
                        int32_t* out_sorted, int32_t* out_count, void* stream);

/* One generation step of the window (model/influentialRS.py:440-449: temp <- [temp[1:L-1], next, target]) applied to its
 * sorted exclusion list in place: one occurrence of removed_ids[m*removed_stride] (the id that slid out) leaves, the pick
 * inserted_ids[m] enters; ids outside [item_base, item_base+N) and PAD are ignored.  Replaces re-sorting every window at
 * every step (at 8 GPUs every rank keeps all 32,768 windows: 0.3 ms per step). */
int irs_exclusions_update(int32_t* sorted, int32_t* count, const int64_t* removed_ids, int64_t removed_stride,
                          const int64_t* inserted_ids, int M, int Lx, int64_t item_base, int64_t N, void* stream);

/* ---- a5+a7 : full-catalog scoring fused with the visited-item mask and top-k ------------------
 * s[m,j] = h[m,:] . W[j,:] + bias[j];  for each row the k best (score desc, item id asc) among
 * columns not listed in excl_sorted.  Logits never reach HBM.
 * replaces  self.project(x) -> softmax -> topk(100) -> history filter -> [0]
 *           model/influentialRS.py:214,418-429 (softmax is monotone; D7 extension: best item not in
 *           the window), and sort -> +1 -> delete_item_in_history -> [:top_k]
 *           model/sas.py:380-386, model/caser.py:291-298.
 * h rows are ld_h floats apart.  vals [M,k] float, items [M,k] int64 (= column + item_base).
 * k == 1 costs one pass over W; k > 1 costs two (threshold, then collect).  1 <= k <= 1024. */
size_t irs_score_topk_workspace_bytes(int M, int64_t N, int d, int k);
int irs_score_topk(const float* h, int64_t ld_h, const float* W, const float* bias, int64_t item_base,
                   const int32_t* excl_sorted, const int32_t* excl_count, int Lx, int k,
                   float* vals, int64_t* items, int M, int64_t N, int d,
                   void* workspace, size_t workspace_bytes, void* stream);

/* ---- a5+a7 on the tensor cores (tcgen05, sm_100a) : arg-max of the catalog scores -------------
 * Same contract as irs_score_topk with k == 1, for d <= 128.  `prepared` is the catalog matrix W
 * re-tiled once per weight version by irs_scorer_prepare_weights (bf16 hi/lo split in the shared-
 * memory image the MMA consumes; irs_scorer_prepared_bytes(N, d) bytes).  Scores are accumulated
 * as three bf16 tcgen05.mma (hi*hi + hi*lo + lo*hi) in fp32; every candidate within the error band
 * of the leader is re-scored with the exact fp32 FMA chain, so values and winners are those of
 * irs_score_topk.  `variant` bit 1 (value 2, the production setting): ONE bf16 MMA per K step (hi*hi only, a third of
 * the tensor work and half of the weight traffic) with the candidate band widened to a rigorous bound of the bf16
 * rounding error, 2 * 2^-8 |h_m| max_j|W_j| -- the exact re-scoring then sees a few more candidates but the winners are
 * still the fp32 winners.  variant 0: three MMAs (hi*hi + hi*lo + lo*hi) and a 1e-4 band.  Bit 0 swaps the descriptor
 * strides (bring-up only).
 * replaces  model/influentialRS.py:214,418-429 (see irs_score_topk). */
size_t irs_scorer_prepared_bytes(int64_t N, int d);
int irs_scorer_prepare_weights(const float* W, int64_t N, int d, void* prepared, void* stream);
size_t irs_score_argmax_tc_workspace_bytes(int M, int64_t N, int d);
int irs_score_argmax_tc(const float* h, int64_t ld_h, const float* W, const void* prepared, const float* bias,
                        int64_t item_base, const int32_t* excl_sorted, const int32_t* excl_count, int Lx,
                        float* vals, int64_t* items, int M, int64_t N, int d, int variant,
                        void* workspace, size_t workspace_bytes, void* stream);

/* The same arg-max over a ROW-SHARDED catalog, one process per shard, in two phases around one max-reduction:
 *   phase 1  scores the shard (W, prepared, bias, item_base describe the shard) and writes lead[0..M) = the shard's best
 *            tensor-core score of every row (-inf if no live column) and lead[M] = the shard's rounding-error scale
 *            (max_j |W_j|^2); the candidate keys stay in `workspace`;
 *   caller   max-reduces lead[0..M] over the shards (ncclAllReduce, ncclMax);
 *   phase 2  (same arguments, same workspace, lead_global = the reduced vector) re-scores exactly only the candidates
 *            inside the error band of the GLOBAL leader: a shard that cannot hold a row's winner returns (-inf, -1) for
 *            it without reading W.  Merging the shards' (vals, items) with irs_topk_merge gives the winners of
 *            irs_score_argmax_tc over the whole catalog; at 8 shards the exact re-scoring does an eighth of the work.
 * (new: the reference gathers full logits on one GPU, pipeline.py:43-44) */
int irs_score_argmax_tc_phase1(const float* h, int64_t ld_h, const float* W, const void* prepared, const float* bias,
                               int64_t item_base, const int32_t* excl_sorted, const int32_t* excl_count, int Lx,
                               float* lead, int M, int64_t N, int d, int variant,
                               void* workspace, size_t workspace_bytes, void* stream);
int irs_score_argmax_tc_phase2(const float* h, int64_t ld_h, const float* W, const void* prepared, const float* bias,
                               int64_t item_base, const int32_t* excl_sorted, const int32_t* excl_count, int Lx,
                               const float* lead_global, float* vals, int64_t* items, int M, int64_t N, int d, int variant,
                               void* workspace, size_t workspace_bytes, void* stream);

/* ---- a5/a12/a13 on the tensor cores : top-k (k > 1) of the catalog scores, d <= 256 ---------------
 * Same contract, values, item ids and tie order as irs_score_topk.  Pass 1 = the fused scorer with ONE bf16 tcgen05 MMA per
 * K step and an epilogue that keeps only the best score of every 32-column chunk ([M, N/32] floats; the [M,N] scores never
 * exist).  Pass 2 (one CTA per row) = radix-select of the k-th largest chunk maximum tau, then every chunk whose maximum is
 * within the rigorous bf16 rounding bound of tau is re-scored column by column with the fp32 FMA chain of the CUDA-core
 * engine and the k best (score desc, id asc) are emitted.  `prepared` = irs_scorer_prepare_weights(W) (d <= 256).
 * replaces  softmax + topk(100) + filter  model/influentialRS.py:418-434 (sample=True; irs_topk_sample then draws the pick),
 *           sort + delete_item_in_history + [:k]  model/sas.py:357-388, model/caser.py:273-299, model/baselines.py:527-550 */
size_t irs_score_topk_tc_workspace_bytes(int M, int64_t N, int d, int k);
int irs_score_topk_tc(const float* h, int64_t ld_h, const float* W, const void* prepared, const float* bias,
                      int64_t item_base, const int32_t* excl_sorted, const int32_t* excl_count, int Lx, int k,
                      float* vals, int64_t* items, int M, int64_t N, int d,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ---- a6/a11 : log-sum-exp over the catalog + gather of selected logits ------------------------
 * lse[m] = log sum_j exp(s[m,j]);  logit[m,t] = s[m, sel[m,t]-item_base]  (sel == 0 -> 0.0)
 * CE loss row = lse - logit.   replaces nn.CrossEntropyLoss over masked_select'ed [M,N] logits
 *           model/influentialRS.py:294-303, and LogSoftmax + 2 gathers model/evaluator.py:194-205 */
size_t irs_score_lse_gather_workspace_bytes(int M, int64_t N, int d, int n_sel);
int irs_score_lse_gather(const float* h, int64_t ld_h, const float* W, const float* bias, int64_t item_base,
                         const int64_t* sel, int n_sel, float* lse, float* logit,
                         int M, int64_t N, int d, void* workspace, size_t workspace_bytes, void* stream);

/* Tensor-core (tcgen05) version of the above for d <= 128: the scores are accumulated as three bf16 MMAs
 * (hi*hi + hi*lo + lo*hi, fp32 accumulation; ~1e-5 relative) and reduced by an online log-sum-exp in the
 * epilogue; the selected logits are computed exactly (fp32 FMA chain), so a cross-entropy row lse - logit
 * carries only the lse's error.  `prepared` as for irs_score_argmax_tc (irs_scorer_prepare_weights). */
size_t irs_score_lse_gather_tc_workspace_bytes(int M, int64_t N, int d);
int irs_score_lse_gather_tc(const float* h, int64_t ld_h, const float* W, const void* prepared, const float* bias,
                            int64_t item_base, const int64_t* sel, int n_sel, float* lse, float* logit,
                            int M, int64_t N, int d, void* workspace, size_t workspace_bytes, void* stream);

/* ---- a8/a11 : rank of a label among non-excluded items, by counting (no sort) -----------------
 * rank[m] = 1 + #{j not excluded : s[m,j] > s_l  or (s[m,j] == s_l and j < l)}, l = label-item_base;
 * rank[m] = 0 if the label itself is excluded (the reference then skips the sample).
 * replaces sort(descending) + _delete_item_in_history + (indices==label).nonzero()
 *           model/influentialRS.py:375-388, model/evaluator.py:121-131,266-286 */
size_t irs_score_rank_workspace_bytes(int M, int64_t N, int d);
int irs_score_rank(const float* h, int64_t ld_h, const float* W, const float* bias, int64_t item_base,
                   const int64_t* label, const int32_t* excl_sorted, const int32_t* excl_count, int Lx,
                   int64_t* rank, int M, int64_t N, int d,
                   void* workspace, size_t workspace_bytes, void* stream);

/* Tensor-core (tcgen05) version of irs_score_rank for d <= 128, same contract and the same (exact) ranks: scores come
 * from three bf16 MMAs; columns further than the rounding-error bound from the label's exact fp32 score are counted in
 * the epilogue, the few inside the bound are listed and re-scored with the exact fp32 FMA chain.  `prepared` as for
 * irs_score_argmax_tc. */
size_t irs_score_rank_tc_workspace_bytes(int M, int64_t N, int d);
int irs_score_rank_tc(const float* h, int64_t ld_h, const float* W, const void* prepared, const float* bias,
                      int64_t item_base, const int64_t* label, const int32_t* excl_sorted, const int32_t* excl_count,
                      int Lx, int64_t* rank, int M, int64_t N, int d,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ---- a8/a11/a12/a13 across catalog shards (SURVEY 8e row 3) -----------------------------------------
 * The reference's only multi-GPU route gathers full [B,L,N] logits on GPU 0 (pipeline.py:43-44,
 * evaluator_pipeline.py:46-47,137-138) before the consumers model/evaluator.py:245-290,292-323 run.  With the catalog
 * row-sharded a rank is  1 + sum over shards of "items of my shard ahead of the label", a log-probability is the label's
 * exact score minus the log-sum-exp merge of the per-shard lse values.
 *
 * irs_score_select: out[m,t] = exact fp32 score of item sel[m,t] (the tile engines' sequential FMA chain), -inf when the
 *   item is 0 (PAD) or outside this shard [item_base, item_base+N): a MAX all-reduce over the shards yields the score. */
int irs_score_select(const float* h, int64_t ld_h, const float* W, const float* bias, int64_t item_base,
                     const int64_t* sel, int n_sel, float* out, int M, int64_t N, int d, void* stream);

/* irs_score_count_ahead: count[m] = #{j in this shard, not excluded : s[m,j] > label_score[m] or (== and item j before
 *   the label's id)}; label[m] is a GLOBAL item id that may belong to another shard; label_excluded[m] = 1 iff the label is
 *   in this shard and in the row's exclusion list.  rank = (sum label_excluded > 0) ? 0 : 1 + sum count over the shards.
 *   fp32 CUDA-core engine, any d. */
size_t irs_score_count_ahead_workspace_bytes(int M, int64_t N, int d);
int irs_score_count_ahead(const float* h, int64_t ld_h, const float* W, const float* bias, int64_t item_base,
                          const int64_t* label, const float* label_score,
                          const int32_t* excl_sorted, const int32_t* excl_count, int Lx,
                          int64_t* count, int32_t* label_excluded, int M, int64_t N, int d,
                          void* workspace, size_t workspace_bytes, void* stream);

/* The same counts on the tensor cores (tcgen05; same exact integers; `prepared` / workspace as for irs_score_rank_tc). */
int irs_score_count_ahead_tc(const float* h, int64_t ld_h, const float* W, const void* prepared, const float* bias,
                             int64_t item_base, const int64_t* label, const float* label_score,
                             const int32_t* excl_sorted, const int32_t* excl_count, int Lx,
                             int64_t* count, int32_t* label_excluded, int M, int64_t N, int d,
                             void* workspace, size_t workspace_bytes, void* stream);

/* ---- a6 backward : softmax-CE gradient with logits recomputed tile by tile --------------------
 * p = exp(s - lse);  g[m,j] = (p - [j == target[m]]) * gscale;   target is a 0-based column, or <0
 * to skip the row.   d_h[m,:] = sum_j g W[j,:];  d_W[j,:] += sum_m g h[m,:];  d_bias[j] += sum_m g.
 * d_h is written; d_W / d_bias are accumulated into (caller zeroes them).
 * replaces autograd of project + CrossEntropyLoss  model/influentialRS.py:214,303,307 */
int irs_score_ce_bwd(const float* h, int64_t ld_h, const float* W, const float* bias,
                     const int64_t* target, const float* lse, float gscale,
                     float* d_h, float* d_W, float* d_bias, int M, int64_t N, int d, void* stream);

/* Tensor-core (tcgen05) version of irs_score_ce_bwd for d <= 128, same contract (d_h written, d_W / d_bias
 * accumulated; any of the three may be NULL).  Logits are recomputed tile by tile as three bf16 MMAs (hi/lo split,
 * fp32 accumulation), the gradient tile g is written back in place over them in tensor memory and multiplied with
 * the streamed tile a second time (d_h = g W, d_W = g^T h) -- two passes of one kernel with the operands swapped.
 * workspace: irs_score_ce_bwd_tc_workspace_bytes(M, N, d) bytes (bf16 hi/lo images of h and W). */
size_t irs_score_ce_bwd_tc_workspace_bytes(int M, int64_t N, int d);
int irs_score_ce_bwd_tc(const float* h, int64_t ld_h, const float* W, const float* bias,
                        const int64_t* target, const float* lse, float gscale,
                        float* d_h, float* d_W, float* d_bias, int M, int64_t N, int d,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- multi-GPU shard merge --------------------------------------------------------------------
 * vals/items [G, M, k] per-shard candidates (as all-gathered) -> best k per row by (score desc,
 * item id asc).  G*k <= 4096. */
int irs_topk_merge(const float* vals, const int64_t* items, int G, int M, int k,
                   float* out_vals, int64_t* out_items, void* stream);

/* ---- a7 sample=True : one draw from the softmax over the k best (model/influentialRS.py:430-434) -------------------------
 * vals/items [G, M, k] per-shard candidates in the layout of irs_topk_merge (G = 1 on one GPU) -> out_items[m], one item
 * per row.  G*k <= 4096.  Per row m:
 *   1. merge the G*k candidates to the best k by (score desc, item id asc), exactly as irs_topk_merge;
 *   2. the finite survivors v_0 >= v_1 >= ... (in that order) get the weights w_i = exp(v_i - v_0), in fp64;
 *   3. S = w_0 + w_1 + ... and C_i = w_0 + ... + w_i, both added one after another in that order (so S = C_last);
 *   4. out = the first survivor with C_i > u*S, or the last finite survivor if rounding leaves none.
 * The draw depends only on the merged list, never on G: sharded and single-GPU picks are equal.
 * u is a 53-bit uniform in [0, 1), a pure function of (seed, step, row_key[m]); with 64-bit unsigned wrap-around,
 * phi = 0x9E3779B97F4A7C15 and fmix64 the murmur3 finaliser
 *   (x ^= x >> 33; x *= 0xff51afd7ed558ccd; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53; x ^= x >> 33):
 *     x = fmix64(seed + phi * (step + 1));  x = fmix64(x + phi * (row_key[m] + 1));  u = (x >> 11) * 2^-53
 * (step and row_key as two's-complement 64-bit words).  Edge rows: no finite candidate (every item excluded) -> -1, what
 * the arg-max returns; any candidate carrying the overflow marker (NaN score or item -2) of irs_score_topk -> -2.
 * replaces  softmax + multinomial over the k survivors (torch's RNG)  model/influentialRS.py:430-434 */
int irs_topk_sample(const float* vals, const int64_t* items, int G, int M, int k,
                    unsigned long long seed, int64_t step, const int64_t* row_key,
                    int64_t* out_items, void* stream);

/* ---- a7 window update (device-side, no host sync) ---------------------------------------------
 * seq[b,:] <- [seq[b,1:L-1], next[b], seq[b,L-1]];  paths[b,step] = (float)next[b]
 * replaces the per-sample shift-left of model/influentialRS.py:436,442-449 (gap_len = 0). */
int irs_window_shift(int64_t* seq, const int64_t* next, float* paths, int B, int L, int P, int step, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* IRS_B200_H_ */
