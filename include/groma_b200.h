/* groma_b200 -- C ABI of the B200-native Groma forward hot path (libgroma_b200.so, sm_100a).
 *
 * Conventions (every entry point):
 *   - returns int32_t status: 0 = GROMA_OK, otherwise a GROMA_ERR_* code; no exceptions cross the boundary
 *   - all pointers are DEVICE pointers unless a parameter says "host"; outputs and workspaces are caller-owned
 *   - `stream` is a cudaStream_t passed as void*; kernels are enqueued on it, nothing synchronises, nothing allocates
 *   - matrices are row-major bf16 (uint16 storage) unless stated; bias / norm / scale vectors are fp32
 *   - thread-compatible: no global mutable state beyond one-time kernel attribute setup
 *
 * Each declaration cites the reference interface it replaces (paths relative to the FoundationVision/Groma tree;
 * $HF = transformers 4.32 as pinned by the reference's pyproject.toml:19).
 */
#ifndef GROMA_B200_H
#define GROMA_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GROMA_OK 0
#define GROMA_ERR_ARG 1
#define GROMA_ERR_ALIGN 2
#define GROMA_ERR_CUDA 3
#define GROMA_ERR_DRIVER 4
#define GROMA_ERR_TMA_ENCODE 5
#define GROMA_ERR_UNSUPPORTED 6

/* epilogue activation / flags of groma_gemm_bf16 */
#define GROMA_ACT_NONE 0
#define GROMA_ACT_GELU 1   /* erf GELU (nn.GELU default) */
#define GROMA_ACT_RELU 2
#define GROMA_ACT_SWIGLU 3 /* columns (2j,2j+1) = (gate_j, up_j) -> out[:, j] = silu(gate)*up ; N_out = N/2 */
#define GROMA_GF_OUT_F32 1
#define GROMA_GF_BIAS_ALONG_M 2
#define GROMA_GF_PARTIAL 4
#define GROMA_GF_CONV_ROWS 8
#define GROMA_GF_CONV_COMPACT 16
#define GROMA_GF_PARTIAL_T 128 /* partials transposed: ws[split][n][m] */
#define GROMA_GF_PDL 64     /* programmatic dependent launch: A tiles are prefetched before waiting for the previous kernel */

/* D[M,N] = sum_{t<num_taps} A[m + a_row_off[t], 0:K] . B[n, t*K : (t+1)*K]   (+ bias, act, *gamma, + residual)
 * tcgen05/TMEM/TMA GEMM.  Replaces every torch.nn.Linear / nn.Conv2d(1x1, 3x3 pad 1) call on the path:
 *   groma/model/groma.py:112-119,389-401 ; groma/model/roi_align.py:128-143,251-264 ; groma/model/ddetr.py:147-151 ;
 *   $HF/models/{dinov2,llama,deformable_detr}/modeling_*.py Linear layers (cuBLAS / cuDNN in the reference).
 * A: [a_rows, lda] bf16, B: [b_rows, ldb] bf16 (lda, ldb multiples of 8; pointers 16-byte aligned).
 * num_taps > 1 = implicit-GEMM convolution over zero-bordered flat NHWC maps (a_row_off = tap row shifts, host array).
 * out[m*ld_m + n*ld_n] bf16 (or fp32 with GROMA_GF_OUT_F32); bias/gamma fp32 per column (per row with BIAS_ALONG_M);
 * residual bf16 with the strides of out.  GROMA_GF_PARTIAL: raw fp32 accumulators to ws[split][M][N] (split_k >= 1).
 * GROMA_GF_CONV_ROWS: rows are pixels of [img][conv_hp][conv_wp] maps, border rows are not written;
 * with GROMA_GF_CONV_COMPACT the row index is that of the un-padded [img][hp-2][wp-2] layout.
 * block_n: 0 = auto, else 16/32/64/128/256. */
int32_t groma_gemm_bf16(const void* A, int64_t a_rows, int64_t lda, const void* B, int64_t b_rows, int64_t ldb,
                        int32_t M, int32_t N, int32_t K, int32_t num_taps, const int32_t* a_row_off /*host*/,
                        void* out, int64_t ld_m, int64_t ld_n, int32_t flags, int32_t act, const float* bias,
                        const float* gamma, const void* residual, float* ws, int32_t split_k,
                        int32_t conv_hp, int32_t conv_wp, int32_t block_n, void* stream);

/* LLaMA attention input in ONE launch: x[B*T, K] @ w_qkv[3*H*D, K]^T (rows of w_qkv = [q heads | k heads | v heads]) with the
 * rotate-half RoPE of q and k and the KV-cache append done in the GEMM epilogue -- the [B*T, 3*H*D] intermediate of
 * groma_gemm_bf16 + groma_rope_kv never exists.  Replaces q_proj/k_proj/v_proj + apply_rotary_pos_emb + the cache torch.cat
 * of $HF/models/llama/modeling_llama.py:199-246 (called from groma/model/groma.py:389-397).  Values are bit-identical to the
 * two-launch form: the projection is rounded to bf16, rotated in fp32, rounded again.
 * q_out [B*T, H*D] bf16; cache_k / cache_v [B, H, ctx_cap, D] bf16; cos_t / sin_t fp32 [max_pos, D/2]; token t of every
 * sequence sits at position pos0 + t (pos0 + T <= ctx_cap).  D must be 128 and H even; block_n = 256 (one CTA per
 * 128x256 tile) or 512 (cta_group::2 pair, 256x256). */
int32_t groma_gemm_qkv_rope(const void* x, int64_t ldx, const void* w_qkv, int64_t ldw, int32_t B, int32_t T, int32_t H,
                            int32_t D, int32_t K, void* q_out, void* cache_k, void* cache_v, const float* cos_t,
                            const float* sin_t, int32_t pos0, int64_t ctx_cap, int32_t block_n, void* stream);

/* out = epilogue(sum_s ws[s][M][N]) -- the deferred epilogue of a GROMA_GF_PARTIAL GEMM (same chain as above). */
int32_t groma_splitk_reduce(const float* ws, int32_t splits, int32_t M, int32_t N, int32_t act, int32_t flags,
                            const float* bias, const float* gamma, const void* residual, void* out, int64_t ld_m,
                            int64_t ld_n, void* stream);

/* softmax(QK^T*scale + mask)V, bf16, head_dim 32/64/128, online softmax, fp32 accumulate.
 * Replaces $HF/models/llama/modeling_llama.py:199-289 (eager attention, causal + key padding),
 * $HF/models/dinov2/modeling_dinov2.py:153-179 and $HF/models/deformable_detr/modeling_deformable_detr.py:453-516.
 * q[b*q_bs + i*q_rs + h*D + d], k[b*k_bs + h*k_hs + j*k_rs + d] (v alike), o[b*o_bs + i*o_rs + h*D + d].
 * causal: key j visible to query i iff j <= q_pos0 + i.  kv_len (optional, int32[B]): keys >= kv_len[b] masked. */
int32_t groma_attention(const void* q, int64_t q_bs, int64_t q_rs, const void* k, int64_t k_bs, int64_t k_hs,
                        int64_t k_rs, const void* v, int64_t v_bs, int64_t v_hs, int64_t v_rs, void* o, int64_t o_bs,
                        int64_t o_rs, const int32_t* kv_len, int32_t B, int32_t H, int32_t Sq, int32_t Sk, int32_t D,
                        int32_t causal, int32_t q_pos0, float scale, void* stream);

/* The same attention on the tcgen05 tensor cores (TMA-fed, S/O accumulators in TMEM), head_dim 64 / 128.
 * q/k/v are 2-D bf16 row-major views [rows, cols] (row stride ld); element (b, i|j, h, d) lives at
 *   q: row b*q_batch_rows + i,                 col h*q_head_cols + d
 *   k: row b*k_batch_rows + h*k_head_rows + j, col h*k_head_cols + d      (v alike)
 * -- covers the KV cache [B,H,cap,D] and fused qkv activations [B*S, 3*H*D] without copies.  o: [B*Sq, o_ld], col h*D + d. */
int32_t groma_attention_tc(const void* q, int64_t q_rows, int64_t q_cols, int64_t q_ld, int32_t q_batch_rows, int32_t q_head_cols,
                           const void* k, int64_t k_rows, int64_t k_cols, int64_t k_ld, int32_t k_batch_rows, int32_t k_head_rows,
                           int32_t k_head_cols, const void* v, int64_t v_rows, int64_t v_cols, int64_t v_ld, int32_t v_batch_rows,
                           int32_t v_head_rows, int32_t v_head_cols, void* o, int64_t o_ld, const int32_t* kv_len, int32_t B,
                           int32_t H, int32_t Sq, int32_t Sk, int32_t D, int32_t causal, int32_t q_pos0, float scale, void* stream);

/* Single-query (decode) attention over the KV cache: every cached position < kv_len[b] is visible (the all-ones mask of
 * groma/model/groma.py:376-379).  q, out [B, H*D]; cache_k/v [B, H, cap, D]; D = 128.  HBM-bound SIMT kernel. */
int32_t groma_decode_attention(const void* q, const void* cache_k, const void* cache_v, void* out, const int32_t* kv_len,
                               int32_t B, int32_t H, int32_t D, int64_t cap, float scale, int32_t pdl, void* stream);

/* groma_decode_reduce_rope_kv + groma_decode_attention in one launch (decode step, D = 128): q and the new token's K/V row
 * are reduced from the qkv GEMM's split-K partials ws[splits][B][3*H*D], rotated (rotate-half RoPE at position *pos_ptr,
 * $HF/models/llama/modeling_llama.py:138-168), the K/V row is appended to the cache at *pos_ptr (the tuple-cache torch.cat of
 * groma.py:376-379) and the attention over kv_len[b] positions follows; bit-identical to the two separate calls. */
int32_t groma_decode_rope_attention(const float* ws, int32_t splits, void* cache_k, void* cache_v, void* out,
                                    const int32_t* kv_len, const int32_t* pos_ptr, const float* cos_t, const float* sin_t,
                                    int32_t B, int32_t H, int32_t D, int64_t cap, float scale, int32_t pdl, void* stream);

/* y = w * bf16(h * rsqrt(mean(h^2)+eps)), h = bf16(x + residual) (h_out optional).  LlamaRMSNorm,
 * $HF/models/llama/modeling_llama.py:53-70 (+ the residual add of :292-340). */
int32_t groma_rmsnorm(const void* x, const void* residual, const float* w, void* y, void* h_out, int64_t rows,
                      int32_t dim, float eps, void* stream);

/* y = LayerNorm(x (+ residual)) * w + b over the last dim.  nn.LayerNorm call sites: modeling_dinov2.py:356-372,
 * modeling_deformable_detr.py:699-706,782-803 (post-LN), groma/model/ddetr.py:25-45 (channel LN == LN over NHWC C),
 * groma/model/roi_align.py:254-261, ddetr_transformer.py:311-314. */
int32_t groma_layernorm(const void* x, const void* residual, const float* w, const float* b, void* y, int64_t rows,
                        int32_t dim, float eps, int64_t x_row_stride, int64_t y_row_stride, void* stream);

/* y = relu(GroupNorm_G(x)) over NHWC [B, P, C]; mmcv ConvModule norm+act (mmcv/cnn/bricks/conv_module.py:196-206)
 * as used by groma/model/roi_align.py:133-143.  part: fp32 scratch [B*chunks*G*2]; stats: fp32 [B*G*2] (mean, rstd). */
int32_t groma_groupnorm_relu(const void* x, const float* gamma, const float* beta, void* y, float* part, float* stats,
                             int32_t B, int64_t P, int32_t C, int32_t G, float eps, int32_t chunks, void* stream);
/* The two halves of the call above: statistics only (stats [B,G,2] = mean, rstd) and apply + ReLU with given statistics.  The
 * fusion rounds of MLVLFuseModule (groma/model/roi_align.py:118-126,180-193) keep the RAW conv outputs and let the next round's
 * groma_fuse_shuffle_gn apply norm + act tap by tap; only the last round's maps are materialised with groma_groupnorm_apply_relu. */
int32_t groma_groupnorm_stats(const void* x, float* part, float* stats, int32_t B, int64_t P, int32_t C, int32_t G, float eps,
                              int32_t chunks, void* stream);
int32_t groma_groupnorm_apply_relu(const void* x, const float* stats, const float* gamma, const float* beta, void* y, int32_t B,
                                   int64_t P, int32_t C, int32_t G, void* stream);

/* Multi-scale deformable attention forward; twin of mmcv `ms_deform_attn_forward`
 * (mmcv/ops/csrc/pytorch/pybind.cpp:162,765; kernel common/cuda/ms_deform_attn_cuda_kernel.cuh:203-256) with the
 * softmax over (levels*points) and the sampling-location arithmetic of modeling_deformable_detr.py:586-610 fused in.
 * value [B,S,nH,32] bf16; proj [B*Q, nH*L*P*2 + nH*L*P] fp32 (offsets | logits); ref [B,Q,ref_dim] fp32;
 * out [B,Q,nH*32] bf16; level_hw host int32[2L] (h,w), level_start host int32[L]. */
int32_t groma_msda_forward(const void* value, const float* proj, const float* ref, void* out, int32_t B, int32_t Q,
                           int32_t S, int32_t n_heads, int32_t n_levels, int32_t n_points, int32_t ref_dim,
                           const int32_t* level_hw /*host*/, const int32_t* level_start /*host*/, void* stream);

/* RoIAlign forward (avg, aligned flag); twin of mmcv `roi_align_forward` (pybind.cpp:191,611; kernel
 * common/cuda/roi_align_cuda_kernel.cuh:17-108).  input NHWC bf16 [N,H,W,C]; rois fp32 [K,5] (batch, x1,y1,x2,y2);
 * output [K, ph+2p, pw+2p, C] bf16 with p = out_pad (0/1) zero border. */
int32_t groma_roi_align_forward(const void* input, const float* rois, void* output, int32_t K, int32_t C, int32_t H,
                                int32_t W, int32_t pooled_h, int32_t pooled_w, float spatial_scale,
                                int32_t sampling_ratio, int32_t aligned, int32_t out_pad, void* stream);

/* Batched greedy NMS; twin of mmcv `nms` (pybind.cpp:175,596; nms_cuda_kernel.cuh:18-74, nms_cuda.cu:5-54) plus the
 * score filter / max_num of mmcv/ops/nms.py:14-33, for all images of groma/model/groma.py:257-280 in one launch.
 * boxes [B,N,4] xyxy fp32, scores [B,N] fp32, counts int32[B] (optional valid prefix length per image).
 * keep int64 [B,max_out] (original indices, score order, -1 padded); num_keep int32[B];
 * argmax_idx int32[B] = first index of the max score (the reference's fallback when nothing is kept). */
int32_t groma_nms_batched(const float* boxes, const float* scores, const int32_t* counts, int32_t B, int32_t N,
                          float iou_threshold, float score_threshold, int32_t offset, int32_t max_num, int64_t* keep,
                          int32_t max_out, int32_t* num_keep, int32_t* argmax_idx, void* stream);

/* torch.topk(scores, k, dim=1)[1] (ddetr_transformer.py:556): indices of the k largest, descending. */
int32_t groma_topk_desc(const float* scores, int64_t ld, int32_t B, int32_t N, int32_t k, int64_t* out_idx, void* stream);

/* Two-stage proposal gather + sigmoid + sine embedding (ddetr_transformer.py:432-446,556-566). */
int32_t groma_ddetr_select(const float* delta, const float* proposals, const int64_t* topk, float* ref_out,
                           void* pos_out, int32_t B, int32_t S, int32_t k, int32_t num_pos_feats, void* stream);

/* Final box/score heads (ddetr_transformer.py:696-715 restricted to what inference reads, groma.py:246-249,268). */
int32_t groma_ddetr_finalize(const float* d4, const float* d5, const float* ref0, const float* coco, const float* sa1b,
                             float* pred_cxcywh, float* pred_xyxy, float* score, int32_t B, int32_t Q,
                             int64_t out_stride_boxes, int64_t out_stride_scores, void* stream);

/* zero rows of x [B,S,D] where valid[s]==0 (ddetr_transformer.py:424-426). */
int32_t groma_mask_rows(void* x, const uint8_t* valid, int32_t B, int32_t S, int32_t D, void* stream);

/* Region-encoder resampling (groma/model/roi_align.py:118-126,215-228 and :150-178). */
int32_t groma_upsample_coords(const void* tokens, int32_t skip, int32_t g, int32_t C, void* out, int32_t B, int32_t Ho,
                              int32_t Wo, int32_t ld, const float* xs, const float* ys, void* stream);
int32_t groma_fuse_shuffle(const void* tar, const void* top, const void* down, void* out, int32_t B, int32_t C,
                           int32_t Ht, int32_t Wt, int32_t Htop, int32_t Wtop, int32_t Hdn, int32_t Wdn, void* stream);
/* Same shuffle over the previous round's raw conv outputs: relu(GroupNorm_G) with per-level statistics and the round's shared
 * gamma / beta (mmcv ConvModule norm + act, conv_module.py:196-206) is applied to every tap and rounded to bf16 first, so the
 * result is bit-identical to groma_groupnorm_apply_relu on each map followed by groma_fuse_shuffle. */
int32_t groma_fuse_shuffle_gn(const void* tar, const void* top, const void* down, void* out, int32_t B, int32_t C,
                              int32_t Ht, int32_t Wt, int32_t Htop, int32_t Wtop, int32_t Hdn, int32_t Wdn,
                              const float* stats_tar, const float* stats_top, const float* stats_down, const float* gamma,
                              const float* beta, int32_t G, void* stream);

/* DINOv2 embeddings (modeling_dinov2.py:57-149): im2col of 14x14 patches and CLS/pos-embed assembly. */
int32_t groma_vit_patchify(const float* images, void* patches, int32_t B, int32_t S, int32_t ld, void* stream);
int32_t groma_vit_embed(const void* patch, const float* cls, const float* pos, void* out, int32_t B, int32_t NP,
                        int32_t C, void* stream);

/* groma.py:227-242: mean of the last hidden states (CLS dropped) and the 2x2 space-to-depth token merge. */
int32_t groma_mean_tokens(const void* a0, const void* a1, const void* a2, const void* a3, int32_t n, void* out,
                          int32_t B, int32_t T, int32_t C, int32_t skip, void* stream);
int32_t groma_space_to_depth(const void* in, void* out, int32_t B, int32_t g, int32_t C, void* stream);

/* groma.py:165-174,360-369: split-vocabulary embedding lookup and visual-token splice (row gather / scatter). */
int32_t groma_gather_rows(const int64_t* idx, const void* t0, const void* t1, int64_t split, void* out, int64_t n,
                          int32_t D, void* stream);
int32_t groma_scatter_rows(const int64_t* idx, const void* src, void* out, int64_t n, int32_t D, void* stream);

int32_t groma_add(const void* a, const void* b, void* c, int64_t n, void* stream);
int32_t groma_add_bcast(const void* a, const void* b, void* c, int64_t rows, int64_t period, int32_t D, void* stream);

/* rotate-half RoPE on fused QKV rows + KV-cache append (modeling_llama.py:138-168,225-289). */
int32_t groma_rope_kv(const void* qkv, void* q_out, void* cache_k, void* cache_v, const float* cos_t,
                      const float* sin_t, int32_t B, int32_t T, int32_t H, int32_t D, int32_t pos0,
                      const int32_t* pos_ptr /*device, optional: overrides pos0*/, int64_t ctx_cap, void* stream);

/* out = act(x[M,K] @ w[N,K]^T + b) for K <= 64 in fp32 (roi_align.py:255: Linear(4,256) on the fp32 boxes). */
int32_t groma_linear_smallk(const float* x, const float* w, const float* b, void* out, int64_t M, int32_t N, int32_t K,
                            int32_t relu, void* stream);

/* device-side decode bookkeeping (*pos += 1; kv_len[b] += 1) so a decode step is CUDA-graph capturable. */
int32_t groma_decode_advance(int32_t* pos, int32_t* kv_len, int32_t B, void* stream);

/* Fused decode epilogues over token-major split-K partials ws[split][token][feature] (GROMA_GF_PARTIAL_T); pdl != 0
 * launches them with programmatic stream serialisation (they wait for their producer in-kernel).
 *   reduce_norm   : x = bf16(sum + x) in place; y = LlamaRMSNorm(x)            (modeling_llama.py:292-340,53-70)
 *   reduce_swiglu : out[:, j] = silu(sum[2j]) * sum[2j+1]                        (modeling_llama.py:171-184)
 *   reduce_rope_kv: RoPE(q,k) at *pos_ptr, q -> q_out, k/v -> cache[b,h,*pos_ptr] (modeling_llama.py:138-168,225-289) */
int32_t groma_decode_reduce_norm(const float* ws, int32_t splits, int32_t B, int32_t N, void* x, const float* w, void* y,
                                 float eps, int32_t pdl, void* stream);
int32_t groma_decode_reduce_swiglu(const float* ws, int32_t splits, int32_t B, int32_t N, void* out, int32_t pdl, void* stream);
/* Tail of a decode step in one launch: logits[b, :] = sum_s ws[s][b][:] (fp32 [B, V], what lm_head returns,
 * groma/model/groma.py:399-402), ids[b] = first maximal index (HF greedy_search's torch.argmax), then *pos += 1 and
 * kv_len[b] += 1 for the next step.  Same values as groma_splitk_reduce + groma_argmax + groma_decode_advance. */
int32_t groma_decode_head_argmax(const float* ws, int32_t splits, int32_t B, int32_t V, float* logits, int64_t* ids,
                                 int32_t* pos, int32_t* kv_len, int32_t pdl, void* stream);
int32_t groma_decode_reduce_rope_kv(const float* ws, int32_t splits, int32_t B, int32_t H, int32_t D, void* q_out, void* cache_k,
                                    void* cache_v, const float* cos_t, const float* sin_t, const int32_t* pos_ptr, int64_t cap,
                                    int32_t pdl, void* stream);

/* greedy next-token argmax over fp32 logits (HF greedy_search). */
int32_t groma_argmax(const float* logits, int64_t* out, int32_t rows, int32_t V, int64_t ld, void* stream);

int32_t groma_cast_f32_bf16(const float* a, void* b, int64_t n, void* stream);
int32_t groma_cast_bf16_f32(const void* a, float* b, int64_t n, void* stream);

/* ---- image preprocessing in front of the ViT (SURVEY.md §8f N3) ----------------------------------------------------------
 * Replaces, per image, the reference's CPU pass  PIL `Image.resize((448, 448))` (BICUBIC, uint8; groma/eval/run_groma.py:78,
 * groma/data/datasets/groma.py:94) + `BitImageProcessor.preprocess` with do_resize=False, do_center_crop=False (rescale 1/255,
 * ImageNet mean/std, CHW float32; run_groma.py:79, run_ddetr.py:39-45).
 * img: uint8 RGB, HWC, row_stride bytes between rows (device).  The resize reproduces Pillow's two-pass fixed-point resampler
 * bit for bit.  lut: float32 [3][256] = normalised value of every byte per channel (host computes it once with the processor's
 * mean/std).  tmp: uint8 [H][out_size][3] scratch.  coef: int32 scratch of GROMA_PREPROCESS_COEF_INTS(out_size).
 * out_f32: float32 [3][out_size][out_size] pixel_values (may be null), out_u8: resized uint8 [out_size][out_size][3] (may be null).
 * Sides up to 15 x out_size. */
#define GROMA_PREPROCESS_COEF_INTS(out_size) (2 * (out_size) * (2 + 64))
int32_t groma_preprocess_image(const uint8_t* img, int32_t H, int32_t W, int64_t row_stride, const float* lut,
                               int32_t out_size, uint8_t* tmp, int32_t* coef, float* out_f32, uint8_t* out_u8, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GROMA_B200_H */
