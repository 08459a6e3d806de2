/*
 * actionmesh_b200 — C ABI of the B200-native (sm_100a) Stage-I denoising hot path of ActionMesh.
 *
 * The reference (facebookresearch/actionmesh) is pure Python on top of PyTorch library kernels; it has no FFI of its
 * own.  Each entry point below therefore cites the reference *call site* whose arithmetic it replaces (paths relative
 * to the reference checkout).  The Python host side (actionmesh_b200/*.py) binds these with ctypes and mirrors the
 * reference's operator interfaces (AttentionProcessor.__call__, ActionMeshDenoiser.forward, SchedulerFlow.denoise,
 * ImageEncoder.encode_images); see INTEGRATION.md for the reference-side binding.
 *
 * Conventions
 *  - every function returns 0 on success, a negative amb error code otherwise; amb_last_error() gives the message;
 *  - plain pointers and sizes only (no torch types); all pointers are DEVICE pointers unless stated;
 *  - the caller allocates every output; the library keeps no caller memory;
 *  - every launch is asynchronous on the given cudaStream_t (passed as void*); no hidden synchronisation;
 *  - bf16 tensors are passed as const void* / void* (uint16 storage);
 *  - "ld*" arguments are row strides in ELEMENTS.
 */
#ifndef ACTIONMESH_B200_H_
#define ACTIONMESH_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AMB_ABI_VERSION 14

typedef void* amb_stream_t; /* cudaStream_t */

/* ---- plumbing -------------------------------------------------------------------------------------------------- */
const char* amb_last_error(void);
int amb_abi_version(void);
int amb_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- K9: CFG combine + Euler flow step + observed-frame mask ------------------------------------------------------
 * Replaces actionmesh/scheduler/guidance.py:95-118 (aggregate_cfg) and actionmesh/scheduler/scheduler.py:238-248
 * (flow step + masked in-place write, incl. the per-step `assert unobserved.any()` D2H sync, which is dropped).
 *   v   = p[0] + sum_i scales[i] * (p[i+1] - p[i])               (fp32 arithmetic on bf16 predictions)
 *   x_f = x_f + dt_signed * v      for every frame f with frame_update[f] != 0     (x fp32, in place)
 * pred element (branch k, frame f, e) lives at pred + k*branch_stride + f*frame_stride + frame_offset + e.
 */
int amb_cfg_euler_step(float* latents, const void* pred_bf16, int n_branches, const float* scales_host,
                       float dt_signed, const uint8_t* frame_update, int n_frames, int64_t n_per_frame,
                       int64_t branch_stride, int64_t frame_stride, int64_t frame_offset, amb_stream_t stream);

/* ---- LayerNorm (affine, fp32 statistics) ---------------------------------------------------------------------------
 * Replaces diffusers FP32LayerNorm at actionmesh/model/utils/block.py:64,83,98,107 and nn.LayerNorm at
 * actionmesh/model/temporal_denoiser.py:108,239; also DinoV2's LayerNorms (transformers modeling_dinov2).
 * x: (rows, cols) bf16 or fp32 (x_fp32), y: bf16 or fp32 (y_fp32).  cols in {256, 512, 1024, 2048, 4096}.
 */
int amb_layernorm(const void* x, int x_fp32, int64_t ldx, const float* gamma, const float* beta, void* y, int y_fp32,
                  int64_t ldy, int64_t rows, int cols, float eps, amb_stream_t stream);

/* ---- small elementwise helpers -------------------------------------------------------------------------------------
 * cast: fp32 -> bf16 (latents before proj_in, temporal_denoiser.py:205-206; context before to_k/to_v).
 * timestep embedding: diffusers Timesteps(num_channels=C, flip_sin_to_cos=False, downscale_freq_shift=0) as used at
 *   temporal_denoiser.py:57-61,209-213: t_r = t[r % n_t] * (1 - mask[r]) (mask may be NULL);
 *   out[r] = [sin(t_r*w_j) | cos(t_r*w_j)], w_j = exp(-ln(1e4) * j / (C/2)).
 * add_bias_rows: y[r, :] += bias, y bf16 or fp32 (A.5: zero-context cross-attention collapses to to_out.0.bias, block.py:146).
 */
int amb_cast_f32_bf16(const float* src, void* dst_bf16, int64_t n, amb_stream_t stream);
/* patchify: im2col for DinoV2's Conv2d(3, D, P, stride P) patch embedding (HF modeling_dinov2 Dinov2PatchEmbeddings, called
 * from actionmesh/model/image_encoder.py:53): pixels (T,3,H,W) fp32 -> bf16 rows (t,py,px) x cols (c,ky,kx), zero padded to
 * kpad (multiple of 64) columns so the projection runs on amb_gemm_bf16. */
int amb_patchify(const float* pixels, void* out_bf16, int n_images, int height, int width, int patch, int kpad,
                 amb_stream_t stream);
int amb_timestep_embedding(const float* t, int n_t, const float* mask, int rows, int channels, void* out_bf16,
                           amb_stream_t stream);
int amb_add_bias_rows(void* y, int y_fp32, int64_t ldy, const float* bias, int64_t rows, int cols, amb_stream_t stream);

/* ---- image preprocessing for the DinoV2 encoder (SURVEY 8(f) rank 3; on row a2's path) -------------------------------
 * Replaces the host BitImageProcessor call at actionmesh/model/image_encoder.py:48-51 (transformers < 5, requirements.txt:10:
 * PIL bicubic resize -> centre crop -> x 1/255 -> mean/std -> CHW).  Pillow's uint8 resize is a two-pass separable integer
 * convolution (libImaging/Resample.c): int32 coefficients with 22 fractional bits, accumulator seeded with 1 << 21,
 * (acc >> 22) clamped to [0, 255], uint8 between the passes; both passes are reproduced bit-exactly.
 *  resize_h_u8: src (n, in_h, in_w, channels_in in {3,4}) u8 -> dst (n, n_rows, out_w, 3) u8 for source rows [y0, y0+n_rows);
 *    bounds (out_w, 2) = (first source column, tap count), coeffs (out_w, ksize) — host-built, already restricted to the
 *    cropped output window.  All table entries must address columns inside [0, in_w).
 *  resize_v_normalize: src as written by resize_h_u8 -> dst (n, 3, out_h, out_w) fp32 = (lut256[u8] - mean[c]) / std[c];
 *    bounds (out_h, 2) in SOURCE row numbers, every tap inside [y0, y0+n_rows); mean/std are HOST pointers to 3 floats;
 *    dst_u8 (optional, may be NULL) receives the resized+cropped uint8 image (n, out_h, out_w, 3). */
int amb_resize_h_u8(const uint8_t* src, int n_images, int in_h, int in_w, int channels_in, int y0, int n_rows,
                    const int32_t* bounds, const int32_t* coeffs, int ksize, int out_w, uint8_t* dst, amb_stream_t stream);
int amb_resize_v_normalize(const uint8_t* src, int n_images, int n_rows, int y0, int out_w, const int32_t* bounds,
                           const int32_t* coeffs, int ksize, int out_h, const float* lut256, const float* mean3_host,
                           const float* std3_host, float* dst, uint8_t* dst_u8, amb_stream_t stream);

/* ---- frame preprocessing before the encoders (SURVEY 8(f) rank 3, second half) -------------------------------------------
 * Replaces the host numpy/PIL arithmetic of ImagePreprocessor.process_images (actionmesh/preprocessing/image_processor.py:
 * 26-146): RGBA frames are composited on a white background, cropped to the (shared or per-frame) foreground bounding box
 * and padded to a square with a margin.
 *  alpha_stats: rgba (n, h, w, 4) u8 -> stats (n, 5) int32 = xmin, ymin, xmax, ymax of alpha > 0 (:57-64; xmax = -1 when the
 *    frame is fully transparent) and the number of pixels with alpha > 127 (is_valid_alpha, :15-23).
 *  composite_crop_pad: -> out (n, box_h + 2 pad_y, box_w + 2 pad_x, 3) u8.  Inside the box: the float32 composite of :44-52 in
 *    the reference's operation order, times 255, truncated like `(img * 255).astype(uint8)` (:143-145); outside: 255.
 *    The uint8 result is bit-identical to the reference's PIL output. */
int amb_alpha_stats(const uint8_t* rgba, int n_images, int height, int width, int32_t* stats, amb_stream_t stream);
int amb_composite_crop_pad(const uint8_t* rgba, int n_images, int height, int width, int box_x, int box_y, int box_w, int box_h,
                           int pad_x, int pad_y, uint8_t* out, amb_stream_t stream);

/* ---- ActionBench evaluation (SURVEY 8(f) rank 4) ----------------------------------------------------------------------
 * Replaces scipy's KDTree.query at actionbench/chamfer.py:44-50,78-82: for each of n_query points (xyz fp32, row-major) the
 * Euclidean distance to and the index of its nearest point among n_reference points.  scratch_u64: n_query * 8 bytes of
 * device memory; out_dist / out_index: either may be NULL.  Ties resolve to the lowest index. */
int amb_nearest_neighbors(const float* query, int n_query, const float* reference, int n_reference, void* scratch_u64,
                          float* out_dist, int32_t* out_index, amb_stream_t stream);

/* Gradient ICP (actionbench/icp.py:53-112, gradient_icp), batched over n_problems cloud pairs x 24 starts.
 * pred (F, n_pred, 3), gt (F, n_gt, 3) fp32; r_init (24, 3, 3) the canonical start rotations (icp.py:18-49).  Per
 * (problem f, start r) the parameters are r6d[6], T[3], s[3] (in that order, 12 floats), R = r_init[r] @ rot6d(r6d) and
 * the prediction moves to x = (s ⊙ p) @ R + T; the loss is pytorch3d's chamfer_distance (mean squared nearest-neighbour
 * distance, pred->gt plus gt->pred).  Distances are exact fp32 differences; every sum runs in a fixed order, so results
 * are deterministic and a batch of F problems equals F single calls bit for bit.
 *  workspace_bytes: device scratch both functions need (amb_icp_workspace_bytes).
 *  icp_chamfer_grad: params (F, 24, 12) -> out_loss (F, 24) and out_grad (F, 24, 12), the gradient of each start's loss.
 *  gradient_icp: n_iter iterations of torch's Adam (betas 0.9/0.999, eps 1e-8) on the mean of the 24 losses from r6d =
 *    (1,0,0,0,1,0), T = 0, s = 1.  step_size / bc2_sqrt: (n_iter) fp32 device tables of lr / (1 - 0.9^t) and
 *    sqrt(1 - 0.999^t), t = 1..n_iter.  The best start of each problem is tracked like the reference: the first start
 *    with the minimum loss of an iteration replaces the best only if strictly lower, and the best is stored as the R that
 *    produced that loss with T and s AFTER that iteration's Adam step (icp.py:96-106).  Outputs: out_rot (F, 3, 3),
 *    out_t (F, 3), out_s (F, 3), out_loss (F), out_start (F, int32); loss_trace (n_iter, F, 24) may be NULL.
 *    The host does no work per iteration beyond two kernel launches. */
int amb_icp_workspace_bytes(int n_problems, int n_pred, int n_gt, size_t* bytes);
int amb_icp_chamfer_grad(const float* pred, const float* gt, int n_problems, int n_pred, int n_gt, const float* r_init,
                         const float* params, void* workspace, size_t workspace_bytes, float* out_loss, float* out_grad,
                         amb_stream_t stream);
int amb_gradient_icp(const float* pred, const float* gt, int n_problems, int n_pred, int n_gt, const float* r_init,
                     int n_iter, const float* step_size, const float* bc2_sqrt, void* workspace, size_t workspace_bytes,
                     float* out_rot, float* out_t, float* out_s, float* out_loss, int32_t* out_start, float* loss_trace,
                     amb_stream_t stream);
/* Per-problem transform (pytorch3d Scale(s).compose(Rotate(R), Translate(T)).transform_points):
 * out[f, i] = points[f, i] @ (diag(s_f) R_f) + T_f; points/out (F, n_points, 3), rot (F, 3, 3), t and s (F, 3). */
int amb_transform_points(const float* points, int n_problems, int n_points, const float* rot, const float* t,
                         const float* s, float* out, amb_stream_t stream);

/* ---- Stage II (temporal autoencoder) helpers — first "next" row of SURVEY 8(f) -----------------------------------------
 * alpha_rows: the (source_alpha, target_alpha) token of actionmesh/model/temporal_autoencoder.py:233-237 (TimestepEmbedder,
 *   model/utils/embeddings.py:56-132), fp32, written to n_rows rows `row_stride` elements apart.
 * point_embedding: FrequencyPositionalEmbedding of the query vertices (+ normals), temporal_autoencoder.py:240-243,
 *   embeddings.py:15-53, as fp32 rows zero-padded to kpad columns for the proj_query GEMM.
 * displacement_out: 2*sigmoid(-logits) - 1 on the first out_dim columns (temporal_autoencoder.py:160,269).
 * split3_bf16 / softmax_split3: the reference runs the vertex-query cross-attention block with autocast DISABLED (fp32,
 *   temporal_autoencoder.py:264-266).  Here that block runs on the bf16 tensor cores at fp32-grade accuracy by splitting
 *   every operand x = hi + lo (two bf16) and concatenating along K: activations as [hi | lo | hi] (w_pattern = 0),
 *   weights as [hi | hi | lo] (w_pattern = 1), so one amb_gemm_bf16 call evaluates a_hi w_hi + a_lo w_hi + a_hi w_lo
 *   with fp32 accumulation.  split3_bf16 cuts `cols` in segments of `seg` columns (each becomes 3*seg output columns);
 *   softmax_split3 does the row softmax of fp32 scores (n valid columns, scaled by `scale`) and writes the probabilities
 *   as the activation split with each part n_pad wide (zeros in the padding). */
int amb_alpha_rows(float source_alpha, float target_alpha, int size, float* out, int64_t row_stride, int n_rows,
                   amb_stream_t stream);
int amb_point_embedding(const float* points, int n_points, int in_dim, int extra, int num_freqs, int include_pi,
                        float* out, int kpad, amb_stream_t stream);
int amb_displacement_out(const float* logits, int64_t ld, int n_points, int out_dim, float* out, amb_stream_t stream);
int amb_split3_bf16(const float* src, int64_t ld_src, int64_t rows, int cols, int seg, int w_pattern, void* dst_bf16,
                    int64_t ld_dst, amb_stream_t stream);
int amb_softmax_split3(const float* scores, int64_t ld_s, int rows, int n, int n_pad, float scale, void* dst_bf16,
                       int64_t ld_dst, amb_stream_t stream);

/* ---- tcgen05 GEMM with fused epilogues: C = epi(A · Wᵀ) ----------------------------------------------------------------
 * Replaces every nn.Linear on the path (cuBLAS in the reference): proj_in/proj_out/time_proj
 * (temporal_denoiser.py:206,213-214,242), linear_skip on cat[skip,h] without materialising the concat (block.py:131-133,
 * a2/k_split), to_q/to_k/to_v with the head split, RMS qk-norm and RoPE of attention_processor.py:92-130 fused in the
 * epilogue, to_out + residual (attention_processor.py:147, block.py:137,146), FeedForward GELU(erf) MLP (block.py:152).
 * A:(m,k) bf16 row-major, W:(n,k) bf16 row-major (nn.Linear layout), fp32 accumulation in TMEM.
 * k % 64 == 0, n % 64 == 0.
 */
typedef struct amb_gemm_args {
  const void* a;        /* bf16 (m, k) */
  int64_t lda;
  const void* a2;       /* optional second A source supplying columns k >= k_split (NULL = unused) */
  int64_t lda2;
  int32_t k_split;      /* multiple of 64 */
  const void* w;        /* bf16 (n, k) */
  int64_t ldw;
  void* c;              /* bf16 or fp32 (m', n) */
  int64_t ldc;
  int32_t c_fp32;
  int32_t m, n, k;
  const float* bias;    /* (n) or NULL */
  const void* residual; /* (m', n) bf16/fp32 or NULL; added after the activation; may alias c */
  int64_t ldr;
  int32_t res_fp32;
  int32_t act;          /* 0 none, 1 GELU(erf) */
  const float* col_scale; /* (n) or NULL: per-column scale applied after bias/act, before residual (DinoV2 LayerScale) */
  /* output row remap: dst_row = (row / grp_rows) * grp_stride + row % grp_rows + row_off  (grp_rows == 0: identity) */
  int32_t grp_rows, grp_stride, row_off;
  /* per-head (128 columns) RMSNorm for columns [0, norm_cols): weight norm_w0 for col < norm_seg, norm_w1 otherwise
   * (norm_cols may be 0 with rope_cols > 0: RoPE without q/k norm, as in the Stage-II blocks) */
  int32_t norm_cols, norm_seg;
  const float* norm_w0;
  const float* norm_w1;
  float norm_eps;
  /* interleaved-pair RoPE for columns [0, rope_cols): cos/sin tables (n_pos, 64) fp32, pos = row / rope_rows_per_pos */
  int32_t rope_cols;
  const float* rope_cos;
  const float* rope_sin;
  int32_t rope_rows_per_pos;
  /* optional second output: the same final values rounded to bf16, (m', n) row-major with row stride ldc2 (plain epilogue only).
   * Used with the fp32 residual stream: the fp32 result continues the stream, the bf16 copy is the GEMM operand of the
   * long-skip linear (block.py:131-133), so no separate cast pass is needed. */
  void* c2;
  int64_t ldc2;
} amb_gemm_args;

int amb_gemm_bf16(const amb_gemm_args* args, amb_stream_t stream);

/* ---- tcgen05 flash attention forward ------------------------------------------------------------------------------
 * Replaces F.scaled_dot_product_attention at actionmesh/model/utils/attention_processor.py:133-139 (non-causal, no
 * mask, dropout 0) for the inflated self-attention (S = T*(N+1)) and the per-frame cross-attention (S_k = 257), and
 * DinoV2's attention (head_dim 64).  Strided 4-D views so q/k/v are read straight out of the fused QKV GEMM output and
 * o is written in (b, s, h*d) order for to_out.  Strides in elements; the innermost (d) stride is 1.
 * kv may be split in `kv_chunks` equal chunks of `sk_chunk` keys whose base pointers are k + c*k_chunk_stride (used by
 * the frame-sharded window: chunk c is rank c's all-gathered K/V).  kv_chunks == 1 for the plain case.
 */
typedef struct amb_attn_args {
  const void* q;
  const void* k;
  const void* v;
  void* o;
  int64_t q_stride_b, q_stride_h, q_stride_s;
  int64_t k_stride_b, k_stride_h, k_stride_s;
  int64_t v_stride_b, v_stride_h, v_stride_s;
  int64_t o_stride_b, o_stride_h, o_stride_s;
  int32_t batch, heads, sq, sk, head_dim;
  float scale; /* softmax scale, 1/sqrt(head_dim) in the reference */
  int32_t kv_chunks;
  int32_t sk_chunk;
  int64_t k_chunk_stride, v_chunk_stride;
} amb_attn_args;

int amb_flash_attn_fwd(const amb_attn_args* args, amb_stream_t stream);

/* fp32 attention for short sequences, head_dim 64 (the DinoV2 encoder, which the reference runs in fp32 outside autocast:
 * actionmesh/pipeline.py:664-667, model/image_encoder.py:38-55 -> HF Dinov2SelfAttention's scaled_dot_product_attention).
 * q, k, v: fp32, element (frame f, token s, head h, d) at ptr[(f * seq + s) * ld + h * 64 + d]; out likewise with ldo.
 * seq <= 320.  No mask, non-causal; softmax(scale * q k^T) v with fp32 arithmetic throughout (CUDA cores). */
int amb_attn_small_f32(const float* q, const float* k, const float* v, int64_t ld, int frames, int seq, int heads, float scale,
                       float* out, int64_t ldo, amb_stream_t stream);

/* Debug only: device buffer (5 roles x 16 iterations x 8 events of int64 clock64 stamps) receiving the role timeline of
 * CTA (0,0,0) of the head_dim-128 attention kernel; NULL switches tracing off (the default). */
int amb_debug_set_attn_trace(void* device_buffer);

#ifdef __cplusplus
}
#endif
#endif /* ACTIONMESH_B200_H_ */
