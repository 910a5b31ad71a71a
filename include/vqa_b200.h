/*
 * vqa_b200.h -- C ABI of libvqa_b200.so, the B200-native (sm_100a) VQAScore engine.
 *
 * This is the drop-in boundary for the scoring hot path of linzhiqiu/t2v_metrics: one call computes, for a batch of
 * (image, question) pairs, the score the reference's VQAScoreModel.forward() returns
 * (t2v_metrics/models/vqascore_models/vqa_model.py:10-18, called from t2v_metrics/score.py:104-106).
 * For CLIP-FlanT5 that is exp(-mean CE(logits, labels)) of T5ForConditionalGeneration on the spliced
 * [text | 576 CLIP patch features | text] sequence (v3.0 clip_t5_model.py; arithmetic in
 * transformers/models/t5/modeling_t5.py:992-1133 and transformers/models/clip/modeling_clip.py:647-696).
 *
 * Conventions
 *   - plain C types only; every pointer documented as HOST or DEVICE memory;
 *   - the caller owns all buffers (weights, inputs, outputs, workspace); the library never frees caller memory and
 *     keeps only borrowed device pointers to the bound weights;
 *   - all work is enqueued on the given CUDA stream (passed as void* = cudaStream_t); no internal device sync;
 *   - every function returns 0 on success or a negative vqa_status; vqa_last_error() gives the message;
 *   - a handle belongs to one device and one in-flight call; distinct handles are independent.
 */
#ifndef VQA_B200_H
#define VQA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VQA_B200_ABI_VERSION 1

typedef enum {
    VQA_OK = 0,
    VQA_ERR_INVALID_ARG = -1,
    VQA_ERR_MISSING_WEIGHT = -2,
    VQA_ERR_CUDA = -3,
    VQA_ERR_WORKSPACE = -4,
    VQA_ERR_UNSUPPORTED = -5
} vqa_status;

typedef enum { VQA_DTYPE_BF16 = 0, VQA_DTYPE_F32 = 1, VQA_DTYPE_I32 = 2 } vqa_dtype;

/* CLIP-FlanT5 architecture description (replaces the HF config objects the reference loads in
 * t2v_metrics/models/vqascore_models/mm_utils.py:182-241). */
typedef struct {
    /* CLIP ViT vision tower (transformers/models/clip/modeling_clip.py) */
    int32_t image_size;       /* 336 */
    int32_t patch_size;       /* 14 */
    int32_t vit_hidden;       /* 1024 */
    int32_t vit_heads;        /* 16 (head_dim must be 64) */
    int32_t vit_mlp;          /* 4096 */
    int32_t vit_layers_run;   /* encoder layers executed = select_layer -2 -> num_hidden_layers - 1 = 23 */
    float   vit_ln_eps;       /* 1e-5 */
    /* T5 encoder-decoder (transformers/models/t5/modeling_t5.py) */
    int32_t d_model;          /* 4096 (xxl) / 2048 (xl) */
    int32_t n_heads;          /* 64 / 32 (d_kv must be 64) */
    int32_t d_ff;             /* 10240 / 5120 */
    int32_t enc_layers;       /* 24 */
    int32_t dec_layers;       /* 24 */
    int32_t vocab;            /* 32128 */
    int32_t rel_buckets;      /* 32 */
    int32_t rel_max_distance; /* 128 */
    float   t5_ln_eps;        /* 1e-6 */
    int32_t image_token_id;   /* -200, t2v_metrics/constants.py:7 */
    int32_t pad_token_id;     /* 0 */
    int32_t decoder_start_id; /* 0 */
    int32_t emulate_bf16_rounding; /* bit flags. 1: the small decoder kernels round scores / bias adds to bf16 where the reference's eager path
                                      does. 2: the tcgen05 attention forms the reference's bf16 score tensors before the softmax (off: fp32
                                      scores). 4: fuse the encoder's T5LayerNorms into the GEMMs around them -- needs t5.enc.{i}.qkv_g / wi_g
                                      (= qkv . diag(ln0), wi . diag(ln1)); the o / wo epilogues emit row sums of squares, the qkv / wi
                                      epilogues apply rsqrt(mean(x^2) + eps) to their accumulator rows */
    int32_t cross_attention_mode;  /* 0: absorbed (q.(Wk x) = (Wk^T q).x, needs t5.dec.{i}.ckT); 1: project K/V of all
                                      encoder rows in every decoder layer, as modeling_t5.py:297-299 does */
} vqa_clipt5_config;

/* A named device tensor handed to vqa_bind_weights (borrowed pointer, bf16, row-major contiguous). */
typedef struct {
    const char* name;  /* HOST string, canonical engine name (see INTEGRATION.md for the HF -> engine mapping) */
    const void* data;  /* DEVICE pointer */
    int64_t shape[4];
    int32_t ndim;
    int32_t dtype;     /* vqa_dtype; weights must be VQA_DTYPE_BF16 */
} vqa_tensor;

/* Qwen2.5-VL architecture description (vision tower + language model; transformers/models/qwen2_5_vl/
 * configuration_qwen2_5_vl.py:51-64,106-125; 7B values in comments). The vision tower's 80-wide heads are laid out
 * zero-padded to 128 columns per head in the fused qkv / proj weights, and its MLP width is padded to a multiple of 128
 * (both done by the host when it fuses the checkpoint tensors, engine.convert_qwen_state_dict). */
typedef struct {
    int32_t vit_depth;        /* 32 */
    int32_t vit_hidden;       /* 1280 */
    int32_t vit_heads;        /* 16 */
    int32_t vit_head_dim;     /* 80 (real head width; stored padded to 128) */
    int32_t vit_mlp;          /* 3420 (stored padded to 3456) */
    int32_t patch_dim;        /* 3 * temporal_patch(2) * 14 * 14 = 1176 */
    int32_t spatial_merge;    /* 2 */
    int32_t out_hidden;       /* 3584 */
    uint64_t fullatt_mask;    /* bit l set: vision block l attends over whole frames (7,15,23,31), else 112-px windows */
    int32_t hidden;           /* 3584 */
    int32_t layers;           /* 28 */
    int32_t heads;            /* 28 (head_dim must be 128) */
    int32_t kv_heads;         /* 4 */
    int32_t mlp;              /* 18944 */
    int32_t vocab;            /* 152064 */
    float   rms_eps;          /* 1e-6 */
    int32_t emulate_bf16_rounding;
} vqa_qwen25vl_config;

typedef struct vqa_handle vqa_handle;

/* ABI / build info ("vqa_b200 abi=1 sm_100a ..."). Never fails. */
const char* vqa_version(void);

/* Create an engine for a CLIP-FlanT5 model on CUDA device `device`. */
int vqa_create_clipt5(const vqa_clipt5_config* cfg, int device, vqa_handle** out);

/* Borrow device pointers of the model weights. May be called several times; names are matched exactly.
 * Replaces model_cls.from_pretrained(...).to(device, bf16) (mm_utils.py:201,228) -- loading stays in the host. */
int vqa_bind_weights(vqa_handle* h, const vqa_tensor* tensors, int32_t n);

/* Check that every weight the forward needs is bound with the right shape. */
int vqa_finalize_weights(vqa_handle* h);

/* Bytes of device workspace vqa_clipt5_score needs for up to `batch` pairs, `n_images` distinct images,
 * text length `text_len` (ids per row incl. the image slot) and `label_len` target tokens. */
size_t vqa_clipt5_workspace_bytes(vqa_handle* h, int32_t batch, int32_t n_images, int32_t text_len,
                                  int32_t label_len);

/* Score `batch` (image, question) pairs.
 *   pixels      DEVICE [n_images, 3, image_size, image_size], dtype pixel_dtype (F32 or BF16): CLIPImageProcessor output
 *   image_index DEVICE int32 [batch] -> which image each pair uses, or NULL for identity (n_images == batch)
 *   input_ids   DEVICE int32 [batch, text_len], image slot = cfg.image_token_id, right-padded with pad_token_id
 *   text_lens   DEVICE int32 [batch] valid ids per row
 *   labels      DEVICE int32 [batch, label_len], -100 = ignored (padding)
 *   out_scores  DEVICE float [batch] : exp(-mean CE)  (v3.0 CLIPT5Model.forward)
 *   out_logprobs DEVICE float [batch, label_len] per-token log-probabilities, or NULL
 *   workspace   DEVICE, >= vqa_clipt5_workspace_bytes(...)
 *   stream      cudaStream_t
 */
int vqa_clipt5_score(vqa_handle* h, const void* pixels, int32_t pixel_dtype, int32_t n_images,
                     const int32_t* image_index, const int32_t* input_ids, const int32_t* text_lens,
                     const int32_t* labels, int32_t batch, int32_t text_len, int32_t label_len, float* out_scores,
                     float* out_logprobs, void* workspace, size_t workspace_bytes, void* stream);

/* ---- Qwen2.5-VL (replaces Qwen2VLModel.forward's per-sample generate(max_new_tokens=1, output_scores=True) +
 * softmax(scores / T)[answer_id], t2v_metrics/models/vqascore_models/qwen2vl_model.py:160-167,190-289) ---- */
int vqa_create_qwen25vl(const vqa_qwen25vl_config* cfg, int device, vqa_handle** out);

/* Rotary metadata (HOST arrays, copied): for frequency index i < n_half the rotation angle of a token is
 * position[axis[i]] * inv_freq[i]. Text: n_half = 64, axis = mrope sections (t,h,w) (modeling_qwen2_5_vl.py:650-662),
 * inv_freq = rope_theta^(-2i/128). Vision: n_half = head_dim/2 = 40, axis = [h]*20 + [w]*20, inv_freq = 10000^(-2i/40). */
int vqa_qwen25vl_set_rope(vqa_handle* h, const float* text_inv_freq, const int32_t* text_axis, int32_t text_half,
                          const float* vis_inv_freq, const int32_t* vis_axis, int32_t vis_half);

size_t vqa_qwen25vl_workspace_bytes(vqa_handle* h, int32_t batch, int32_t seq_len, int32_t n_patches);

/* Score `batch` prompts in one prefill. All index arrays are DEVICE int32 and are produced by the host's mirror of the
 * reference's index logic (rot_pos_emb :382-409, get_window_index :411-451, get_rope_index :1024-1133):
 *   pixel_patches  [n_patches, patch_dim] (F32 or BF16), all images concatenated, processor (merge-block) order
 *   vis_pos_hw     [2, n_patches]  (h, w) index of every patch, already in WINDOW order
 *   window_index   [n_patches / merge^2]  window order of the 2x2 patch groups;  reverse_index = argsort(window_index)
 *   cu_window      [n_windows + 1], cu_frames [n_frames + 1]  cumulative patch counts (window order)
 *   input_ids      [batch, seq_len] right-padded; seq_lens [batch]
 *   feat_index     [batch, seq_len] row of the merged vision features for image-token positions, -1 elsewhere
 *   position_ids   [3, batch*seq_len] (t, h, w) mRoPE positions
 *   answer_ids     [batch] the answer's first token id
 *   repetition_penalty  1.0 = off; otherwise HF's RepetitionPenaltyLogitsProcessor over each sample's prompt ids is applied to the
 *                  fp32 logits before the temperature (generation/utils.py:2762-2770; the checkpoint's generation_config.json
 *                  decides it in the reference, SURVEY F8)
 *   out_probs      [batch] softmax(processed last-position logits / temperature)[answer_id]; out_logprobs optional
 */
int vqa_qwen25vl_score(vqa_handle* h, const void* pixel_patches, int32_t pixel_dtype, int32_t n_patches,
                       const int32_t* vis_pos_hw, const int32_t* window_index, const int32_t* reverse_index,
                       const int32_t* cu_window, int32_t n_windows, int32_t max_window_len, const int32_t* cu_frames,
                       int32_t n_frames, int32_t max_frame_len, const int32_t* input_ids, const int32_t* seq_lens,
                       const int32_t* feat_index, const int32_t* position_ids, const int32_t* answer_ids, int32_t batch,
                       int32_t seq_len, float temperature, float repetition_penalty, float* out_probs, float* out_logprobs,
                       void* workspace, size_t workspace_bytes, void* stream);

/* Trace output (reference forward_with_trace, qwen2vl_model.py:303-493, top-5 at :439-447): the k <= 8 most probable next tokens of every
 * prompt of the LAST scoring call on this handle (vqa_qwen25vl_score: total_rows = batch * seq_len; vqa_qwen25vl_score_packed: its
 * total_rows) with the same n_patches and the same workspace -- its final hidden states and, when repetition_penalty != 1, its prompt-token
 * bitmap are still there -- under the same processing as the score: bf16 logits -> fp32 -> repetition penalty -> 1/T -> softmax over the
 * whole vocabulary. out_ids / out_probs: DEVICE [batch, k], most probable first; out_ids[b][0] is the token generate(max_new_tokens=1,
 * do_sample=False) would emit. This call materialises [batch, vocab] bf16 logits of that one position in the workspace -- a debugging
 * aid; the scoring path never stores logits. */
int vqa_qwen25vl_topk(vqa_handle* h, int32_t batch, int64_t total_rows, int32_t n_patches, int32_t k, float temperature,
                      float repetition_penalty, int32_t* out_ids, float* out_probs, void* workspace, size_t workspace_bytes, void* stream);

/* KV-prefix sharing (SURVEY 8(f)1; reference score.py:104-106 repeats one image across N texts and qwen2vl_model.py:190 re-runs the whole
 * prompt per text). The language-model tokens are given as PACKED rows: sequences stored back to back (cu_seqlens [n_seq + 1]); the
 * [chat prefix + vision tokens] of an image is ONE sequence (kv_prefix = -1), each prompt's remaining tokens are a sequence of their own whose
 * kv_prefix names the shared one: its rows attend to all prefix rows, then causally to themselves. Causality makes this exact (a prefix
 * row never sees a suffix), and the prefix rows go through every layer once per image instead of once per prompt.
 *   input_ids / feat_index [total_rows], position_ids [3, total_rows]: as in vqa_qwen25vl_score, in packed row order
 *   pair_row [n_prompts]: packed row of each prompt's last token; pair_seq [n_prompts]: the sequence holding it
 *   max_seq_len: longest sequence; max_prompt_len: longest prefix + suffix (repetition-penalty bitmap) */
size_t vqa_qwen25vl_packed_workspace_bytes(vqa_handle* h, int32_t n_prompts, int64_t total_rows, int32_t n_patches);
int vqa_qwen25vl_score_packed(vqa_handle* h, const void* pixel_patches, int32_t pixel_dtype, int32_t n_patches, const int32_t* vis_pos_hw,
                              const int32_t* window_index, const int32_t* reverse_index, const int32_t* cu_window, int32_t n_windows,
                              int32_t max_window_len, const int32_t* cu_frames, int32_t n_frames, int32_t max_frame_len,
                              const int32_t* input_ids, const int32_t* feat_index, const int32_t* position_ids, int32_t total_rows,
                              const int32_t* cu_seqlens, const int32_t* kv_prefix, int32_t n_seq, int32_t max_seq_len, const int32_t* pair_row,
                              const int32_t* pair_seq, const int32_t* answer_ids, int32_t n_prompts, int32_t max_prompt_len, float temperature,
                              float repetition_penalty, float* out_probs, float* out_logprobs, void* workspace, size_t workspace_bytes,
                              void* stream);

/* Number of kernels the last vqa_clipt5_score call launched (for bench.py's gpu_launches). */
int64_t vqa_last_launch_count(vqa_handle* h);

/* Optional device-side timing of the forward: with profiling on, every launch of vqa_clipt5_score is bracketed by CUDA
 * events on the caller's stream. After the caller synchronised the stream, vqa_profile_read returns, per category
 * {0 gemm, 1 attention, 2 norm, 3 other} (arrays of 4): device ms, algorithmic FLOPs (2MNK / 4*S*S*d), algorithmic bytes
 * (GEMM: A and W read once, C written once, residual read once) and scope counts of the LAST call. Used by bench.py for the
 * roofline object. */
int vqa_set_profile(vqa_handle* h, int32_t enable);
int vqa_profile_read(vqa_handle* h, float* ms, double* flops, double* bytes, int64_t* scopes);

/* Parity investigation aids: byte offsets, inside the caller-owned workspace of a call with the same sizes, of intermediate tensors
 * that the reference exposes too (encoder_last_hidden_state, decoder_hidden_states[-1], ...). Valid after the stream has passed
 * the scoring call. CLIP-FlanT5 (n >= 6): {encoder output, decoder output (both after the final T5LayerNorm), projector output,
 * encoder / decoder residual streams, last vision-tower hidden state (fp32)}. Qwen2.5-VL (n >= 4): {last-position hidden state after the
 * final norm, merged vision features, residual stream, last-position residual}. */
int vqa_clipt5_debug_layout(vqa_handle* h, int32_t batch, int32_t n_images, int32_t text_len, int32_t label_len, size_t* offsets,
                            int32_t n);
int vqa_qwen25vl_debug_layout(vqa_handle* h, int32_t batch, int32_t seq_len, int32_t n_patches, size_t* offsets, int32_t n);

/* Process-wide override of the GEMM tile order (tuning): group_rows > 0 = A rows per M group, chunk_rows > 0 = W rows per
 * L2-resident chunk, chunk_rows < 0 = one chunk; 0 = automatic. */
int vqa_set_gemm_schedule(int32_t group_rows, int32_t chunk_rows);

/* Tuning aid: number of clusters of `cluster_size` CTAs of the 256-wide GEMM kernel (one CTA per SM) the current device can hold at once
 * (cudaOccupancyMaxActiveClusters); negative vqa_status on error. */
int vqa_debug_max_active_clusters(int32_t cluster_size);

const char* vqa_last_error(vqa_handle* h);
void vqa_destroy(vqa_handle* h);

/* ---- image pre-processing on the device (SURVEY 8(f)2) ----
 * Replaces expand2square (t2v_metrics/models/vqascore_models/mm_utils.py:128-139) + the CLIP image processor of the v3.0 wrapper
 * (PIL BICUBIC resize of the shortest edge to out_size, centre crop, /255, (x - mean) / std): bit-identical to Pillow's integer
 * resampling (Resample.c) and to the fp32 normalisation of oracle/clipt5_oracle.py:clip_preprocess.
 *   src        DEVICE, the decoded images as packed HWC uint8 RGB, image i at byte offsets[i], heights[i] x widths[i] x 3
 *   offsets / heights / widths   HOST arrays [n_images]
 *   pad_to_square  1 = image_aspect_ratio 'pad' (centre on a max(h, w) square of `background`), 0 = plain resize + centre crop
 *   out        DEVICE [n_images, 3, out_size, out_size], out_dtype VQA_DTYPE_F32 or VQA_DTYPE_BF16
 *   workspace  DEVICE, >= vqa_clip_preprocess_workspace_bytes(...) (0 = bad arguments, see vqa_last_error(NULL))
 *   host_staging  optional HOST buffer of the same size, ideally pinned: the geometry + tap tables are written there and copied
 *              with ONE asynchronous cudaMemcpyAsync; the caller must leave it untouched until `stream` has passed this call.
 *              NULL: the tables are copied from the library's pageable memory (the runtime stages that copy synchronously). */
size_t vqa_clip_preprocess_workspace_bytes(const int32_t* heights, const int32_t* widths, int32_t n_images, int32_t out_size,
                                           int32_t pad_to_square);
int vqa_clip_preprocess(const void* src, const int64_t* offsets, const int32_t* heights, const int32_t* widths, int32_t n_images,
                        int32_t out_size, int32_t pad_to_square, const uint8_t* background, const float* mean, const float* stdv,
                        void* out, int32_t out_dtype, void* workspace, size_t workspace_bytes, void* host_staging, void* stream);

/* Qwen2.5-VL still-image pre-processing on the device: smart_resize (qwen_vl_utils / image_processing_qwen2_vl.py:62-87) + PIL-exact
 * bicubic resize + /255 + normalise + frame duplication + 14x14 patch rows in 2x2 merge-block order
 * (image_processing_qwen2_vl.py:191-220). vqa_qwen_preprocess_plan is host-only: grid_hw [n][2] = (h, w) patch grid of each image,
 * total_patches = rows of `out`, workspace_bytes = device scratch needed. out: DEVICE [total_patches, 3*temporal_patch*patch^2]. */
int vqa_qwen_preprocess_plan(const int32_t* heights, const int32_t* widths, int32_t n_images, int32_t patch, int32_t merge,
                             int64_t min_pixels, int64_t max_pixels, int32_t* grid_hw, int64_t* total_patches, size_t* workspace_bytes);
int vqa_qwen_preprocess(const void* src, const int64_t* offsets, const int32_t* heights, const int32_t* widths, int32_t n_images,
                        int32_t patch, int32_t temporal_patch, int32_t merge, int64_t min_pixels, int64_t max_pixels, const float* mean,
                        const float* stdv, void* out, int32_t out_dtype, void* workspace, size_t workspace_bytes, void* host_staging,
                        void* stream);

/* Host-only helper (no GPU needed): the 22-bit fixed-point bicubic tap table of one resize axis (in_size -> out_size, output
 * pixels [first, first + count)), exactly as vqa_clip_preprocess builds it after Pillow's precompute_coeffs /
 * normalize_coeffs_8bpc. bounds [count][2] = (first source index, taps used); kk [count][ksize]; returns ksize (0 = bad
 * arguments). Either output pointer may be NULL. */
int32_t vqa_resample_table(int32_t in_size, int32_t out_size, int32_t first, int32_t count, int32_t* bounds, int32_t* kk);

/* Qwen2.5-VL video pre-processing on the device: for each video, smart_resize with its own pixel bounds, resize of every frame, /255,
 * normalise, consecutive frames paired into temporal patches (a count that is not a multiple of temporal_patch repeats the last frame)
 * and 14x14 patch rows in 2x2 merge-block order -- what Qwen2VLVideoProcessor(do_resize=False) does to qwen_vl_utils' frames.
 *   src        DEVICE, video v = frames[v] packed HWC uint8 RGB frames of heights[v] x widths[v], back to back from byte offsets[v]
 *   policy[v]  VQA_RESAMPLE_PIL (frames handed over as images: Pillow's bicubic, bit-exact) or VQA_RESAMPLE_TORCHVISION (decoded video
 *              files: torchvision's antialiased bicubic on uint8 tensors, fp32 taps and intermediate, clamp + round-half-even)
 *   min_pixels / max_pixels  HOST [n_videos], the smart_resize bounds of each video
 *   grid_thw   HOST [n_videos][3] (plan only) = (ceil(frames / temporal_patch), h / patch, w / patch)
 *   out        DEVICE [total_patches, 3*temporal_patch*patch^2], video v's rows after those of videos 0..v-1
 * vqa_qwen_video_preprocess_plan is host-only. At most 65535 frames per call. workspace / host_staging as for vqa_clip_preprocess. */
#define VQA_RESAMPLE_PIL 0
#define VQA_RESAMPLE_TORCHVISION 1
int vqa_qwen_video_preprocess_plan(const int32_t* heights, const int32_t* widths, const int32_t* frames, const int32_t* policy,
                                   int32_t n_videos, int32_t patch, int32_t temporal_patch, int32_t merge, const int64_t* min_pixels,
                                   const int64_t* max_pixels, int32_t* grid_thw, int64_t* total_patches, size_t* workspace_bytes);
int vqa_qwen_video_preprocess(const void* src, const int64_t* offsets, const int32_t* heights, const int32_t* widths, const int32_t* frames,
                              const int32_t* policy, int32_t n_videos, int32_t patch, int32_t temporal_patch, int32_t merge,
                              const int64_t* min_pixels, const int64_t* max_pixels, const float* mean, const float* stdv, void* out,
                              int32_t out_dtype, void* workspace, size_t workspace_bytes, void* host_staging, void* stream);

/* Host-only helper: the fp32 tap table of one axis of the VQA_RESAMPLE_TORCHVISION resize, exactly as vqa_qwen_video_preprocess builds
 * it. bounds [count][2] = (first source index, taps used); taps [count][ksize]; *fma = 1 when the pass over this axis accumulates
 * acc = fma(px, tap, acc), 0 when it computes acc + round(px * tap); returns ksize (0 = bad arguments). Pointers may be NULL. */
int32_t vqa_resample_table_tv(int32_t in_size, int32_t out_size, int32_t first, int32_t count, int32_t* bounds, float* taps, int32_t* fma);

/* ---- kernel-level entry points (used by tests/ and bench.py to exercise single kernels through the same ABI) ---- */

/* C[M,N] = epilogue(A[M,K] . W[N,K]^T); all DEVICE bf16 row-major. epilogue: 0 store, 1 quick_gelu, 2 gelu(erf),
 * 3 gated gelu_new (W = [gate; up] with `gate_up_offset` rows between them, C is [M, N/2]), 5 relu.
 * bias [N] / residual [M, ldr] may be NULL. variant: 0 auto, else (BLOCK_N * 10 + cta_group), e.g. 2562, 2561, 641. */
int vqa_op_gemm_bf16(const void* A, int32_t lda, const void* W, int32_t ldw, int32_t w_rows, void* C, int32_t ldc,
                     int32_t M, int32_t N, int32_t K, const void* bias, const void* residual, int32_t ldr,
                     int32_t epilogue, int32_t gate_up_offset, int32_t variant, void* stream);

/* vqa_op_gemm_bf16 with the fused-RMSNorm hooks the encoder uses when emulate_bf16_rounding & 4 (T5LayerNorm, modeling_t5.py:55-68, folded
 * into the GEMMs around it). ssq_in DEVICE float [M, stride] or NULL: partial sums of squares of the rows of A; the epilogue multiplies
 * accumulator row m by rsqrt(sum_i ssq_in[m][i] / norm_dim + eps) before the Linear's bf16 rounding (W must carry the norm's gain:
 * W . diag(gamma)). ssq_out DEVICE float [M, stride] or NULL (epilogue 0 only): receives the partial sums of squares of the bf16 rows this
 * launch stores, slots [0, *parts_out); the caller zeroes the buffer first. stride % 4 == 0. No bias. */
int vqa_op_gemm_bf16_normfuse(const void* A, int32_t lda, const void* W, int32_t ldw, int32_t w_rows, void* C, int32_t ldc, int32_t M, int32_t N,
                              int32_t K, const void* residual, int32_t ldr, int32_t epilogue, int32_t gate_up_offset, const float* ssq_in,
                              float* ssq_out, int32_t stride, int32_t norm_dim, float eps, int32_t* parts_out, void* stream);

/* Fused lm_head + log-softmax gather: logprob[m] = (h[m].W[label[m]]) - logsumexp_n(h[m].W[n]); logits never stored.
 * scratch: DEVICE float, >= 4*M*ceil(N/128) + M floats. */
int vqa_op_lmhead_logprob(const void* H, int32_t ldh, const void* W, int32_t ldw, int32_t M, int32_t N, int32_t K,
                          const int32_t* labels, float* logprob, float* scratch, void* stream);

/* Bidirectional attention, head_dim 64, packed qkv [B*S, 3*H*64] -> out [B*S, H*64].
 * bias_table: DEVICE float [H, 2S-1] (index key - query + S - 1) or NULL; seq_lens DEVICE int32 [B] or NULL.
 * bias_const_from > 0: the caller guarantees bias_table[h][.] is constant for |key - query| >= bias_const_from on each side (T5's
 * relative_attention_max_distance, modeling_t5.py:189-234), which lets far key tiles fold the bias into one FFMA; 0: no assumption.
 * round_scores != 0: reproduce the bf16 tensors the reference's eager attention forms before its fp32 softmax (q.k^T as bf16, then the
 * bf16 `scores += position_bias`, modeling_t5.py:308-331); 0: scores and bias stay fp32. */
int vqa_op_attention_d64(const void* qkv, void* out, int32_t B, int32_t S, int32_t H, const int32_t* seq_lens,
                         const float* bias_table, float scale, int32_t bias_const_from, int32_t round_scores, void* stream);

/* T5LayerNorm / nn.LayerNorm on [rows, D] bf16. beta == NULL selects T5 RMS norm. */
int vqa_op_norm(const void* x, const void* gamma, const void* beta, void* y, int32_t rows, int32_t D, float eps,
                void* stream);

/* head_dim-128 attention on a packed buffer [rows, ld]: q heads at q_col0 + h*128, k/v heads at k_col0/v_col0 + (h/kv_group)*128.
 * cu_seqlens [n_seq+1] (variable-length sequences) or NULL with fixed stride S and optional seq_lens [n_seq]. */
int vqa_op_attention_d128(const void* qkv, int32_t ld, int64_t rows, int32_t q_col0, int32_t k_col0, int32_t v_col0, void* out,
                          int32_t ldo, int32_t n_seq, int32_t max_len, int32_t S, int32_t q_heads, int32_t kv_group,
                          const int32_t* cu_seqlens, const int32_t* seq_lens, float scale, int32_t causal, void* stream);

/* vqa_op_attention_d128 in variable-length mode with its extras: kv_prefix [n_seq] (or NULL): sequence b also attends to all rows of sequence
 * kv_prefix[b] >= 0, placed in front of its own keys; pair_sequences: two consecutive sequences (each <= 64 rows) share one 128-row tile under a
 * block-diagonal mask (non-causal only); output head h is written at column h * o_head_stride, first d_out (multiple of 8) head dims only. */
int vqa_op_attention_d128_ex(const void* qkv, int32_t ld, int64_t rows, int32_t q_col0, int32_t k_col0, int32_t v_col0, void* out, int32_t ldo,
                             int32_t n_seq, int32_t max_len, int32_t q_heads, int32_t kv_group, const int32_t* cu_seqlens, const int32_t* kv_prefix,
                             float scale, int32_t causal, int32_t pair_sequences, int32_t o_head_stride, int32_t d_out, void* stream);

/* Skinny GEMM (M <= 128): K cut into `splits` slices that run as one launch, fp32 partial tiles in `workspace` (splits * M * N floats), then one
 * reduction kernel: C = [residual +] bf16(A W^T + bias). splits == 0: the library picks (returned in *splits_out, may be 1). */
int vqa_op_gemm_bf16_splitk(const void* A, int32_t lda, const void* W, int32_t ldw, int32_t w_rows, void* C, int32_t ldc, int32_t M, int32_t N,
                            int32_t K, const void* bias, const void* residual, int32_t ldr, int32_t splits, void* workspace,
                            size_t workspace_bytes, int32_t* splits_out, void* stream);

/* vqa_op_gemm_bf16 with the plain store epilogue, output columns written in groups: logical column c -> (c / group_in) * group_out + c % group_in. */
int vqa_op_gemm_bf16_grouped(const void* A, int32_t lda, const void* W, int32_t ldw, int32_t w_rows, void* C, int32_t ldc, int32_t M, int32_t N,
                             int32_t K, const void* bias, int32_t group_in, int32_t group_out, int32_t variant, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VQA_B200_H */
