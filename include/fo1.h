/*
 * fo1.h -- C ABI of libfo1.so, the B200 (sm_100a) engine for the VLM-FO1 inference hot path.
 *
 * Plain C types only: device pointers, sizes, a cudaStream_t passed as void*.  Every entry point
 * returns 0 on success or a negative fo1_status; fo1_last_error() returns a message for the calling
 * thread.  Nothing here allocates on the hot path: callers own inputs/outputs and hand the library a
 * workspace; the model-level handle owns its weights and one arena sized when the model is created.
 * All entry points enqueue on the given stream and return (asynchronous) unless stated otherwise.
 *
 * Each declaration cites the reference interface (om-ai-lab/VLM-FO1 @ e6bef8d) it replaces.
 * The reference has no FFI of its own (pure PyTorch); INTEGRATION.md shows the ctypes binding a
 * maintainer adds under vlm_fo1/model/.
 */
#ifndef FO1_H_
#define FO1_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FO1_ABI_VERSION 2

typedef enum {
  FO1_OK = 0,
  FO1_ERR_INVALID_ARG = -1,
  FO1_ERR_CUDA = -2,
  FO1_ERR_UNSUPPORTED = -3,
  FO1_ERR_WORKSPACE = -4,
  FO1_ERR_NOT_FOUND = -5,
  FO1_ERR_STATE = -6
} fo1_status;

typedef enum { FO1_BF16 = 0, FO1_F32 = 1, FO1_I32 = 2, FO1_I64 = 3, FO1_U8 = 4, FO1_F16 = 5 } fo1_dtype;

int fo1_abi_version(void);
/* Message describing the last failure on this thread ("" if none). */
const char* fo1_last_error(void);
/* Number of kernels this library has launched since load / since the last reset (all threads). */
uint64_t fo1_launch_count(void);
void fo1_launch_count_reset(void);
/* Optional per-launch profiler: CUDA events recorded around the library's GEMM / attention / HFRE launches on
 * the launching stream.  enable(1) clears and starts recording, enable(0) stops; collect() synchronises the
 * device and writes a JSON object {tag: {launches, ms, flops, bytes, max_ms}} (algorithmic flops / bytes). */
void fo1_profile_enable(int on);
int fo1_profile_collect(char* buf, size_t cap);

/* ------------------------------------------------------------------------------------------------
 * HFRE -- Hybrid Fine-grained Region Encoder.
 * Replaces HFREModule.__call__ (vlm_fo1/model/multimodal_visual_prompt_encoder/
 * hybrid_finegrained_region_encoder.py:275-468) as called from encode_regions
 * (vlm_fo1/model/language_model/omchat_qwen2_5_vl.py:101-106): ROIAlign(7x7, adaptive sampling,
 * aligned=False) + mean over bins on every pyramid level of both towers, channel concat, and the
 * sinusoidal box embedding -- WITHOUT materialising the up-sampled/concatenated map (:338-350).
 * ---------------------------------------------------------------------------------------------- */

/* One feature level: bf16, channels-last [H][W][C] in device memory, C % 8 == 0, 16-byte aligned. */
typedef struct {
  const void* data;
  int32_t H, W, C;
  int32_t up_H, up_W;     /* grid the reference bilinearly up-samples this level to before ROIAlign
                             (F.interpolate align_corners=False, :341-346); == H, W when it does not */
  float spatial_scale;    /* ROIAlign spatial_scale on that (up-sampled) grid: 0.25 aux (:357),
                             1/14 taps (:267), 1/3.5 .. 1/28 FPN (:245-253) */
  int32_t box_set;        /* 0: aux boxes, 1: primary-tower ("vt") boxes */
  int32_t out_offset;     /* first output channel written by this level */
} fo1_hfre_level;

#define FO1_HFRE_MAX_LEVELS 8

/* One image's work. */
typedef struct {
  fo1_hfre_level levels[FO1_HFRE_MAX_LEVELS];
  int32_t n_levels;
  int32_t n_boxes;
  const float* boxes_aux;  /* [n_boxes][4] xyxy, aux-tensor pixels (device) */
  const float* boxes_vt;   /* [n_boxes][4] xyxy, primary-tower pixels (device); may equal boxes_aux */
  float* out;              /* [n_boxes][out_dim] fp32 (device) */
  void* out_bf16;          /* optional [n_boxes][out_dim] bf16 copy for the projector GEMM, or NULL */
  float pos_img_w, pos_img_h; /* normaliser of the box embedding (:447-448): grid * 14 */
  int32_t pos_box_set;     /* which boxes feed the embedding (:442-452): 1 = vt */
} fo1_hfre_image;

typedef struct {
  int32_t out_dim;          /* D = mm_region_hidden_size (5888 variant B, 8960 variant A) */
  int32_t roi_size;         /* 7 (omchat_arch.py:18) */
  int32_t apply_pos_embed;  /* mm_apply_position_embedding, bbox_based */
  int32_t algo;             /* 0 = auto (gather below 8 boxes per image on average, else sweep), 1 = per-box gather,
                               3 = map sweep, row sums on mma.sync; other values are rejected */
} fo1_hfre_params;

/* Bytes of device workspace fo1_hfre_forward needs for these images (host-side arithmetic only). */
size_t fo1_hfre_workspace_bytes(const fo1_hfre_image* images, int32_t n_images, const fo1_hfre_params* p);
/* Enqueue HFRE for n_images images.  `images` is a HOST array (device pointers inside). */
int fo1_hfre_forward(const fo1_hfre_image* images, int32_t n_images, const fo1_hfre_params* p,
                     void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Dense contraction: D[M,N] = epilogue(A[M,K] . W[N,K]^T) -- bf16 operands, fp32 accumulate in TMEM
 * (tcgen05.mma, operands staged by TMA).  Replaces every nn.Linear / 1x1 conv / patch-embed on the
 * path (modeling_qwen2_5_vl.py:88-111, 176-177, 151-155, 731-734, 633-635; modeling_davit.py:62-66,
 * 157-158, 235-236; simple_fpn.py:143-175; multimodal_projector/builder.py:100-106).
 * ---------------------------------------------------------------------------------------------- */
typedef enum {
  FO1_EPI_NONE = 0,
  FO1_EPI_GELU = 1,          /* exact erf GELU (nn.GELU default) */
  FO1_EPI_SILU = 2
} fo1_epilogue_act;

typedef struct {
  int32_t M, N, K;
  const void* A; int64_t lda;      /* bf16 [M][K], row stride lda elements (lda*2 % 16 == 0) */
  const void* W; int64_t ldw;      /* bf16 [N][K] (nn.Linear weight layout) */
  void* D; int64_t ldd;            /* output [M][N], bf16 or fp32 */
  int32_t d_dtype;                 /* FO1_BF16 or FO1_F32 */
  const void* bias;                /* optional [N], bias_dtype */
  int32_t bias_dtype;              /* FO1_BF16 or FO1_F32 */
  int32_t act;                     /* fo1_epilogue_act, applied after bias */
  const void* residual; int64_t ldr; /* optional bf16 [M][N] added after act */
  int32_t gated;                   /* 1: W rows interleave [32 gate | 32 up] blocks -> D[M][N/2] =
                                      act(gate)*up  (Qwen2MLP, modeling_qwen2_5_vl.py:84-85,638-640) */
  int32_t tile_n;                  /* 0 = library heuristic; 32 / 64 / 128 / 256 pins the tile width (tuning, tests) */
  int32_t split_k;                 /* with tile_n != 0: number of K splits reduced in-kernel (>= 1); 0 = 1 */
} fo1_gemm_desc;

int fo1_gemm_bf16(const fo1_gemm_desc* d, void* stream);



/* ------------------------------------------------------------------------------------------------
 * Variable-length softmax attention over packed token rows (replaces flash_attn_varlen_func at
 * modeling_qwen2_5_vl.py:205 and _flash_attention_forward at :895, and DaViT's window attention
 * modeling_davit.py:261-268) on tcgen05 / TMEM with TMA-fed K/V rings.  q/k/v/o: bf16 rows with the given
 * pitches (elements, multiples of 8; 16-byte aligned bases); head h of a row starts at h*head_dim.
 * cu_seqlens: device int32 [n_seqs+1]; total_rows = cu_seqlens[n_seqs] (the host passes it: it sizes the grid).
 * head_dim in {32, 64, 80, 128}.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  const void* q; const void* k; const void* v; void* o;
  int64_t ldq, ldk, ldv, ldo;
  const int32_t* cu_seqlens;
  int32_t n_seqs, max_seqlen;
  int32_t q_heads, kv_heads, head_dim;
  float scale;
  int32_t causal;
  int32_t total_rows;
} fo1_attn_desc;
int fo1_attention_varlen(const fo1_attn_desc* d, void* stream);

/* DaViT channel-group attention (ChannelAttention.forward, modeling_davit.py:151-172) for n_images maps of n_tokens tokens:
 * qkv bf16 [n_images][n_tokens][3*channels] (q | k | v as the fused Linear emits them), groups * 32 == channels;
 * out bf16 [n_images][n_tokens][channels] = (softmax_c2((q N^-0.5)^T k) v^T)^T per group of 32 channels.  Both contractions
 * run on tcgen05 (the Gram over the token axis with MN-major operands straight from the TMA tiles); partial Grams of the
 * token chunks live in `workspace` and are summed in a fixed order (bit-reproducible, no atomics). */
size_t fo1_channel_attention_workspace_bytes(int32_t n_images, int32_t n_tokens, int32_t channels);
int fo1_channel_attention(const void* qkv, int32_t n_images, int32_t n_tokens, int32_t channels, int32_t groups, void* out,
                          void* workspace, size_t workspace_bytes, void* stream);

/* DaViT conditional position encoding (PreNorm(None, DepthWiseConv2d), modeling_davit.py:29-48, 72-99): y = x + dwconv3x3(x) + bias over
 * NHWC bf16 maps [n_images][height][width][channels]; w9 bf16 [9][channels] (tap-major repack of [channels][1][3][3]), bias bf16
 * [channels].  channels % 8 == 0; x and y must not alias.  Exposed for the parity test of the kernel; fo1_davit_forward runs the same code. */
int fo1_dwconv3x3_residual(const void* x, const void* w9, const void* bias, void* y, int32_t n_images, int32_t height, int32_t width,
                           int32_t channels, void* stream);

/* Single-query GQA attention of one decode step over the K/V cache (the per-step attention of the HF generate loop,
 * modeling_qwen2_5_vl.py:731-780 with past_key_values; mm_utils.py:640-654 drives it).  The step's own K/V must already
 * sit in the cache at index cache_len[b].  head_dim 128, q_heads / kv_heads <= 8.  Exposed so the parity tests can
 * check the kernel directly; fo1_llm_generate runs the same code. */
typedef struct {
  const void* q; int64_t ldq;        /* bf16 [n_seqs][q_heads*128] (rotated), row stride ldq elements */
  const void* k_cache;               /* bf16 [n_seqs][cap][kv_heads*128] */
  const void* v_cache;
  const int32_t* cache_len;          /* device [n_seqs]: keys 0 .. cache_len[b] (inclusive) are attended */
  int32_t n_seqs, cap, q_heads, kv_heads, head_dim;
  float scale;
  void* out; int64_t ldo;            /* bf16 [n_seqs][q_heads*128] */
  void* workspace;                   /* fp32 partials, fo1_decode_attention_workspace_bytes(n_seqs, q_heads) */
  size_t workspace_bytes;
} fo1_decode_attn_desc;
size_t fo1_decode_attention_workspace_bytes(int32_t n_seqs, int32_t q_heads);
int fo1_decode_attention(const fo1_decode_attn_desc* d, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Model-level engine.  One handle per GPU / rank; calls on one handle are not re-entrant.
 * Weights are BORROWED device pointers (the caller keeps them alive): the Python loader prepares
 * them once (layout changes listed in DESIGN.md section "weights") from the checkpoint tensors that
 * vlm_fo1/model/builder.py:90-131 loads.
 * ---------------------------------------------------------------------------------------------- */
typedef struct fo1_model fo1_model;

typedef struct {
  /* primary tower: Qwen2.5-VL ViT (configuration_qwen2_5_vl.py:30-66) */
  int32_t vit_depth, vit_hidden, vit_heads, vit_inter, vit_inter_pad, vit_out_hidden;
  int32_t vit_patch, vit_merge, vit_temporal, vit_in_ch, vit_window;
  int32_t vit_n_fullatt; int32_t vit_fullatt[8];   /* fullatt_block_indexes, also the tap layers */
  /* aux tower: DaViT (davit/configs.py:70-136) */
  int32_t davit_dims[4], davit_depths[4], davit_heads[4], davit_groups[4], davit_window;
  /* SimpleFPN on the last tap (simple_fpn.py:100-216) */
  int32_t fpn_out;                 /* 512; 0 = FPN absent (variant A) */
  /* region projector / image projector (multimodal_projector/builder.py:39-115) */
  int32_t region_dim;              /* mm_region_hidden_size */
  int32_t proj_aux_layers;         /* mlpNx_gelu depth; 1 = linear */
  int32_t proj_img_layers;         /* 0 = identity */
  /* LLM: Qwen2.5 decoder (configuration_qwen2_5_vl.py:193-253) */
  int32_t llm_layers, llm_hidden, llm_heads, llm_kv_heads, llm_head_dim, llm_inter, llm_vocab;
  int32_t mrope_section[3];
  float rope_theta, rms_eps;
  int32_t tie_embeddings;
} fo1_model_config;

int fo1_model_create(const fo1_model_config* cfg, fo1_model** out);
/* Entries of the handle's cache of device-side integer tables (window indices, cu_seqlens ...).  The cache is trimmed
 * only at the entry of a forward, never while one is using its tables; exposed for the test of that rule. */
int fo1_int_cache_entries(fo1_model* m);
/* Which decode path the handle's last fo1_generate took: 1 = the persistent kernel (decode_mega.cu, the whole greedy loop as one
 * cooperative launch), 0 = the per-kernel CUDA graph, -1 = no generate yet.  Reported by bench.py next to the decode roofline. */
int fo1_last_decode_path(fo1_model* m);
void fo1_model_destroy(fo1_model* m);
/* Register one prepared weight (device pointer, borrowed).  Names: see DESIGN.md / vlm-fo1_b200/weights.py. */
int fo1_model_set_weight(fo1_model* m, const char* name, const void* dev_ptr, int32_t dtype, int32_t ndim,
                         const int64_t* shape);
/* Check that every weight the configured towers need is present with the right shape. */
int fo1_model_finalize(fo1_model* m);

/* Primary tower forward over a batch of images (replaces Qwen2_5_VlVisionTower.forward ->
 * custom_forward + extract_multi_level_features, qwen2_5_vl_encoder.py:86-158, 37-80, 228-257).
 * pixel_values[b]: device fp32 [gh*gw][in_ch*temporal*patch*patch] as Qwen2VLImageProcessor emits it;
 * grid_hw: host int32 [B][2].  Outputs (device, caller-owned, bf16):
 *   img_feats : [sum_b gh*gw/merge^2][out_hidden]   merged tokens, images back to back, raster order
 *   taps[t]   : [sum_b gh*gw][hidden] for each full-attention layer t -- image b's slice is its
 *               channels-last map [gh][gw][hidden] (un-windowed; what HFRE / SimpleFPN read). */
int fo1_vit_forward(fo1_model* m, const float* const* pixel_values, const int32_t* grid_hw, int32_t n_images,
                    void* img_feats, void* const* taps, void* stream);
/* Integer bookkeeping of the tower, exposed for bit-exact parity tests against
 * get_window_index / rot_pos_emb (modeling_qwen2_5_vl.py:436-504).  Host outputs, sized by the caller:
 * window_index [gh*gw/merge^2], cu_window_seqlens [<= n_windows+1] (count returned), pos_hw [gh*gw][2]
 * in window order. */
int fo1_vit_window_index(const fo1_model_config* cfg, int32_t gh, int32_t gw, int32_t* window_index,
                         int32_t* cu_window_seqlens, int32_t* n_cu, int32_t* pos_hw);

/* Aux tower forward (replaces DavitVisionTower.forward -> DaViT.forward_features,
 * davit_aux_encoder.py:54-73, modeling_davit.py:478-506) for n_images images of the SAME size H x W.
 * images[b]: device fp32 [3][H][W] (CLIP-normalised).  stage_out[s]: bf16 [B][H_s][W_s][C_s], s = 0..3. */
int fo1_davit_forward(fo1_model* m, const float* const* images, int32_t H, int32_t W, int32_t n_images,
                      void* const* stage_out, void* stream);

/* SimpleFPN (replaces SimpleFP.forward, simple_fpn.py:197-216) on n_images last-tap maps of the SAME grid.
 * tap: bf16 [B][gh][gw][hidden] ; level_out[l]: bf16 [B][gh*f][gw*f][fpn_out], f = 4, 2, 1, 1/2. */
int fo1_fpn_forward(fo1_model* m, const void* tap, int32_t gh, int32_t gw, int32_t n_images, void* const* level_out,
                    void* stream);

/* Region projector mm_projector_aux (omchat_qwen2_5_vl.py:107): bf16 [n][region_dim] -> bf16 [n][llm_hidden]. */
int fo1_region_project(fo1_model* m, const void* feats, int32_t n, void* out, void* stream);
/* Image projector mm_projector (encode_images, omchat_qwen2_5_vl.py:58-66; multimodal_projector/builder.py:39-76) for the
 * `linear` / `mlpNx_gelu` types: bf16 [n][vit_out_hidden] -> bf16 [n][llm_hidden].  The released checkpoint uses
 * `identity` (proj_img_layers = 0): the call is then an error and the caller passes the tower output through. */
int fo1_image_project(fo1_model* m, const void* feats, int32_t n, void* out, void* stream);


/* ------------------------------------------------------------------------------------------------
 * Device-side image pre-processing (SURVEY.md section 8f rank 1): uint8 RGB [H][W][3] in device memory -> the tensors the two
 * host processors produce, bit-identical (integer resize; float32 normalisation in the processors' operation order).
 * ---------------------------------------------------------------------------------------------- */
/* PIL's bicubic resize of an 8-bit image (what Qwen2VLImageProcessor / CLIPImageProcessor call: mm_utils.py:615, :596 ->
 * PIL Image.resize(BICUBIC)): horizontal pass then vertical pass with the uint8 intermediate.  bounds: host-computed, DEVICE
 * int32 [out][2] = (first input index, count); coef: DEVICE int32 [out][ksize], 22 fractional bits (PIL's normalised
 * coefficients; vlm-fo1_b200/preprocess.py computes them).  tmp: [H][out_w][3] bytes when both axes change.  A pass whose
 * size does not change is skipped (its tables may be NULL). */
int fo1_resize_bicubic_u8(const void* img, int32_t H, int32_t W, int32_t out_h, int32_t out_w, const int32_t* h_bounds,
                          const int32_t* h_coef, int32_t h_ksize, const int32_t* v_bounds, const int32_t* v_coef, int32_t v_ksize,
                          void* tmp, void* out, void* stream);
/* Qwen2VLImageProcessor's rescale + normalise + patchify (2x2-merge order, frame repeated over the temporal patch) of an image
 * whose sides are already multiples of patch*merge: -> fp32 [H/patch * W/patch][3*temporal*patch*patch].  mean / std: HOST [3]. */
int fo1_preprocess_primary_u8(const void* img, int32_t H, int32_t W, int32_t patch, int32_t merge, int32_t temporal, const float* mean,
                              const float* std, float* pixel_values, void* stream);
/* CLIPImageProcessor's rescale + normalise + channels-first (davit/image_processing_clip.py:344-358): -> fp32 [3][H][W]. */
int fo1_preprocess_aux_u8(const void* img, int32_t H, int32_t W, const float* mean, const float* std, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------
 * LLM half: embedding splice, M-RoPE bookkeeping, prefill and greedy decode.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t image_token_id;        /* config.image_token_id (151655) */
  int32_t video_token_id;        /* config.video_token_id (151656) */
  int32_t vision_start_token_id; /* config.vision_start_token_id (151652) */
  int32_t merge;                 /* vision_config.spatial_merge_size */
  int32_t image_placeholder;     /* IMAGE_TOKEN_INDEX  (-200, vlm_fo1/constants.py) */
  int32_t region_placeholder;    /* DEFAULT_REGION_INDEX (-300) */
} fo1_splice_cfg;

/* Integer work of prepare_inputs_labels_for_qwen2_5_vl_multimodal (omchat_qwen2_5_vl.py:291-373, 434-458)
 * + get_rope_index (modeling_qwen2_5_vl.py:1546-1721) for ONE sample (host only, bit-exact):
 * every image placeholder expands to that image's gh*gw/merge^2 feature rows (ids <- image_token_id), every
 * region placeholder keeps one slot (id stays region_placeholder); then the 3-axis position ids.
 * Outputs (host, capacity elements each; position_ids 3*capacity laid out [3][capacity]):
 *   new_ids, src_kind (0 text / 1 image row / 2 region row), src_index (token id / row in the image- /
 *   region-feature matrix of this sample), position_ids, *rope_delta, *out_len.
 * Returns FO1_ERR_WORKSPACE if capacity is too small (out_len then holds the needed length). */
int fo1_splice_plan(const int64_t* input_ids, int32_t n_ids, const int32_t* image_grid_hw, int32_t n_images,
                    int32_t n_regions, const fo1_splice_cfg* cfg, int64_t* new_ids, int32_t* src_kind,
                    int32_t* src_index, int32_t* position_ids, int32_t* rope_delta, int32_t* out_len,
                    int32_t capacity);

/* The same integer work for a whole BATCH of prompts in one launch, on the device (SURVEY.md section 8f rank 2): all pointers
 * are DEVICE int32 arrays.  ids / id_off: the prompts' ids concatenated + offsets [n_samples+1]; grids / img_off: (gh, gw) of
 * every image + offsets [n_samples+1]; n_regions [n_samples]; out_off [n_samples+1]: row offsets of the spliced sequences
 * (L_b = n_ids_b - n_img_b + sum gh*gw/merge^2, host arithmetic); img_row_off / reg_row_off [n_samples]: first row of the
 * sample in the batch's image- / region-feature matrices (added to src_index).  Outputs over total_rows = out_off[n_samples]:
 * new_ids, src_kind, src_index [total_rows], position_ids [3][total_rows], rope_delta / status [n_samples] (status 0 or a
 * fo1_status per sample).  Bit-identical to fo1_splice_plan sample by sample. */
int fo1_splice_plan_batch(const int32_t* ids, const int32_t* id_off, const int32_t* grids, const int32_t* img_off,
                          const int32_t* n_regions, const int32_t* out_off, const int32_t* img_row_off,
                          const int32_t* reg_row_off, int32_t n_samples, int64_t total_rows, const fo1_splice_cfg* cfg,
                          int32_t* new_ids, int32_t* src_kind, int32_t* src_index, int32_t* position_ids, int32_t* rope_delta,
                          int32_t* status, void* stream);

/* extract_predictions_to_indexes (vlm_fo1/mm_utils.py:346-369) over the decoded TOKEN IDS of a batch, on the device, for
 * tokenizers that hold "<ground>", "</ground>", "<objects>", "</objects>" and every "<regionN>" as single tokens: tokens DEVICE
 * int32 [n_samples][ld], lens [n_samples]; region_ids DEVICE [n_region_ids] (id of <region0>, <region1>, ...); newline_bitmap
 * DEVICE, bit t set iff the text of token t contains a newline ("." of the reference's regex does not cross one), or NULL.
 * records DEVICE [n_samples][max_records][3] = (first label token, label end token (exclusive), N or -1 for a label without
 * regions), n_records DEVICE [n_samples]. */
int fo1_parse_predictions(const int32_t* tokens, int64_t ld, const int32_t* lens, int32_t n_samples, int32_t ground_start_id,
                          int32_t ground_end_id, int32_t objects_start_id, int32_t objects_end_id, const int32_t* region_ids,
                          int32_t n_region_ids, const uint32_t* newline_bitmap, int32_t vocab, int32_t* records, int32_t max_records,
                          int32_t* n_records, void* stream);

/* inputs_embeds[r] = embed_tokens[src_index[r]] | img_feats[src_index[r]] | region_feats[src_index[r]]
 * (omchat_qwen2_5_vl.py:333-368).  src_kind / src_index: device int32 [n_rows]; feature matrices bf16
 * [*, llm_hidden] with indices already offset per sample by the caller. */
int fo1_llm_build_embeds(fo1_model* m, const int32_t* src_kind, const int32_t* src_index, int32_t n_rows,
                         const void* img_feats, const void* region_feats, void* inputs_embeds, void* stream);

typedef struct {
  int32_t n_seqs;
  const int32_t* seq_lens;        /* host [n_seqs]: L_b, prompt length after the splice */
  const void* inputs_embeds;      /* device bf16 [sum L_b][llm_hidden], sequences packed back to back */
  const int32_t* position_ids;    /* device int32 [3][sum L_b] */
  const int32_t* rope_deltas;     /* host [n_seqs] */
  int32_t max_new_tokens;
  const int32_t* stop_ids;        /* host [n_stop_ids]: generation stops after emitting one of these */
  int32_t n_stop_ids;
  int32_t pad_id;
  int32_t* out_tokens;            /* device int32 [n_seqs][max_new_tokens], pad_id after the stop token */
  int32_t* out_lens;              /* device int32 [n_seqs], counts the stop token */
  float* prefill_logits;          /* optional device fp32 [n_seqs][vocab]: logits at the last prompt position */
  float* all_logits;              /* optional device fp32 [sum L_b][vocab]: logits at every prompt position */
  int32_t early_exit_interval;    /* host polls "all sequences stopped" every k decode steps (0 = never) */
  int32_t steps_run;              /* out: decode iterations actually executed */
  const int32_t* rope_deltas_device; /* optional DEVICE [n_seqs] (what fo1_splice_plan_batch wrote); overrides rope_deltas when set */
} fo1_generate_desc;

/* Prefill + greedy decode (replaces OmChatQwen25VLForCausalLM.forward / HF generate's greedy loop /
 * DynamicCache for this path: omchat_qwen2_5_vl.py:466-532, modeling_qwen2_5_vl.py:1126-1242, 1848-1876).
 * The K/V cache and the decode loop state live on the device; the host only launches. */
int fo1_llm_generate(fo1_model* m, fo1_generate_desc* d, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FO1_H_ */
