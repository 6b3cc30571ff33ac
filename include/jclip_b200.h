/* jclip_b200.h -- C ABI of libjclip_b200.so: the B200-native (sm_100a) hot path of
 * Dokumushikun/jittor-clip-fewshot behind plain pointers and sizes.
 *
 * The reference has no FFI / plugin boundary: it is 100 % Python on top of Jittor, and the seam of the
 * hot path is a handful of Python callables.  Each entry point below names the reference callable it
 * stands in for (paths relative to the reference checkout); INTEGRATION.md shows the ctypes binding a
 * maintainer of the reference would add at each of those seams.
 *
 * Conventions
 *   - every function returns 0 (JCB_OK) or a negative JCB_E_* code; it never throws or aborts.  The
 *     message of the last failure on a context is returned by jcb_last_error().
 *   - "dev" pointers are CUDA device pointers on the context's device; "host" pointers are ordinary
 *     (preferably page-locked) host memory.  The caller allocates every output.
 *   - device work is enqueued on the context's stream (jcb_ctx_set_stream; default: a private
 *     non-blocking stream) and the call returns without waiting, except the *_host entry points and
 *     jcb_sync, which block until their results are in host memory.
 *   - a context and the objects created from it may be used by one host thread at a time.
 *   - there is no CPU fallback: without a CUDA device of compute capability 10.0 context creation fails.
 */
#ifndef JCLIP_B200_H_
#define JCLIP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define JCB_OK 0
#define JCB_E_INVALID (-1)     /* bad argument / unsupported shape */
#define JCB_E_CUDA (-2)        /* CUDA runtime or driver error */
#define JCB_E_STATE (-3)       /* call order (e.g. encode before finalize) */
#define JCB_E_NO_DEVICE (-4)   /* no sm_100 device */
#define JCB_E_KERNEL (-5)      /* a kernel reported a device-side status (pipeline timeout) */
#define JCB_E_NOMEM (-6)

#define JCB_ABI_VERSION 4

typedef struct jcb_ctx jcb_ctx;
typedef struct jcb_vit jcb_vit;
typedef struct jcb_text jcb_text;

/* image element types accepted by the encoder */
#define JCB_IMG_F32 0   /* float32, the reference's dtype (T.ToTensor -> float32) */
#define JCB_IMG_BF16 1
#define JCB_IMG_U8 2    /* uint8 0..255, scaled by 1/255 on the device */
/* not pixels but the conv1 patch matrix [n_views * (R/P)^2, 3 * P * P] written by jcb_tta_patches (view generator fused
 * with ToTensor / tfm_clip / im2col), device-resident, in the tower's 16-bit operand type; apply_clip_norm is ignored */
#define JCB_IMG_PATCHES_BF16 3
#define JCB_IMG_PATCHES_F16 4

/* LoRA target projections (reference test.py:625-640 `enable_lora` items q, k, v, o) */
#define JCB_PROJ_Q 0
#define JCB_PROJ_K 1
#define JCB_PROJ_V 2
#define JCB_PROJ_O 3

/* which fused score the head ranks by (reference test.py:1729-1736 names) */
#define JCB_SCORE_LOGITS 0  /* LP++ logits after logit_normalize            test.py:1721-1722 */
#define JCB_SCORE_CS 1      /* cosine_similarity   (hand text)              test.py:1729 */
#define JCB_SCORE_CS1 2     /* cosine_similarity1  (prompt-tuned text)      test.py:1730  <- what test.py:1738 ranks */
#define JCB_SCORE_CS2 3     /* (cs + cs1) / 2                               test.py:1733 */
#define JCB_SCORE_CS3 4     /* cosine_similarity3  (zero-shot tower)        test.py:1731 */
#define JCB_SCORE_CS4 5     /* (cs2 + cs3) / 2                              test.py:1734 */
#define JCB_SCORE_CS5 6     /* cs4 + 0.5 * logits  (LP++ fusion)            test.py:1735  <- BASELINE config 4 */
#define JCB_SCORE_COUNT 7

int jcb_abi_version(void);

/* ---------------------------------------------------------------- context ------------------- */
/* One per process / GPU.  Replaces `jt.flags.use_cuda = 1` (reference test.py:25). */
int jcb_ctx_create(int device, jcb_ctx** out);
int jcb_ctx_destroy(jcb_ctx* ctx);
/* Use the caller's CUDA stream (a cudaStream_t / CUstream cast to void*), e.g. torch's current stream. */
int jcb_ctx_set_stream(jcb_ctx* ctx, void* cuda_stream);
/* Upper bound on the views processed per pass through the tower (workspace = ~1.2 MB per view); a batch
 * is split into the fewest equal passes that respect it.  Default 16384 for device-resident input
 * (measured on B200: larger passes are faster, intermediates never fit L2 anyway) and min(2048, bound)
 * for host input, so that the copy of pass i+1 overlaps the compute of pass i.  Both bounds count views of a tower
 * of up to 64 tokens (ViT-B/32: 50); a tower of T > 64 tokens runs min(bound, bound * 64 / T) views per pass, about
 * the same number of token rows (ViT-B/16, 197 tokens: 5322 views of the default 16384). */
int jcb_ctx_set_chunk_views(jcb_ctx* ctx, int64_t chunk_views);
int jcb_ctx_set_host_chunk_views(jcb_ctx* ctx, int64_t chunk_views);
/* Opt-in schedule for the image tower (default off; env JCB_CLS_ONLY_LAST_BLOCK=1 sets the initial value): run the
 * LAST transformer block on the class-token row of every view only.  `encode_image` returns
 * ln_post(x[:, 0, :]) @ proj (jclip/model.py:121-124), so after that block's keys and values no other token row
 * reaches the result; the reference computes them anyway.  Embeddings agree with the full schedule to rounding
 * (different attention summation order for that one row).  Ignored by jcb_vit_debug_tokens consumers that read
 * other rows of the last block: with the option on, only row 0 of every view is defined there.  Applies to towers
 * of up to 64 tokens only (the class-token attention scores at most 64 keys); a longer tower such as ViT-B/16 runs
 * the full last block with the option on or off. */
int jcb_ctx_set_cls_only_last_block(jcb_ctx* ctx, int on);
/* Element type of every 16-bit GEMM operand of the towers packed AFTER this call (weights, the residual copy the
 * LayerNorm-folded GEMMs read, q|k|v, softmax numerators, attention output, MLP hidden); accumulation is fp32 in
 * TMEM either way and tcgen05.mma kind::f16 runs both at the same rate.
 *   JCB_OPERAND_F16  (default; env JCB_OPERANDS=f16): 11-bit significands -- end to end the x100 logits stay within
 *                    1e-2 of the fp32 reference (BASELINE north star; measured 0.005-0.008), conversions saturate at
 *                    +-65504 instead of overflowing.
 *   JCB_OPERAND_BF16 (env JCB_OPERANDS=bf16): the north star's literal wording; 8-bit significands put the logits
 *                    0.02-0.07 off (DESIGN.md section 3).
 * A tower keeps the type it was finalized with (jcb_vit_operand_type); re-finalize to change it. */
#define JCB_OPERAND_BF16 0
#define JCB_OPERAND_F16 1
int jcb_ctx_set_operand_type(jcb_ctx* ctx, int operand_type);
int jcb_ctx_get_operand_type(const jcb_ctx* ctx);
/* How the towers packed AFTER this call carry their LoRA adapters (reference LinearLoRA.execute, test.py:378-398):
 *   JCB_LORA_MERGED  (default; env JCB_LORA=merged): W' = W + s B A in fp32, rounded to 16 bits once at pack time
 *                    (the `merged` branch, test.py:310-313, :386); the tower runs exactly the zero-shot schedule.
 *   JCB_LORA_APPLIED (env JCB_LORA=applied): y = W x + b + s B (A x), the branch the reference evaluates in eval mode
 *                    (test.py:388-398; SURVEY.md App. B: Jittor's eval() never merges).  Base weights stay un-merged;
 *                    per layer one narrow GEMM U = x [A_q; A_k; A_v]^T, and the projection GEMM accumulates
 *                    U [s B_q | s B_k | s B_v]^T into the same TMEM accumulator through a second TMA operand pair
 *                    (likewise out_proj for 'o' adapters).  The ranks of q, k, v of one layer must sum to <= 64 (r <= 64
 *                    for 'o').  This schedule keeps the LayerNorms as stand-alone passes (the folded epilogues would
 *                    need the low-rank term pre-divided by the row's 1 / sigma), so it is the slower of the two; it
 *                    exists for callers that swap adapters per request.  It is also the mode that serves several
 *                    adapter sets from one image tower, chosen per image (LoRA slots, jcb_vit_set_lora_slot).
 * A tower keeps the mode it was finalized with (jcb_vit_lora_mode / jcb_text_lora_mode). */
#define JCB_LORA_MERGED 0
#define JCB_LORA_APPLIED 1
int jcb_ctx_set_lora_mode(jcb_ctx* ctx, int mode);
int jcb_ctx_get_lora_mode(const jcb_ctx* ctx);
/* Give the grow-only scratch of the context (tower pass buffers, view-generator scratch, host-input staging) back to
 * the device allocator; it is re-reserved on demand.  Waits for the device.  JCB_E_STATE while submissions are in flight. */
int jcb_ctx_trim(jcb_ctx* ctx);
/* Wait for the context's stream and report any device-side kernel status. */
int jcb_sync(jcb_ctx* ctx);
const char* jcb_last_error(const jcb_ctx* ctx);
/* Device properties the host side reports next to measurements. */
int jcb_ctx_info(const jcb_ctx* ctx, int* num_sms, int* cc_major, int* cc_minor, size_t* workspace_bytes);
/* Number of kernels this library has launched on the context so far (bench.py's gpu_launches). */
int64_t jcb_ctx_launch_count(const jcb_ctx* ctx);

/* Per-kernel-class timing with CUDA events recorded on the launch stream around every launch of the
 * library (what bench.py's roofline uses).  jcb_ctx_profile(ctx, 1) resets and starts; (ctx, 0) waits for
 * the stream and folds the event pairs into per-class totals, read with jcb_ctx_profile_read:
 *   total_ms over the `timed_launches` launches that got an event pair (at most 32768 per session),
 *   `launches` seen, and the ALGORITHMIC flops / bytes of all `launches` (DESIGN.md section 5). */
#define JCB_KC_IM2COL 0
#define JCB_KC_GEMM_PATCH 1
#define JCB_KC_EMBED_LN 2
#define JCB_KC_GEMM_QKV 3
#define JCB_KC_ATTENTION 4
#define JCB_KC_GEMM_OUT 5
#define JCB_KC_LAYERNORM 6
#define JCB_KC_GEMM_FC1 7
#define JCB_KC_GEMM_FC2 8
#define JCB_KC_TAIL 9
#define JCB_KC_MTA 10
#define JCB_KC_HEAD 11
#define JCB_KC_OTHER 12
#define JCB_KC_TTA 13
#define JCB_KC_GEMM_LORA 14   /* LoRA applied: the narrow down-projection GEMMs */
#define JCB_KC_COUNT 15
int jcb_ctx_profile(jcb_ctx* ctx, int enable);
int jcb_ctx_profile_read(const jcb_ctx* ctx, int kernel_class, double* total_ms, int64_t* launches,
                         int64_t* timed_launches, double* flops, double* bytes);
const char* jcb_kernel_class_name(int kernel_class);

/* ---------------------------------------------------------------- image tower ---------------- */
typedef struct jcb_vit_config {
  int32_t layers;      /* 12   number of visual.*.attn.in_proj_weight keys   jclip/model.py:240-243 */
  int32_t width;       /* 768  visual.conv1.weight.shape[0]                  jclip/model.py:238 */
  int32_t patch;       /* 32   visual.conv1.weight.shape[-1]                 jclip/model.py:244 */
  int32_t resolution;  /* 224  patch * sqrt(pos_emb rows - 1)                jclip/model.py:245-247 */
  int32_t embed_dim;   /* 512  visual.proj.shape[1] */
  int32_t vpt_tokens;  /* 0, or 4 for the IVLP / VPT tower of `clip1.load_vlp` (jclip/model1.py:161-164, :192-196):
                          learnable tokens `visual.VPT` appended after the positional embedding, before ln_pre */
} jcb_vit_config;

/* Stands in for `build_model(state_dict)` restricted to the image tower (jclip/model.py:235-285). */
int jcb_vit_create(jcb_ctx* ctx, const jcb_vit_config* cfg, jcb_vit** out);
int jcb_vit_destroy(jcb_vit* vit);
/* Load one fp32 tensor of the CLIP state dict by its reference key name ("visual.conv1.weight",
 * "visual.transformer.resblocks.3.attn.in_proj_weight", ...; jclip/model.py:235-285 / load_parameters).
 * `data` is host memory with `numel` floats; it is copied.  Unknown keys return JCB_E_INVALID. */
int jcb_vit_set_param(jcb_vit* vit, const char* name, const float* data, int64_t numel);
/* Attach one LoRA adapter (reference LinearLoRA, test.py:340-398): A [r, width], B [width, r] host fp32,
 * scaling = alpha / sqrt(r) (test.py:288-289).  Replaces any adapter already on (layer, proj). */
int jcb_vit_set_lora(jcb_vit* vit, int layer, int proj, const float* A, const float* B, int r, float scaling);
/* LoRA slots: a tower holds adapter sets 0 .. G-1 (G <= JCB_MAX_LORA_SLOTS) and a call picks one per view
 * (jcb_encode_image_slots) or per image (jcb_pipeline_slots): view v is encoded exactly -- bit for bit -- as if the tower
 * carried only slot s[v], in applied mode.  Slot 0 is what jcb_vit_set_lora sets (jcb_vit_set_lora_slot with slot 0 is
 * the same call); G = 1 + the highest slot given an adapter (or declared, jcb_vit_set_lora_slot_count) since the last
 * jcb_vit_clear_lora, which clears all slots.
 * More than one slot needs JCB_LORA_APPLIED: jcb_vit_finalize returns JCB_E_INVALID in merged mode, and also when a
 * slot's q, k, v ranks of one layer sum to more than 64 or its 'o' rank exceeds 64.  A slot without an adapter on some
 * (layer, projection) runs the plain projection there.  Per layer and projection the device holds one 64-row down block
 * and one 64-column up block per slot; a 256-row GEMM tile multiplies the up blocks of the slots its rows use (measured
 * on a B200 with one slot per image of 65 views: +2 to +3 % per step for G = 2 to 8; DESIGN.md section 4). */
#define JCB_MAX_LORA_SLOTS 8
int jcb_vit_set_lora_slot(jcb_vit* vit, int slot, int layer, int proj, const float* A, const float* B, int r, float scaling);
/* Declare slots 0 .. n_slots-1 even if the highest of them has no adapter (an adapter set that is empty, e.g. the
 * plain tower next to adapted ones): G = max(G, n_slots).  1 <= n_slots <= JCB_MAX_LORA_SLOTS; cleared by
 * jcb_vit_clear_lora like the adapters. */
int jcb_vit_set_lora_slot_count(jcb_vit* vit, int n_slots);
/* G: the number of slots the next jcb_vit_finalize packs (1 without jcb_vit_set_lora_slot / _slot_count). */
int jcb_vit_lora_slots(const jcb_vit* vit);
int jcb_vit_clear_lora(jcb_vit* vit);
/* Pack the weights for the device: W' = W + scaling * B A in fp32, then bf16 (GEMM operands); LayerNorm /
 * bias / embedding / final projection parameters stay fp32.  Must be called after the last set_param /
 * set_lora and before jcb_encode_image; may be called again after the adapters change. */
int jcb_vit_finalize(jcb_vit* vit);
/* JCB_OPERAND_* the device weights were packed with by the last jcb_vit_finalize. */
int jcb_vit_operand_type(const jcb_vit* vit);
/* JCB_LORA_* the adapters were packed with by the last jcb_vit_finalize. */
int jcb_vit_lora_mode(const jcb_vit* vit);

/* `CLIP.encode_image(image)` (jclip/model.py:199-200 -> VisionTransformer.execute :104-126).
 *   images_dev   [n_views, 3, R, R] on the device, element type `img_dtype`
 *   apply_clip_norm != 0 fuses `tfm_clip` = ImageNormalize(mean, std) (test.py:1301, applied at :1705)
 *   normalize   != 0 fuses `f / f.norm(dim=-1, keepdim=True)` (test.py:1706)
 *   out_dev      [n_views, embed_dim] float32 */
int jcb_encode_image(jcb_vit* vit, const void* images_dev, int img_dtype, int64_t n_views, int apply_clip_norm,
                     int normalize, float* out_dev);
/* jcb_encode_image with a LoRA slot per view: slot_of_view_host [n_views] int32 host array, each in [0, G).  It is
 * validated before anything is launched (JCB_E_INVALID for a NULL array or a slot outside the tower's G, out_dev
 * untouched) and copied to the device once per call.  A tower with one slot runs jcb_encode_image. */
int jcb_encode_image_slots(jcb_vit* vit, const void* images_dev, int img_dtype, int64_t n_views,
                           const int32_t* slot_of_view_host, int apply_clip_norm, int normalize, float* out_dev);
/* Same with host buffers: host->device copies of the image chunks (overlapped with compute on a second
 * stream) and the device->host copy of the embeddings happen inside the call; it returns when out_host
 * is valid.  This is the call the end-to-end measurement times. */
int jcb_encode_image_host(jcb_vit* vit, const void* images_host, int img_dtype, int64_t n_views,
                          int apply_clip_norm, int normalize, float* out_host);

/* Final token tensor of the tower [n_views * tokens, width] fp32 before ln_post (tests / debugging). */
int jcb_vit_debug_tokens(jcb_vit* vit, const void* images_dev, int img_dtype, int64_t n_views, int apply_clip_norm,
                         float* tokens_out_dev);

/* ---------------------------------------------------------------- text tower ----------------- */
/* `CLIP.encode_text` (jclip/model.py:202-215), SURVEY.md section 8 "next" row f3: it runs once per run to build the
 * cached text embeddings (clip_classifier, test.py:920-940: 403 classes x the templates), reusing the image
 * tower's kernels with a causal attention mask. */
typedef struct jcb_text_config {
  int32_t layers;          /* 12  number of transformer.resblocks.*                jclip/model.py:269-273 */
  int32_t width;           /* 512 ln_final.weight.shape[0]                         jclip/model.py:267 */
  int32_t context_length;  /* 77  positional_embedding.shape[0]                    jclip/model.py:265 */
  int32_t vocab_size;      /* 49408 token_embedding.weight.shape[0]                jclip/model.py:266 */
  int32_t embed_dim;       /* 512 text_projection.shape[1]                         jclip/model.py:264 */
} jcb_text_config;
int jcb_text_create(jcb_ctx* ctx, const jcb_text_config* cfg, jcb_text** out);
int jcb_text_destroy(jcb_text* text);
/* keys: token_embedding.weight, positional_embedding, transformer.resblocks.{i}.*, ln_final.{weight,bias},
 * text_projection (jclip/model.py:235-285) */
int jcb_text_set_param(jcb_text* text, const char* name, const float* data, int64_t numel);
/* LoRA on the text blocks (apply_lora with encoder 'text' / 'both', test.py:611-623) */
int jcb_text_set_lora(jcb_text* text, int layer, int proj, const float* A, const float* B, int r, float scaling);
int jcb_text_clear_lora(jcb_text* text);
int jcb_text_finalize(jcb_text* text);
int jcb_text_operand_type(const jcb_text* text);
int jcb_text_lora_mode(const jcb_text* text);
/* tokens_dev [n_seq, context_length] int64 (what `clip.tokenize` returns); out_dev [n_seq, embed_dim] float32;
 * normalize != 0 fuses `/ norm(dim=-1)` (test.py:929) */
int jcb_encode_text(jcb_text* text, const int64_t* tokens_dev, int64_t n_seq, int normalize, float* out_dev);
/* The averaging step of `clip_classifier` (test.py:931-934): out[c] = normalise(mean of emb rows offsets[c] ..
 * offsets[c+1]) for unit-norm template embeddings emb_dev [n, dim]; offsets_dev [n_classes + 1] int32. */
int jcb_class_mean(jcb_ctx* ctx, const float* emb_dev, const int32_t* offsets_dev, int32_t n_classes, int32_t dim,
                   float* out_dev);

/* ---------------------------------------------------------------- TTA views ------------------ */
/* The step upstream of encode_image: the reference builds, per test image, 1 centre view + N random crops on
 * the CPU with PIL (JtDataset.__getitem__, test.py:1547-1560; transforms test.py:1898-1903, ood.py:1084-1089,
 * jclip/clip.py:102-135).  A view = take a box of a decoded uint8 image, resample it (Pillow's ImagingResample,
 * reproduced bit for bit), keep an S x S window, optionally mirror it. */
typedef struct jcb_src_image {
  int64_t offset;             /* byte offset of this image ([height, width, 3] uint8, RGB interleaved) in src_dev */
  int32_t height, width;
} jcb_src_image;
#define JCB_FILTER_BILINEAR 0 /* PIL.Image.BILINEAR: RandomResizedCrop's interpolation */
#define JCB_FILTER_BICUBIC 1  /* PIL.Image.BICUBIC : Resize(256) of the centre view, jclip/clip.py:130-135 */
typedef struct jcb_view_job {
  int32_t image;                      /* index into images[] */
  int32_t top, left, crop_h, crop_w;  /* `img.crop((left, top, left + crop_w, top + crop_h))` */
  int32_t out_h, out_w;               /* `.resize((out_w, out_h), filter)` */
  int32_t off_y, off_x;               /* window kept of the resized crop: CenterCrop offsets, 0 for random crops */
  int32_t filter, flip, reserved;
} jcb_view_job;
/* out_dev [n_jobs, 3, size, size] uint8 (planar, the layout jcb_encode_image / jcb_pipeline take with
 * JCB_IMG_U8).  images / jobs are host arrays; they are validated and copied.  When src_dev is 4-byte aligned the
 * source is read as whole aligned 32-bit words, so the buffer must be readable up to the next multiple of 4 bytes
 * past the last image (any cudaMalloc / torch allocation is); an unaligned src_dev takes a slower byte-wise path.
 * cuda_stream: the stream to enqueue on (a cudaStream_t cast to void*), NULL = the context's stream.  The generator has
 * its own scratch, so a batch may be generated on a second stream while the towers work on the previous one; the caller
 * orders the streams (src_dev ready before, out_dev consumed after) with its own events. */
int jcb_tta_views(jcb_ctx* ctx, void* cuda_stream, const uint8_t* src_dev, const jcb_src_image* images, int32_t n_images,
                  const jcb_view_job* jobs, int64_t n_jobs, int32_t size, uint8_t* out_dev);
/* The same views, delivered as what the image tower's first GEMM reads: out_patches_dev [n_jobs * (size/patch)^2,
 * 3 * patch^2] 16-bit of `operand_type`, row = (view, py, px), column = (c, i, j) (jclip/model.py:105-108 as im2col),
 * value = round16(u8 / 255) or, with apply_clip_norm, round16((u8 / 255 - mean_c) / std_c) (test.py:1301) -- bit-identical
 * to jcb_tta_views followed by jcb_im2col, without the uint8 view tensor or the im2col pass.  Feed it to
 * jcb_encode_image / jcb_pipeline with img_dtype JCB_IMG_PATCHES_*. */
int jcb_tta_patches(jcb_ctx* ctx, void* cuda_stream, const uint8_t* src_dev, const jcb_src_image* images, int32_t n_images,
                    const jcb_view_job* jobs, int64_t n_jobs, int32_t size, int32_t patch, int32_t apply_clip_norm,
                    int32_t operand_type, void* out_patches_dev);

/* ---------------------------------------------------------------- MTA ------------------------ */
typedef struct jcb_mta_params {
  float lambda_y;     /* 0.2   test.py:1395 */
  float lambda_q;     /* 4     test.py:1396 */
  float th;           /* 1e-6  test.py:1421 */
  float temperature;  /* 1     test.py:1398 */
  double k_frac;      /* 0.3   test.py:1405 */
  int32_t max_iter;   /* 5     test.py:1397 */
  int32_t reserved;
} jcb_mta_params;
void jcb_mta_default_params(jcb_mta_params* p);

/* `solve_mta(image_features, text_features)` batched over images (test.py:1391-1461; ood.py:751-820).
 *   feats_dev    [n_images, n_views, dim] float32 unit rows, view 0 = un-augmented image
 *   text_dev     [dim, n_classes] float32  (the orientation the reference passes: `text_features.t()`)
 *   out_mode_dev [n_images, dim]            the mode, unit norm            (test.py:1461)
 *   out_logits_dev [n_images, n_classes] or NULL: 100 * mode @ text         (ood.py:819)
 *   params NULL = reference constants
 * JCB_E_INVALID, before anything is allocated or launched, for n_views outside [1, 2048], n_classes < 1, dim not a
 * multiple of 32 in [32, 1024], a non-finite parameter, lambda_y <= 0, temperature <= 0, th < 0, max_iter < 1 or
 * k_frac outside [0, 1] (the reference averages at most n_views - 1 neighbours).  n_views = 1 is accepted and gives
 * what the reference gives: its bandwidth is the mean of no distances, so the mode is all NaN. */
int jcb_mta(jcb_ctx* ctx, const float* feats_dev, const float* text_dev, int64_t n_images, int32_t n_views,
            int32_t n_classes, int32_t dim, const jcb_mta_params* params, float* out_mode_dev,
            float* out_logits_dev);
/* jcb_mta plus the solver's state per image, for tests and debugging; each output may be NULL (skipped):
 *   out_bw_dev       [n_images, n_views]           the bandwidths                                (test.py:1403-1408)
 *   out_y_dev        [n_images, n_views]           the inlierness weights the last mode loop used (test.py:1434)
 *   out_affinity_dev [n_images, n_views, n_views]  A = P P^T, P = softmax(100 X T / temperature)  (test.py:1411)
 * The mode and logits are the ones jcb_mta returns for the same arguments. */
int jcb_mta_debug(jcb_ctx* ctx, const float* feats_dev, const float* text_dev, int64_t n_images, int32_t n_views,
                  int32_t n_classes, int32_t dim, const jcb_mta_params* params, float* out_mode_dev,
                  float* out_logits_dev, float* out_bw_dev, float* out_y_dev, float* out_affinity_dev);

/* ---------------------------------------------------------------- head ----------------------- */
typedef struct jcb_head_weights {   /* Channel_LP parameters, test.py:1223-1228, all device fp32 */
  const float* scale1;  /* [dim] */
  const float* bias1;   /* [dim] */
  const float* fc_w;    /* [n_classes, dim] */
  const float* fc_b;    /* [n_classes] */
} jcb_head_weights;

/* Per-image body of evaluate_base after the three solve_mta calls (test.py:1710-1738):
 * Channel_LP x2 -> logit_normalize x3 -> cosine logits x3 -> fusion -> top-k of `rank_by`.
 *   m_*_dev [n_images, dim] modes; T_*_dev [n_classes, dim] text features (un-transposed, unit rows)
 *   out_topk_dev [n_images, k] int32 (k <= 8); out_scores_dev [n_images, n_classes] or NULL (the ranked
 *   score); out_all_dev [n_images, JCB_SCORE_COUNT, n_classes] or NULL. */
int jcb_head(jcb_ctx* ctx, const float* m_pt_dev, const float* m_hand_dev, const float* m_zs_dev,
             const float* T_pt_dev, const float* T_hand_dev, const float* T_zs_dev, const jcb_head_weights* lp,
             int64_t n_images, int32_t n_classes, int32_t dim, int32_t rank_by, int32_t k, int32_t* out_topk_dev,
             float* out_scores_dev, float* out_all_dev);

/* `scale * f @ T.t()` then topk (evaluate_new test.py:1770-1774; OOD argmax ood.py:875-877 with k = 1). */
int jcb_cosine_topk(jcb_ctx* ctx, const float* feats_dev, const float* text_dev /* [n_classes, dim] */,
                    int64_t n, int32_t n_classes, int32_t dim, float scale, int32_t k, int32_t* out_topk_dev,
                    float* out_scores_dev);
/* `Channel_LP.execute(features)` (test.py:1229-1234): out [n, n_classes]. */
int jcb_channel_lp(jcb_ctx* ctx, const float* feats_dev, int64_t n, int32_t n_classes, int32_t dim,
                   const jcb_head_weights* lp, float* out_dev);
/* `logit_normalize(logit)` (test.py:1304-1308): global unbiased std, per-row mean. */
int jcb_logit_normalize(jcb_ctx* ctx, const float* in_dev, int64_t n, int32_t n_classes, float* out_dev);

/* ---------------------------------------------------------------- whole hot path ------------- */
typedef struct jcb_pipeline_args {
  /* inputs */
  const void* images;       /* [n_images, n_views, 3, R, R]; device or host pointer (see images_on_host) */
  int32_t img_dtype;
  int32_t images_on_host;   /* 1: page-locked host memory, copied chunk by chunk inside the call */
  int64_t n_images;
  int32_t n_views;          /* V = N + 1 (reference test.py:1700) */
  int32_t apply_clip_norm;
  const float* text_pt_dev;     /* [n_classes, dim] prompt-tuned text features   (test.py:1684-1686) */
  const float* text_hand_dev;   /* [n_classes, dim] hand-template text features  (test.py:1678) */
  const float* text_zs_dev;     /* [n_classes, dim] zero-shot tower text features (test.py:1679) */
  const float* text_pt_t_dev;   /* the same three, transposed [dim, n_classes] (what solve_mta receives) */
  const float* text_hand_t_dev;
  const float* text_zs_t_dev;
  jcb_head_weights lp;
  int32_t n_classes;
  int32_t rank_by;
  int32_t k;
  int32_t topk_on_host;     /* 1: out_topk is host memory and the call blocks until it is valid */
  /* outputs */
  int32_t* out_topk;        /* [n_images, k] */
  float* out_feats_dev;     /* optional [n_images * n_views, dim] unit view embeddings, or NULL */
  float* out_scores_dev;    /* optional [n_images, n_classes], or NULL */
} jcb_pipeline_args;

/* encode_image over every view -> L2 normalise -> solve_mta x3 -> head -> top-k: the loop body of
 * evaluate_base (test.py:1692-1742) for a batch of images, one image tower (`vit`) feeding all three
 * MTA solves.  `vit_zs` may be NULL (single tower) or a second tower for the zero-shot branch
 * (test.py:1711-1713). */
int jcb_pipeline(jcb_vit* vit, jcb_vit* vit_zs, const jcb_pipeline_args* args);
/* jcb_pipeline with a LoRA slot per image: slot_of_image_host [n_images] int32 host array, each in [0, G) of `vit`; every
 * view of image i runs slot slot_of_image_host[i] of `vit` (jcb_vit_set_lora_slot), while `vit_zs` runs its own slot 0.
 * Validated before anything is launched, like jcb_encode_image_slots.  These calls are never captured into or served
 * from the CUDA graphs of jcb_ctx_set_graphs. */
int jcb_pipeline_slots(jcb_vit* vit, jcb_vit* vit_zs, const jcb_pipeline_args* args, const int32_t* slot_of_image_host);

/* Small calls (n_images * n_views <= max_views, default 1024; device work only; no out_feats / out_scores) are served
 * from CUDA graphs: the second jcb_pipeline call with the same towers, shapes and operand pointers is captured, later ones
 * replay it with a single launch (the reference's own loop calls the path once per image, test.py:1692-1742: ~210
 * launches for ~0.6 ms of GPU work).  Results are bit-identical to the un-captured path.  on = 0 (or env JCB_GRAPHS=0)
 * disables and drops the captured graphs; max_views = 0 keeps the current threshold. */
int jcb_ctx_set_graphs(jcb_ctx* ctx, int on, int64_t max_views);
int jcb_ctx_graph_stats(const jcb_ctx* ctx, int64_t* captured, int64_t* launched, int64_t* failed);

/* The same for a STREAM of batches (the reference's `for images in loader:` loop, test.py:1692): submit enqueues
 * everything jcb_pipeline does -- the host->device copies of the view chunks, the tower, MTA, head and, with
 * topk_on_host, the device->host copy of the top-k -- and returns without waiting; jcb_pipeline_wait blocks until
 * the submission `ticket` has completed (its out_topk is valid) and reports device-side errors.  Submitting batch
 * k+1 before waiting for batch k overlaps the uploads of k+1 with the compute of k.  `images` and `out_topk` of a
 * submission must stay valid and untouched until its wait returns; tickets complete in submission order; at most
 * JCB_MAX_INFLIGHT submissions may be un-waited (JCB_E_STATE otherwise). */
#define JCB_MAX_INFLIGHT 4
int jcb_pipeline_submit(jcb_vit* vit, jcb_vit* vit_zs, const jcb_pipeline_args* args, int64_t* ticket);
/* jcb_pipeline_submit with per-image LoRA slots (jcb_pipeline_slots); the slot array is copied before the call returns. */
int jcb_pipeline_submit_slots(jcb_vit* vit, jcb_vit* vit_zs, const jcb_pipeline_args* args, const int32_t* slot_of_image_host,
                              int64_t* ticket);
int jcb_pipeline_wait(jcb_ctx* ctx, int64_t ticket);

/* ---------------------------------------------------------------- building blocks (tests) ---- */
/* GEMM epilogues fused into the tcgen05 kernel (csrc/kernels.h GemmEpilogue) */
#define JCB_EPI_BIAS_16 0            /* out16 = acc + bias                                   (QKV projection) */
#define JCB_EPI_BIAS_GELU_16 1       /* out16 = quickgelu(acc + bias)   jclip/model.py:27   (MLP c_fc) */
#define JCB_EPI_BIAS_RESID_F32 2     /* out32 += acc + bias             jclip/model.py:60-61 */
#define JCB_EPI_F32 4                /* out32 = acc (+ bias) */
#define JCB_EPI_LNFOLD_16 5          /* out16 = r[m] acc - r[m] mu[m] colsum[n] + bias[n]: LayerNorm folded into the GEMM */
#define JCB_EPI_LNFOLD_GELU_16 6     /* quickgelu of that */
#define JCB_EPI_RESID_LNPREP_SHORT 7 /* out32 += acc + bias; out2_16 = out32 - shift[m]; stats[m, n / 256] = (sum, sumsq) of out2 */
#define JCB_EPI_RESID_LNPREP_LONG 8  /* same, staging tuned for long K */
/* C[M,N] = A[M,K] * B[N,K]^T, A / B 16-bit operands of `operand_type`, with the fused epilogues of the tower
 * (jclip/model.py:38-39, :59-62, jclip/mha.py:129-146, :461).  The LayerNorm-fold fields are what the tower passes
 * between its GEMMs (csrc/api.cu tower_blocks): tests drive the epilogues directly through them. */
typedef struct jcb_gemm_args {
  const void* A_dev;        /* [M, K] row-major */
  const void* B_dev;        /* [N, K] row-major (nn.Linear weight layout) */
  int32_t M, N, K;
  int32_t operand_type;     /* JCB_OPERAND_* */
  const float* bias_dev;    /* [N] or NULL */
  int32_t epilogue;         /* JCB_EPI_* */
  int32_t stats_slots;      /* partial-sum slots per row (N / 256 of the producer) */
  void* out_dev;            /* 16-bit or fp32 according to the epilogue */
  int64_t ldo;
  float* stats_dev;         /* LNFOLD: in, LNPREP: out; [M, stats_slots, 2] */
  const float* colsum_dev;  /* LNFOLD: S[N] = sum_k of the rounded folded weight */
  void* out2_dev;           /* LNPREP: centred 16-bit copy [M, N] */
  const float* stats_in_dev;   /* LNPREP: previous LayerNorm point's statistics / shift, or NULL (shift 0) */
  const float* shift_in_dev;
  float* shift_out_dev;     /* LNPREP: [M] or NULL */
  int64_t stats_in_row_stride;
  /* optional second operand pair accumulated into the same tile: C = A B^T + A2 B2^T (LoRA applied, test.py:388-398) */
  const void* A2_dev;       /* [M, K2] row-major, leading dimension lda2; NULL / K2 = 0: none */
  const void* B2_dev;       /* [N, K2] row-major, leading dimension ldb2 */
  int32_t K2;               /* multiple of 64 */
  int64_t lda2, ldb2;
} jcb_gemm_args;
int jcb_gemm(jcb_ctx* ctx, const jcb_gemm_args* args);
/* Weight preparation of a LayerNorm-folded GEMM: Wf[n,k] = round16(gamma[k] W[n,k]); S[n] = sum_k Wf[n,k];
 * c[n] = sum_k beta[k] W[n,k] + bias[n]   (LN(x) W^T + b = r (x Wf^T) - r mu S + c; jclip/model.py:17-21, :59-62) */
int jcb_fold_ln(jcb_ctx* ctx, const float* W_dev, const float* gamma_dev, const float* beta_dev, const float* bias_dev,
                int32_t N, int32_t K, int32_t operand_type, void* Wf_dev, float* S_dev, float* c_dev);
int jcb_layernorm(jcb_ctx* ctx, const float* x_dev, int64_t rows, int32_t width, const float* gamma_dev,
                  const float* beta_dev, int32_t operand_type, void* out16_dev);
/* `tfm_clip` + the patch extraction of conv1 (test.py:1301, jclip/model.py:105-108): images_dev [n_views, 3, R, R]
 * (JCB_IMG_*) -> patches16_dev [n_views * (R/P)^2, 3 * P * P], row = (view, py, px), column = (c, i, j). */
int jcb_im2col(jcb_ctx* ctx, const void* images_dev, int32_t img_dtype, int64_t n_views, int32_t resolution,
               int32_t patch, int32_t apply_clip_norm, int32_t operand_type, void* patches16_dev);
/* softmax(q k^T / 8 [+ causal mask]) v per (sequence, head) (jclip/mha.py:55-83; mask jclip/model.py:189-193):
 * qkv16_dev [n_views * tokens, 3 * 64 * heads] -> out16_dev [n_views * tokens, 64 * heads]; tokens <= 256 without the
 * mask, tokens <= 128 with it (JCB_E_INVALID otherwise) */
int jcb_attention(jcb_ctx* ctx, const void* qkv16_dev, int64_t n_views, int32_t tokens, int32_t heads, int32_t causal,
                  int32_t operand_type, void* out16_dev);
/* hits / misses of the process-wide cache of encoded TMA tensor maps (one entry per (pointer, shape) launched) */
void jcb_tensor_map_cache_stats(uint64_t* hits, uint64_t* misses);

/* ---------------------------------------------------------------- DLPack hand-off ------------ */
/* Zero-copy variant of jcb_encode_image taking DLManagedTensor* (dlpack.h ABI v0.x).  Tensors are
 * borrowed: the deleters are never called.  images: [n,3,R,R] f32/bf16/u8 on kDLCUDA; out: [n,E] f32. */
int jcb_encode_image_dlpack(jcb_vit* vit, void* images_dlmanaged, void* out_dlmanaged, int apply_clip_norm,
                            int normalize);

#ifdef __cplusplus
}
#endif
#endif /* JCLIP_B200_H_ */
