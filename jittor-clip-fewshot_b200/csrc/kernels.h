// Host-side launchers of the sm_100a kernels behind the C-ABI (include/jclip_b200.h).
#pragma once
#include <cstddef>
#include <cstdint>
#include <utility>
#include <vector>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace jcb {

// 16-bit operand storage.  Every 16-bit tensor of a tower (weights, raw residual copy, q|k|v, attention output, MLP
// hidden) holds bf16 OR fp16 bits, fixed per tower when it is packed (jcb_ctx_set_operand_type); the pointers are
// typed __nv_bfloat16* for historical reasons and the launchers take `f16` (0 = bf16, 1 = fp16) next to them.
enum TmapDtype : int { TM_F32 = 0, TM_BF16 = 1, TM_F16 = 2 };

// ---- GEMM epilogues (fused into the tcgen05 kernel) -------------------------------------------
enum GemmEpilogue : int {
  EPI_BIAS_BF16 = 0,       // out_bf16[m,n]  = acc + bias[n]                       (QKV projection)
  EPI_BIAS_GELU_BF16 = 1,  // out_bf16[m,n]  = quickgelu(acc + bias[n])            (MLP c_fc)
  EPI_BIAS_RESID_F32 = 2,  // out_f32[m,n]  += acc + bias[n]                       (out_proj / c_proj + residual)
  // 3 was the conv1 scatter epilogue (direct stores); conv1 now leaves through EPI_F32 and the embed kernel scatters
  EPI_F32 = 4,             // out_f32[m,n]   = acc (+ bias[n] if given)            (tests / generic)
  // ---- LayerNorm folded into the GEMMs (no stand-alone LayerNorm pass over the residual stream) ----
  // LN(x) W^T = r (x (g*W)^T) - r mu S + c  with  S[n] = sum_k g[k] W[n,k],  c[n] = sum_k b[k] W[n,k] + bias[n]:
  // the consumer GEMM multiplies the RAW bf16 copy of the residual stream by the gamma-folded weight and applies
  // the per-row (mu, r) in its epilogue; the producer GEMM (a residual epilogue) writes that bf16 copy and the
  // per-row partial sums next to the fp32 residual.
  EPI_LNFOLD_BF16 = 5,       // out_bf16[m,n] = r[m] * acc - r[m] * mu[m] * colsum[n] + bias[n]          (QKV)
  EPI_LNFOLD_GELU_BF16 = 6,  // out_bf16[m,n] = quickgelu(that)                                        (MLP c_fc)
  EPI_RESID_LNPREP_SHORT = 7,  // out_f32 += acc + bias; out2_bf16 = bf16(out_f32); stats[m, n_blk] = (sum, sumsq)
  EPI_RESID_LNPREP_LONG = 8,   // same; staging / ring split tuned for long K (c_proj) instead of HBM-bound short K (out_proj)
};

struct GemmArgs {
  const __nv_bfloat16* A = nullptr;  // [M, K] row-major, leading dimension lda (elements)
  const __nv_bfloat16* B = nullptr;  // [N, K] row-major (nn.Linear weight layout), leading dimension ldb
  int64_t lda = 0, ldb = 0;
  int M = 0, N = 0, K = 0;
  // optional second operand pair accumulated into the same output tile: C = A B^T + A2 B2^T (LoRA in applied form,
  // test.py:388-398: A2 = x A_lora^T [M, K2], B2 = s B_lora [N, K2]); K2 % 64 == 0, 0 = none
  const __nv_bfloat16* A2 = nullptr;
  const __nv_bfloat16* B2 = nullptr;
  int64_t lda2 = 0, ldb2 = 0;
  int K2 = 0;
  const float* bias = nullptr;       // [N] or nullptr
  int epilogue = EPI_BIAS_BF16;
  void* out = nullptr;               // bf16 or fp32 according to the epilogue
  int64_t ldo = 0;
  float* stats = nullptr;            // LNFOLD: in, LNPREP: out.  [M, stats_slots, 2] fp32 partial (sum, sum of squares)
  int stats_slots = 0;               // partial slots per row (= N / 256 of the producer; the consumer adds them up)
  const float* colsum = nullptr;     // LNFOLD: S[N]
  void* out2 = nullptr;              // LNPREP: 16-bit copy of the updated residual [M, N], centred by `shift`
  int64_t ldo2 = 0;
  int f16 = 0;                       // element type of A, B and of 16-bit outputs: 0 = bf16, 1 = fp16
  // LNPREP: out2 = x - shift[row] and stats = partial sums of the centred copy, shift[row] = the row's mean at the
  // previous LayerNorm point = shift_in[row] + sum(stats_in[row, :].sum) / N.  nullptr: shift 0.
  const float* stats_in = nullptr;   // [M * stats_in_row_stride, stats_slots, 2], must not alias `stats`
  const float* shift_in = nullptr;   // [M * stats_in_row_stride]
  float* shift_out = nullptr;        // [M]
  int64_t stats_in_row_stride = 1;
  // LoRA slots (several adapter sets, chosen per view): slot_of_view[v] is the slot of rows [v * slot_rows,
  // (v + 1) * slot_rows) and slot_live the slots that have an adapter in this GEMM.  With K2 > 0, second-pair k-block g
  // belongs to slot g: a 256-row tile multiplies only the k-blocks of slots its rows use.  With K2 == 0 (EPI_BIAS_BF16,
  // the down-projection U = x A^T), output columns [64 g, 64 g + 64) belong to slot g: a row gets exact zeros in the
  // blocks of other slots, and tiles whose column blocks hold no slot of the tile's rows are not computed (nor written).
  // nullptr: none (the kernels without the per-tile slot logic).
  const int* slot_of_view = nullptr;
  int slot_rows = 0;
  uint32_t slot_live = 0;
};
constexpr int LORA_MAX_SLOTS = 8;   // JCB_MAX_LORA_SLOTS

// Persistent TMA + tcgen05 GEMM.  Requires N % 128 == 0 and K % 64 == 0 (every GEMM of the ViT-B/32
// tower satisfies it); any M.  Returns cudaErrorInvalidValue otherwise.
cudaError_t launch_gemm(const GemmArgs& a, int* dev_status, int num_sms, cudaStream_t stream);
// Resolves cuTensorMapEncodeTiled through the runtime (no link-time libcuda dependency).
const char* gemm_init_driver_api();

// ---- row-wise / elementwise kernels ----------------------------------------------------------
// images [B,3,R,R] (fp32 | bf16 | u8) -> patches [B*G*G, 3*P*P] bf16 (K-major rows for the patch GEMM).
// apply_norm: fuse tfm_clip (x - mean_c) / std_c ; u8 input is scaled by 1/255 first.
enum ImageDtype : int { IMG_F32 = 0, IMG_BF16 = 1, IMG_U8 = 2 };
cudaError_t launch_im2col(const void* images, int img_dtype, int64_t n_views, int resolution, int patch,
                          int apply_norm, __nv_bfloat16* patches, cudaStream_t stream, int f16 = 0);
// tokens [B*T, W] fp32: row t==0 of each view := cls + pos[0]; rows 1..T-1-n_vpt already hold patch+pos;
// the last n_vpt rows := vpt[0..n_vpt) (IVLP / VPT prompt tokens, no positional embedding);
// then x := ln_pre(x) written back in place (the residual stream), and y := ln_1(x) as bf16.
cudaError_t launch_embed_ln(float* tokens, int64_t n_views, int T, int W, const float* cls, const float* pos,
                            const float* vpt, int n_vpt, const float* g_pre, const float* b_pre, const float* g1,
                            const float* b1, __nv_bfloat16* y, cudaStream_t stream, float* stats = nullptr,
                            int stats_slots = 0,    // stats != nullptr: y = 16-bit (x - mean) + (sum, sumsq) of it for EPI_LNFOLD_*
                            const float* patch_out = nullptr,    // dense conv1 output [n_views * (T-1-n_vpt), W] (no pos) instead
                                                                 // of patch rows already scattered into `tokens`
                            float* shift = nullptr,              // with stats: the row mean the copy was centred by
                            int f16 = 0);
// y_bf16[r,:] = LayerNorm(x_f32[r,:]) * g + b   (eps 1e-5, biased variance), W == 768 or any W % 128 == 0 <= 1024
cudaError_t launch_layernorm(const float* x, int64_t rows, int W, const float* g, const float* b,
                             __nv_bfloat16* y, cudaStream_t stream, int f16 = 0);
// out[v,:] = (ln_post(tokens[v*T + row_idx[v], :]) @ proj[W,E]) ; optionally / ||.||_2.  row_idx == nullptr: row 0
// (the class token); the text tower passes the EOT position of each sequence.
cudaError_t launch_tail(const float* tokens, int64_t n_views, int T, int W, const float* g, const float* b,
                        const float* proj, int E, int normalize, float* out, cudaStream_t stream,
                        const int* row_idx = nullptr);
// text tower front end (jclip/model.py:203-205): x[s*T + t, :] = tok_emb[ids[s, t], :] + pos[t, :] (fp32 residual
// stream), y = ln_1(x) as bf16, and eot[s] = argmax_t ids[s, t] (first maximum; model.py:213-214)
cudaError_t launch_text_embed_ln(const long long* ids, int64_t n_seq, int T, int W, int vocab, const float* tok_emb,
                                 const float* pos, const float* g1, const float* b1, float* tokens, __nv_bfloat16* y,
                                 int* eot, cudaStream_t stream, float* stats = nullptr, int stats_slots = 0,
                                 float* shift = nullptr, int f16 = 0);
// qkv [B*T, 3W] bf16 (q | k | v, heads = 64-wide column blocks) -> out [B*T, W] bf16
// causal != 0: key j is visible to query i only if j <= i (text tower); T <= 128 with the mask, T <= 256 without.
// Runs the tcgen05 / TMEM kernels (attention_tc.cu): two heads per work item without a mask at T <= 64 and an even head
// count, one head per item up to T = 128, one head and one 128-row query tile per item for 129 <= T <= 256
cudaError_t launch_attention(const __nv_bfloat16* qkv, int64_t n_views, int T, int heads, __nv_bfloat16* out,
                             cudaStream_t stream, int causal, int* dev_status, int num_sms, int f16 = 0);
// query row 0 only (no mask, T <= 64): out [n_views, W] bf16, dense
cudaError_t launch_attention_cls(const __nv_bfloat16* qkv, int64_t n_views, int T, int heads, __nv_bfloat16* out,
                                 cudaStream_t stream, int f16 = 0);
bool attention_tc_supported(int T, int heads, int causal);
cudaError_t launch_attention_tc(const __nv_bfloat16* qkv, int64_t n_views, int T, int heads, __nv_bfloat16* out,
                                cudaStream_t stream, int* dev_status, int num_sms, int f16 = 0, int causal = 0);
// hits / misses of the encoded-tensor-map cache (gemm.cu)
void tmap_cache_stats(uint64_t* hits, uint64_t* misses);
// fp32 -> bf16 cast (weight packing)
cudaError_t launch_cast_bf16(const float* src, __nv_bfloat16* dst, int64_t n, cudaStream_t stream, int f16 = 0);
// W'[rows, cols] (bf16) = W (fp32) + scaling * B[rows, r] @ A[r, cols]   for a row range of a packed weight
cudaError_t launch_merge_lora_cast(const float* W, const float* A, const float* B, int rows, int cols, int r,
                                   float scaling, __nv_bfloat16* dst, cudaStream_t stream, int f16 = 0);

// in place W (fp32) += scaling * B A; and the LayerNorm fold of a weight (see EPI_LNFOLD_* above)
cudaError_t launch_merge_lora_f32(float* W, const float* A, const float* B, int rows, int cols, int r, float scaling,
                                  cudaStream_t stream);
cudaError_t launch_fold_ln(const float* W, const float* gamma, const float* beta, const float* bias, int N, int K,
                           __nv_bfloat16* Wf, float* S, float* c, cudaStream_t stream, int f16 = 0);

// ---- LoRA training (train.cu): the backward pass of the image tower with respect to the adapters --------------
// element types of launch_xty_accumulate's operands
enum TrainElem : int { TR_BF16 = 0, TR_F16 = 1, TR_F32 = 2 };
// training dropout of the LoRA branch input (one (layer, step) of a call; see dropout_keep in train.cu)
struct DropoutArgs {
  unsigned long long seed = 0;
  long long step = 0;
  int layer = 0;
  unsigned thr24 = 0;   // floor(rate * 2^24): an element is kept iff the top 24 bits of its Philox word are >= thr24
  float inv = 1.f;      // 1 / (1 - rate)
};
// the adapters of one projection group: npj = 3 (in_proj: q, k, v) or 1 (out_proj: o); A[p] == nullptr: no adapter
struct LoraGroup {
  int npj = 0;
  const float* A[3] = {nullptr, nullptr, nullptr};   // [r, W] fp32, device
  const float* B[3] = {nullptr, nullptr, nullptr};   // [W, r] fp32, device
  int r[3] = {0, 0, 0};
  int j0[3] = {0, 0, 0};    // first rank column of projection p in the packed intermediate U
  int n0[3] = {0, 0, 0};    // first output row of projection p in the packed weight
  float s[3] = {0.f, 0.f, 0.f};
};
enum LoraPackKind : int { LP_DN = 0, LP_UP = 1, LP_DN_BLK = 2, LP_DN_T = 3, LP_UP_T = 4 };
cudaError_t launch_lora_pack(const LoraGroup& g, int kind, int W, int n_out, int f16, __nv_bfloat16* out, cudaStream_t s);
cudaError_t launch_dropout_fwd(const __nv_bfloat16* x, int64_t M, int W, int npj, int proj0, const DropoutArgs& d, int64_t row0,
                               int f16, __nv_bfloat16* xd, cudaStream_t s);
cudaError_t launch_dropout_bwd_add(const float* dxd, int64_t M, int W, int npj, int proj0, const DropoutArgs& d, int64_t row0,
                                   float* dx, cudaStream_t s);
cudaError_t launch_dropout_mask(const DropoutArgs& d, int proj, int64_t rows, int cols, uint8_t* out, cudaStream_t s);
cudaError_t launch_gelu_bwd(const float* dy, const __nv_bfloat16* h, int64_t n, int h_f16, __nv_bfloat16* dh, cudaStream_t s);
cudaError_t launch_ln_bwd(const float* x, const float* dy, int64_t rows, int W, const float* gamma, float* g, cudaStream_t s);
// qkv [n_views * T, 3W] 16-bit (forward), dout [n_views * T, W] fp32 -> dqkv [n_views * T, 3W] bf16; T <= 64 on the
// FFMA kernel, 65 <= T <= 256 on the tcgen05 kernel (which reports pipeline timeouts in dev_status)
cudaError_t launch_attention_bwd(const __nv_bfloat16* qkv, const float* dout, int64_t n_views, int T, int heads, int f16,
                                 __nv_bfloat16* dqkv, cudaStream_t s, int* dev_status);
// grad row 0 of every view (stride T rows) := d(loss)/d(last block output) through ln_post, proj and the normalisation
cudaError_t launch_tail_bwd(const float* x0, const float* dfeat, int64_t n_views, int W, int E, const float* g, const float* b,
                            const float* proj, int normalize, int T, float* grad, cudaStream_t s);
// acc[I, J] += X[:, :I]^T Y[:, :J] over M rows, split in at most 128 fixed row chunks summed in order (deterministic);
// partial needs 128 * I * J floats
int64_t xty_chunk_rows(int64_t M);
cudaError_t launch_xty_accumulate(const void* X, int xt, int64_t ldx, const void* Y, int yt, int64_t ldy, int64_t M, int I, int J,
                                  float* partial, float* acc, cudaStream_t s);
cudaError_t launch_extract(const float* src, int64_t lds, int r0, int c0, int rows, int cols, float scale, float* out, cudaStream_t s);
cudaError_t launch_transpose_cast(const float* src, int rows, int cols, int f16, __nv_bfloat16* dst, cudaStream_t s);

// ---- MTA + head --------------------------------------------------------------------------------
struct MtaParams {
  float lambda_y = 0.2f, lambda_q = 4.0f, th = 1e-6f, temperature = 1.0f;
  double k_frac = 0.3;
  int max_iter = 5;
};
constexpr int MTA_MAX_SETS = 4;
struct MtaSet {
  const float* feats;   // [I, V, D] unit rows, row 0 of each image = un-augmented view
  const float* text;    // [D, C]  (the orientation the reference passes: text_features.t())
  float* out_mode;      // [I, D]
  float* out_logits;    // [I, C] = 100 * mode @ text, or nullptr
};
// solver state of set 0 written at the end of the solve (jcb_mta_debug); each pointer may be nullptr
struct MtaDebug {
  float* bw;         // [I, V] bandwidths
  float* y;          // [I, V] inlierness weights of the last mode loop
  float* affinity;   // [I, V, V] softmax(100 X T / temperature) softmax(...)^T
};
// the (V, C, D) launch_mta accepts
bool mta_shape_supported(int V, int C, int D);
// bytes of global scratch launch_mta needs (0 when a problem fits in shared memory)
size_t mta_scratch_bytes(int64_t n_problems, int V, int C, int D);
// n_sets independent (feats, text) problems per image in one launch: grid = (I, n_sets)
// softmax(100 X T) runs as a bf16 x 3-limb GEMM on the tensor cores (launch_gemm) for C <= 512 and D % 64 == 0;
// otherwise the fp32 SIMT kernel
cudaError_t launch_mta(const MtaSet* sets, int n_sets, int64_t I, int V, int C, int D, const MtaParams& p,
                       float* scratch, cudaStream_t stream, int* dev_status, int num_sms,
                       const MtaDebug* debug = nullptr);

enum HeadScore : int { SCORE_LOGITS = 0, SCORE_CS = 1, SCORE_CS1 = 2, SCORE_CS2 = 3, SCORE_CS3 = 4, SCORE_CS4 = 5, SCORE_CS5 = 6, SCORE_COUNT = 7 };
// Opt a kernel in to `bytes` of dynamic shared memory on the CURRENT device.  cudaFuncSetAttribute acts on the current
// device's context, so the cache is keyed by (function, device): a process that drives several GPUs through several
// contexts gets the attribute on each of them (a per-process `static bool` would leave the second device at 48 KB).
cudaError_t ensure_dynamic_smem(const void* func, size_t bytes);
template <class F>
inline cudaError_t ensure_dynamic_smem(F* func, size_t bytes) {
  return ensure_dynamic_smem(reinterpret_cast<const void*>(func), bytes);
}

// Launch `kern` as a programmatic dependent of the kernel in front of it in `stream` (ptx.cuh griddep_wait): EVERY kernel
// launched through this MUST call griddep_wait() before its first access to global memory another kernel produced or
// still reads.  cluster_x > 1 adds a run-time cluster dimension.  Opt-in: JCB_PDL=1 (see pdl_enabled in api.cu for why it
// is not the default); otherwise these are ordinary launches and griddep_wait() is a no-op.
bool pdl_enabled();
template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              unsigned cluster_x, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  unsigned n = 0;
  if (cluster_x > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster_x;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  if (pdl_enabled()) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

struct HeadArgs {
  const float *m_pt, *m_hand, *m_zs;  // [I, D] modes
  const float *T_pt, *T_hand, *T_zs;  // [C, D] text features (unit rows)
  const float *scale1, *bias1;        // [D]
  const float *fc_w, *fc_b;           // [C, D], [C]
  int64_t I;
  int C, D;
  int rank_by;                        // HeadScore used for the top-k
  int k;                              // <= 8
  int32_t* out_topk;                  // [I, k]
  float* out_scores;                  // [I, C] (the ranked score) or nullptr
  float* out_all;                     // [I, SCORE_COUNT, C] or nullptr (tests)
  int vec_ok = 0;                     // set by launch_head: banks and fc_w are 16-byte aligned (float4 loads)
};
cudaError_t launch_head(const HeadArgs& a, cudaStream_t stream);
// Stand-alone pieces of the head (drop-in functions of the reference's Python API)
cudaError_t launch_channel_lp(const float* feats, int64_t n, int C, int D, const float* scale1, const float* bias1,
                              const float* fc_w, const float* fc_b, float* out, cudaStream_t stream);
cudaError_t launch_class_mean(const float* emb, const int* offsets, int C, int D, float* out, cudaStream_t stream);
cudaError_t launch_logit_normalize(const float* in, int64_t n, int C, float* out, cudaStream_t stream);
cudaError_t launch_cosine_topk(const float* feats, const float* text, int64_t n, int C, int D, float scale, int k,
                               int32_t* out_topk, float* out_scores, cudaStream_t stream);


// ---- TTA view generator (tta.cu) ---------------------------------------------------------------
struct TtaImage {            // == jcb_src_image
  int64_t offset;            // byte offset of the HWC uint8 image in the packed source buffer
  int32_t height, width;
};
struct TtaJob {              // == jcb_view_job
  int32_t image;
  int32_t top, left, crop_h, crop_w;
  int32_t out_h, out_w, off_y, off_x;
  int32_t filter, flip, reserved;
};
// Validates the jobs and builds the device-side plan (opaque bytes to upload); returns the bytes of
// intermediate scratch the two passes need, or SIZE_MAX with *err set.
size_t tta_plan(const TtaImage* images, int n_images, const TtaJob* jobs, int64_t n_jobs, int S,
                std::vector<uint8_t>* plan_bytes, int* kmax_h, int* kmax_v, int* max_rows, const char** err);
// out_mode 0: out = uint8 [n_jobs, 3, S, S] planar views.  out_mode 1 (bf16) / 2 (fp16): out = the views' rows of the
// conv1 patch matrix [n_jobs * (S / patch)^2, 3 * patch^2] with ToTensor's 1/255 and (apply_norm) tfm_clip applied --
// bit-identical to launch_im2col over the uint8 views.
cudaError_t launch_tta(const uint8_t* src, const void* plan_dev, int64_t n_jobs, int S, int kmax_h, int kmax_v,
                       int max_rows, uint8_t* tmp, void* out, cudaStream_t stream, int out_mode = 0, int patch = 0,
                       int apply_norm = 0);

}  // namespace jcb
