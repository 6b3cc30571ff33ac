// C-ABI of libjclip_b200.so (include/jclip_b200.h): contexts, weight packing, the image-tower schedule
// and the MTA / head entry points.  Everything here is host orchestration; the arithmetic lives in
// gemm.cu, attention.cu, rowwise.cu, mta.cu and head.cu.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <utility>
#include <string>
#include <vector>

#include "../../include/jclip_b200.h"
#include "kernels.h"

using namespace jcb;

namespace jcb {
// Programmatic dependent launch is OPT-IN (JCB_PDL=1).  Measured with it on AND an explicit early trigger
// (griddepcontrol.launch_dependents right after the wait, since removed): one image x 65 views per
// call 1.43 -> 1.39 ms (CUDA graphs) / 1.59 -> 1.43 (no graphs), the batched step +0.5 %, all GPU tests green -- but two
// FULL-SIZE pipeline calls adjacent in the stream (call k's head kernel directly followed by call k + 1's im2col while
// call k is still running) never finish: tools/pdl_first_calls_probe.py, profiles/r02_pdl_hang_probes.log (one GPU, no
// NCCL).  Without the early trigger (dependents are released by the exit of the primary's CTAs) the same probe
// finishes; that form was checked by the probe and a test subset only, hence still not the default.
bool pdl_enabled() {
  static const bool on = [] { const char* e = getenv("JCB_PDL"); return e && e[0] == '1'; }();
  return on;
}
cudaError_t ensure_dynamic_smem(const void* func, size_t bytes) {
  if (bytes <= 48 * 1024) return cudaSuccess;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, size_t> granted;
  std::lock_guard<std::mutex> lock(mu);
  size_t& cur = granted[std::make_pair(func, dev)];
  if (bytes <= cur) return cudaSuccess;
  e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(bytes));
  if (e == cudaSuccess) cur = bytes;
  return e;
}
}  // namespace jcb

// ------------------------------------------------------------------------------------------------
struct PipelineGraph;
struct jcb_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t copy_done[2] = {nullptr, nullptr};
  cudaEvent_t compute_done[2] = {nullptr, nullptr};
  int num_sms = 0, cc_major = 0, cc_minor = 0;
  int* dev_status = nullptr;
  int64_t chunk_views = 16384;       // upper bound of views per pass through the tower (device-resident input)
  int64_t host_chunk_views = 2048;   // same for host input: smaller, so copies of chunk i+1 overlap compute of chunk i
  void* ws = nullptr;
  size_t ws_bytes = 0;
  void* stage[2] = {nullptr, nullptr};  // device staging for host images
  size_t stage_bytes = 0;
  int64_t stage_seq = 0;             // staging uses so far (buffer = seq & 1): persists ACROSS calls, so a call that
  bool stage_recorded[2] = {false, false};  // starts while the previous one still computes cannot overwrite its input
  // asynchronous submissions (jcb_pipeline_submit / jcb_pipeline_wait)
  cudaEvent_t ticket_done[JCB_MAX_INFLIGHT] = {nullptr, nullptr, nullptr, nullptr};
  int* ticket_status = nullptr;      // pinned host, [JCB_MAX_INFLIGHT]: device status word copied behind each submission
  int64_t next_ticket = 0, waited_ticket = 0;
  // jcb_tta_views / jcb_tta_patches: their own scratch (plan + horizontal-pass intermediate), so that a view batch can be
  // generated on a second stream WHILE the towers use `ws` for the previous batch
  void* tta_ws = nullptr;
  size_t tta_ws_bytes = 0;
  cudaStream_t tta_last_stream = nullptr;   // the stream the generator last ran on, and the end of that run: a call on
  cudaEvent_t tta_done = nullptr;           // ANOTHER stream waits for it before it overwrites the shared scratch
  // pinned, double-buffered staging of the per-view plan (no stream synchronisation in the call)
  void* tta_plan_host[2] = {nullptr, nullptr};
  size_t tta_plan_bytes[2] = {0, 0};
  cudaEvent_t tta_plan_copied[2] = {nullptr, nullptr};
  int tta_turn = 0;
  int cls_only_last = 0;             // opt-in: last block of the image tower on the class-token rows only (see tower_blocks)
  bool overlapped = false;           // this submission was enqueued behind an un-waited one: its first upload is hidden
  int64_t launches = 0;
  int operand_f16 = 1;               // 16-bit operand type towers are packed with: 1 = fp16 (default), 0 = bf16
  int lora_applied = 0;              // how towers packed from now on carry their LoRA adapters: 0 = merged into the
                                     // weights (default), 1 = applied as low-rank GEMMs (jcb_ctx_set_lora_mode)
  int32_t* slot_dev = nullptr;       // per-view LoRA slots of the current call (jcb_*_slots), grow-only
  int64_t slot_cap = 0;
  char err[512] = {0};
  // CUDA graphs of whole small pipelines (see PipelineGraph below)
  int graphs_on = 1;
  int64_t graph_max_views = 1024;
  uint64_t ws_gen = 0;               // bumped whenever `ws` is re-allocated: graphs hold pointers into it
  std::vector<struct PipelineGraph*> graphs;
  int64_t graph_captures = 0, graph_launches = 0, graph_failures = 0;
  cudaStream_t capture_stream = nullptr;   // captures run here: the caller's stream may be the legacy default stream,
                                           // which cannot be captured; the graph is LAUNCHED on the caller's stream
  // per-kernel-class CUDA-event profile (jcb_ctx_profile): event pairs recorded on the launch stream
  bool prof_on = false;
  std::vector<cudaEvent_t> prof_ev;           // 2 * PROF_PAIRS events, created on first use
  std::vector<int> prof_cls;                  // class of each recorded pair
  double prof_ms[JCB_KC_COUNT] = {0};
  int64_t prof_n[JCB_KC_COUNT] = {0};         // launches seen (recorded or not)
  int64_t prof_timed[JCB_KC_COUNT] = {0};     // launches with an event pair
  double prof_flops[JCB_KC_COUNT] = {0};
  double prof_bytes[JCB_KC_COUNT] = {0};
};

void graphs_clear_fwd(jcb_ctx* ctx);   // defined next to the pipeline graphs below

namespace {

int fail(jcb_ctx* ctx, int code, const char* fmt, ...) {
  if (ctx) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(ctx->err, sizeof(ctx->err), fmt, ap);
    va_end(ap);
  }
  return code;
}

#define CUDA_TRY(ctx, expr)                                                                          \
  do {                                                                                               \
    cudaError_t _e = (expr);                                                                         \
    if (_e != cudaSuccess)                                                                           \
      return fail((ctx), _e == cudaErrorInvalidValue ? JCB_E_INVALID : JCB_E_CUDA, "%s failed: %s (%s:%d)", \
                  #expr, cudaGetErrorString(_e), __FILE__, __LINE__);                                \
  } while (0)

#define LAUNCH(ctx, expr)    \
  do {                       \
    CUDA_TRY((ctx), (expr)); \
    ++(ctx)->launches;       \
  } while (0)

constexpr size_t PROF_PAIRS = 32768;

// Launch with an optional CUDA-event pair around it (same stream), attributed to kernel class `cls`
// with its algorithmic FLOPs / bytes.  Costs two cudaEventRecord per launch while profiling is on.
#define LAUNCH_P(ctx, cls, flops_, bytes_, expr)                                              \
  do {                                                                                        \
    jcb_ctx* _c = (ctx);                                                                      \
    long _slot = -1;                                                                          \
    if (_c->prof_on) {                                                                        \
      _c->prof_n[(cls)] += 1;                                                                 \
      _c->prof_flops[(cls)] += static_cast<double>(flops_);                                   \
      _c->prof_bytes[(cls)] += static_cast<double>(bytes_);                                   \
      if (_c->prof_cls.size() < PROF_PAIRS) {                                                 \
        _slot = static_cast<long>(_c->prof_cls.size());                                       \
        _c->prof_cls.push_back((cls));                                                        \
        cudaEventRecord(_c->prof_ev[2 * _slot], _c->stream);                                  \
      }                                                                                       \
    }                                                                                         \
    LAUNCH(_c, (expr));                                                                       \
    if (_slot >= 0) cudaEventRecord(_c->prof_ev[2 * _slot + 1], _c->stream);                  \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// Grow-only workspace.  Growth synchronises the stream (buffers may be in use); steady state never does.
int ws_reserve(jcb_ctx* ctx, size_t bytes) {
  if (bytes <= ctx->ws_bytes) return JCB_OK;
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (ctx->ws) cudaFree(ctx->ws);
  ctx->ws = nullptr;
  ctx->ws_bytes = 0;
  ++ctx->ws_gen;
  cudaError_t e = cudaMalloc(&ctx->ws, bytes);
  if (e != cudaSuccess) return fail(ctx, JCB_E_NOMEM, "cudaMalloc(%zu) for the workspace failed: %s", bytes, cudaGetErrorString(e));
  ctx->ws_bytes = bytes;
  return JCB_OK;
}
int stage_reserve(jcb_ctx* ctx, size_t bytes) {
  if (bytes <= ctx->stage_bytes) return JCB_OK;
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy_stream));
  for (int i = 0; i < 2; ++i) {
    if (ctx->stage[i]) cudaFree(ctx->stage[i]);
    ctx->stage[i] = nullptr;
  }
  ctx->stage_bytes = 0;
  for (int i = 0; i < 2; ++i) {
    cudaError_t e = cudaMalloc(&ctx->stage[i], bytes);
    if (e != cudaSuccess) return fail(ctx, JCB_E_NOMEM, "cudaMalloc(%zu) for image staging failed: %s", bytes, cudaGetErrorString(e));
  }
  ctx->stage_bytes = bytes;
  ctx->stage_recorded[0] = ctx->stage_recorded[1] = false;
  return JCB_OK;
}

struct Bump {
  uint8_t* base;
  size_t off = 0;
  explicit Bump(void* p) : base(static_cast<uint8_t*>(p)) {}
  template <typename T>
  T* take(size_t n) {
    T* p = reinterpret_cast<T*>(base + off);
    off += align_up(n * sizeof(T));
    return p;
  }
};

size_t img_elem_bytes(int dt) { return dt == JCB_IMG_F32 ? 4 : dt == JCB_IMG_U8 ? 1 : 2; }
bool is_patches(int dt) { return dt == JCB_IMG_PATCHES_BF16 || dt == JCB_IMG_PATCHES_F16; }

}  // namespace

// ------------------------------------------------------------------------------------------------
struct LoraAdapter {
  std::vector<float> A, B;
  int r = 0;
  float scaling = 0.f;
};

struct LayerDev {
  __nv_bfloat16 *in_w = nullptr, *out_w = nullptr, *fc_w = nullptr, *proj_w = nullptr;
  float *in_b = nullptr, *out_b = nullptr, *fc_b = nullptr, *proj_b = nullptr;
  float *ln1_g = nullptr, *ln1_b = nullptr, *ln2_g = nullptr, *ln2_b = nullptr;
  // LayerNorm folded into the consuming GEMM: gamma-scaled weights, their column sums S and the constants c
  __nv_bfloat16 *in_wf = nullptr, *fc_wf = nullptr;
  float *in_S = nullptr, *in_c = nullptr, *fc_S = nullptr, *fc_c = nullptr;
  // LoRA applied (jcb_ctx_set_lora_mode): the adapters of the packed in_proj / of out_proj side by side,
  // down = [A_q; A_k; A_v; 0] as [LORA_U_COLS, W] and up = [s B_q | s B_k | s B_v | 0] in the rows of its projection as
  // [3W, LORA_K2] ([W, LORA_K2] for out_proj); nullptr when the layer has no adapter there
  // LoRA slots (jcb_vit_set_lora_slot): the same layout once per slot -- slot g's down rows are rows [64 g, 64 g + 64)
  // of the down matrix ([lora_u_cols(G), W]), its up matrix is column block g of the up matrix ([3W | W, 64 G]).
  __nv_bfloat16 *lin_dn = nullptr, *lin_up = nullptr, *lout_dn = nullptr, *lout_up = nullptr;
  uint32_t lin_slots = 0, lout_slots = 0;   // slots with an adapter on in_proj / out_proj of this layer
};
// columns of the low-rank intermediate U = x [A_q; A_k; A_v]^T (the GEMM kernel's minimum N) and the k extent the
// second operand pair of the projection GEMM reads of it (one 64-wide k-block: the ranks of q, k, v together <= 64)
constexpr int LORA_U_COLS = 128;
constexpr int LORA_K2 = 64;
// U of a tower with G slots: one 64-column block per slot, rounded up to the GEMM's N granularity (G = 1: LORA_U_COLS)
int lora_u_cols(int G) { return (LORA_K2 * G + 127) / 128 * 128; }

// What the image tower and the text tower share: a stack of pre-LN transformer blocks with packed-QKV
// attention (+ LoRA adapters merged at pack time), the fp32 staging of the reference state dict and the
// device arena the packed weights live in.
struct TowerBase {
  jcb_ctx* ctx = nullptr;
  int f16 = 0;                                       // operand type the device weights were packed with (jcb_*_finalize)
  int lora_applied = 0;                              // LoRA mode they were packed with
  uint64_t gen = 0;                                  // bumped by every finalize (captured graphs key on it)
  int W = 0, L = 0, heads = 0, tokens = 0;           // width, blocks, heads (W / 64), tokens per sequence
  std::string prefix;                                // state-dict prefix of the blocks
  std::map<std::string, std::vector<float>> host;   // fp32 staging by reference key name
  std::map<std::string, int64_t> expected;          // key -> numel
  std::vector<std::map<int, LoraAdapter>> lora = std::vector<std::map<int, LoraAdapter>>(1);   // [slot][layer * 4 + proj]
  int lora_slots = 1;                               // slots the weights were packed with (the last finalize)
  bool finalized = false;
  void* arena = nullptr;                            // device weights
  size_t arena_bytes = 0;
  std::vector<LayerDev> layers;
};

struct jcb_vit : TowerBase {
  jcb_vit_config cfg{};
  int grid = 0, kpatch = 0;
  __nv_bfloat16* conv_w = nullptr;
  float *vpt = nullptr;
  float *cls = nullptr, *pos = nullptr, *ln_pre_g = nullptr, *ln_pre_b = nullptr, *ln_post_g = nullptr,
        *ln_post_b = nullptr, *proj = nullptr;
};

struct jcb_text : TowerBase {
  jcb_text_config cfg{};
  float *tok_emb = nullptr, *pos = nullptr, *ln_final_g = nullptr, *ln_final_b = nullptr, *text_projection = nullptr;
};

namespace {

int tower_set_param(TowerBase* t, const char* name, const float* data, int64_t numel);
int tower_set_lora(TowerBase* t, int layer, int proj, const float* A, const float* B, int r, float scaling, int slot = 0);

std::string blk(const TowerBase* t, int i, const char* tail) { return t->prefix + std::to_string(i) + "." + tail; }

void expect_blocks(TowerBase* t) {
  const int64_t W = t->W;
  auto& e = t->expected;
  for (int i = 0; i < t->L; ++i) {
    e[blk(t, i, "attn.in_proj_weight")] = 3 * W * W;
    e[blk(t, i, "attn.in_proj_bias")] = 3 * W;
    e[blk(t, i, "attn.out_proj.weight")] = W * W;
    e[blk(t, i, "attn.out_proj.bias")] = W;
    e[blk(t, i, "ln_1.weight")] = W;
    e[blk(t, i, "ln_1.bias")] = W;
    e[blk(t, i, "ln_2.weight")] = W;
    e[blk(t, i, "ln_2.bias")] = W;
    e[blk(t, i, "mlp.c_fc.weight")] = 4 * W * W;
    e[blk(t, i, "mlp.c_fc.bias")] = 4 * W;
    e[blk(t, i, "mlp.c_proj.weight")] = 4 * W * W;
    e[blk(t, i, "mlp.c_proj.bias")] = W;
  }
}

void build_expected(jcb_vit* v) {
  const int64_t W = v->cfg.width, P = v->cfg.patch, E = v->cfg.embed_dim, T = v->tokens;
  auto& e = v->expected;
  e["visual.conv1.weight"] = W * 3 * P * P;
  e["visual.class_embedding"] = W;
  e["visual.positional_embedding"] = (T - v->cfg.vpt_tokens) * W;
  if (v->cfg.vpt_tokens > 0) e["visual.VPT"] = static_cast<int64_t>(v->cfg.vpt_tokens) * W;
  e["visual.ln_pre.weight"] = W;
  e["visual.ln_pre.bias"] = W;
  e["visual.ln_post.weight"] = W;
  e["visual.ln_post.bias"] = W;
  e["visual.proj"] = W * E;
  expect_blocks(v);
}

// workspace layout for one chunk of n views
struct TowerWs {
  __nv_bfloat16* big;     // patches [n*G*G, 3PP]  /  MLP hidden [n*T, 4W]  (never live together)
  float* tokens;          // residual stream [n*T, W] fp32
  __nv_bfloat16* ln_out;  // [n*T, W]
  __nv_bfloat16* qkv;     // [n*T, 3W]
  __nv_bfloat16* attn;    // [n*T, W]
  __nv_bfloat16* lora_u;  // [n*T, LORA_U_COLS]  LoRA applied: x A^T of the projection about to run
  // LayerNorm fold: per-row partial (sum, sum of squares) [n*T, W/256, 2] of the centred 16-bit copy of the residual
  // stream and the per-row shift [n*T] it was centred by; two of each, because the producer GEMM of LayerNorm point
  // i + 1 reads the statistics of point i while its other tiles already write those of point i + 1
  float* stats[2];
  float* shift[2];
};
size_t tower_ws_bytes_dims(size_t W, size_t T, size_t GG, size_t KP, int64_t n, size_t u_cols = LORA_U_COLS) {
  const size_t big = std::max(n * GG * KP, n * T * 4 * W) * 2;
  return align_up(big) + align_up(n * T * W * 4) + align_up(n * T * W * 2) + align_up(n * T * 3 * W * 2) +
         align_up(n * T * W * 2) + align_up(n * T * u_cols * 2) + 2 * align_up(n * T * ((W + 255) / 256) * 8) +
         2 * align_up(n * T * 4);
}
size_t tower_ws_bytes(const jcb_vit* v, int64_t n) {
  return tower_ws_bytes_dims(v->W, v->tokens, static_cast<size_t>(v->grid) * v->grid, v->kpatch, n, lora_u_cols(v->lora_slots));
}
TowerWs tower_ws_carve_dims(size_t W, size_t T, size_t GG, size_t KP, int64_t n, Bump& b, size_t u_cols = LORA_U_COLS) {
  TowerWs w;
  w.big = b.take<__nv_bfloat16>(std::max(n * GG * KP, n * T * 4 * W));
  w.tokens = b.take<float>(n * T * W);
  w.ln_out = b.take<__nv_bfloat16>(n * T * W);
  w.qkv = b.take<__nv_bfloat16>(n * T * 3 * W);
  w.attn = b.take<__nv_bfloat16>(n * T * W);
  w.lora_u = b.take<__nv_bfloat16>(n * T * u_cols);
  for (int i = 0; i < 2; ++i) w.stats[i] = b.take<float>(n * T * ((W + 255) / 256) * 2);
  for (int i = 0; i < 2; ++i) w.shift[i] = b.take<float>(n * T);
  return w;
}
TowerWs tower_ws_carve(const jcb_vit* v, int64_t n, Bump& b) {
  return tower_ws_carve_dims(v->W, v->tokens, static_cast<size_t>(v->grid) * v->grid, v->kpatch, n, b, lora_u_cols(v->lora_slots));
}

// LayerNorm-fold plumbing of one GEMM launch: the consumer (EPI_LNFOLD_*) reads `stats` / `colsum`; the producer
// (EPI_RESID_LNPREP_*) writes `stats` / `shift_out` / the centred copy `out2` and reads the previous point's
// `stats_in` / `shift_in` (row r of this GEMM = row r * in_stride there).
struct LnArgs {
  float* stats = nullptr;
  int slots = 0;
  const float* colsum = nullptr;
  void* out2 = nullptr;
  const float* stats_in = nullptr;
  const float* shift_in = nullptr;
  float* shift_out = nullptr;
  int64_t in_stride = 1;
  // second operand pair of the GEMM (LoRA applied): out = A B^T + A2 B2^T
  const __nv_bfloat16* A2 = nullptr;
  const __nv_bfloat16* B2 = nullptr;
  int K2 = 0;
  int64_t lda2 = 0, ldb2 = 0;
  // LoRA slots (GemmArgs::slot_of_view)
  const int* slot_of_view = nullptr;
  int slot_rows = 0;
  uint32_t slot_live = 0;
};

int run_gemm(jcb_ctx* ctx, int cls, int f16, const __nv_bfloat16* A, const __nv_bfloat16* B, int M, int N, int K,
             const float* bias, int epi, void* out, int64_t ldo, const LnArgs& ln = LnArgs()) {
  GemmArgs g;
  g.stats = ln.stats; g.stats_slots = ln.slots; g.colsum = ln.colsum; g.out2 = ln.out2; g.ldo2 = N;   // out2 / stats are dense
  g.stats_in = ln.stats_in; g.shift_in = ln.shift_in; g.shift_out = ln.shift_out; g.stats_in_row_stride = ln.in_stride;
  g.A = A; g.B = B; g.lda = K; g.ldb = K; g.M = M; g.N = N; g.K = K; g.f16 = f16;
  g.A2 = ln.A2; g.B2 = ln.B2; g.K2 = ln.K2; g.lda2 = ln.lda2; g.ldb2 = ln.ldb2;
  g.slot_of_view = ln.slot_of_view; g.slot_rows = ln.slot_rows; g.slot_live = ln.slot_live;
  g.bias = bias; g.epilogue = epi; g.out = out; g.ldo = ldo;
  // algorithmic bytes: A + B read once, C written once (read-modify-write for the residual epilogue)
  const bool lnprep = epi == EPI_RESID_LNPREP_SHORT || epi == EPI_RESID_LNPREP_LONG;
  const double out_b = (epi == EPI_BIAS_BF16 || epi == EPI_BIAS_GELU_BF16 || epi == EPI_LNFOLD_BF16 || epi == EPI_LNFOLD_GELU_BF16)
                           ? 2.0 : (epi == EPI_BIAS_RESID_F32 ? 8.0 : (lnprep ? 10.0 : 4.0));
  // with LoRA slots a row needs one slot's k-block (projection) / column block (down-projection) of the K2 / N extent
  const int K2a = ln.slot_of_view && ln.K2 > 0 ? LORA_K2 : ln.K2;
  const int Na = ln.slot_of_view && ln.K2 == 0 ? LORA_K2 : N;
  const double bytes = 2.0 * M * (K + K2a) + 2.0 * N * (K + ln.K2) + out_b * M * N;
  LAUNCH_P(ctx, cls, 2.0 * M * Na * (K + K2a), bytes, launch_gemm(g, ctx->dev_status, ctx->num_sms, ctx->stream));
  return JCB_OK;
}

// L pre-LN blocks on `n` sequences of t->tokens tokens: w.ln_out holds ln_1 of block 0 on entry, w.tokens the
// fp32 residual stream; on exit w.tokens is the output of the last block (reference jclip/model.py:59-62).
// slot_dev (LoRA applied, towers with several slots): the slot of each of the n sequences, on the device; nullptr = slot 0.
int tower_blocks(TowerBase* t, int64_t n, const TowerWs& w, int causal, bool cls_row0 = false, const int* slot_dev = nullptr) {
  jcb_ctx* ctx = t->ctx;
  cudaStream_t s = ctx->stream;
  const int W = t->W, T = t->tokens, f16 = t->f16;
  const int M = static_cast<int>(n * T);
  const double MW = static_cast<double>(M) * W;
  int rc;
  if (t->layers[0].in_wf != nullptr) {
    // Both LayerNorms folded into the GEMMs (towers packed with merged or no LoRA): w.ln_out holds the CENTRED 16-bit
    // copy of the residual stream (x - shift[row]), w.stats[cur] its per-row partial sums and w.shift[cur] the shift
    // (written by the embed kernel for block 0, then by the residual epilogue of the producing GEMM), and no
    // stand-alone pass reads the fp32 residual stream.
    //   ln_1 (c_proj of block l-1 -> QKV of block l): c_proj's 48 k-blocks per tile hide the heavier epilogue;
    //       measured net gain (-1.5 ms / step).
    //   ln_2 (out_proj -> c_fc): out_proj is HBM-bound and pays 12 instead of 10 bytes per element (6.9 -> 9.3 ms),
    //       c_fc's epilogue gets one FMA heavier (+0.3 ms); the 4.0 ms ln_2 pass disappears.  A net loss while c_fc
    //       ran a 4-stage operand ring (its heavier epilogue then stalled an already starved main loop); with 5 stages
    //       a net gain: 75.7-76.0 vs 77.2-78.7 ms / step with ln_1 folded alone (same B200).
    const int slots = (W + 255) / 256;
    const bool cls_only = cls_row0 && ctx->cls_only_last && !causal && T <= 64;
    int cur = 0;   // which of w.stats / w.shift describes the copy in w.ln_out
    auto consumer = [&]() { LnArgs a; a.stats = w.stats[cur]; a.slots = slots; return a; };
    auto producer = [&](int64_t in_stride) {
      LnArgs a;
      a.stats = w.stats[cur ^ 1]; a.slots = slots; a.out2 = w.ln_out; a.shift_out = w.shift[cur ^ 1];
      a.stats_in = w.stats[cur]; a.shift_in = w.shift[cur]; a.in_stride = in_stride;
      cur ^= 1;
      return a;
    };
    for (int l = 0; l < t->L; ++l) {
      const LayerDev& L = t->layers[l];
      {
        LnArgs a = consumer();
        a.colsum = L.in_S;
        if ((rc = run_gemm(ctx, JCB_KC_GEMM_QKV, f16, w.ln_out, L.in_wf, M, 3 * W, W, L.in_c, EPI_LNFOLD_BF16, w.qkv, 3 * W, a))) return rc;
      }
      if (cls_only && l + 1 == t->L) {
        // Opt-in (jcb_ctx_set_cls_only_last_block, default off): the caller of the image tower reads nothing but
        // ln_post(x[:, 0, :]) @ proj (jclip/model.py:121-124), so after the last block's K and V only the class-token
        // row of every view is live.  Attention, out_proj, ln_2, c_fc and c_proj of that block run on n rows instead
        // of n * T: the same GEMM kernels with M = n, the residual stream addressed as [n, T * W] (leading dimension
        // T * W: row v = class token of view v), the 16-bit copy / row statistics / MLP hidden dense.  Per output
        // element the GEMM arithmetic is identical (same k order); the 0.53 GFLOP per view it skips (6 % of the
        // tower) were never part of the result.  Not the default: bench.py's headline numbers run the full block.
        const int Mc = static_cast<int>(n);
        LAUNCH_P(ctx, JCB_KC_ATTENTION, 4.0 * n * t->heads * T * 64, static_cast<double>(n) * T * W * 4 + static_cast<double>(n) * W * 4,
                 launch_attention_cls(w.qkv, n, T, t->heads, w.attn, s, f16));
        {
          LnArgs a = producer(T);   // row v of this GEMM = token row v * T of the previous LayerNorm point
          if ((rc = run_gemm(ctx, JCB_KC_GEMM_OUT, f16, w.attn, L.out_w, Mc, W, W, L.out_b, EPI_RESID_LNPREP_SHORT, w.tokens,
                             static_cast<int64_t>(T) * W, a))) return rc;
        }
        {
          LnArgs a = consumer();
          a.colsum = L.fc_S;
          if ((rc = run_gemm(ctx, JCB_KC_GEMM_FC1, f16, w.ln_out, L.fc_wf, Mc, 4 * W, W, L.fc_c, EPI_LNFOLD_GELU_BF16, w.big, 4 * W, a))) return rc;
        }
        if ((rc = run_gemm(ctx, JCB_KC_GEMM_FC2, f16, w.big, L.proj_w, Mc, W, 4 * W, L.proj_b, EPI_BIAS_RESID_F32, w.tokens,
                           static_cast<int64_t>(T) * W))) return rc;
        break;
      }
      LAUNCH_P(ctx, JCB_KC_ATTENTION, 4.0 * n * t->heads * T * T * 64, MW * (6 + 2),
               launch_attention(w.qkv, n, T, t->heads, w.attn, s, causal, ctx->dev_status, ctx->num_sms, f16));
      {
        LnArgs a = producer(1);
        if ((rc = run_gemm(ctx, JCB_KC_GEMM_OUT, f16, w.attn, L.out_w, M, W, W, L.out_b, EPI_RESID_LNPREP_SHORT, w.tokens, W, a))) return rc;
      }
      {
        LnArgs a = consumer();
        a.colsum = L.fc_S;
        if ((rc = run_gemm(ctx, JCB_KC_GEMM_FC1, f16, w.ln_out, L.fc_wf, M, 4 * W, W, L.fc_c, EPI_LNFOLD_GELU_BF16, w.big, 4 * W, a))) return rc;
      }
      if (l + 1 < t->L) {
        LnArgs a = producer(1);
        if ((rc = run_gemm(ctx, JCB_KC_GEMM_FC2, f16, w.big, L.proj_w, M, W, 4 * W, L.proj_b, EPI_RESID_LNPREP_LONG, w.tokens, W, a))) return rc;
      } else if ((rc = run_gemm(ctx, JCB_KC_GEMM_FC2, f16, w.big, L.proj_w, M, W, 4 * W, L.proj_b, EPI_BIAS_RESID_F32, w.tokens, W))) {
        return rc;
      }
    }
    return JCB_OK;
  }
  // LoRA applied (jcb_ctx_set_lora_mode; the form the reference evaluates, test.py:388-398: W x + b + s B (A x)):
  // U = x [A_q; A_k; A_v]^T as one narrow GEMM, then the projection GEMM accumulates U (s B)^T into the same TMEM
  // tile through its second operand pair -- the base weights stay un-merged, an adapter swap re-packs 2 x r rows.
  // Several slots, chosen per sequence (slot_dev): U holds one 64-column block per slot, zero outside the row's own
  // slot, and the projection GEMM multiplies, per 256-row tile, the k-blocks of the slots present in it (gemm.cu SLOTS).
  // Without slot_dev a multi-slot tower runs slot 0 alone: its 64 columns of U and k-block 0 of the up matrix.
  const int G = t->lora_slots;
  const int u_cols = lora_u_cols(G);
  auto lora_pair = [&](const __nv_bfloat16* x, const __nv_bfloat16* dn, const __nv_bfloat16* up, uint32_t live, LnArgs* a) -> int {
    if (!slot_dev) {
      if (!(live & 1u)) return JCB_OK;
      int rc2 = run_gemm(ctx, JCB_KC_GEMM_LORA, f16, x, dn, M, LORA_U_COLS, W, nullptr, EPI_BIAS_BF16, w.lora_u, LORA_U_COLS);
      if (rc2) return rc2;
      a->A2 = w.lora_u; a->B2 = up; a->K2 = LORA_K2; a->lda2 = LORA_U_COLS; a->ldb2 = static_cast<int64_t>(LORA_K2) * G;
      return JCB_OK;
    }
    if (!live) return JCB_OK;
    LnArgs d;
    d.slot_of_view = slot_dev; d.slot_rows = T; d.slot_live = live;
    int rc2 = run_gemm(ctx, JCB_KC_GEMM_LORA, f16, x, dn, M, u_cols, W, nullptr, EPI_BIAS_BF16, w.lora_u, u_cols, d);
    if (rc2) return rc2;
    a->A2 = w.lora_u; a->B2 = up; a->K2 = LORA_K2 * G; a->lda2 = u_cols; a->ldb2 = LORA_K2 * G;
    a->slot_of_view = slot_dev; a->slot_rows = T; a->slot_live = live;
    return JCB_OK;
  };
  for (int l = 0; l < t->L; ++l) {
    const LayerDev& L = t->layers[l];
    {
      LnArgs a;
      if ((rc = lora_pair(w.ln_out, L.lin_dn, L.lin_up, L.lin_slots, &a))) return rc;
      if ((rc = run_gemm(ctx, JCB_KC_GEMM_QKV, f16, w.ln_out, L.in_w, M, 3 * W, W, L.in_b, EPI_BIAS_BF16, w.qkv, 3 * W, a))) return rc;
    }
    LAUNCH_P(ctx, JCB_KC_ATTENTION, 4.0 * n * t->heads * T * T * 64, MW * (6 + 2),
             launch_attention(w.qkv, n, T, t->heads, w.attn, s, causal, ctx->dev_status, ctx->num_sms, f16));
    {
      LnArgs a;
      if ((rc = lora_pair(w.attn, L.lout_dn, L.lout_up, L.lout_slots, &a))) return rc;
      if ((rc = run_gemm(ctx, JCB_KC_GEMM_OUT, f16, w.attn, L.out_w, M, W, W, L.out_b, EPI_BIAS_RESID_F32, w.tokens, W, a))) return rc;
    }
    LAUNCH_P(ctx, JCB_KC_LAYERNORM, 0, MW * (4 + 2), launch_layernorm(w.tokens, M, W, L.ln2_g, L.ln2_b, w.ln_out, s, f16));
    if ((rc = run_gemm(ctx, JCB_KC_GEMM_FC1, f16, w.ln_out, L.fc_w, M, 4 * W, W, L.fc_b, EPI_BIAS_GELU_BF16, w.big, 4 * W))) return rc;
    if ((rc = run_gemm(ctx, JCB_KC_GEMM_FC2, f16, w.big, L.proj_w, M, W, 4 * W, L.proj_b, EPI_BIAS_RESID_F32, w.tokens, W))) return rc;
    if (l + 1 < t->L) {
      const LayerDev& Nx = t->layers[l + 1];
      LAUNCH_P(ctx, JCB_KC_LAYERNORM, 0, MW * (4 + 2), launch_layernorm(w.tokens, M, W, Nx.ln1_g, Nx.ln1_b, w.ln_out, s, f16));
    }
  }
  return JCB_OK;
}

// The image tower on `n` views resident on the device.  Schedule = VisionTransformer.execute
// (reference jclip/model.py:104-126) with every elementwise op fused into a neighbouring kernel.
int tower_forward(jcb_vit* v, const void* images, int dt, int64_t n, int apply_norm, const TowerWs& w,
                  const int* slot_dev = nullptr) {
  jcb_ctx* ctx = v->ctx;
  cudaStream_t s = ctx->stream;
  const int W = v->cfg.width, T = v->tokens, GG = v->grid * v->grid, KP = v->kpatch;
  const int M = static_cast<int>(n * T);
  // conv1 as im2col + GEMM; epilogue scatters to token rows 1..T-1 and adds the positional embedding
  const double MW = static_cast<double>(M) * W;  // elements of one [tokens, width] tensor
  const double img_b = static_cast<double>(n) * 3 * v->cfg.resolution * v->cfg.resolution;
  // input already is the patch matrix (jcb_tta_patches: view generator fused with the front end): no im2col pass
  const __nv_bfloat16* patches = is_patches(dt) ? static_cast<const __nv_bfloat16*>(images) : w.big;
  if (!is_patches(dt))
    LAUNCH_P(ctx, JCB_KC_IM2COL, 0, img_b * img_elem_bytes(dt) + img_b * 2,
             launch_im2col(images, dt, n, v->cfg.resolution, v->cfg.patch, apply_norm, w.big, s, v->f16));
  // conv1 output as a dense [n * GG, W] fp32 matrix through the TMA-store epilogue, parked in the (not yet used)
  // QKV buffer; the embed kernel moves each row to its token slot while adding the positional embedding.  The
  // scatter epilogue (EPI_PATCH_F32: direct stores, one row per thread) ran the GEMM at 0.81-1.0 of the others' rate.
  float* patch_out = reinterpret_cast<float*>(w.qkv);
  int rc = run_gemm(ctx, JCB_KC_GEMM_PATCH, v->f16, patches, v->conv_w, static_cast<int>(n * GG), W, KP, nullptr, EPI_F32, patch_out, W);
  if (rc) return rc;
  // class token + positional embedding + ln_pre (residual stream) + layer 0's ln_1
  LAUNCH_P(ctx, JCB_KC_EMBED_LN, 0, MW * (4 + 4 + 2), launch_embed_ln(w.tokens, n, T, W, v->cls, v->pos, v->vpt, v->cfg.vpt_tokens, v->ln_pre_g, v->ln_pre_b, v->layers[0].ln1_g,
                              v->layers[0].ln1_b, w.ln_out, s, v->layers[0].in_wf ? w.stats[0] : nullptr, (W + 255) / 256,
                              patch_out, w.shift[0], v->f16));
  return tower_blocks(v, n, w, 0, /*cls_row0=*/true, slot_dev);   // the tail reads token row 0 only
}

// Views per pass through the tower.  Host input of a blocking call is cut into small passes so that the upload of
// pass i+1 hides behind the compute of pass i; a submission queued behind a running one (jcb_pipeline_submit) hides
// its WHOLE upload behind that one's compute and keeps the large, more efficient passes of device-resident input.
// The bounds count views of a tower of up to 64 tokens; a longer tower gets proportionally fewer views per pass, so
// that a pass holds about the same number of token rows (and workspace) whatever the patch size.
int64_t token_rows_bound(int64_t bound, int T) { return std::max<int64_t>(1, std::min(bound, bound * 64 / T)); }

int64_t views_bound(const jcb_ctx* ctx, bool on_host, int T) {
  return token_rows_bound(
      (on_host && !ctx->overlapped) ? std::min(ctx->host_chunk_views, ctx->chunk_views) : ctx->chunk_views, T);
}

int64_t balanced_chunk(int64_t n, int64_t bound) {
  if (n <= bound) return n;
  const int64_t passes = (n + bound - 1) / bound;
  return (n + passes - 1) / passes;
}

int check_vit(jcb_vit* v) {
  if (!v) return JCB_E_INVALID;
  if (!v->finalized) return fail(v->ctx, JCB_E_STATE, "jcb_vit_finalize has not been called");
  return JCB_OK;
}

// encode `n` views (device-resident when !on_host) into out_dev [n, E]; ws_extra bytes at the start of
// the workspace are reserved for the caller.  slot_dev: the LoRA slot of each view on the device (slots_prepare), or nullptr.
int encode_views(jcb_vit* v, const void* images, int dt, bool on_host, int64_t n, int apply_norm, int normalize,
                 float* out_dev, size_t ws_extra, const int* slot_dev = nullptr) {
  jcb_ctx* ctx = v->ctx;
  if (dt < 0 || dt > JCB_IMG_PATCHES_F16) return fail(ctx, JCB_E_INVALID, "unknown image dtype %d", dt);
  if (is_patches(dt)) {
    if (on_host) return fail(ctx, JCB_E_INVALID, "patch-matrix input must be device-resident");
    if ((dt == JCB_IMG_PATCHES_F16) != (v->f16 != 0))
      return fail(ctx, JCB_E_INVALID, "patch matrix is %s but the tower was packed with %s operands",
                  dt == JCB_IMG_PATCHES_F16 ? "fp16" : "bf16", v->f16 ? "fp16" : "bf16");
  }
  if (n < 0) return fail(ctx, JCB_E_INVALID, "negative view count");
  if (n == 0) return JCB_OK;
  if (!images || !out_dev) return fail(ctx, JCB_E_INVALID, "null image / output pointer");
  // balanced chunks: the fewest passes that respect the bound, all (nearly) the same size, so no pass
  // runs the 148 SMs on a sliver of work
  const int64_t chunk = balanced_chunk(n, views_bound(ctx, on_host, v->tokens));
  int rc = ws_reserve(ctx, ws_extra + tower_ws_bytes(v, chunk));
  if (rc) return rc;
  Bump b(static_cast<uint8_t*>(ctx->ws) + ws_extra);
  TowerWs w = tower_ws_carve(v, chunk, b);
  // bytes of one view: [3, R, R] pixels, or its G^2 rows of the patch matrix (the same 3 R^2 elements, 16-bit)
  const size_t view_bytes = static_cast<size_t>(3) * v->cfg.resolution * v->cfg.resolution * img_elem_bytes(dt);
  if (on_host && (rc = stage_reserve(ctx, chunk * view_bytes))) return rc;
  // Host input: the upload of pass i+1 overlaps the compute of pass i, but nothing hides the FIRST upload, so
  // the first pass is a quarter of the others (its copy is 4x shorter; it is too short to matter for the GEMMs).
  // (not needed when the call is queued behind a running submission: that one's compute hides it)
  const int64_t lead = (on_host && n > chunk && !ctx->overlapped) ? std::max<int64_t>(chunk / 4, 1) : 0;
  const int64_t body = lead ? balanced_chunk(n - lead, chunk) : chunk;
  int64_t ci = 0;
  for (int64_t off = 0; off < n; ++ci) {
    const int64_t m = std::min(ci == 0 && lead ? lead : body, n - off);
    const void* src = static_cast<const uint8_t*>(images) + off * view_bytes;
    int buf = 0;
    if (on_host) {
      buf = static_cast<int>(ctx->stage_seq++ & 1);
      // the pass that last read this staging buffer (possibly of the previous, still running call) must be done
      if (ctx->stage_recorded[buf]) CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->compute_done[buf], 0));
      CUDA_TRY(ctx, cudaMemcpyAsync(ctx->stage[buf], src, m * view_bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
      CUDA_TRY(ctx, cudaEventRecord(ctx->copy_done[buf], ctx->copy_stream));
      CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->stream, ctx->copy_done[buf], 0));
      src = ctx->stage[buf];
    }
    if ((rc = tower_forward(v, src, dt, m, apply_norm, w, slot_dev ? slot_dev + off : nullptr))) return rc;
    LAUNCH_P(ctx, JCB_KC_TAIL, 2.0 * m * v->cfg.width * v->cfg.embed_dim,
             static_cast<double>(m) * (v->cfg.width + v->cfg.embed_dim) * 4, launch_tail(w.tokens, m, v->tokens, v->cfg.width, v->ln_post_g, v->ln_post_b, v->proj,
                            v->cfg.embed_dim, normalize, out_dev + off * v->cfg.embed_dim, ctx->stream));
    if (on_host) {
      CUDA_TRY(ctx, cudaEventRecord(ctx->compute_done[buf], ctx->stream));
      ctx->stage_recorded[buf] = true;
    }
    off += m;
  }
  return JCB_OK;
}

int sync_and_check(jcb_ctx* ctx) {
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  int st = 0;
  CUDA_TRY(ctx, cudaMemcpy(&st, ctx->dev_status, sizeof(int), cudaMemcpyDeviceToHost));
  if (st != 0) {
    int zero = 0;
    cudaMemcpy(ctx->dev_status, &zero, sizeof(int), cudaMemcpyHostToDevice);
    return fail(ctx, JCB_E_KERNEL, "device-side kernel status %d (101 producer / 102 mma / 103 epilogue pipeline timeout)", st);
  }
  return JCB_OK;
}

// LoRA slots of one call: `host` holds n_entries slots, each repeated for `repeat` consecutive views (1 per view, or V
// per image).  Validated on the host before anything is launched, then copied to the device once, on the context's
// stream (a pageable copy: the caller's array may be reused as soon as the call returns).  *dev = nullptr when the tower
// has one slot: every entry is 0 and the call runs the single-slot schedule.
int slots_prepare(jcb_vit* v, const int32_t* host, int64_t n_entries, int64_t repeat, const int32_t** dev) {
  jcb_ctx* ctx = v->ctx;
  *dev = nullptr;
  if (!host) return fail(ctx, JCB_E_INVALID, "null LoRA slot array");
  const int G = v->lora_slots;
  for (int64_t i = 0; i < n_entries; ++i)
    if (host[i] < 0 || host[i] >= G)
      return fail(ctx, JCB_E_INVALID, "LoRA slot %d of entry %lld out of range: the tower carries %d slot(s)", host[i],
                  static_cast<long long>(i), G);
  if (G == 1 || n_entries <= 0) return JCB_OK;
  const int64_t n = n_entries * repeat;
  if (n > ctx->slot_cap) {   // growth: a queued submission may still read the old array
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->slot_dev) cudaFree(ctx->slot_dev);
    ctx->slot_dev = nullptr;
    ctx->slot_cap = 0;
    cudaError_t e = cudaMalloc(&ctx->slot_dev, static_cast<size_t>(n) * sizeof(int32_t));
    if (e != cudaSuccess) return fail(ctx, JCB_E_NOMEM, "cudaMalloc for the LoRA slot array failed: %s", cudaGetErrorString(e));
    ctx->slot_cap = n;
  }
  std::vector<int32_t> per_view;
  if (repeat > 1) {
    per_view.resize(static_cast<size_t>(n));
    for (int64_t i = 0; i < n; ++i) per_view[i] = host[i / repeat];
    host = per_view.data();
  }
  CUDA_TRY(ctx, cudaMemcpyAsync(ctx->slot_dev, host, static_cast<size_t>(n) * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
  *dev = ctx->slot_dev;
  return JCB_OK;
}

}  // namespace

// ================================================================================================
extern "C" {

int jcb_abi_version(void) { return JCB_ABI_VERSION; }

int jcb_ctx_create(int device, jcb_ctx** out) {
  if (!out) return JCB_E_INVALID;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return JCB_E_NO_DEVICE;
  if (device < 0 || device >= count) return JCB_E_INVALID;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return JCB_E_CUDA;
  if (prop.major != 10) return JCB_E_NO_DEVICE;  // kernels are sm_100a only: tcgen05 / TMEM / TMA
  jcb_ctx* ctx = new jcb_ctx();
  ctx->device = device;
  ctx->num_sms = prop.multiProcessorCount;
  {
    const char* env_cls = getenv("JCB_CLS_ONLY_LAST_BLOCK");
    ctx->cls_only_last = (env_cls && env_cls[0] == '1') ? 1 : 0;
    const char* env_op = getenv("JCB_OPERANDS");   // "bf16" | "f16" (default): see jcb_ctx_set_operand_type
    ctx->operand_f16 = (env_op && (env_op[0] == 'b' || env_op[0] == 'B')) ? 0 : 1;
    const char* env_lm = getenv("JCB_LORA");       // "applied" | "merged" (default): see jcb_ctx_set_lora_mode
    ctx->lora_applied = (env_lm && (env_lm[0] == 'a' || env_lm[0] == 'A')) ? 1 : 0;
    const char* env_g = getenv("JCB_GRAPHS");
    ctx->graphs_on = (env_g && env_g[0] == '0') ? 0 : 1;
  }
  ctx->cc_major = prop.major;
  ctx->cc_minor = prop.minor;
  DeviceGuard g(device);
  bool ok = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) == cudaSuccess;
  ctx->own_stream = ok;
  ok = ok && cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
  for (int i = 0; i < 2 && ok; ++i) {
    ok = cudaEventCreateWithFlags(&ctx->copy_done[i], cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&ctx->compute_done[i], cudaEventDisableTiming) == cudaSuccess;
  }
  for (int i = 0; ok && i < JCB_MAX_INFLIGHT; ++i)
    ok = cudaEventCreateWithFlags(&ctx->ticket_done[i], cudaEventDisableTiming | cudaEventBlockingSync) == cudaSuccess;
  ok = ok && cudaHostAlloc(reinterpret_cast<void**>(&ctx->ticket_status), JCB_MAX_INFLIGHT * sizeof(int), cudaHostAllocDefault) == cudaSuccess;
  ok = ok && cudaMalloc(&ctx->dev_status, sizeof(int)) == cudaSuccess &&
       cudaMemset(ctx->dev_status, 0, sizeof(int)) == cudaSuccess;
  const char* derr = ok ? gemm_init_driver_api() : "context setup failed";
  if (!ok || derr) {
    jcb_ctx_destroy(ctx);
    return JCB_E_CUDA;
  }
  *out = ctx;
  return JCB_OK;
}

int jcb_ctx_destroy(jcb_ctx* ctx) {
  if (!ctx) return JCB_OK;
  DeviceGuard g(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  if (ctx->copy_stream) cudaStreamSynchronize(ctx->copy_stream);
  graphs_clear_fwd(ctx);
  if (ctx->capture_stream) cudaStreamDestroy(ctx->capture_stream);
  if (ctx->ws) cudaFree(ctx->ws);
  if (ctx->tta_ws) cudaFree(ctx->tta_ws);
  for (int i = 0; i < 2; ++i) {
    if (ctx->stage[i]) cudaFree(ctx->stage[i]);
    if (ctx->copy_done[i]) cudaEventDestroy(ctx->copy_done[i]);
    if (ctx->compute_done[i]) cudaEventDestroy(ctx->compute_done[i]);
  }
  if (ctx->dev_status) cudaFree(ctx->dev_status);
  if (ctx->slot_dev) cudaFree(ctx->slot_dev);
  for (int i = 0; i < JCB_MAX_INFLIGHT; ++i)
    if (ctx->ticket_done[i]) cudaEventDestroy(ctx->ticket_done[i]);
  if (ctx->ticket_status) cudaFreeHost(ctx->ticket_status);
  for (int i = 0; i < 2; ++i) {
    if (ctx->tta_plan_host[i]) cudaFreeHost(ctx->tta_plan_host[i]);
    if (ctx->tta_plan_copied[i]) cudaEventDestroy(ctx->tta_plan_copied[i]);
  }
  if (ctx->tta_done) cudaEventDestroy(ctx->tta_done);
  for (auto e : ctx->prof_ev)
    if (e) cudaEventDestroy(e);
  if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  delete ctx;
  return JCB_OK;
}

int jcb_ctx_set_stream(jcb_ctx* ctx, void* cuda_stream) {
  if (!ctx) return JCB_E_INVALID;
  DeviceGuard g(ctx->device);
  cudaStream_t ns = static_cast<cudaStream_t>(cuda_stream);
  if (ns == ctx->stream) return JCB_OK;
  CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  ctx->stream = ns;
  ctx->own_stream = false;
  return JCB_OK;
}

int jcb_ctx_set_chunk_views(jcb_ctx* ctx, int64_t chunk_views) {
  if (!ctx || chunk_views < 1 || chunk_views > 40000) return ctx ? fail(ctx, JCB_E_INVALID, "chunk_views out of range") : JCB_E_INVALID;
  ctx->chunk_views = chunk_views;
  return JCB_OK;
}

int jcb_ctx_set_host_chunk_views(jcb_ctx* ctx, int64_t chunk_views) {
  if (!ctx || chunk_views < 1 || chunk_views > 40000) return ctx ? fail(ctx, JCB_E_INVALID, "chunk_views out of range") : JCB_E_INVALID;
  ctx->host_chunk_views = chunk_views;
  return JCB_OK;
}

int jcb_ctx_set_cls_only_last_block(jcb_ctx* ctx, int on) {
  if (!ctx) return JCB_E_INVALID;
  ctx->cls_only_last = on ? 1 : 0;
  return JCB_OK;
}

int jcb_ctx_set_operand_type(jcb_ctx* ctx, int operand_type) {
  if (!ctx) return JCB_E_INVALID;
  if (operand_type != JCB_OPERAND_BF16 && operand_type != JCB_OPERAND_F16)
    return fail(ctx, JCB_E_INVALID, "operand_type must be JCB_OPERAND_BF16 (0) or JCB_OPERAND_F16 (1)");
  ctx->operand_f16 = operand_type == JCB_OPERAND_F16 ? 1 : 0;
  return JCB_OK;
}

int jcb_ctx_get_operand_type(const jcb_ctx* ctx) { return ctx ? (ctx->operand_f16 ? JCB_OPERAND_F16 : JCB_OPERAND_BF16) : JCB_E_INVALID; }

int jcb_ctx_set_lora_mode(jcb_ctx* ctx, int mode) {
  if (!ctx) return JCB_E_INVALID;
  if (mode != JCB_LORA_MERGED && mode != JCB_LORA_APPLIED)
    return fail(ctx, JCB_E_INVALID, "lora mode must be JCB_LORA_MERGED (0) or JCB_LORA_APPLIED (1)");
  ctx->lora_applied = mode == JCB_LORA_APPLIED ? 1 : 0;
  return JCB_OK;
}

int jcb_ctx_get_lora_mode(const jcb_ctx* ctx) { return ctx ? (ctx->lora_applied ? JCB_LORA_APPLIED : JCB_LORA_MERGED) : JCB_E_INVALID; }

int jcb_vit_lora_mode(const jcb_vit* v) { return v ? (v->lora_applied ? JCB_LORA_APPLIED : JCB_LORA_MERGED) : JCB_E_INVALID; }

int jcb_text_lora_mode(const jcb_text* t) { return t ? (t->lora_applied ? JCB_LORA_APPLIED : JCB_LORA_MERGED) : JCB_E_INVALID; }

int jcb_vit_operand_type(const jcb_vit* v) { return v ? (v->f16 ? JCB_OPERAND_F16 : JCB_OPERAND_BF16) : JCB_E_INVALID; }

int jcb_text_operand_type(const jcb_text* t) { return t ? (t->f16 ? JCB_OPERAND_F16 : JCB_OPERAND_BF16) : JCB_E_INVALID; }

int jcb_ctx_trim(jcb_ctx* ctx) {
  if (!ctx) return JCB_E_INVALID;
  DeviceGuard g(ctx->device);
  if (ctx->next_ticket > ctx->waited_ticket) return fail(ctx, JCB_E_STATE, "jcb_ctx_trim: submissions are still in flight");
  CUDA_TRY(ctx, cudaDeviceSynchronize());
  graphs_clear_fwd(ctx);
  if (ctx->ws) cudaFree(ctx->ws);
  ctx->ws = nullptr;
  ctx->ws_bytes = 0;
  ++ctx->ws_gen;
  if (ctx->tta_ws) cudaFree(ctx->tta_ws);
  ctx->tta_ws = nullptr;
  ctx->tta_ws_bytes = 0;
  for (int i = 0; i < 2; ++i) {
    if (ctx->stage[i]) cudaFree(ctx->stage[i]);
    ctx->stage[i] = nullptr;
  }
  ctx->stage_bytes = 0;
  ctx->stage_recorded[0] = ctx->stage_recorded[1] = false;
  if (ctx->slot_dev) cudaFree(ctx->slot_dev);
  ctx->slot_dev = nullptr;
  ctx->slot_cap = 0;
  return JCB_OK;
}

int jcb_sync(jcb_ctx* ctx) {
  if (!ctx) return JCB_E_INVALID;
  DeviceGuard g(ctx->device);
  return sync_and_check(ctx);
}

const char* jcb_last_error(const jcb_ctx* ctx) { return ctx ? ctx->err : "null context"; }

int jcb_ctx_info(const jcb_ctx* ctx, int* num_sms, int* cc_major, int* cc_minor, size_t* workspace_bytes) {
  if (!ctx) return JCB_E_INVALID;
  if (num_sms) *num_sms = ctx->num_sms;
  if (cc_major) *cc_major = ctx->cc_major;
  if (cc_minor) *cc_minor = ctx->cc_minor;
  if (workspace_bytes) *workspace_bytes = ctx->ws_bytes + 2 * ctx->stage_bytes;
  return JCB_OK;
}

int64_t jcb_ctx_launch_count(const jcb_ctx* ctx) { return ctx ? ctx->launches : 0; }


int jcb_ctx_profile(jcb_ctx* ctx, int enable) {
  if (!ctx) return JCB_E_INVALID;
  DeviceGuard g(ctx->device);
  if (enable) {
    if (ctx->prof_ev.empty()) {
      ctx->prof_ev.resize(2 * PROF_PAIRS, nullptr);
      for (auto& e : ctx->prof_ev)
        if (cudaEventCreate(&e) != cudaSuccess) return fail(ctx, JCB_E_CUDA, "cudaEventCreate failed");
      ctx->prof_cls.reserve(PROF_PAIRS);
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->prof_cls.clear();
    for (int i = 0; i < JCB_KC_COUNT; ++i) {
      ctx->prof_ms[i] = 0; ctx->prof_n[i] = 0; ctx->prof_timed[i] = 0; ctx->prof_flops[i] = 0; ctx->prof_bytes[i] = 0;
    }
    ctx->prof_on = true;
  } else if (ctx->prof_on) {
    ctx->prof_on = false;
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    for (size_t i = 0; i < ctx->prof_cls.size(); ++i) {
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, ctx->prof_ev[2 * i], ctx->prof_ev[2 * i + 1]) == cudaSuccess) {
        ctx->prof_ms[ctx->prof_cls[i]] += ms;
        ctx->prof_timed[ctx->prof_cls[i]] += 1;
      }
    }
    ctx->prof_cls.clear();
  }
  return JCB_OK;
}

int jcb_ctx_profile_read(const jcb_ctx* ctx, int kernel_class, double* total_ms, int64_t* launches,
                         int64_t* timed_launches, double* flops, double* bytes) {
  if (!ctx || kernel_class < 0 || kernel_class >= JCB_KC_COUNT) return JCB_E_INVALID;
  if (total_ms) *total_ms = ctx->prof_ms[kernel_class];
  if (launches) *launches = ctx->prof_n[kernel_class];
  if (timed_launches) *timed_launches = ctx->prof_timed[kernel_class];
  if (flops) *flops = ctx->prof_flops[kernel_class];
  if (bytes) *bytes = ctx->prof_bytes[kernel_class];
  return JCB_OK;
}

const char* jcb_kernel_class_name(int kernel_class) {
  static const char* names[JCB_KC_COUNT] = {"im2col", "gemm_patch", "embed_ln", "gemm_qkv", "attention", "gemm_out",
                                            "layernorm", "gemm_fc1", "gemm_fc2", "tail", "mta", "head", "other", "tta_views",
                                            "gemm_lora"};
  return kernel_class >= 0 && kernel_class < JCB_KC_COUNT ? names[kernel_class] : "?";
}

// ------------------------------------------------------------------------------------------------
int jcb_vit_create(jcb_ctx* ctx, const jcb_vit_config* cfg, jcb_vit** out) {
  if (!ctx || !cfg || !out) return JCB_E_INVALID;
  *out = nullptr;
  if (cfg->layers < 1 || cfg->layers > 64) return fail(ctx, JCB_E_INVALID, "layers=%d unsupported", cfg->layers);
  if (cfg->width % 256 != 0 || cfg->width > 1024 || cfg->width < 256)
    return fail(ctx, JCB_E_INVALID, "width=%d unsupported (need a multiple of 256 in [256, 1024])", cfg->width);
  if (cfg->patch % 16 != 0 || cfg->resolution % cfg->patch != 0)
    return fail(ctx, JCB_E_INVALID, "patch=%d / resolution=%d unsupported", cfg->patch, cfg->resolution);
  if (cfg->embed_dim != 512) return fail(ctx, JCB_E_INVALID, "embed_dim=%d unsupported (512 only)", cfg->embed_dim);
  if (cfg->vpt_tokens < 0 || cfg->vpt_tokens > 14) return fail(ctx, JCB_E_INVALID, "vpt_tokens=%d unsupported", cfg->vpt_tokens);
  jcb_vit* v = new jcb_vit();
  v->ctx = ctx;
  v->cfg = *cfg;
  v->grid = cfg->resolution / cfg->patch;
  v->tokens = v->grid * v->grid + 1 + cfg->vpt_tokens;
  v->heads = cfg->width / 64;  // jclip/model.py:152
  v->W = cfg->width;
  v->L = cfg->layers;
  v->prefix = "visual.transformer.resblocks.";
  v->kpatch = 3 * cfg->patch * cfg->patch;
  if (v->tokens > 256 || v->heads % 4 != 0 || v->kpatch % 64 != 0) {
    delete v;
    return fail(ctx, JCB_E_INVALID, "tokens=%d (max 256) / heads=%d (multiple of 4) unsupported", v->tokens, v->heads);
  }
  build_expected(v);
  *out = v;
  return JCB_OK;
}

int jcb_vit_destroy(jcb_vit* v) {
  if (!v) return JCB_OK;
  DeviceGuard g(v->ctx->device);
  cudaStreamSynchronize(v->ctx->stream);
  graphs_clear_fwd(v->ctx);      // captured pipelines point into this tower's weights
  if (v->arena) cudaFree(v->arena);
  delete v;
  return JCB_OK;
}

int jcb_vit_set_param(jcb_vit* v, const char* name, const float* data, int64_t numel) {
  return tower_set_param(v, name, data, numel);
}

int jcb_vit_set_lora(jcb_vit* v, int layer, int proj, const float* A, const float* B, int r, float scaling) {
  return tower_set_lora(v, layer, proj, A, B, r, scaling);
}

int jcb_vit_set_lora_slot(jcb_vit* v, int slot, int layer, int proj, const float* A, const float* B, int r, float scaling) {
  return tower_set_lora(v, layer, proj, A, B, r, scaling, slot);
}

int jcb_vit_set_lora_slot_count(jcb_vit* v, int n_slots) {
  if (!v) return JCB_E_INVALID;
  if (n_slots < 1 || n_slots > JCB_MAX_LORA_SLOTS)
    return fail(v->ctx, JCB_E_INVALID, "set_lora_slot_count: %d slots out of range (1 .. %d)", n_slots, JCB_MAX_LORA_SLOTS);
  if (static_cast<size_t>(n_slots) > v->lora.size()) {   // the new slots carry no adapter: plain projections
    v->lora.resize(n_slots);
    v->finalized = false;
  }
  return JCB_OK;
}

int jcb_vit_lora_slots(const jcb_vit* v) { return v ? static_cast<int>(v->lora.size()) : JCB_E_INVALID; }

int jcb_vit_clear_lora(jcb_vit* v) {
  if (!v) return JCB_E_INVALID;
  v->lora.assign(1, {});
  v->finalized = false;
  return JCB_OK;
}

}  // extern "C"

namespace {

// Uploads a tower's staged fp32 parameters into its device arena: GEMM operands as bf16 (LoRA merged in fp32
// first: W' = W + s * B A, reference test.py:310-313 / :388-398), everything else fp32.
struct Packer {
  TowerBase* t;
  jcb_ctx* ctx;
  Bump b{nullptr};
  void* tmp = nullptr;
  float *tmp_w = nullptr, *tmp_A = nullptr, *tmp_B = nullptr;
  explicit Packer(TowerBase* tower) : t(tower), ctx(tower->ctx) {}
  ~Packer() { if (tmp) cudaFree(tmp); }

  int begin(size_t arena_bytes, size_t max_tensor_elems) {
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    t->f16 = ctx->operand_f16;   // the tower keeps the operand type it was packed with until the next finalize
    t->lora_applied = ctx->lora_applied;
    ++t->gen;
    if (!t->arena || t->arena_bytes < arena_bytes) {
      if (t->arena) cudaFree(t->arena);
      t->arena = nullptr;
      cudaError_t e = cudaMalloc(&t->arena, arena_bytes);
      if (e != cudaSuccess) return fail(ctx, JCB_E_NOMEM, "cudaMalloc(%zu) for weights failed: %s", arena_bytes, cudaGetErrorString(e));
      t->arena_bytes = arena_bytes;
    }
    const size_t W = t->W;
    const size_t tmp_bytes = align_up(max_tensor_elems * 4) + 2 * align_up(256 * W * 4);
    cudaError_t e = cudaMalloc(&tmp, tmp_bytes);
    if (e != cudaSuccess) return fail(ctx, JCB_E_NOMEM, "cudaMalloc(%zu) for packing failed: %s", tmp_bytes, cudaGetErrorString(e));
    tmp_w = static_cast<float*>(tmp);
    tmp_A = reinterpret_cast<float*>(static_cast<uint8_t*>(tmp) + align_up(max_tensor_elems * 4));
    tmp_B = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(tmp_A) + align_up(256 * W * 4));
    b = Bump(t->arena);
    return JCB_OK;
  }
  int up_f32(const std::string& key, float** dst) {
    const std::vector<float>& h = t->host[key];
    *dst = b.take<float>(h.size());
    CUDA_TRY(ctx, cudaMemcpyAsync(*dst, h.data(), h.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    return JCB_OK;
  }
  // bf16 weight [rows, cols]; `adapters` lists (row offset, adapter) pairs merged in fp32 before the cast
  int up_bf16(const std::string& key, size_t rows, size_t cols, __nv_bfloat16** dst,
              const std::vector<std::pair<size_t, const LoraAdapter*>>& adapters) {
    cudaStream_t s = ctx->stream;
    const std::vector<float>& h = t->host[key];
    *dst = b.take<__nv_bfloat16>(h.size());
    CUDA_TRY(ctx, cudaMemcpyAsync(tmp_w, h.data(), h.size() * 4, cudaMemcpyHostToDevice, s));
    LAUNCH(ctx, launch_cast_bf16(tmp_w, *dst, static_cast<int64_t>(rows * cols), s, t->f16));
    for (auto& ad : adapters) {
      const LoraAdapter* a = ad.second;
      CUDA_TRY(ctx, cudaMemcpyAsync(tmp_A, a->A.data(), a->A.size() * 4, cudaMemcpyHostToDevice, s));
      CUDA_TRY(ctx, cudaMemcpyAsync(tmp_B, a->B.data(), a->B.size() * 4, cudaMemcpyHostToDevice, s));
      // rows [off, off + W) of the packed weight: W' = W + s * B A
      LAUNCH(ctx, launch_merge_lora_cast(tmp_w + ad.first * cols, tmp_A, tmp_B, t->W, static_cast<int>(cols), a->r,
                                         a->scaling, *dst + ad.first * cols, s, t->f16));
      CUDA_TRY(ctx, cudaStreamSynchronize(s));  // the staging buffers are reused by the next adapter
    }
    CUDA_TRY(ctx, cudaStreamSynchronize(s));
    return JCB_OK;
  }
  // LayerNorm fold of one weight: merged fp32 W (LoRA adapters applied in place) -> gamma-scaled bf16 Wf, S, c
  int up_folded(const std::string& key, size_t rows, size_t cols,
                const std::vector<std::pair<size_t, const LoraAdapter*>>& adapters, const float* gamma_dev,
                const float* beta_dev, const float* bias_dev, __nv_bfloat16** wf, float** S, float** c) {
    cudaStream_t s = ctx->stream;
    const std::vector<float>& h = t->host[key];
    *wf = b.take<__nv_bfloat16>(h.size());
    *S = b.take<float>(rows);
    *c = b.take<float>(rows);
    CUDA_TRY(ctx, cudaMemcpyAsync(tmp_w, h.data(), h.size() * 4, cudaMemcpyHostToDevice, s));
    for (auto& ad : adapters) {
      const LoraAdapter* a = ad.second;
      CUDA_TRY(ctx, cudaMemcpyAsync(tmp_A, a->A.data(), a->A.size() * 4, cudaMemcpyHostToDevice, s));
      CUDA_TRY(ctx, cudaMemcpyAsync(tmp_B, a->B.data(), a->B.size() * 4, cudaMemcpyHostToDevice, s));
      LAUNCH(ctx, launch_merge_lora_f32(tmp_w + ad.first * cols, tmp_A, tmp_B, t->W, static_cast<int>(cols), a->r,
                                        a->scaling, s));
      CUDA_TRY(ctx, cudaStreamSynchronize(s));
    }
    LAUNCH(ctx, launch_fold_ln(tmp_w, gamma_dev, beta_dev, bias_dev, static_cast<int>(rows), static_cast<int>(cols), *wf,
                               *S, *c, s, t->f16));
    CUDA_TRY(ctx, cudaStreamSynchronize(s));
    return JCB_OK;
  }
  // LoRA applied: the adapters of one projection GEMM side by side (see LayerDev), once per slot.  `slots[g]` =
  // (row offset of the projection inside the packed weight, adapter) of slot g; rows = rows of the packed weight.  s is
  // folded into the up matrix.  *live = the slots with an adapter here.
  int up_lora_applied(const std::vector<std::vector<std::pair<size_t, const LoraAdapter*>>>& slots, size_t rows,
                      __nv_bfloat16** dn, __nv_bfloat16** up, uint32_t* live) {
    *dn = *up = nullptr;
    *live = 0;
    const int G = static_cast<int>(slots.size());
    for (int g = 0; g < G; ++g)
      if (!slots[g].empty()) *live |= 1u << g;
    if (!*live) return JCB_OK;
    cudaStream_t s = ctx->stream;
    const size_t W = t->W, u_cols = lora_u_cols(G), k2 = static_cast<size_t>(LORA_K2) * G;
    std::vector<float> hd(u_cols * W, 0.f), hu(rows * k2, 0.f);
    for (int g = 0; g < G; ++g) {
      int r_total = 0;
      for (auto& ad : slots[g]) r_total += ad.second->r;
      if (r_total > LORA_K2 && G == 1)
        return fail(ctx, JCB_E_INVALID, "LoRA applied: the ranks of one projection GEMM sum to %d (max %d); use JCB_LORA_MERGED",
                    r_total, LORA_K2);
      if (r_total > LORA_K2)
        return fail(ctx, JCB_E_INVALID, "LoRA slot %d: the ranks of one projection GEMM sum to %d (max %d)", g, r_total, LORA_K2);
      size_t j0 = static_cast<size_t>(LORA_K2) * g;   // slot g: rows [64 g, 64 g + 64) of down, columns of up
      for (auto& ad : slots[g]) {
        const LoraAdapter* a = ad.second;
        for (int j = 0; j < a->r; ++j) std::copy(a->A.begin() + j * W, a->A.begin() + (j + 1) * W, hd.begin() + (j0 + j) * W);
        for (size_t n = 0; n < W; ++n)
          for (int j = 0; j < a->r; ++j) hu[(ad.first + n) * k2 + j0 + j] = a->scaling * a->B[n * a->r + j];
        j0 += a->r;
      }
    }
    *dn = b.take<__nv_bfloat16>(hd.size());
    *up = b.take<__nv_bfloat16>(hu.size());
    CUDA_TRY(ctx, cudaMemcpyAsync(tmp_w, hd.data(), hd.size() * 4, cudaMemcpyHostToDevice, s));
    LAUNCH(ctx, launch_cast_bf16(tmp_w, *dn, static_cast<int64_t>(hd.size()), s, t->f16));
    CUDA_TRY(ctx, cudaStreamSynchronize(s));   // hd / tmp_w are reused
    CUDA_TRY(ctx, cudaMemcpyAsync(tmp_w, hu.data(), hu.size() * 4, cudaMemcpyHostToDevice, s));
    LAUNCH(ctx, launch_cast_bf16(tmp_w, *up, static_cast<int64_t>(hu.size()), s, t->f16));
    CUDA_TRY(ctx, cudaStreamSynchronize(s));
    return JCB_OK;
  }
  int pack_blocks() {
    const size_t W = t->W;
    t->layers.assign(t->L, LayerDev());
    const bool applied = t->lora_applied != 0;
    const std::vector<std::pair<size_t, const LoraAdapter*>> none;
    const size_t G = t->lora.size();
    int rc;
    for (int li = 0; li < t->L; ++li) {
      LayerDev& Ld = t->layers[li];
      std::vector<std::vector<std::pair<size_t, const LoraAdapter*>>> in_ad(G), out_ad(G);   // per slot
      for (size_t g = 0; g < G; ++g) {
        for (int p = 0; p < 3; ++p) {  // packed in_proj rows: q 0:W, k W:2W, v 2W:3W  (test.py:491-501)
          auto it = t->lora[g].find(li * 4 + p);
          if (it != t->lora[g].end()) in_ad[g].push_back({p * W, &it->second});
        }
        auto ito = t->lora[g].find(li * 4 + JCB_PROJ_O);
        if (ito != t->lora[g].end()) out_ad[g].push_back({0, &ito->second});
      }
      // merged mode has one slot (jcb_vit_finalize)
      if ((rc = up_bf16(blk(t, li, "attn.in_proj_weight"), 3 * W, W, &Ld.in_w, applied ? none : in_ad[0]))) return rc;
      if ((rc = up_bf16(blk(t, li, "attn.out_proj.weight"), W, W, &Ld.out_w, applied ? none : out_ad[0]))) return rc;
      if (applied) {
        if ((rc = up_lora_applied(in_ad, 3 * W, &Ld.lin_dn, &Ld.lin_up, &Ld.lin_slots))) return rc;
        if ((rc = up_lora_applied(out_ad, W, &Ld.lout_dn, &Ld.lout_up, &Ld.lout_slots))) return rc;
      }
      if ((rc = up_bf16(blk(t, li, "mlp.c_fc.weight"), 4 * W, W, &Ld.fc_w, {}))) return rc;
      if ((rc = up_bf16(blk(t, li, "mlp.c_proj.weight"), W, 4 * W, &Ld.proj_w, {}))) return rc;
      if ((rc = up_f32(blk(t, li, "attn.in_proj_bias"), &Ld.in_b))) return rc;
      if ((rc = up_f32(blk(t, li, "attn.out_proj.bias"), &Ld.out_b))) return rc;
      if ((rc = up_f32(blk(t, li, "mlp.c_fc.bias"), &Ld.fc_b))) return rc;
      if ((rc = up_f32(blk(t, li, "mlp.c_proj.bias"), &Ld.proj_b))) return rc;
      if ((rc = up_f32(blk(t, li, "ln_1.weight"), &Ld.ln1_g))) return rc;
      if ((rc = up_f32(blk(t, li, "ln_1.bias"), &Ld.ln1_b))) return rc;
      if ((rc = up_f32(blk(t, li, "ln_2.weight"), &Ld.ln2_g))) return rc;
      if ((rc = up_f32(blk(t, li, "ln_2.bias"), &Ld.ln2_b))) return rc;
      if (!applied) {   // LoRA applied runs the stand-alone LayerNorm schedule (tower_blocks)
        if ((rc = up_folded(blk(t, li, "attn.in_proj_weight"), 3 * W, W, in_ad[0], Ld.ln1_g, Ld.ln1_b, Ld.in_b, &Ld.in_wf,
                            &Ld.in_S, &Ld.in_c))) return rc;
        if ((rc = up_folded(blk(t, li, "mlp.c_fc.weight"), 4 * W, W, {}, Ld.ln2_g, Ld.ln2_b, Ld.fc_b, &Ld.fc_wf, &Ld.fc_S,
                            &Ld.fc_c))) return rc;
      }
    }
    return JCB_OK;
  }
  int end() {
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    if (b.off > t->arena_bytes) return fail(ctx, JCB_E_STATE, "internal: weight arena overflow (%zu > %zu)", b.off, t->arena_bytes);
    t->lora_slots = static_cast<int>(t->lora.size());
    t->finalized = true;
    return JCB_OK;
  }
};

size_t blocks_arena_bytes(size_t W, size_t L, size_t G = 1) {
  // packed weights + biases / LayerNorm vectors, plus the LayerNorm-folded copies of in_proj / c_fc (Wf, S, c)
  // (LoRA applied: the down / up matrices of in_proj and out_proj for G slots; the folded copies are not packed then)
  return L * (align_up(3 * W * W * 2) + align_up(W * W * 2) + 2 * align_up(4 * W * W * 2) + 8 * align_up(4 * W * 4) +
              align_up(3 * W * W * 2) + align_up(4 * W * W * 2) + 4 * align_up(4 * W * 4) +
              2 * align_up(lora_u_cols(static_cast<int>(G)) * W * 2) + align_up(3 * W * LORA_K2 * G * 2) +
              align_up(W * LORA_K2 * G * 2));
}

int tower_set_param(TowerBase* t, const char* name, const float* data, int64_t numel) {
  if (!t || !name || !data) return JCB_E_INVALID;
  auto it = t->expected.find(name);
  if (it == t->expected.end()) return fail(t->ctx, JCB_E_INVALID, "unknown parameter '%s'", name);
  if (it->second != numel)
    return fail(t->ctx, JCB_E_INVALID, "parameter '%s': expected %lld elements, got %lld", name,
                static_cast<long long>(it->second), static_cast<long long>(numel));
  t->host[name].assign(data, data + numel);
  t->finalized = false;
  return JCB_OK;
}

int tower_set_lora(TowerBase* t, int layer, int proj, const float* A, const float* B, int r, float scaling, int slot) {
  if (!t || !A || !B) return JCB_E_INVALID;
  if (layer < 0 || layer >= t->L || proj < 0 || proj > 3 || r < 1 || r > 256)
    return fail(t->ctx, JCB_E_INVALID, "set_lora: layer=%d proj=%d r=%d out of range", layer, proj, r);
  if (slot < 0 || slot >= JCB_MAX_LORA_SLOTS)
    return fail(t->ctx, JCB_E_INVALID, "set_lora_slot: slot %d out of range (0 .. %d)", slot, JCB_MAX_LORA_SLOTS - 1);
  if (static_cast<size_t>(slot) >= t->lora.size()) t->lora.resize(slot + 1);
  LoraAdapter& a = t->lora[slot][layer * 4 + proj];
  const int64_t W = t->W;
  a.A.assign(A, A + r * W);
  a.B.assign(B, B + W * r);
  a.r = r;
  a.scaling = scaling;
  t->finalized = false;
  return JCB_OK;
}

int tower_missing(TowerBase* t) {
  for (auto& kv : t->expected)
    if (!t->host.count(kv.first)) return fail(t->ctx, JCB_E_STATE, "parameter '%s' was never set", kv.first.c_str());
  return JCB_OK;
}

}  // namespace

extern "C" {

int jcb_vit_finalize(jcb_vit* v) {
  if (!v) return JCB_E_INVALID;
  jcb_ctx* ctx = v->ctx;
  DeviceGuard g(ctx->device);
  int rc = tower_missing(v);
  if (rc) return rc;
  const size_t G = v->lora.size();
  if (G > 1) {   // several slots: every slot's rank limits are checked before anything is packed
    if (!ctx->lora_applied)
      return fail(ctx, JCB_E_INVALID, "%zu LoRA slots need JCB_LORA_APPLIED (applied mode); merged mode packs one adapter set", G);
    for (size_t s = 0; s < G; ++s)
      for (int li = 0; li < v->L; ++li) {
        int r_qkv = 0;
        for (int p = 0; p < 3; ++p) {
          auto it = v->lora[s].find(li * 4 + p);
          if (it != v->lora[s].end()) r_qkv += it->second.r;
        }
        auto ito = v->lora[s].find(li * 4 + JCB_PROJ_O);
        const int r_o = ito != v->lora[s].end() ? ito->second.r : 0;
        if (r_qkv > LORA_K2 || r_o > LORA_K2)
          return fail(ctx, JCB_E_INVALID, "LoRA slot %zu, layer %d: the ranks of q, k, v sum to %d and r(o) = %d (max %d each)", s,
                      li, r_qkv, r_o, LORA_K2);
      }
  }
  const size_t W = v->cfg.width, E = v->cfg.embed_dim, T = v->tokens, KP = v->kpatch, L = v->cfg.layers;
  // arena: bf16 GEMM operands, then fp32 vectors
  const size_t bytes = align_up(W * KP * 2) + blocks_arena_bytes(W, L, G) + 9 * align_up(std::max(W * E, T * W) * 4);
  Packer pk(v);
  if ((rc = pk.begin(bytes, std::max(4 * W * W, W * KP)))) return rc;
  if ((rc = pk.up_bf16("visual.conv1.weight", W, KP, &v->conv_w, {}))) return rc;
  if ((rc = pk.up_f32("visual.class_embedding", &v->cls))) return rc;
  if ((rc = pk.up_f32("visual.positional_embedding", &v->pos))) return rc;
  if (v->cfg.vpt_tokens > 0 && (rc = pk.up_f32("visual.VPT", &v->vpt))) return rc;
  if ((rc = pk.up_f32("visual.ln_pre.weight", &v->ln_pre_g))) return rc;
  if ((rc = pk.up_f32("visual.ln_pre.bias", &v->ln_pre_b))) return rc;
  if ((rc = pk.up_f32("visual.ln_post.weight", &v->ln_post_g))) return rc;
  if ((rc = pk.up_f32("visual.ln_post.bias", &v->ln_post_b))) return rc;
  if ((rc = pk.up_f32("visual.proj", &v->proj))) return rc;
  if ((rc = pk.pack_blocks())) return rc;
  return pk.end();
}

// ------------------------------------------------------------------------------------------------ text tower
int jcb_text_create(jcb_ctx* ctx, const jcb_text_config* cfg, jcb_text** out) {
  if (!ctx || !cfg || !out) return JCB_E_INVALID;
  *out = nullptr;
  if (cfg->layers < 1 || cfg->layers > 64) return fail(ctx, JCB_E_INVALID, "layers=%d unsupported", cfg->layers);
  if (cfg->width % 128 != 0 || cfg->width < 256 || cfg->width > 1024 || (cfg->width != 512 && cfg->width != 768 && cfg->width != 1024))
    return fail(ctx, JCB_E_INVALID, "text width=%d unsupported (512, 768 or 1024)", cfg->width);
  if (cfg->context_length < 1 || cfg->context_length > 128)
    return fail(ctx, JCB_E_INVALID, "context_length=%d unsupported (max 128: one attention tile per head)", cfg->context_length);
  if (cfg->embed_dim != 512) return fail(ctx, JCB_E_INVALID, "embed_dim=%d unsupported (512 only)", cfg->embed_dim);
  if (cfg->vocab_size < 1) return fail(ctx, JCB_E_INVALID, "vocab_size=%d", cfg->vocab_size);
  jcb_text* t = new jcb_text();
  t->ctx = ctx;
  t->cfg = *cfg;
  t->W = cfg->width;
  t->L = cfg->layers;
  t->heads = cfg->width / 64;                       // jclip/model.py:268 transformer_heads = width // 64
  t->tokens = cfg->context_length;
  t->prefix = "transformer.resblocks.";
  const int64_t W = t->W;
  t->expected["token_embedding.weight"] = static_cast<int64_t>(cfg->vocab_size) * W;
  t->expected["positional_embedding"] = static_cast<int64_t>(cfg->context_length) * W;
  t->expected["ln_final.weight"] = W;
  t->expected["ln_final.bias"] = W;
  t->expected["text_projection"] = W * cfg->embed_dim;
  expect_blocks(t);
  *out = t;
  return JCB_OK;
}

int jcb_text_destroy(jcb_text* t) {
  if (!t) return JCB_OK;
  DeviceGuard g(t->ctx->device);
  cudaStreamSynchronize(t->ctx->stream);
  if (t->arena) cudaFree(t->arena);
  delete t;
  return JCB_OK;
}

int jcb_text_set_param(jcb_text* t, const char* name, const float* data, int64_t numel) {
  return tower_set_param(t, name, data, numel);
}

int jcb_text_set_lora(jcb_text* t, int layer, int proj, const float* A, const float* B, int r, float scaling) {
  return tower_set_lora(t, layer, proj, A, B, r, scaling);
}

int jcb_text_clear_lora(jcb_text* t) {
  if (!t) return JCB_E_INVALID;
  t->lora.assign(1, {});
  t->finalized = false;
  return JCB_OK;
}

int jcb_text_finalize(jcb_text* t) {
  if (!t) return JCB_E_INVALID;
  jcb_ctx* ctx = t->ctx;
  DeviceGuard g(ctx->device);
  int rc = tower_missing(t);
  if (rc) return rc;
  const size_t W = t->W, E = t->cfg.embed_dim, T = t->tokens, V = t->cfg.vocab_size, L = t->L;
  const size_t bytes = blocks_arena_bytes(W, L) + align_up(V * W * 4) + align_up(T * W * 4) + 2 * align_up(W * 4) + align_up(W * E * 4);
  Packer pk(t);
  if ((rc = pk.begin(bytes, 4 * W * W))) return rc;
  if ((rc = pk.up_f32("token_embedding.weight", &t->tok_emb))) return rc;
  if ((rc = pk.up_f32("positional_embedding", &t->pos))) return rc;
  if ((rc = pk.up_f32("ln_final.weight", &t->ln_final_g))) return rc;
  if ((rc = pk.up_f32("ln_final.bias", &t->ln_final_b))) return rc;
  if ((rc = pk.up_f32("text_projection", &t->text_projection))) return rc;
  if ((rc = pk.pack_blocks())) return rc;
  return pk.end();
}

// `CLIP.encode_text(text)` (jclip/model.py:202-215): token + positional embedding, L causal blocks, ln_final on the
// EOT token (the highest id of each sequence), @ text_projection.
int jcb_encode_text(jcb_text* t, const int64_t* tokens_dev, int64_t n_seq, int normalize, float* out_dev) {
  if (!t) return JCB_E_INVALID;
  jcb_ctx* ctx = t->ctx;
  if (!t->finalized) return fail(ctx, JCB_E_STATE, "jcb_text_finalize has not been called");
  if (n_seq < 0) return fail(ctx, JCB_E_INVALID, "negative sequence count");
  if (n_seq == 0) return JCB_OK;
  if (!tokens_dev || !out_dev) return fail(ctx, JCB_E_INVALID, "null token / output pointer");
  DeviceGuard g(ctx->device);
  const int W = t->W, T = t->tokens, E = t->cfg.embed_dim;
  const int64_t chunk = balanced_chunk(n_seq, std::max<int64_t>(1, ctx->chunk_views * 50 / T));
  const size_t eot_b = align_up(static_cast<size_t>(chunk) * 4);
  int rc = ws_reserve(ctx, eot_b + tower_ws_bytes_dims(W, T, 0, 0, chunk));
  if (rc) return rc;
  int* eot = static_cast<int*>(ctx->ws);
  Bump b(static_cast<uint8_t*>(ctx->ws) + eot_b);
  TowerWs w = tower_ws_carve_dims(W, T, 0, 0, chunk, b);
  for (int64_t off = 0; off < n_seq; off += chunk) {
    const int64_t m = std::min(chunk, n_seq - off);
    const double MW = static_cast<double>(m) * T * W;
    LAUNCH_P(ctx, JCB_KC_EMBED_LN, 0, MW * (4 + 4 + 2),
             launch_text_embed_ln(reinterpret_cast<const long long*>(tokens_dev) + off * T, m, T, W, t->cfg.vocab_size,
                                  t->tok_emb, t->pos, t->layers[0].ln1_g, t->layers[0].ln1_b, w.tokens, w.ln_out, eot,
                                  ctx->stream, t->layers[0].in_wf ? w.stats[0] : nullptr, (W + 255) / 256,
                                  w.shift[0], t->f16));
    if ((rc = tower_blocks(t, m, w, 1))) return rc;
    LAUNCH_P(ctx, JCB_KC_TAIL, 2.0 * m * W * E, static_cast<double>(m) * (W + E) * 4,
             launch_tail(w.tokens, m, T, W, t->ln_final_g, t->ln_final_b, t->text_projection, E, normalize,
                         out_dev + off * E, ctx->stream, eot));
  }
  return JCB_OK;
}

int jcb_encode_image(jcb_vit* v, const void* images_dev, int img_dtype, int64_t n_views, int apply_clip_norm,
                     int normalize, float* out_dev) {
  int rc = check_vit(v);
  if (rc) return rc;
  DeviceGuard g(v->ctx->device);
  return encode_views(v, images_dev, img_dtype, false, n_views, apply_clip_norm, normalize, out_dev, 0);
}

int jcb_encode_image_slots(jcb_vit* v, const void* images_dev, int img_dtype, int64_t n_views,
                           const int32_t* slot_of_view_host, int apply_clip_norm, int normalize, float* out_dev) {
  int rc = check_vit(v);
  if (rc) return rc;
  DeviceGuard g(v->ctx->device);
  const int32_t* slot_dev = nullptr;
  if ((rc = slots_prepare(v, slot_of_view_host, n_views, 1, &slot_dev))) return rc;
  return encode_views(v, images_dev, img_dtype, false, n_views, apply_clip_norm, normalize, out_dev, 0, slot_dev);
}

int jcb_encode_image_host(jcb_vit* v, const void* images_host, int img_dtype, int64_t n_views, int apply_clip_norm,
                          int normalize, float* out_host) {
  int rc = check_vit(v);
  if (rc) return rc;
  jcb_ctx* ctx = v->ctx;
  DeviceGuard g(ctx->device);
  if (n_views == 0) return JCB_OK;
  if (n_views < 0 || !out_host) return fail(ctx, JCB_E_INVALID, "bad arguments");
  const size_t out_bytes = align_up(static_cast<size_t>(n_views) * v->cfg.embed_dim * 4);
  if ((rc = ws_reserve(ctx, out_bytes + tower_ws_bytes(v, balanced_chunk(n_views, token_rows_bound(std::min(ctx->host_chunk_views, ctx->chunk_views), v->tokens)))))) return rc;
  float* out_dev = static_cast<float*>(ctx->ws);
  if ((rc = encode_views(v, images_host, img_dtype, true, n_views, apply_clip_norm, normalize, out_dev, out_bytes)))
    return rc;
  CUDA_TRY(ctx, cudaMemcpyAsync(out_host, out_dev, static_cast<size_t>(n_views) * v->cfg.embed_dim * 4,
                                cudaMemcpyDeviceToHost, ctx->stream));
  return sync_and_check(ctx);
}

int jcb_vit_debug_tokens(jcb_vit* v, const void* images_dev, int img_dtype, int64_t n_views, int apply_clip_norm,
                         float* tokens_out_dev) {
  int rc = check_vit(v);
  if (rc) return rc;
  jcb_ctx* ctx = v->ctx;
  DeviceGuard g(ctx->device);
  if (n_views < 1 || n_views > ctx->chunk_views) return fail(ctx, JCB_E_INVALID, "debug_tokens: 1 <= n_views <= chunk_views");
  if ((rc = ws_reserve(ctx, tower_ws_bytes(v, n_views)))) return rc;
  Bump b(ctx->ws);
  TowerWs w = tower_ws_carve(v, n_views, b);
  if ((rc = tower_forward(v, images_dev, img_dtype, n_views, apply_clip_norm, w))) return rc;
  CUDA_TRY(ctx, cudaMemcpyAsync(tokens_out_dev, w.tokens, static_cast<size_t>(n_views) * v->tokens * v->cfg.width * 4,
                                cudaMemcpyDeviceToDevice, ctx->stream));
  return JCB_OK;
}

// ------------------------------------------------------------------------------------------------
namespace {
// Grow-only scratch of the view generator.  Growth waits for the whole device (a view batch may be in flight on a
// stream this context does not know); steady state never does.
int tta_ws_reserve(jcb_ctx* ctx, size_t bytes) {
  if (bytes <= ctx->tta_ws_bytes) return JCB_OK;
  CUDA_TRY(ctx, cudaDeviceSynchronize());
  if (ctx->tta_ws) cudaFree(ctx->tta_ws);
  ctx->tta_ws = nullptr;
  ctx->tta_ws_bytes = 0;
  cudaError_t e = cudaMalloc(&ctx->tta_ws, bytes);
  if (e != cudaSuccess) return fail(ctx, JCB_E_NOMEM, "cudaMalloc(%zu) for the view generator failed: %s", bytes, cudaGetErrorString(e));
  ctx->tta_ws_bytes = bytes;
  return JCB_OK;
}

int tta_run(jcb_ctx* ctx, cudaStream_t stream, const uint8_t* src_dev, const jcb_src_image* images, int32_t n_images,
            const jcb_view_job* jobs, int64_t n_jobs, int32_t size, int out_mode, int patch, int apply_norm, void* out_dev) {
  if (n_jobs < 0 || n_images < 0 || size < 8 || size > 1024) return fail(ctx, JCB_E_INVALID, "jcb_tta: bad sizes");
  if (n_jobs == 0) return JCB_OK;
  if (!src_dev || !images || !jobs || !out_dev) return fail(ctx, JCB_E_INVALID, "jcb_tta: null pointer");
  static_assert(sizeof(jcb_src_image) == sizeof(TtaImage) && sizeof(jcb_view_job) == sizeof(TtaJob), "ABI structs");
  DeviceGuard g(ctx->device);
  const int64_t BATCH = 16384;   // views per launch pair (grid.y limit; bounds the intermediate scratch)
  const size_t out_view_bytes = static_cast<size_t>(3) * size * size * (out_mode == 0 ? 1 : 2);
  // one reservation for the whole call: a later batch must not move the scratch an earlier batch's kernels still use
  std::vector<std::vector<uint8_t>> plans;
  struct Meta { int kh, kv, mr; size_t tmp_bytes; };
  std::vector<Meta> metas;
  size_t need = 0;
  for (int64_t j0 = 0; j0 < n_jobs; j0 += BATCH) {
    const int64_t nj = std::min(BATCH, n_jobs - j0);
    plans.emplace_back();
    Meta m{};
    const char* err = nullptr;
    m.tmp_bytes = tta_plan(reinterpret_cast<const TtaImage*>(images), n_images, reinterpret_cast<const TtaJob*>(jobs + j0), nj,
                           size, &plans.back(), &m.kh, &m.kv, &m.mr, &err);
    if (m.tmp_bytes == SIZE_MAX) return fail(ctx, JCB_E_INVALID, "jcb_tta: %s", err ? err : "invalid job");
    need = std::max(need, align_up(plans.back().size()) + m.tmp_bytes);
    metas.push_back(m);
  }
  // the intermediate's size depends on the (random) crop heights: reserve with 25 % head-room, so that a stream of batches
  // stops growing the scratch (a growth waits for the whole device) after the first one or two
  int rc = tta_ws_reserve(ctx, need > ctx->tta_ws_bytes ? need + need / 4 : need);
  if (rc) return rc;
  if (!ctx->tta_done) CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->tta_done, cudaEventDisableTiming));
  else if (ctx->tta_last_stream != stream) CUDA_TRY(ctx, cudaStreamWaitEvent(stream, ctx->tta_done, 0));
  size_t bi = 0;
  for (int64_t j0 = 0; j0 < n_jobs; j0 += BATCH, ++bi) {
    const int64_t nj = std::min(BATCH, n_jobs - j0);
    const std::vector<uint8_t>& plan = plans[bi];
    const Meta& m = metas[bi];
    uint8_t* plan_dev = static_cast<uint8_t*>(ctx->tta_ws);
    uint8_t* tmp = plan_dev + align_up(plan.size());
    // the plan goes through one of two pinned buffers, so the call never waits for the stream: a buffer is reused only
    // after the upload that last read it has completed (its event; two calls back, normally long done)
    const int t = ctx->tta_turn;
    ctx->tta_turn ^= 1;
    if (ctx->tta_plan_copied[t]) CUDA_TRY(ctx, cudaEventSynchronize(ctx->tta_plan_copied[t]));
    else CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->tta_plan_copied[t], cudaEventDisableTiming));
    if (ctx->tta_plan_bytes[t] < plan.size()) {
      if (ctx->tta_plan_host[t]) cudaFreeHost(ctx->tta_plan_host[t]);
      ctx->tta_plan_host[t] = nullptr;
      ctx->tta_plan_bytes[t] = 0;
      CUDA_TRY(ctx, cudaMallocHost(&ctx->tta_plan_host[t], plan.size()));
      ctx->tta_plan_bytes[t] = plan.size();
    }
    memcpy(ctx->tta_plan_host[t], plan.data(), plan.size());
    CUDA_TRY(ctx, cudaMemcpyAsync(plan_dev, ctx->tta_plan_host[t], plan.size(), cudaMemcpyHostToDevice, stream));
    CUDA_TRY(ctx, cudaEventRecord(ctx->tta_plan_copied[t], stream));
    void* out = static_cast<uint8_t*>(out_dev) + j0 * out_view_bytes;
    if (stream == ctx->stream) {
      LAUNCH_P(ctx, JCB_KC_TTA, 0, static_cast<double>(nj) * out_view_bytes,
               launch_tta(src_dev, plan_dev, nj, size, m.kh, m.kv, m.mr, tmp, out, stream, out_mode, patch, apply_norm));
    } else {   // a caller-chosen stream: the per-class event profile belongs to the context's stream
      LAUNCH(ctx, launch_tta(src_dev, plan_dev, nj, size, m.kh, m.kv, m.mr, tmp, out, stream, out_mode, patch, apply_norm));
    }
    ++ctx->launches;  // two kernels per call
  }
  CUDA_TRY(ctx, cudaEventRecord(ctx->tta_done, stream));
  ctx->tta_last_stream = stream;
  return JCB_OK;
}
}  // namespace

int jcb_tta_views(jcb_ctx* ctx, void* cuda_stream, const uint8_t* src_dev, const jcb_src_image* images, int32_t n_images,
                  const jcb_view_job* jobs, int64_t n_jobs, int32_t size, uint8_t* out_dev) {
  if (!ctx) return JCB_E_INVALID;
  return tta_run(ctx, cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->stream, src_dev, images, n_images, jobs,
                 n_jobs, size, 0, 0, 0, out_dev);
}

int jcb_tta_patches(jcb_ctx* ctx, void* cuda_stream, const uint8_t* src_dev, const jcb_src_image* images, int32_t n_images,
                    const jcb_view_job* jobs, int64_t n_jobs, int32_t size, int32_t patch, int32_t apply_clip_norm,
                    int32_t operand_type, void* out_patches_dev) {
  if (!ctx) return JCB_E_INVALID;
  if (operand_type != JCB_OPERAND_BF16 && operand_type != JCB_OPERAND_F16) return fail(ctx, JCB_E_INVALID, "jcb_tta_patches: bad operand_type");
  if (patch < 4 || patch % 4 != 0 || size % patch != 0) return fail(ctx, JCB_E_INVALID, "jcb_tta_patches: patch=%d must divide size=%d and be a multiple of 4", patch, size);
  return tta_run(ctx, cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->stream, src_dev, images, n_images, jobs,
                 n_jobs, size, operand_type == JCB_OPERAND_F16 ? 2 : 1, patch, apply_clip_norm, out_patches_dev);
}

// ------------------------------------------------------------------------------------------------
void jcb_mta_default_params(jcb_mta_params* p) {
  if (!p) return;
  p->lambda_y = 0.2f; p->lambda_q = 4.0f; p->th = 1e-6f; p->temperature = 1.0f; p->k_frac = 0.3; p->max_iter = 5;
  p->reserved = 0;
}

namespace {
MtaParams to_params(const jcb_mta_params* p) {
  MtaParams m;
  if (p) {
    m.lambda_y = p->lambda_y; m.lambda_q = p->lambda_q; m.th = p->th; m.temperature = p->temperature;
    m.k_frac = p->k_frac; m.max_iter = p->max_iter;
  }
  return m;
}

// Arguments of jcb_mta / jcb_mta_debug, checked before the workspace is sized from them.  Parameters are rejected where
// the solver would stop meaning what the reference computes: temperature and lambda_y divide (test.py:1411, :1434); the
// reference's loops run at least once (`while True`), the kernels' would run max_iter < 1 times and return view 0; the
// reference averages sorted_dist[:, 1:k+1], at most V - 1 neighbours, where the kernels divide by k -- k_frac <= 1 keeps
// k = int(k_frac (V - 1)) <= V - 1.
int check_mta_args(jcb_ctx* ctx, const char* fn, const float* feats, const float* text, const float* out_mode,
                   int64_t n_images, int32_t V, int32_t C, int32_t D, const jcb_mta_params* p) {
  if (n_images < 0 || !feats || !text || !out_mode) return fail(ctx, JCB_E_INVALID, "%s: bad arguments", fn);
  if (!mta_shape_supported(V, C, D))
    return fail(ctx, JCB_E_INVALID, "%s: unsupported n_views=%d n_classes=%d dim=%d (need 1 <= n_views <= 2048, n_classes >= 1, "
                "dim a multiple of 32 in [32, 1024])", fn, V, C, D);
  if (!p) return JCB_OK;
  if (!std::isfinite(p->lambda_y) || !std::isfinite(p->lambda_q) || !std::isfinite(p->th) || !std::isfinite(p->temperature) ||
      !std::isfinite(p->k_frac))
    return fail(ctx, JCB_E_INVALID, "%s: non-finite parameter", fn);
  if (p->lambda_y <= 0.f) return fail(ctx, JCB_E_INVALID, "%s: lambda_y=%g must be > 0", fn, p->lambda_y);
  if (p->temperature <= 0.f) return fail(ctx, JCB_E_INVALID, "%s: temperature=%g must be > 0", fn, p->temperature);
  if (p->th < 0.f) return fail(ctx, JCB_E_INVALID, "%s: th=%g must be >= 0", fn, p->th);
  if (p->max_iter < 1) return fail(ctx, JCB_E_INVALID, "%s: max_iter=%d must be >= 1", fn, p->max_iter);
  if (!(p->k_frac >= 0.0 && p->k_frac <= 1.0)) return fail(ctx, JCB_E_INVALID, "%s: k_frac=%g must be in [0, 1]", fn, p->k_frac);
  return JCB_OK;
}
}  // namespace

// fp32 work of one solve_mta: P = softmax(100 X T) (2 V C D), the two V x V Gram matrices over the upper triangle
// (V^2 (C + D)) and <= 50 density / mode passes over X (4 V D each): the figure the MTA profile class reports
static double mta_flops(double I, double V, double C, double D) { return I * (2 * V * C * D + V * V * (C + D) + 50 * 4 * V * D); }

static int mta_run(jcb_ctx* ctx, const char* fn, const float* feats_dev, const float* text_dev, int64_t n_images,
                   int32_t n_views, int32_t n_classes, int32_t dim, const jcb_mta_params* params, float* out_mode_dev,
                   float* out_logits_dev, const MtaDebug* debug) {
  if (!ctx) return JCB_E_INVALID;
  int rc = check_mta_args(ctx, fn, feats_dev, text_dev, out_mode_dev, n_images, n_views, n_classes, dim, params);
  if (rc) return rc;
  DeviceGuard g(ctx->device);
  const size_t scratch = mta_scratch_bytes(n_images, n_views, n_classes, dim);
  if ((rc = ws_reserve(ctx, scratch))) return rc;
  MtaSet set{feats_dev, text_dev, out_mode_dev, out_logits_dev};
  LAUNCH_P(ctx, JCB_KC_MTA, mta_flops(n_images, n_views, n_classes, dim), static_cast<double>(n_images) * (n_views + 1) * dim * 4,
           launch_mta(&set, 1, n_images, n_views, n_classes, dim, to_params(params),
                      scratch ? static_cast<float*>(ctx->ws) : nullptr, ctx->stream, ctx->dev_status, ctx->num_sms, debug));
  return JCB_OK;
}

int jcb_mta(jcb_ctx* ctx, const float* feats_dev, const float* text_dev, int64_t n_images, int32_t n_views,
            int32_t n_classes, int32_t dim, const jcb_mta_params* params, float* out_mode_dev, float* out_logits_dev) {
  return mta_run(ctx, "jcb_mta", feats_dev, text_dev, n_images, n_views, n_classes, dim, params, out_mode_dev, out_logits_dev,
                 nullptr);
}

int jcb_mta_debug(jcb_ctx* ctx, const float* feats_dev, const float* text_dev, int64_t n_images, int32_t n_views,
                  int32_t n_classes, int32_t dim, const jcb_mta_params* params, float* out_mode_dev, float* out_logits_dev,
                  float* out_bw_dev, float* out_y_dev, float* out_affinity_dev) {
  const MtaDebug debug{out_bw_dev, out_y_dev, out_affinity_dev};
  return mta_run(ctx, "jcb_mta_debug", feats_dev, text_dev, n_images, n_views, n_classes, dim, params, out_mode_dev,
                 out_logits_dev, &debug);
}

int jcb_head(jcb_ctx* ctx, const float* m_pt, const float* m_hand, const float* m_zs, const float* T_pt,
             const float* T_hand, const float* T_zs, const jcb_head_weights* lp, int64_t n_images, int32_t n_classes,
             int32_t dim, int32_t rank_by, int32_t k, int32_t* out_topk, float* out_scores, float* out_all) {
  if (!ctx) return JCB_E_INVALID;
  if (!m_pt || !m_hand || !m_zs || !T_pt || !T_hand || !T_zs || !lp || !out_topk || n_images < 0)
    return fail(ctx, JCB_E_INVALID, "jcb_head: null argument");
  DeviceGuard g(ctx->device);
  HeadArgs a;
  a.m_pt = m_pt; a.m_hand = m_hand; a.m_zs = m_zs; a.T_pt = T_pt; a.T_hand = T_hand; a.T_zs = T_zs;
  a.scale1 = lp->scale1; a.bias1 = lp->bias1; a.fc_w = lp->fc_w; a.fc_b = lp->fc_b;
  a.I = n_images; a.C = n_classes; a.D = dim; a.rank_by = rank_by; a.k = k;
  a.out_topk = out_topk; a.out_scores = out_scores; a.out_all = out_all;
  LAUNCH_P(ctx, JCB_KC_HEAD, 0, static_cast<double>(n_images) * (3 * dim + k) * 4, launch_head(a, ctx->stream));
  return JCB_OK;
}

int jcb_cosine_topk(jcb_ctx* ctx, const float* feats, const float* text, int64_t n, int32_t n_classes, int32_t dim,
                    float scale, int32_t k, int32_t* out_topk, float* out_scores) {
  if (!ctx) return JCB_E_INVALID;
  if (!feats || !text || n < 0 || (!out_topk && !out_scores)) return fail(ctx, JCB_E_INVALID, "jcb_cosine_topk: bad arguments");
  DeviceGuard g(ctx->device);
  LAUNCH(ctx, launch_cosine_topk(feats, text, n, n_classes, dim, scale, k, out_topk, out_scores, ctx->stream));
  return JCB_OK;
}

int jcb_channel_lp(jcb_ctx* ctx, const float* feats, int64_t n, int32_t n_classes, int32_t dim,
                   const jcb_head_weights* lp, float* out) {
  if (!ctx) return JCB_E_INVALID;
  if (!feats || !lp || !out || n < 0) return fail(ctx, JCB_E_INVALID, "jcb_channel_lp: bad arguments");
  DeviceGuard g(ctx->device);
  LAUNCH(ctx, launch_channel_lp(feats, n, n_classes, dim, lp->scale1, lp->bias1, lp->fc_w, lp->fc_b, out, ctx->stream));
  return JCB_OK;
}

int jcb_class_mean(jcb_ctx* ctx, const float* emb_dev, const int32_t* offsets_dev, int32_t n_classes, int32_t dim,
                   float* out_dev) {
  if (!ctx) return JCB_E_INVALID;
  if (!emb_dev || !offsets_dev || !out_dev || n_classes < 0 || dim < 1) return fail(ctx, JCB_E_INVALID, "jcb_class_mean: bad arguments");
  DeviceGuard g(ctx->device);
  LAUNCH(ctx, launch_class_mean(emb_dev, offsets_dev, n_classes, dim, out_dev, ctx->stream));
  return JCB_OK;
}

int jcb_logit_normalize(jcb_ctx* ctx, const float* in, int64_t n, int32_t n_classes, float* out) {
  if (!ctx) return JCB_E_INVALID;
  if (!in || !out || n < 0) return fail(ctx, JCB_E_INVALID, "jcb_logit_normalize: bad arguments");
  DeviceGuard g(ctx->device);
  LAUNCH(ctx, launch_logit_normalize(in, n, n_classes, out, ctx->stream));
  return JCB_OK;
}

// ------------------------------------------------------------------------------------------------
namespace {
// Everything jcb_pipeline does, enqueued on the context's streams without waiting for any of it.
// with_slots: a jcb_pipeline_slots call, slot_of_image = its per-image LoRA slots of `vit` (host)
int pipeline_enqueue(jcb_vit* vit, jcb_vit* vit_zs, const jcb_pipeline_args* a, bool with_slots = false,
                     const int32_t* slot_of_image = nullptr) {
  int rc = check_vit(vit);
  if (rc) return rc;
  jcb_ctx* ctx = vit->ctx;
  if (vit_zs && ((rc = check_vit(vit_zs)) || vit_zs->ctx != ctx)) return rc ? rc : fail(ctx, JCB_E_INVALID, "vit_zs belongs to another context");
  if (!a || !a->images || !a->out_topk || !a->text_pt_dev || !a->text_hand_dev || !a->text_zs_dev ||
      !a->text_pt_t_dev || !a->text_hand_t_dev || !a->text_zs_t_dev)
    return fail(ctx, JCB_E_INVALID, "jcb_pipeline: null argument");
  if (a->n_images < 0 || a->n_views < 1 || a->k < 1 || a->k > 8) return fail(ctx, JCB_E_INVALID, "jcb_pipeline: bad sizes");
  if (with_slots && !slot_of_image) return fail(ctx, JCB_E_INVALID, "jcb_pipeline_slots: null LoRA slot array");
  if (a->n_images == 0) return JCB_OK;
  DeviceGuard g(ctx->device);
  const int32_t* slot_dev = nullptr;   // per view; vit_zs runs its own slot 0
  if (with_slots && (rc = slots_prepare(vit, slot_of_image, a->n_images, a->n_views, &slot_dev))) return rc;
  const int E = vit->cfg.embed_dim, C = a->n_classes, V = a->n_views;
  const int64_t I = a->n_images, NV = I * V;
  // persistent part of the workspace: [feats] [feats_zs] [modes x3] [topk] [mta scratch]
  const size_t feats_b = align_up(static_cast<size_t>(NV) * E * 4);
  const size_t modes_b = align_up(static_cast<size_t>(I) * E * 4);
  const size_t topk_b = align_up(static_cast<size_t>(I) * a->k * 4);
  const size_t scratch_b = align_up(mta_scratch_bytes(3 * I, V, C, E));
  const bool own_feats = a->out_feats_dev == nullptr;
  const size_t head_bytes = (own_feats ? feats_b : 0) + (vit_zs ? feats_b : 0) + 3 * modes_b + topk_b + scratch_b;
  // ONE reservation for everything below: the persistent part and the larger of the two towers' pass workspaces.
  // (encode_views reserves again per tower; if the second tower needed MORE than the first, ws_reserve would free
  // the buffer the first tower's embeddings, the modes and the scratch were carved from.)
  {
    const int64_t chunk = balanced_chunk(NV, views_bound(ctx, a->images_on_host != 0, vit->tokens));
    size_t tower_b = tower_ws_bytes(vit, chunk);
    if (vit_zs) tower_b = std::max(tower_b, tower_ws_bytes(vit_zs, balanced_chunk(NV, views_bound(ctx, a->images_on_host != 0, vit_zs->tokens))));
    if ((rc = ws_reserve(ctx, head_bytes + tower_b))) return rc;
  }
  Bump b(ctx->ws);
  const void* ws_at_carve = ctx->ws;
  float* feats = own_feats ? b.take<float>(static_cast<size_t>(NV) * E) : a->out_feats_dev;
  float* feats_zs = vit_zs ? b.take<float>(static_cast<size_t>(NV) * E) : feats;
  float* m_pt = b.take<float>(static_cast<size_t>(I) * E);
  float* m_hand = b.take<float>(static_cast<size_t>(I) * E);
  float* m_zs = b.take<float>(static_cast<size_t>(I) * E);
  int32_t* topk_dev = a->topk_on_host ? b.take<int32_t>(static_cast<size_t>(I) * a->k) : a->out_topk;
  if (!a->topk_on_host) b.take<int32_t>(static_cast<size_t>(I) * a->k);
  float* scratch = scratch_b ? b.take<float>(scratch_b / 4) : nullptr;
  if (b.off > head_bytes) return fail(ctx, JCB_E_STATE, "internal: pipeline workspace overflow");

  // encode_image + L2 normalise over every view                      test.py:1705-1706 (:1711-1712)
  if ((rc = encode_views(vit, a->images, a->img_dtype, a->images_on_host != 0, NV, a->apply_clip_norm, 1, feats, head_bytes,
                         slot_dev))) return rc;
  if (vit_zs && (rc = encode_views(vit_zs, a->images, a->img_dtype, a->images_on_host != 0, NV, a->apply_clip_norm, 1, feats_zs, head_bytes))) return rc;
  if (ctx->ws != ws_at_carve) return fail(ctx, JCB_E_STATE, "internal: the workspace moved while the pipeline held pointers into it");
  // solve_mta x3 in one launch                                        test.py:1708-1709, :1713
  MtaSet sets[3] = {{feats, a->text_pt_t_dev, m_pt, nullptr},
                    {feats, a->text_hand_t_dev, m_hand, nullptr},
                    {feats_zs, a->text_zs_t_dev, m_zs, nullptr}};
  LAUNCH_P(ctx, JCB_KC_MTA, 3.0 * mta_flops(I, V, C, E), 3.0 * I * (V + 1) * E * 4, launch_mta(sets, 3, I, V, C, E, MtaParams(), scratch, ctx->stream, ctx->dev_status, ctx->num_sms));
  // Channel_LP, logit_normalize, fusion, top-k                        test.py:1710-1738
  HeadArgs h;
  h.m_pt = m_pt; h.m_hand = m_hand; h.m_zs = m_zs;
  h.T_pt = a->text_pt_dev; h.T_hand = a->text_hand_dev; h.T_zs = a->text_zs_dev;
  h.scale1 = a->lp.scale1; h.bias1 = a->lp.bias1; h.fc_w = a->lp.fc_w; h.fc_b = a->lp.fc_b;
  h.I = I; h.C = C; h.D = E; h.rank_by = a->rank_by; h.k = a->k;
  h.out_topk = topk_dev; h.out_scores = a->out_scores_dev; h.out_all = nullptr;
  LAUNCH_P(ctx, JCB_KC_HEAD, 10.0 * I * C * E, static_cast<double>(I) * (3 * E + a->k) * 4, launch_head(h, ctx->stream));
  if (a->topk_on_host)
    CUDA_TRY(ctx, cudaMemcpyAsync(a->out_topk, topk_dev, static_cast<size_t>(I) * a->k * 4, cudaMemcpyDeviceToHost, ctx->stream));
  return JCB_OK;
}
}  // namespace

// ------------------------------------------------------------------------------------------------
// CUDA graphs for SMALL pipelines.  The reference calls the path once per image (test.py:1692-1742: 1 image x 65 views):
// ~210 kernel launches for ~0.6 ms of GPU work, i.e. bound by launch latency on the host.  The launch sequence of
// jcb_pipeline depends only on (towers, shapes, operand pointers), so the second call with the same key is captured
// into a graph (input copied into a graph-owned staging buffer, top-k read from a graph-owned buffer) and later calls
// replay it with one launch.  Only device work is captured: no allocation, no synchronisation (the first call with a
// key ran normally and reserved the workspace).  Graphs are dropped when the workspace moves, a tower is re-packed or
// destroyed, or a schedule option changes.  jcb_ctx_set_graphs(ctx, 0) / JCB_GRAPHS=0 turn the mechanism off.
struct PipelineGraph {
  // key
  const jcb_vit *vit = nullptr, *vit_zs = nullptr;
  uint64_t vit_gen = 0, zs_gen = 0, ws_gen = 0;
  int64_t I = 0;
  int V = 0, dt = 0, apply_norm = 0, C = 0, rank_by = 0, k = 0, cls_only = 0;
  const void* ptrs[10] = {nullptr};   // text banks (6) + head weights (4)
  cudaStream_t stream = nullptr;
  // state
  int seen = 0;
  cudaGraphExec_t exec = nullptr;
  void* in_stage = nullptr;
  int32_t* topk_dev = nullptr;
  uint64_t last_use = 0;
};

namespace {
void graph_free(PipelineGraph* g) {
  if (g->exec) cudaGraphExecDestroy(g->exec);
  if (g->in_stage) cudaFree(g->in_stage);
  if (g->topk_dev) cudaFree(g->topk_dev);
  delete g;
}
void graphs_clear(jcb_ctx* ctx) {
  if (ctx->graphs.empty()) return;
  cudaStreamSynchronize(ctx->stream);
  for (auto* g : ctx->graphs) graph_free(g);
  ctx->graphs.clear();
}
bool graph_key_equal(const PipelineGraph& g, const jcb_ctx* ctx, const jcb_vit* vit, const jcb_vit* vit_zs, const jcb_pipeline_args* a) {
  if (g.vit != vit || g.vit_zs != vit_zs || g.vit_gen != vit->gen || g.zs_gen != (vit_zs ? vit_zs->gen : 0) ||
      g.I != a->n_images || g.V != a->n_views || g.dt != a->img_dtype ||
      g.apply_norm != a->apply_clip_norm || g.C != a->n_classes || g.rank_by != a->rank_by || g.k != a->k ||
      g.cls_only != ctx->cls_only_last || g.stream != ctx->stream)
    return false;
  const void* p[10] = {a->text_pt_dev, a->text_hand_dev, a->text_zs_dev, a->text_pt_t_dev, a->text_hand_t_dev, a->text_zs_t_dev,
                       a->lp.scale1, a->lp.bias1, a->lp.fc_w, a->lp.fc_b};
  for (int i = 0; i < 10; ++i)
    if (g.ptrs[i] != p[i]) return false;
  return true;
}

// returns JCB_OK with *handled = true when the call was served by a graph
int pipeline_try_graph(jcb_vit* vit, jcb_vit* vit_zs, const jcb_pipeline_args* a, bool* handled) {
  *handled = false;
  jcb_ctx* ctx = vit->ctx;
  if (!ctx->graphs_on || ctx->prof_on || !a || a->n_images < 1 || a->out_feats_dev || a->out_scores_dev ||
      static_cast<int64_t>(a->n_images) * a->n_views > ctx->graph_max_views || ctx->next_ticket > ctx->waited_ticket)
    return JCB_OK;
  if (check_vit(vit) != JCB_OK || (vit_zs && (check_vit(vit_zs) != JCB_OK || vit_zs->ctx != ctx))) return JCB_OK;   // the normal path reports it
  static uint64_t tick = 0;
  PipelineGraph* g = nullptr;
  for (size_t i = 0; i < ctx->graphs.size();) {
    PipelineGraph* c = ctx->graphs[i];
    if (c->ws_gen != ctx->ws_gen && c->exec) {     // the workspace moved under a captured graph: drop it
      cudaStreamSynchronize(ctx->stream);
      graph_free(c);
      ctx->graphs.erase(ctx->graphs.begin() + static_cast<long>(i));
      continue;
    }
    if (graph_key_equal(*c, ctx, vit, vit_zs, a)) g = c;
    ++i;
  }
  if (!g) {
    if (ctx->graphs.size() >= 16) {   // forget the least recently used shape
      size_t lru = 0;
      for (size_t i = 1; i < ctx->graphs.size(); ++i)
        if (ctx->graphs[i]->last_use < ctx->graphs[lru]->last_use) lru = i;
      cudaStreamSynchronize(ctx->stream);
      graph_free(ctx->graphs[lru]);
      ctx->graphs.erase(ctx->graphs.begin() + static_cast<long>(lru));
    }
    g = new PipelineGraph();
    g->vit = vit; g->vit_zs = vit_zs; g->vit_gen = vit->gen; g->zs_gen = vit_zs ? vit_zs->gen : 0;
    g->I = a->n_images; g->V = a->n_views; g->dt = a->img_dtype; g->apply_norm = a->apply_clip_norm; g->C = a->n_classes;
    g->rank_by = a->rank_by; g->k = a->k; g->cls_only = ctx->cls_only_last; g->stream = ctx->stream;
    const void* p[10] = {a->text_pt_dev, a->text_hand_dev, a->text_zs_dev, a->text_pt_t_dev, a->text_hand_t_dev, a->text_zs_t_dev,
                         a->lp.scale1, a->lp.bias1, a->lp.fc_w, a->lp.fc_b};
    for (int i = 0; i < 10; ++i) g->ptrs[i] = p[i];
    ctx->graphs.push_back(g);
  }
  g->last_use = ++tick;
  if (g->seen++ <= 0) return JCB_OK;          // first call with this key (or a key that failed to capture): the normal path
  DeviceGuard guard(ctx->device);
  const size_t in_bytes = static_cast<size_t>(a->n_images) * a->n_views * 3 * vit->cfg.resolution * vit->cfg.resolution *
                          img_elem_bytes(a->img_dtype);
  const size_t topk_bytes = static_cast<size_t>(a->n_images) * a->k * sizeof(int32_t);
  if (!g->exec) {
    g->ws_gen = ctx->ws_gen;
    if (!g->in_stage && cudaMalloc(&g->in_stage, in_bytes) != cudaSuccess) { cudaGetLastError(); g->seen = 0; return JCB_OK; }
    if (!g->topk_dev && cudaMalloc(reinterpret_cast<void**>(&g->topk_dev), topk_bytes) != cudaSuccess) { cudaGetLastError(); g->seen = 0; return JCB_OK; }
    jcb_pipeline_args inner = *a;
    inner.images = g->in_stage;
    inner.images_on_host = 0;
    inner.topk_on_host = 0;
    inner.out_topk = g->topk_dev;
    const uint64_t ws_before = ctx->ws_gen;
    const int64_t launches_before = ctx->launches;
    if (!ctx->capture_stream && cudaStreamCreateWithFlags(&ctx->capture_stream, cudaStreamNonBlocking) != cudaSuccess) {
      cudaGetLastError(); ctx->capture_stream = nullptr; ++ctx->graph_failures; g->seen = 0; return JCB_OK;
    }
    cudaStream_t user_stream = ctx->stream;
    if (cudaStreamBeginCapture(ctx->capture_stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
      cudaGetLastError(); ++ctx->graph_failures; g->seen = 0; return JCB_OK;
    }
    ctx->stream = ctx->capture_stream;
    const int rc = pipeline_enqueue(vit, vit_zs, &inner);
    ctx->stream = user_stream;
    cudaGraph_t graph = nullptr;
    const cudaError_t ce = cudaStreamEndCapture(ctx->capture_stream, &graph);
    if (rc != JCB_OK || ce != cudaSuccess || graph == nullptr || ctx->ws_gen != ws_before) {
      cudaGetLastError();
      if (graph) cudaGraphDestroy(graph);
      ctx->launches = launches_before;
      ++ctx->graph_failures;
      g->seen = -1000000;                      // this key cannot be captured: stay on the normal path
      return JCB_OK;
    }
    const cudaError_t ie = cudaGraphInstantiate(&g->exec, graph, 0);
    cudaGraphDestroy(graph);
    ctx->launches = launches_before;           // captured, not launched
    if (ie != cudaSuccess) { cudaGetLastError(); g->exec = nullptr; ++ctx->graph_failures; g->seen = -1000000; return JCB_OK; }
    ++ctx->graph_captures;
  }
  CUDA_TRY(ctx, cudaMemcpyAsync(g->in_stage, a->images, in_bytes, cudaMemcpyDefault, ctx->stream));
  CUDA_TRY(ctx, cudaGraphLaunch(g->exec, ctx->stream));
  CUDA_TRY(ctx, cudaMemcpyAsync(a->out_topk, g->topk_dev, topk_bytes, cudaMemcpyDefault, ctx->stream));
  ++ctx->graph_launches;
  ++ctx->launches;
  *handled = true;
  return JCB_OK;
}
}  // namespace

int jcb_pipeline(jcb_vit* vit, jcb_vit* vit_zs, const jcb_pipeline_args* a) {
  if (vit && a) {
    bool handled = false;
    int rc = pipeline_try_graph(vit, vit_zs, a, &handled);
    if (rc) return rc;
    if (handled) return a->topk_on_host ? sync_and_check(vit->ctx) : JCB_OK;
  }
  int rc = pipeline_enqueue(vit, vit_zs, a);
  if (rc) return rc;
  if (a->n_images > 0 && a->topk_on_host) return sync_and_check(vit->ctx);
  return JCB_OK;
}

int jcb_pipeline_slots(jcb_vit* vit, jcb_vit* vit_zs, const jcb_pipeline_args* a, const int32_t* slot_of_image_host) {
  int rc = pipeline_enqueue(vit, vit_zs, a, true, slot_of_image_host);   // never served from a captured graph
  if (rc) return rc;
  if (a->n_images > 0 && a->topk_on_host) return sync_and_check(vit->ctx);
  return JCB_OK;
}

}  // extern "C"
void graphs_clear_fwd(jcb_ctx* ctx) { graphs_clear(ctx); }
extern "C" {

int jcb_ctx_set_graphs(jcb_ctx* ctx, int on, int64_t max_views) {
  if (!ctx) return JCB_E_INVALID;
  if (max_views < 0) return fail(ctx, JCB_E_INVALID, "jcb_ctx_set_graphs: negative max_views");
  DeviceGuard g(ctx->device);
  ctx->graphs_on = on ? 1 : 0;
  if (max_views > 0) ctx->graph_max_views = max_views;
  if (!on) graphs_clear(ctx);
  return JCB_OK;
}

int jcb_ctx_graph_stats(const jcb_ctx* ctx, int64_t* captured, int64_t* launched, int64_t* failed) {
  if (!ctx) return JCB_E_INVALID;
  if (captured) *captured = ctx->graph_captures;
  if (launched) *launched = ctx->graph_launches;
  if (failed) *failed = ctx->graph_failures;
  return JCB_OK;
}

}  // extern "C"
namespace {
int pipeline_submit(jcb_vit* vit, jcb_vit* vit_zs, const jcb_pipeline_args* a, bool with_slots, const int32_t* slot_of_image,
                    int64_t* ticket) {
  int rc = check_vit(vit);
  if (rc) return rc;
  jcb_ctx* ctx = vit->ctx;
  if (!ticket) return fail(ctx, JCB_E_INVALID, "jcb_pipeline_submit: null ticket");
  if (ctx->next_ticket - ctx->waited_ticket >= JCB_MAX_INFLIGHT)
    return fail(ctx, JCB_E_STATE, "jcb_pipeline_submit: %d submissions already in flight; call jcb_pipeline_wait first",
                JCB_MAX_INFLIGHT);
  ctx->overlapped = ctx->next_ticket > ctx->waited_ticket;
  rc = pipeline_enqueue(vit, vit_zs, a, with_slots, slot_of_image);
  ctx->overlapped = false;
  if (rc) return rc;
  DeviceGuard g(ctx->device);
  const int slot = static_cast<int>(ctx->next_ticket % JCB_MAX_INFLIGHT);
  // the device status word as of the end of this submission travels to the host behind it: waiting needs no
  // stream-wide synchronisation (which would also wait for the submissions queued after this one)
  CUDA_TRY(ctx, cudaMemcpyAsync(&ctx->ticket_status[slot], ctx->dev_status, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(ctx, cudaEventRecord(ctx->ticket_done[slot], ctx->stream));
  *ticket = ctx->next_ticket++;
  return JCB_OK;
}
}  // namespace
extern "C" {

int jcb_pipeline_submit(jcb_vit* vit, jcb_vit* vit_zs, const jcb_pipeline_args* a, int64_t* ticket) {
  return pipeline_submit(vit, vit_zs, a, false, nullptr, ticket);
}

int jcb_pipeline_submit_slots(jcb_vit* vit, jcb_vit* vit_zs, const jcb_pipeline_args* a, const int32_t* slot_of_image_host,
                              int64_t* ticket) {
  return pipeline_submit(vit, vit_zs, a, true, slot_of_image_host, ticket);
}

int jcb_pipeline_wait(jcb_ctx* ctx, int64_t ticket) {
  if (!ctx) return JCB_E_INVALID;
  if (ticket < 0 || ticket >= ctx->next_ticket) return fail(ctx, JCB_E_INVALID, "jcb_pipeline_wait: unknown ticket %lld", static_cast<long long>(ticket));
  if (ticket < ctx->waited_ticket) return JCB_OK;   // tickets complete in order; this one was covered by a later wait
  DeviceGuard g(ctx->device);
  const int slot = static_cast<int>(ticket % JCB_MAX_INFLIGHT);
  CUDA_TRY(ctx, cudaEventSynchronize(ctx->ticket_done[slot]));
  ctx->waited_ticket = ticket + 1;
  const int st = ctx->ticket_status[slot];
  if (st != 0) {
    cudaMemsetAsync(ctx->dev_status, 0, sizeof(int), ctx->stream);
    return fail(ctx, JCB_E_KERNEL, "device-side kernel status %d (101 producer / 102 mma / 103 epilogue pipeline timeout, 104 smem alignment)", st);
  }
  return JCB_OK;
}

// ------------------------------------------------------------------------------------------------
int jcb_gemm(jcb_ctx* ctx, const jcb_gemm_args* g) {
  if (!ctx) return JCB_E_INVALID;
  if (!g || !g->A_dev || !g->B_dev || !g->out_dev) return fail(ctx, JCB_E_INVALID, "jcb_gemm: null pointer");
  if (g->epilogue == 3) return fail(ctx, JCB_E_INVALID, "jcb_gemm: epilogue 3 (conv1 scatter) no longer exists");
  if (g->operand_type != JCB_OPERAND_BF16 && g->operand_type != JCB_OPERAND_F16) return fail(ctx, JCB_E_INVALID, "jcb_gemm: bad operand_type");
  DeviceGuard guard(ctx->device);
  LnArgs ln;
  ln.stats = g->stats_dev; ln.slots = g->stats_slots; ln.colsum = g->colsum_dev; ln.out2 = g->out2_dev;
  ln.stats_in = g->stats_in_dev; ln.shift_in = g->shift_in_dev; ln.shift_out = g->shift_out_dev;
  ln.in_stride = g->stats_in_row_stride > 0 ? g->stats_in_row_stride : 1;
  if (g->K2 > 0) {
    ln.A2 = static_cast<const __nv_bfloat16*>(g->A2_dev); ln.B2 = static_cast<const __nv_bfloat16*>(g->B2_dev);
    ln.K2 = g->K2; ln.lda2 = g->lda2 > 0 ? g->lda2 : g->K2; ln.ldb2 = g->ldb2 > 0 ? g->ldb2 : g->K2;
  }
  return run_gemm(ctx, JCB_KC_OTHER, g->operand_type == JCB_OPERAND_F16, static_cast<const __nv_bfloat16*>(g->A_dev),
                  static_cast<const __nv_bfloat16*>(g->B_dev), g->M, g->N, g->K, g->bias_dev, g->epilogue, g->out_dev, g->ldo, ln);
}

int jcb_fold_ln(jcb_ctx* ctx, const float* W_dev, const float* gamma_dev, const float* beta_dev, const float* bias_dev,
                int32_t N, int32_t K, int32_t operand_type, void* Wf_dev, float* S_dev, float* c_dev) {
  if (!ctx) return JCB_E_INVALID;
  if (!W_dev || !gamma_dev || !beta_dev || !bias_dev || !Wf_dev || !S_dev || !c_dev || N < 1 || K < 1)
    return fail(ctx, JCB_E_INVALID, "jcb_fold_ln: bad arguments");
  DeviceGuard g(ctx->device);
  LAUNCH(ctx, launch_fold_ln(W_dev, gamma_dev, beta_dev, bias_dev, N, K, static_cast<__nv_bfloat16*>(Wf_dev), S_dev, c_dev,
                             ctx->stream, operand_type == JCB_OPERAND_F16));
  return JCB_OK;
}

int jcb_layernorm(jcb_ctx* ctx, const float* x, int64_t rows, int32_t width, const float* gamma, const float* beta,
                  int32_t operand_type, void* out) {
  if (!ctx) return JCB_E_INVALID;
  if (!x || !gamma || !beta || !out) return fail(ctx, JCB_E_INVALID, "jcb_layernorm: null pointer");
  DeviceGuard g(ctx->device);
  LAUNCH(ctx, launch_layernorm(x, rows, width, gamma, beta, static_cast<__nv_bfloat16*>(out), ctx->stream,
                               operand_type == JCB_OPERAND_F16));
  return JCB_OK;
}

int jcb_im2col(jcb_ctx* ctx, const void* images, int32_t img_dtype, int64_t n_views, int32_t resolution,
               int32_t patch, int32_t apply_clip_norm, int32_t operand_type, void* patches) {
  if (!ctx) return JCB_E_INVALID;
  if (!images || !patches) return fail(ctx, JCB_E_INVALID, "jcb_im2col: null pointer");
  if (img_dtype < 0 || img_dtype > 2 || n_views < 0) return fail(ctx, JCB_E_INVALID, "jcb_im2col: bad dtype / count");
  DeviceGuard g(ctx->device);
  LAUNCH(ctx, launch_im2col(images, img_dtype, n_views, resolution, patch, apply_clip_norm,
                            static_cast<__nv_bfloat16*>(patches), ctx->stream, operand_type == JCB_OPERAND_F16));
  return JCB_OK;
}

int jcb_attention(jcb_ctx* ctx, const void* qkv, int64_t n_views, int32_t tokens, int32_t heads, int32_t causal,
                  int32_t operand_type, void* out) {
  if (!ctx) return JCB_E_INVALID;
  if (!qkv || !out) return fail(ctx, JCB_E_INVALID, "jcb_attention: null pointer");
  DeviceGuard g(ctx->device);
  LAUNCH(ctx, launch_attention(static_cast<const __nv_bfloat16*>(qkv), n_views, tokens, heads,
                               static_cast<__nv_bfloat16*>(out), ctx->stream, causal, ctx->dev_status, ctx->num_sms,
                               operand_type == JCB_OPERAND_F16));
  return JCB_OK;
}

void jcb_tensor_map_cache_stats(uint64_t* hits, uint64_t* misses) { tmap_cache_stats(hits, misses); }

// ------------------------------------------------------------------------------------------------
// Minimal DLPack (dlpack.h v0.8) structures: enough to borrow a tensor.
namespace {
struct DLDevice { int32_t device_type; int32_t device_id; };
struct DLDataType { uint8_t code; uint8_t bits; uint16_t lanes; };
struct DLTensor {
  void* data; DLDevice device; int32_t ndim; DLDataType dtype; int64_t* shape; int64_t* strides; uint64_t byte_offset;
};
struct DLManagedTensor { DLTensor dl_tensor; void* manager_ctx; void (*deleter)(DLManagedTensor*); };
constexpr int kDLCUDA = 2, kDLUInt = 1, kDLFloat = 2, kDLBfloat = 4;
bool dl_contiguous(const DLTensor& t) {
  if (!t.strides) return true;
  int64_t expect = 1;
  for (int i = t.ndim - 1; i >= 0; --i) {
    if (t.shape[i] != 1 && t.strides[i] != expect) return false;
    expect *= t.shape[i];
  }
  return true;
}
}  // namespace

int jcb_encode_image_dlpack(jcb_vit* v, void* images_dlmanaged, void* out_dlmanaged, int apply_clip_norm, int normalize) {
  int rc = check_vit(v);
  if (rc) return rc;
  jcb_ctx* ctx = v->ctx;
  if (!images_dlmanaged || !out_dlmanaged) return fail(ctx, JCB_E_INVALID, "null DLManagedTensor");
  const DLTensor& in = static_cast<DLManagedTensor*>(images_dlmanaged)->dl_tensor;
  const DLTensor& out = static_cast<DLManagedTensor*>(out_dlmanaged)->dl_tensor;
  if (in.device.device_type != kDLCUDA || out.device.device_type != kDLCUDA || in.device.device_id != ctx->device ||
      out.device.device_id != ctx->device)
    return fail(ctx, JCB_E_INVALID, "DLPack tensors must live on CUDA device %d", ctx->device);
  int dt;
  if (in.dtype.code == kDLFloat && in.dtype.bits == 32) dt = JCB_IMG_F32;
  else if (in.dtype.code == kDLBfloat && in.dtype.bits == 16) dt = JCB_IMG_BF16;
  else if (in.dtype.code == kDLUInt && in.dtype.bits == 8) dt = JCB_IMG_U8;
  else return fail(ctx, JCB_E_INVALID, "unsupported image dtype (code %d, bits %d)", in.dtype.code, in.dtype.bits);
  const int R = v->cfg.resolution;
  if (in.ndim != 4 || in.shape[1] != 3 || in.shape[2] != R || in.shape[3] != R || !dl_contiguous(in))
    return fail(ctx, JCB_E_INVALID, "images must be contiguous [n, 3, %d, %d] (got ndim %d, shape [%lld, %lld, %lld, %lld], strides [%lld, %lld, %lld, %lld])",
                R, R, in.ndim, in.ndim > 0 ? (long long)in.shape[0] : -1LL, in.ndim > 1 ? (long long)in.shape[1] : -1LL,
                in.ndim > 2 ? (long long)in.shape[2] : -1LL, in.ndim > 3 ? (long long)in.shape[3] : -1LL,
                in.strides && in.ndim > 0 ? (long long)in.strides[0] : -1LL, in.strides && in.ndim > 1 ? (long long)in.strides[1] : -1LL,
                in.strides && in.ndim > 2 ? (long long)in.strides[2] : -1LL, in.strides && in.ndim > 3 ? (long long)in.strides[3] : -1LL);
  if (out.ndim != 2 || out.shape[0] != in.shape[0] || out.shape[1] != v->cfg.embed_dim || out.dtype.code != kDLFloat ||
      out.dtype.bits != 32 || !dl_contiguous(out))
    return fail(ctx, JCB_E_INVALID, "out must be contiguous float32 [n, %d]", v->cfg.embed_dim);
  DeviceGuard g(ctx->device);
  return encode_views(v, static_cast<const uint8_t*>(in.data) + in.byte_offset, dt, false, in.shape[0], apply_clip_norm,
                      normalize, reinterpret_cast<float*>(static_cast<uint8_t*>(out.data) + out.byte_offset), 0);
}

}  // extern "C"
