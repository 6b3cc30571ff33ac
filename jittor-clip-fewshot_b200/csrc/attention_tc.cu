// Image-tower attention on the 5th-generation tensor cores: softmax(Q K^T / sqrt(64)) V for T <= 64 tokens per
// sequence, two heads per work item, operands moved by TMA and multiplied by tcgen05.mma, scores / probabilities /
// outputs held in TMEM.  The kernel streams 8 B per element of [T, W] and is bound by HBM; the mma.sync kernel
// (attention.cu) it replaces on this path spent 2/3 of its time in the shared-memory pipe (ldmatrix of K and V by
// every warp) -- here no operand crosses the LSU at all.
//
//   work item = (sequence, pair of adjacent heads A | B); persistent CTAs, 2 per SM, 256 TMEM columns each
//   warp 0   TMA producer : six 4-D boxes per item -- Q, K, V of both heads, each [64 tokens][64] bf16 with 128-byte
//                           swizzle; token rows >= T are out of bounds of the tensor map -> zero filled, never read
//                           from HBM
//   warp 1   MMA issuer   : S[128,128] = [Q_A;Q_B] [K_A;K_B]^T   (UMMA 128x128x16 x4, both operands K-major smem);
//                           the diagonal 64x64 blocks are the two heads' scores, the off-diagonal blocks are ignored.
//                           O[128,64] = P [V_A;V_B]              (UMMA 128x64x16 x8, A = P from TMEM, B = V MN-major
//                           smem); P is block diagonal (zeros written once), so each head sees only its own keys.
//   warps 2-5 softmax + epilogue : thread = query row = TMEM lane.  tcgen05.ld the row's 64 scores, fp32 softmax
//                           (exp2, 1/8 scale folded in, keys >= T masked), P as bf16 pairs back to TMEM (tcgen05.st);
//                           then O * 1/rowsum -> bf16 -> swizzled smem -> one 4-D TMA store per item (rows >= T clipped).
//
//
// MODE 1 (text tower, or any T in 65..128): work item = (sequence, ONE head); the 128 tile rows are the head's token
// rows 0..127 (two 64-token boxes per matrix, rows >= T zero-filled), S = Q K^T is the head's full 128 x 128 score
// matrix, P is dense, and the softmax applies the causal mask of the text tower (key j visible to query i iff j <= i,
// jclip/model.py:189-193 build_attention_mask) on the fly.  Same shared-memory / TMEM layout and MMA sequence.
//
// LONG FORM (attention_tcgen05_long_kernel, 129 <= T <= 256, no mask: the ViT-B/16 image tower, 197 / 201 tokens):
// work item = (sequence, head, query tile qt in {0, 1}); the two query tiles of a head are adjacent items, so they run
// on neighbouring CTAs at the same time and the second read of the head's K and V hits L2.  Q = two 64-token boxes at
// tokens 128 qt + {0, 64}, K and V = the head's whole key range, ceil(T / 64) boxes each (boxes wholly beyond T are
// neither loaded nor multiplied: the K / V box at token 192 for T <= 192, and Q box 1 of tile 1).
//   S[128, 64 nkb] = Q K^T      (UMMA 128 x 64nkb x 16, x4; S fills up to 256 TMEM columns)
//   softmax                      two passes over S in 32-column chunks (maximum, then exponentials), exact: the whole
//                                row stays on chip, no online rescaling; P as 16-bit pairs over the score columns already
//                                read (P column j <- scores 2j, 2j + 1; columns 0..127)
//   O[128, 64] = P V            (UMMA 128x64x16, 4 nkb steps, A = P from TMEM, B = V MN-major) into score columns
//                                128..191 (read before P was published), then O / rowsum -> 16 bits -> TMA store
// Everything aliases into 256 TMEM columns, so two CTAs (one 80 KB Q | K | V stage + 16 KB output staging each) share
// an SM; the next item's scores wait until the epilogue has read O (tmem_free barrier).  One CTA per SM with two
// Q | K | V stages measured 1.076 against 0.874 ms for this form (T = 197, 12 heads, 2048 sequences; DESIGN.md section 4).
//
// The 16-bit element type (bf16 | fp16) of Q, K, V, P and the output is the template parameter F16.
//
// Reference: jclip/mha.py:55-83 scaled_dot_product_attention (attn_mask None for the vision tower,
// jclip/model.py:99; dropout 0 in eval), head split jclip/mha.py:351-362 / test.py:584-590.
#include <cstdlib>
#include <map>
#include <mutex>
#include <cudaTypedefs.h>

#include "kernels.h"
#include "ptx.cuh"

namespace jcb {

void* gemm_encode_tiled_fn();  // gemm.cu: cuTensorMapEncodeTiled resolved through the runtime

namespace {

constexpr int HD = 64;                    // head dim
constexpr int TILE = 64 * HD * 2;         // one head's [64 tokens][64] bf16 tile: 8 KB
constexpr int MAT_BYTES = 2 * TILE;       // both heads of a pair: 16 KB
constexpr int STAGE_BYTES = 3 * MAT_BYTES;  // Q | K | V
constexpr int NSTAGE = 2;
constexpr int OUT_BYTES = MAT_BYTES;      // bf16 output staging, same [2][64][128 B] swizzled shape
constexpr int BAR_BYTES = 128;
constexpr int ATC_SMEM = NSTAGE * STAGE_BYTES + OUT_BYTES + BAR_BYTES;   // 114816 B -> two CTAs per SM
constexpr int ATC_THREADS = 192;
constexpr int TMEM_COLS = 256;
constexpr uint32_t S_COL = 0, P_COL = 128, O_COL = 192;

struct AtcDev {
  long long n_items;   // sequences * head pairs (MODE 0) / sequences * heads (MODE 1)
  int pairs;           // work items per sequence
  int T;
  int causal;          // MODE 1 only
  int* status;
};

// TCT = the token count as a compile-time constant (50 = plain tower, 54 = IVLP / VPT tower) so the softmax touches only
// the valid keys; 0 = run-time T (any T <= 64).
template <int TCT, bool F16, int MODE>
__global__ void __launch_bounds__(ATC_THREADS, 2)
attention_tcgen05_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmOut,
                         const AtcDev p) {
  extern __shared__ __align__(1024) uint8_t atc_smem[];
  uint8_t* ring = atc_smem;
  uint8_t* ostage = atc_smem + NSTAGE * STAGE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(ostage + OUT_BYTES);
  uint64_t* full_bar = bars;            // [NSTAGE] TMA -> MMA
  uint64_t* empty_bar = bars + NSTAGE;  // [NSTAGE] MMA (P V done) -> TMA
  uint64_t* s_full = bars + 2 * NSTAGE;       // scores in TMEM          MMA -> softmax
  uint64_t* p_full = bars + 2 * NSTAGE + 1;   // probabilities in TMEM   softmax (128 arrivals) -> MMA
  uint64_t* o_full = bars + 2 * NSTAGE + 2;   // outputs in TMEM         MMA -> epilogue
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * NSTAGE + 3);

  const int warp_idx = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    if ((smem_u32(atc_smem) & 1023u) != 0u) atomicCAS(p.status, 0, JCB_DEV_SMEM_ALIGN);
    tma_prefetch_desc(&tmQKV);
    tma_prefetch_desc(&tmOut);
    for (int s = 0; s < NSTAGE; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(p_full, 128);
    mbar_init(o_full, 1);
    fence_mbar_init();
    fence_proxy_async_smem();
  }
  if (warp_idx == 1) {
    tmem_alloc(tmem_ptr_smem, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_ptr_smem);
  griddep_wait();               // programmatic dependent launch (ptx.cuh): nothing global is touched above

  if (warp_idx == 0) {
    // ===================================================================== TMA producer
    if (elect_one()) {
      int it = 0;
      for (long long item = blockIdx.x; item < p.n_items; item += gridDim.x, ++it) {
        const int stage = it % NSTAGE;
        const uint32_t phase = static_cast<uint32_t>(it / NSTAGE) & 1u;
        if (!mbar_wait(&empty_bar[stage], phase ^ 1u, p.status, JCB_DEV_TIMEOUT_PRODUCER)) break;
        const int view = static_cast<int>(item / p.pairs);
        const int hp = static_cast<int>(item % p.pairs);
        uint8_t* dst = ring + stage * STAGE_BYTES;
        mbar_arrive_expect_tx(&full_bar[stage], STAGE_BYTES);
        // coordinates: (d, 64-wide column block of the [T, 3W] row, token, sequence); blocks: q | k | v heads
#pragma unroll
        for (int m = 0; m < 3; ++m)
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            if (MODE == 0)   // head 2 hp + h, tokens 0..63
              tma_load_4d(dst + m * MAT_BYTES + h * TILE, &tmQKV, &full_bar[stage], 0, 2 * m * p.pairs + 2 * hp + h, 0, view);
            else             // head hp, tokens 64 h .. 64 h + 63
              tma_load_4d(dst + m * MAT_BYTES + h * TILE, &tmQKV, &full_bar[stage], 0, m * p.pairs + hp, 64 * h, view);
          }
      }
    }
  } else if (warp_idx == 1) {
    // ===================================================================== MMA issuer
    if (elect_one()) {
      constexpr uint32_t idesc_s = umma_idesc_f32acc(F16, 128, 128);
      constexpr uint32_t idesc_o = umma_idesc_f32acc(F16, 128, 64, /*b_mn_major=*/true);
      int it = 0;
      for (long long item = blockIdx.x; item < p.n_items; item += gridDim.x, ++it) {
        const int stage = it % NSTAGE;
        const uint32_t phase = static_cast<uint32_t>(it / NSTAGE) & 1u;
        const uint32_t iphase = static_cast<uint32_t>(it) & 1u;
        if (!mbar_wait(&full_bar[stage], phase, p.status, JCB_DEV_TIMEOUT_MMA)) break;
        tc_fence_after();
        const uint32_t sq = smem_u32(ring + stage * STAGE_BYTES);
        const uint64_t dq = umma_desc_sw128(sq);
        const uint64_t dk = umma_desc_sw128(sq + MAT_BYTES);
        // the score columns are free: the softmax warps finished reading the previous item's scores before they
        // published its probabilities, which this thread waited for below
#pragma unroll
        for (int k = 0; k < HD / 16; ++k)
          umma_bf16(tmem_base + S_COL, dq + static_cast<uint64_t>(2 * k), dk + static_cast<uint64_t>(2 * k), idesc_s,
                    k != 0 ? 1u : 0u);
        umma_commit(s_full);
        if (!mbar_wait(p_full, iphase, p.status, JCB_DEV_TIMEOUT_MMA)) break;
        tc_fence_after();
        const uint64_t dv = umma_desc_sw128_mn(sq + 2 * MAT_BYTES);
        // 128 keys (64 of head A, 64 of head B) in steps of 16: 8 TMEM columns of P, 16 rows (2048 B) of V per step
#pragma unroll
        for (int ks = 0; ks < 8; ++ks)
          umma_bf16_ts(tmem_base + O_COL, tmem_base + P_COL + static_cast<uint32_t>(8 * ks),
                       dv + static_cast<uint64_t>(ks * (2048 >> 4)), idesc_o, ks != 0 ? 1u : 0u);
        umma_commit(&empty_bar[stage]);   // Q, K, V of this stage have been read
        umma_commit(o_full);
      }
    }
  } else {
    // ===================================================================== softmax + epilogue (warps 2..5)
    const int q = warp_idx & 3;              // TMEM lane quarter this warp may access
    const int head = q >> 1;                 // rows 0..63 = head A, 64..127 = head B
    const int row = (q & 1) * 32 + lane;     // token row within the head
    const bool leader = warp_idx == 2 && lane == 0;
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const float scale_log2 = 0.125f * 1.4426950408889634f;  // 1/sqrt(64) * log2(e)
    // the other head's half of this row's probabilities stays zero for the whole kernel (block-diagonal P)
    if (MODE == 0) {
      uint32_t z[32];
#pragma unroll
      for (int i = 0; i < 32; ++i) z[i] = 0u;
      tmem_st_32x32b_x32(lane_base + P_COL + static_cast<uint32_t>((1 - head) * 32), z);
      tmem_st_wait();
    }
    int it = 0;
    bool ok = true;
    for (long long item = blockIdx.x; item < p.n_items && ok; item += gridDim.x, ++it) {
      const uint32_t iphase = static_cast<uint32_t>(it) & 1u;
      ok = mbar_wait(s_full, iphase, p.status, JCB_DEV_TIMEOUT_EPILOGUE);
      ok = __all_sync(0xffffffffu, ok);
      if (!ok) break;
      tc_fence_after();
      const int T = TCT > 0 ? TCT : p.T;
      float sum;
      if (MODE == 0) {
        uint32_t sv[64];
        tmem_ld_32x32b_x32(lane_base + S_COL + static_cast<uint32_t>(head * 64), *reinterpret_cast<uint32_t(*)[32]>(&sv[0]));
        tmem_ld_32x32b_x32(lane_base + S_COL + static_cast<uint32_t>(head * 64 + 32), *reinterpret_cast<uint32_t(*)[32]>(&sv[32]));
        tmem_ld_wait();
        // row maximum over the valid keys and the exponentials' sum, each as four independent chains (a single chain of
        // 64 dependent FMNMX / FADD was a quarter of the per-item critical path); 1/8 and log2(e) ride in the FMA
        float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
        for (int c = 0; c < 64; ++c)
          if (c < T) m4[c & 3] = fmaxf(m4[c & 3], __uint_as_float(sv[c]));
        const float nmx = -fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])) * scale_log2;
        float s4[4] = {0.f, 0.f, 0.f, 0.f};
        uint32_t pv[32];
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          const float p0 = 2 * c < T ? ex2_approx(fmaf(__uint_as_float(sv[2 * c]), scale_log2, nmx)) : 0.f;
          const float p1 = 2 * c + 1 < T ? ex2_approx(fmaf(__uint_as_float(sv[2 * c + 1]), scale_log2, nmx)) : 0.f;
          s4[c & 3] += p0 + p1;
          pv[c] = pack_h2<F16>(p0, p1);
        }
        sum = (s4[0] + s4[1]) + (s4[2] + s4[3]);
        tmem_st_32x32b_x32(lane_base + P_COL + static_cast<uint32_t>(head * 32), pv);
      } else {
        // one head, 128 key columns: two passes over the scores in TMEM (maximum, then exponentials) keep the row in
        // 32 registers at a time.  Key c is visible to query row r = q * 32 + lane iff c < T and (causal) c <= r;
        // column 0 is always visible, so padding rows (r >= T, all-zero Q) stay finite; they are clipped on store.
        const int r = q * 32 + lane;
        const int lim = p.causal ? (r + 1 < T ? r + 1 : T) : T;   // visible keys: [0, lim)
        float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          uint32_t sv[32];
          tmem_ld_32x32b_x32(lane_base + S_COL + static_cast<uint32_t>(ch * 32), sv);
          tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < 32; ++c)
            if (ch * 32 + c < lim) m4[c & 3] = fmaxf(m4[c & 3], __uint_as_float(sv[c]));
        }
        const float nmx = -fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])) * scale_log2;
        float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          uint32_t pv[32];
#pragma unroll
          for (int ch = 0; ch < 2; ++ch) {
            uint32_t sv[32];
            tmem_ld_32x32b_x32(lane_base + S_COL + static_cast<uint32_t>(hf * 64 + ch * 32), sv);
            tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < 16; ++c) {
              const int k0 = hf * 64 + ch * 32 + 2 * c;
              const float p0 = k0 < lim ? ex2_approx(fmaf(__uint_as_float(sv[2 * c]), scale_log2, nmx)) : 0.f;
              const float p1 = k0 + 1 < lim ? ex2_approx(fmaf(__uint_as_float(sv[2 * c + 1]), scale_log2, nmx)) : 0.f;
              s4[c & 3] += p0 + p1;
              pv[ch * 16 + c] = pack_h2<F16>(p0, p1);
            }
          }
          tmem_st_32x32b_x32(lane_base + P_COL + static_cast<uint32_t>(hf * 32), pv);
        }
        sum = (s4[0] + s4[1]) + (s4[2] + s4[3]);
      }
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(p_full);
      const float inv = 1.0f / sum;

      ok = mbar_wait(o_full, iphase, p.status, JCB_DEV_TIMEOUT_EPILOGUE);
      ok = __all_sync(0xffffffffu, ok);
      if (!ok) break;
      tc_fence_after();
      uint32_t ov[64];
      tmem_ld_32x32b_x32(lane_base + O_COL, *reinterpret_cast<uint32_t(*)[32]>(&ov[0]));
      tmem_ld_32x32b_x32(lane_base + O_COL + 32, *reinterpret_cast<uint32_t(*)[32]>(&ov[32]));
      // the previous item's store must have finished reading the staging tile before it is overwritten
      if (leader) bulk_wait_read<0>();
      named_bar_sync(1, 128);
      tmem_ld_wait();
      uint8_t* rowp = ostage + head * TILE + row * 128;
#pragma unroll
      for (int j = 0; j < 8; ++j) {  // 16-byte piece j of this row, XOR-swizzled by row % 8
        uint4 o;
        o.x = pack_h2<F16>(__uint_as_float(ov[8 * j + 0]) * inv, __uint_as_float(ov[8 * j + 1]) * inv);
        o.y = pack_h2<F16>(__uint_as_float(ov[8 * j + 2]) * inv, __uint_as_float(ov[8 * j + 3]) * inv);
        o.z = pack_h2<F16>(__uint_as_float(ov[8 * j + 4]) * inv, __uint_as_float(ov[8 * j + 5]) * inv);
        o.w = pack_h2<F16>(__uint_as_float(ov[8 * j + 6]) * inv, __uint_as_float(ov[8 * j + 7]) * inv);
        *reinterpret_cast<uint4*>(rowp + ((j ^ (row & 7)) << 4)) = o;
      }
      fence_proxy_async_smem();
      tc_fence_before();   // this row's TMEM reads are complete before the MMA issuer may overwrite S / O
      named_bar_sync(1, 128);
      if (leader) {
        const int view = static_cast<int>(item / p.pairs);
        const int hp = static_cast<int>(item % p.pairs);
        if (MODE == 0) {
          tma_store_4d(&tmOut, ostage, 0, 2 * hp, 0, view);
          tma_store_4d(&tmOut, ostage + TILE, 0, 2 * hp + 1, 0, view);
        } else {
          tma_store_4d(&tmOut, ostage, 0, hp, 0, view);
          if (p.T > 64) tma_store_4d(&tmOut, ostage + TILE, 0, hp, 64, view);
        }
        bulk_commit();
      }
    }
    if (leader) bulk_wait<0>();
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------------- long form
constexpr int LQ_BYTES = 2 * TILE;                 // 128 query rows
constexpr int LKV_BYTES = 4 * TILE;                // up to 256 key rows, 256 contiguous 128-byte rows
constexpr int LSTAGE_BYTES = LQ_BYTES + 2 * LKV_BYTES;   // Q | K | V: 80 KB
constexpr int LOUT_BYTES = 2 * TILE;
constexpr int ATL_SMEM = LSTAGE_BYTES + LOUT_BYTES + BAR_BYTES;   // 98432 B -> two CTAs per SM
constexpr uint32_t L_S_COL = 0, L_P_COL = 0, L_O_COL = 128;

struct AtlDev {
  long long n_items;   // sequences * heads * 2
  int heads;
  int T;
  int* status;
};

template <bool F16>
__global__ void __launch_bounds__(ATC_THREADS, 2)
attention_tcgen05_long_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmOut,
                              const AtlDev p) {
  extern __shared__ __align__(1024) uint8_t atl_smem[];
  uint8_t* sq = atl_smem;
  uint8_t* ostage = atl_smem + LSTAGE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(ostage + LOUT_BYTES);
  uint64_t* full_bar = bars;        // TMA -> MMA
  uint64_t* empty_bar = bars + 1;   // MMA (P V done) -> TMA
  uint64_t* s_full = bars + 2;      // scores in TMEM          MMA -> softmax
  uint64_t* p_full = bars + 3;      // probabilities in TMEM   softmax (128 arrivals) -> MMA
  uint64_t* o_full = bars + 4;      // outputs in TMEM         MMA -> epilogue
  uint64_t* tmem_free = bars + 5;   // outputs read            epilogue (128 arrivals) -> MMA (next item's scores)
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 6);

  const int warp_idx = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int T = p.T;
  const int nkb = (T + 63) >> 6;   // 64-key boxes that hold valid keys: 3 (T <= 192) or 4

  if (threadIdx.x == 0) {
    if ((smem_u32(atl_smem) & 1023u) != 0u) atomicCAS(p.status, 0, JCB_DEV_SMEM_ALIGN);
    tma_prefetch_desc(&tmQKV);
    tma_prefetch_desc(&tmOut);
    mbar_init(full_bar, 1);
    mbar_init(empty_bar, 1);
    mbar_init(s_full, 1);
    mbar_init(p_full, 128);
    mbar_init(o_full, 1);
    mbar_init(tmem_free, 128);
    fence_mbar_init();
    fence_proxy_async_smem();
  }
  if (warp_idx == 1) {
    tmem_alloc(tmem_ptr_smem, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_ptr_smem);
  griddep_wait();               // programmatic dependent launch (ptx.cuh): nothing global is touched above

  if (warp_idx == 0) {
    // ===================================================================== TMA producer
    if (elect_one()) {
      int it = 0;
      for (long long item = blockIdx.x; item < p.n_items; item += gridDim.x, ++it) {
        if (!mbar_wait(empty_bar, (static_cast<uint32_t>(it) & 1u) ^ 1u, p.status, JCB_DEV_TIMEOUT_PRODUCER)) break;
        const int qt = static_cast<int>(item & 1);
        const long long sh = item >> 1;
        const int seq = static_cast<int>(sh / p.heads);
        const int h = static_cast<int>(sh % p.heads);
        const int nq = 128 * qt + 64 < T ? 2 : 1;
        mbar_arrive_expect_tx(full_bar, static_cast<uint32_t>((nq + 2 * nkb) * TILE));
        // coordinates: (d, 64-wide column block of the [T, 3W] row, token, sequence); blocks: q | k | v heads
        for (int b = 0; b < nq; ++b)
          tma_load_4d(sq + b * TILE, &tmQKV, full_bar, 0, h, 128 * qt + 64 * b, seq);
        for (int b = 0; b < nkb; ++b) {
          tma_load_4d(sq + LQ_BYTES + b * TILE, &tmQKV, full_bar, 0, p.heads + h, 64 * b, seq);
          tma_load_4d(sq + LQ_BYTES + LKV_BYTES + b * TILE, &tmQKV, full_bar, 0, 2 * p.heads + h, 64 * b, seq);
        }
      }
    }
  } else if (warp_idx == 1) {
    // ===================================================================== MMA issuer
    if (elect_one()) {
      const uint32_t idesc_s = umma_idesc_f32acc(F16, 128, 64 * nkb);
      constexpr uint32_t idesc_o = umma_idesc_f32acc(F16, 128, 64, /*b_mn_major=*/true);
      const uint32_t sa = smem_u32(sq);
      const uint64_t dq = umma_desc_sw128(sa);
      const uint64_t dk = umma_desc_sw128(sa + LQ_BYTES);
      const uint64_t dv = umma_desc_sw128_mn(sa + LQ_BYTES + LKV_BYTES);
      int it = 0;
      for (long long item = blockIdx.x; item < p.n_items; item += gridDim.x, ++it) {
        const uint32_t iphase = static_cast<uint32_t>(it) & 1u;
        if (!mbar_wait(full_bar, iphase, p.status, JCB_DEV_TIMEOUT_MMA)) break;
        // S, P and O share the columns: the previous item's outputs must have been read out
        if (it > 0 && !mbar_wait(tmem_free, iphase ^ 1u, p.status, JCB_DEV_TIMEOUT_MMA)) break;
        tc_fence_after();
#pragma unroll
        for (int k = 0; k < HD / 16; ++k)
          umma_bf16(tmem_base + L_S_COL, dq + static_cast<uint64_t>(2 * k), dk + static_cast<uint64_t>(2 * k), idesc_s,
                    k != 0 ? 1u : 0u);
        umma_commit(s_full);
        if (!mbar_wait(p_full, iphase, p.status, JCB_DEV_TIMEOUT_MMA)) break;
        tc_fence_after();
        // keys in steps of 16: 8 TMEM columns of P, 16 rows (2048 B) of V per step; the V boxes are contiguous
        for (int ks = 0; ks < 4 * nkb; ++ks)
          umma_bf16_ts(tmem_base + L_O_COL, tmem_base + L_P_COL + static_cast<uint32_t>(8 * ks),
                       dv + static_cast<uint64_t>(ks * (2048 >> 4)), idesc_o, ks != 0 ? 1u : 0u);
        umma_commit(empty_bar);   // Q, K, V have been read
        umma_commit(o_full);
      }
    }
  } else {
    // ===================================================================== softmax + epilogue (warps 2..5)
    const int q = warp_idx & 3;              // TMEM lane quarter this warp may access
    const int r = q * 32 + lane;             // query row within the tile
    const bool leader = warp_idx == 2 && lane == 0;
    const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const float scale_log2 = 0.125f * 1.4426950408889634f;  // 1/sqrt(64) * log2(e)
    int it = 0;
    bool ok = true;
    for (long long item = blockIdx.x; item < p.n_items && ok; item += gridDim.x, ++it) {
      const uint32_t iphase = static_cast<uint32_t>(it) & 1u;
      ok = mbar_wait(s_full, iphase, p.status, JCB_DEV_TIMEOUT_EPILOGUE);
      ok = __all_sync(0xffffffffu, ok);
      if (!ok) break;
      tc_fence_after();
      // pass 1: row maximum over the keys < T, four independent chains.  Rows of tile 1 beyond T hold stale or zero
      // queries; their results are clipped on store.
      float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
      for (int ch = 0; ch < 2 * nkb; ++ch) {
        uint32_t sv[32];
        tmem_ld_32x32b_x32(lane_base + L_S_COL + static_cast<uint32_t>(ch * 32), sv);
        tmem_ld_wait();
        if (ch * 32 + 32 <= T) {
#pragma unroll
          for (int c = 0; c < 32; ++c) m4[c & 3] = fmaxf(m4[c & 3], __uint_as_float(sv[c]));
        } else {
#pragma unroll
          for (int c = 0; c < 32; ++c)
            if (ch * 32 + c < T) m4[c & 3] = fmaxf(m4[c & 3], __uint_as_float(sv[c]));
        }
      }
      const float nmx = -fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])) * scale_log2;
      // pass 2: exponentials per 64-key box; P for keys 64 hf .. 64 hf + 63 goes to columns 32 hf .. 32 hf + 31,
      // whose scores were read in this or the previous box
      float s4[4] = {0.f, 0.f, 0.f, 0.f};
      for (int hf = 0; hf < nkb; ++hf) {
        uint32_t pv[32];
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
          uint32_t sv[32];
          tmem_ld_32x32b_x32(lane_base + L_S_COL + static_cast<uint32_t>(hf * 64 + ch * 32), sv);
          tmem_ld_wait();
#pragma unroll
          for (int c = 0; c < 16; ++c) {
            const int k0 = hf * 64 + ch * 32 + 2 * c;
            const float p0 = k0 < T ? ex2_approx(fmaf(__uint_as_float(sv[2 * c]), scale_log2, nmx)) : 0.f;
            const float p1 = k0 + 1 < T ? ex2_approx(fmaf(__uint_as_float(sv[2 * c + 1]), scale_log2, nmx)) : 0.f;
            s4[c & 3] += p0 + p1;
            pv[ch * 16 + c] = pack_h2<F16>(p0, p1);
          }
        }
        tmem_st_32x32b_x32(lane_base + L_P_COL + static_cast<uint32_t>(hf * 32), pv);
      }
      const float sum = (s4[0] + s4[1]) + (s4[2] + s4[3]);
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(p_full);
      const float inv = 1.0f / sum;

      ok = mbar_wait(o_full, iphase, p.status, JCB_DEV_TIMEOUT_EPILOGUE);
      ok = __all_sync(0xffffffffu, ok);
      if (!ok) break;
      tc_fence_after();
      uint32_t ov[64];
      tmem_ld_32x32b_x32(lane_base + L_O_COL, *reinterpret_cast<uint32_t(*)[32]>(&ov[0]));
      tmem_ld_32x32b_x32(lane_base + L_O_COL + 32, *reinterpret_cast<uint32_t(*)[32]>(&ov[32]));
      tmem_ld_wait();
      tc_fence_before();   // this row's TMEM reads are complete: the next item's scores may overwrite the columns
      mbar_arrive(tmem_free);
      // the previous item's store must have finished reading the staging tile before it is overwritten
      if (leader) bulk_wait_read<0>();
      named_bar_sync(1, 128);
      uint8_t* rowp = ostage + (r >> 6) * TILE + (r & 63) * 128;
#pragma unroll
      for (int j = 0; j < 8; ++j) {  // 16-byte piece j of this row, XOR-swizzled by row % 8
        uint4 o;
        o.x = pack_h2<F16>(__uint_as_float(ov[8 * j + 0]) * inv, __uint_as_float(ov[8 * j + 1]) * inv);
        o.y = pack_h2<F16>(__uint_as_float(ov[8 * j + 2]) * inv, __uint_as_float(ov[8 * j + 3]) * inv);
        o.z = pack_h2<F16>(__uint_as_float(ov[8 * j + 4]) * inv, __uint_as_float(ov[8 * j + 5]) * inv);
        o.w = pack_h2<F16>(__uint_as_float(ov[8 * j + 6]) * inv, __uint_as_float(ov[8 * j + 7]) * inv);
        *reinterpret_cast<uint4*>(rowp + ((j ^ (r & 7)) << 4)) = o;
      }
      fence_proxy_async_smem();
      named_bar_sync(1, 128);
      if (leader) {
        const int qt = static_cast<int>(item & 1);
        const long long sh = item >> 1;
        const int seq = static_cast<int>(sh / p.heads);
        const int h = static_cast<int>(sh % p.heads);
        tma_store_4d(&tmOut, ostage, 0, h, 128 * qt, seq);
        if (128 * qt + 64 < T) tma_store_4d(&tmOut, ostage + TILE, 0, h, 128 * qt + 64, seq);
        bulk_commit();
      }
    }
    if (leader) bulk_wait<0>();
  }

  tc_fence_before();
  __syncthreads();
  if (warp_idx == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

struct HeadsKey {
  const void* base; uint64_t n_seq, T, blocks; int f16;
  bool operator<(const HeadsKey& o) const {
    if (base != o.base) return base < o.base;
    if (n_seq != o.n_seq) return n_seq < o.n_seq;
    if (T != o.T) return T < o.T;
    if (blocks != o.blocks) return blocks < o.blocks;
    return f16 < o.f16;
  }
};
std::mutex g_heads_mu;
std::map<HeadsKey, CUtensorMap> g_heads_cache;

}  // namespace

// [n_seq, T, blocks, 64] 16-bit elements as a 4-D tensor (d, block, token, sequence); boxes of 64 x 1 x 64 x 1 = one
// head's [64 tokens][64] tile.  The token dimension is T long, so the rows T.. of a box are out of bounds: zero on
// load, dropped on store.  Encoded once per (pointer, shape) and cached (same reason as gemm.cu's cache).  Also used by
// the attention backward (train.cu).
bool make_tmap_heads(CUtensorMap* tm, const void* base, uint64_t n_seq, uint64_t T, uint64_t blocks, int f16) {
  const HeadsKey key{base, n_seq, T, blocks, f16};
  {
    std::lock_guard<std::mutex> lock(g_heads_mu);
    auto it = g_heads_cache.find(key);
    if (it != g_heads_cache.end()) { *tm = it->second; return true; }
  }
  auto encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(gemm_encode_tiled_fn());
  if (!encode) return false;
  const uint64_t row_bytes = blocks * HD * 2;
  cuuint64_t gdim[4] = {HD, blocks, T, n_seq};
  cuuint64_t gstride[3] = {HD * 2, row_bytes, T * row_bytes};
  cuuint32_t box[4] = {HD, 1, 64, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = encode(tm, f16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4,
                      const_cast<void*>(base), gdim, gstride, box, estr,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return false;
  std::lock_guard<std::mutex> lock(g_heads_mu);
  if (g_heads_cache.size() >= 2048) g_heads_cache.clear();
  g_heads_cache.emplace(key, *tm);
  return true;
}

namespace {

template <int TCT, int MODE>
cudaError_t launch_atc(const CUtensorMap& tmQKV, const CUtensorMap& tmOut, const AtcDev& p, int f16, int num_sms,
                       cudaStream_t stream) {
  auto kernel = f16 ? attention_tcgen05_kernel<TCT, true, MODE> : attention_tcgen05_kernel<TCT, false, MODE>;
  cudaError_t e = ensure_dynamic_smem(kernel, ATC_SMEM);
  if (e != cudaSuccess) return e;
  const long long max_ctas = 2LL * num_sms;
  const unsigned grid = static_cast<unsigned>(p.n_items < max_ctas ? p.n_items : max_ctas);
  return launch_pdl(kernel, dim3(grid), dim3(ATC_THREADS), ATC_SMEM, stream, 1, tmQKV, tmOut, p);
}

cudaError_t launch_atl(const CUtensorMap& tmQKV, const CUtensorMap& tmOut, const AtlDev& p, int f16, int num_sms,
                       cudaStream_t stream) {
  auto kernel = f16 ? attention_tcgen05_long_kernel<true> : attention_tcgen05_long_kernel<false>;
  cudaError_t e = ensure_dynamic_smem(kernel, ATL_SMEM);
  if (e != cudaSuccess) return e;
  const long long max_ctas = 2LL * num_sms;
  const unsigned grid = static_cast<unsigned>(p.n_items < max_ctas ? p.n_items : max_ctas);
  return launch_pdl(kernel, dim3(grid), dim3(ATC_THREADS), ATL_SMEM, stream, 1, tmQKV, tmOut, p);
}

}  // namespace

// two heads per 128-row tile (T <= 64, no mask, even head count), one head per tile (T <= 128, optional causal mask)
// or one head and one of two 128-row query tiles per item (129 <= T <= 256, no mask)
bool attention_tc_supported(int T, int heads, int causal) {
  if (T < 1 || heads < 1) return false;
  if (!causal && T <= 64 && heads % 2 == 0) return true;
  if (T <= 128) return true;
  return !causal && T <= 256;
}

cudaError_t launch_attention_tc(const __nv_bfloat16* qkv, int64_t n_views, int T, int heads, __nv_bfloat16* out,
                                cudaStream_t stream, int* dev_status, int num_sms, int f16, int causal) {
  if (!attention_tc_supported(T, heads, causal) || dev_status == nullptr || num_sms < 1) return cudaErrorInvalidValue;
  if (n_views == 0) return cudaSuccess;
  if ((reinterpret_cast<uintptr_t>(qkv) & 15) || (reinterpret_cast<uintptr_t>(out) & 15)) return cudaErrorInvalidValue;
  CUtensorMap tmQKV, tmOut;
  if (!make_tmap_heads(&tmQKV, qkv, static_cast<uint64_t>(n_views), static_cast<uint64_t>(T), 3ull * heads, f16))
    return cudaErrorInvalidValue;
  if (!make_tmap_heads(&tmOut, out, static_cast<uint64_t>(n_views), static_cast<uint64_t>(T), static_cast<uint64_t>(heads), f16))
    return cudaErrorInvalidValue;
  if (T > 128) {
    AtlDev p;
    p.n_items = static_cast<long long>(n_views) * heads * 2;
    p.heads = heads;
    p.T = T;
    p.status = dev_status;
    return launch_atl(tmQKV, tmOut, p, f16, num_sms, stream);
  }
  const bool paired = !causal && T <= 64 && heads % 2 == 0;
  AtcDev p;
  p.pairs = paired ? heads / 2 : heads;
  p.n_items = static_cast<long long>(n_views) * p.pairs;
  p.T = T;
  p.causal = causal ? 1 : 0;
  p.status = dev_status;
  if (!paired) return launch_atc<0, 1>(tmQKV, tmOut, p, f16, num_sms, stream);
  if (T == 50) return launch_atc<50, 0>(tmQKV, tmOut, p, f16, num_sms, stream);
  if (T == 54) return launch_atc<54, 0>(tmQKV, tmOut, p, f16, num_sms, stream);
  return launch_atc<0, 0>(tmQKV, tmOut, p, f16, num_sms, stream);
}

}  // namespace jcb
