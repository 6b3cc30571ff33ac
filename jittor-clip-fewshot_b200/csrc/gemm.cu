// Persistent, warp-specialised 16-bit-operand (bf16 | fp16) GEMM for sm_100a:   C[M,N] = A[M,K] * B[N,K]^T  (+ fused epilogue)
//
//   warp 0      TMA producer   : cp.async.bulk.tensor 2-D tiles (128B swizzle) into a STAGES-deep smem ring
//   warp 1      MMA issuer     : one elected thread issues tcgen05.mma (kind::f16: bf16 or fp16 operands -> fp32)
//                                accumulating in TMEM;
//                                tcgen05.commit releases smem slots / publishes accumulator stages
//   warps 2..5  epilogue       : tcgen05.ld TMEM -> registers, bias / QuickGELU / residual / pos-embed,
//                                vectorised global stores; TMEM accumulators are double buffered so the
//                                epilogue of tile i overlaps the main loop of tile i+1
//
// CTA pairs (cluster 2x1x1, tcgen05 cta_group::2): UMMA 256 x BN x 16 across two SMs.  Each CTA stages its 128 rows
// of A and HALF of the B tile (BN/2 rows); the tensor core reads both halves.  Per CTA and k-block that is 32 KB of
// TMA writes + 8 KB/MMA of operand reads = 128 B/cycle, exactly the shared-memory bandwidth of an SM.  A single-CTA
// UMMA 128 x BN x 16 would demand 48 KB written + 12 KB/MMA read = 192 B/cycle of a 128 B/cycle SMEM: its tensor pipe
// cannot exceed ~66 % (measured 64 %, profiles/r01a), so that form was removed.
//
// This replaces the reference's fp32 `nn.Linear` calls on the hot path: packed QKV projection
// (jclip/mha.py:129-146, test.py:557-559), attention out-proj (jclip/mha.py:461, test.py:594), MLP
// c_fc / c_proj (jclip/model.py:38-39) and the patch-embed conv lowered to an im2col GEMM
// (jclip/model.py:105-108).  Residual adds (jclip/model.py:60-61), QuickGELU (jclip/model.py:27) and the
// positional-embedding add (jclip/model.py:114) are fused into the epilogues.
#include <cstdio>
#include <mutex>
#include <unordered_map>
#include <cudaTypedefs.h>

#include "kernels.h"
#include "ptx.cuh"

namespace jcb {

namespace {

constexpr int BLOCK_M = 128;  // rows of A (and of the accumulator) per CTA
constexpr int BLOCK_K = 64;   // 64 bf16 = 128 B = one swizzle atom row
constexpr int UMMA_K = 16;
// epilogue warps: 4 (one per TMEM lane quarter, all BN columns each); 8 (two per quarter, half the columns each) is
// supported by the tile configuration but never pays: the epilogues are idle more than half of every tile
// (clock64 role timeline of CTA 0, DESIGN.md) -- measured c_fc 1284 (8 warps) vs 1337 (4 warps) TFLOP/s.
#ifndef JCB_GELU_WARPS
#define JCB_GELU_WARPS 4
#endif
__host__ __device__ constexpr int epi_warps_of(int epi) {
  return (epi == EPI_BIAS_GELU_BF16 || epi == EPI_LNFOLD_GELU_BF16) ? JCB_GELU_WARPS : 4;
}

// chunks converted per generic->async proxy fence / per batch of TMA stores = staging buffers per epilogue warp.
// Every epilogue fences every 2 chunks and leaves the ring 5 stages (160 KB in flight per SM).  The role timeline
// (clock64 stamps of CTA 0, DESIGN.md) shows why staging must not eat a ring stage: with 4 stages the c_fc GEMM's MMA
// issuer waits for operands (157 cycles per UMMA instead of the pipe's 135-138) while its GELU epilogue idles 4.4 k of
// every 7.8 k cycles -- the loads are latency-bound (~1.7 us under load), so bytes in flight set the rate.  Measured on B200
// (tools/gpu_ab.sh): c_fc 1309 -> 1432 TFLOP/s with 5 stages; 6 stages with per-chunk fences gain 3 % on QKV but
// cost the HBM-bound out_proj 10 %.  (JCB_* macros: A/B builds via build.py --variant.)
#ifndef JCB_GELU_GROUP
#define JCB_GELU_GROUP 2
#endif
#ifndef JCB_GROUP
#define JCB_GROUP 2
#endif
#ifndef JCB_SMEM_KB
#define JCB_SMEM_KB 200
#endif
__host__ __device__ constexpr int group_of(int epi) { return (epi == EPI_BIAS_GELU_BF16 || epi == EPI_LNFOLD_GELU_BF16) ? JCB_GELU_GROUP : JCB_GROUP; }
__host__ __device__ constexpr bool is_lnprep(int epi) { return epi == EPI_RESID_LNPREP_SHORT || epi == EPI_RESID_LNPREP_LONG; }
__host__ __device__ constexpr bool is_lnfold(int epi) { return epi == EPI_LNFOLD_BF16 || epi == EPI_LNFOLD_GELU_BF16; }
__host__ __device__ constexpr bool out_is_bf16(int epi) { return epi == EPI_BIAS_BF16 || epi == EPI_BIAS_GELU_BF16 || is_lnfold(epi); }
// LNPREP (residual epilogue that also reads the old residual through TMA loads): NB fp32 chunk buffers per warp,
// loads issued D chunks ahead, NH bf16 chunk buffers.  SHORT (out_proj, HBM-bound, 12 k-blocks per tile): deep
// prefetch, 3 ring stages.  LONG (c_proj, 48 k-blocks per tile, tensor-bound): shallow prefetch, 5 ring stages.
#ifndef JCB_LNS_NB
#define JCB_LNS_NB 5
#endif
#ifndef JCB_LNS_D
#define JCB_LNS_D 3
#endif
#ifndef JCB_LNS_NH
#define JCB_LNS_NH 2
#endif
__host__ __device__ constexpr int lnprep_nb(int epi) { return epi == EPI_RESID_LNPREP_SHORT ? JCB_LNS_NB : 2; }
__host__ __device__ constexpr int lnprep_d(int epi) { return epi == EPI_RESID_LNPREP_SHORT ? JCB_LNS_D : 1; }
__host__ __device__ constexpr int lnprep_nh(int epi) { return epi == EPI_RESID_LNPREP_SHORT ? JCB_LNS_NH : 1; }

constexpr int CTAS = 2;       // CTAs of a pair (one cluster) sharing each 256-row UMMA

template <int BN, int EPI>
struct TileCfg {
  static constexpr int EPI_WARPS = epi_warps_of(EPI);
  static constexpr int NUM_THREADS = 64 + 32 * EPI_WARPS;
  static constexpr int HALVES = EPI_WARPS / 4;     // column slices of the tile, one per warp of a lane quarter
  static constexpr int CW = BN / HALVES;           // columns handled by one epilogue warp
  static constexpr int GROUP = group_of(EPI) / HALVES;
  // per epilogue warp: 32-row x 128-B swizzled chunks (GROUP of them, or NB + NH for the LNPREP epilogues)
  static constexpr int WARP_STAGING = (is_lnprep(EPI) ? lnprep_nb(EPI) + lnprep_nh(EPI) : GROUP) * 4096;
  static constexpr int STAGING_BYTES = EPI_WARPS * WARP_STAGING;
  static constexpr int SMEM_TOTAL = is_lnprep(EPI) ? 220 * 1024 : JCB_SMEM_KB * 1024;  // operand ring + epilogue staging
  static constexpr int VEC_FLOATS = (is_lnfold(EPI) ? 2 : 1) * CW;             // per-warp bias (+ column-sum) slice
  static constexpr int BAR_BYTES = 512;
  static constexpr int B_ROWS = BN / CTAS;  // rows of the B tile this CTA stages
  static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
  static constexpr int B_BYTES = B_ROWS * BLOCK_K * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (SMEM_TOTAL - STAGING_BYTES) / STAGE_BYTES;
  static constexpr int TMEM_COLS = 2 * BN;  // two accumulator stages; power of two for BN in {128,256}
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + STAGING_BYTES + EPI_WARPS * VEC_FLOATS * 4 + BAR_BYTES + 1024;  // + per-warp vectors + barriers + align slack
};

struct GemmDev {
  int M, N, K;
  int K2;                // k extent of the SECOND operand pair (tmA2 / tmB2) accumulated into the same tile; 0 = none
  const float* bias;
  void* out;
  long long ldo;
  int* status;
  float* stats;          // LNFOLD: in / LNPREP: out, [M, stats_slots, 2]
  int stats_slots;
  const float* colsum;   // LNFOLD
  // LNPREP: the bf16 / fp16 copy of the updated residual row is written CENTRED, x - shift[row], where shift is the
  // row's mean as of the previous LayerNorm point (previous shift + previous mean of the centred copy): the 16-bit
  // rounding then acts on |x - mean| instead of |x|, and the one-pass variance E[x'^2] - E[x']^2 has nothing to cancel.
  const float* stats_in;     // [M_in, stats_slots, 2] partial sums of the previous centred copy (nullptr: shift 0)
  const float* shift_in;     // [M_in] previous shift
  float* shift_out;          // [M] new shift (written by the n_blk == 0 tiles)
  long long stats_in_stride; // row r of this GEMM = row r * stride of stats_in / shift_in (class-token-only last block)
  uint32_t idesc;            // tcgen05 instruction descriptor (operand formats, M, N)
  // LoRA slots (SLOTS instantiations only; see GemmArgs::slot_of_view)
  const int* slot_of_view;   // slot of view v = rows [v * slot_rows, (v + 1) * slot_rows)
  int slot_rows;
  uint32_t slot_live;        // slots that have an adapter in this GEMM
};

// Slots present among the rows of the CTA pair's 256-row tile m_blk, restricted to p.slot_live.  The producer, the MMA
// issuer and the epilogue derive the same mask from the same inputs, so they agree on the k-blocks / tiles of a tile.
__device__ __forceinline__ uint32_t tile_slot_mask(const GemmDev& p, int m_blk, int tile_m) {
  const int r0 = m_blk * tile_m;
  const int r1 = min(r0 + tile_m, p.M) - 1;
  uint32_t mask = 0;
  for (int v = r0 / p.slot_rows; v <= r1 / p.slot_rows; ++v) mask |= 1u << __ldg(p.slot_of_view + v);
  return mask & p.slot_live;
}

// F16 selects the element type of 16-bit OUTPUTS (the conversion instruction of the epilogue); the operand formats
// the tensor core assumes travel in p.idesc, so the fp32-output epilogues need no second instantiation.
// SLOTS: several LoRA adapter sets, chosen per view (GemmArgs::slot_of_view).  With K2 > 0 (projection GEMM) second-pair
// k-block g is slot g's up-projection and a tile loads / multiplies only the k-blocks of the slots its rows use; with
// K2 == 0 (the down-projection GEMM) output column block [64 g, 64 g + 64) is slot g's: rows of other slots get exact
// zeros there, and N tiles that hold no slot of the tile's rows are skipped (the projection GEMM never reads them).
template <int BN, int EPI, bool F16, bool SLOTS>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(64 + 32 * epi_warps_of(EPI), 1)
gemm_tcgen05_2cta_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                         const __grid_constant__ CUtensorMap tmOut, const __grid_constant__ CUtensorMap tmOut2,
                         const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB2,
                         const GemmDev p) {
  using Cfg = TileCfg<BN, EPI>;
  constexpr int STAGES = Cfg::STAGES;
  constexpr int GROUP = Cfg::GROUP;
  constexpr int WARP_STAGING = Cfg::WARP_STAGING;
  constexpr int STAGING_BYTES = Cfg::STAGING_BYTES;
  constexpr int EPI_WARPS = Cfg::EPI_WARPS;
  constexpr int CW = Cfg::CW;
  extern __shared__ uint8_t smem_raw[];
  // 128B-swizzled TMA/UMMA tiles need 1024-byte alignment in the shared address space.
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + ((1024u - (raw_addr & 1023u)) & 1023u);
  uint8_t* ring = smem;
  uint8_t* staging = smem + STAGES * Cfg::STAGE_BYTES;   // 1024-B aligned (STAGE_BYTES is a multiple of 1024)
  float* s_bias_all = reinterpret_cast<float*>(staging + STAGING_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(staging + STAGING_BYTES + EPI_WARPS * Cfg::VEC_FLOATS * 4);
  uint64_t* full_bar = bars;                         // [STAGES]  TMA -> MMA       (the leader CTA's copy is used)
  uint64_t* empty_bar = bars + STAGES;               // [STAGES]  MMA -> TMA       (each CTA its own)
  uint64_t* tmem_full_bar = bars + 2 * STAGES;       // [2]  MMA -> epilogue       (each CTA its own)
  uint64_t* tmem_empty_bar = bars + 2 * STAGES + 2;  // [2]  epilogue -> MMA       (the leader CTA's copy is used)
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);
  uint64_t* load_bar = bars + 2 * STAGES + 5;        // [EPI_WARPS][8]  LNPREP: old-residual chunk landed in staging

  const int warp_idx = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = cluster_ctarank();
  const bool leader = cta_rank == 0;

  // one work unit = one CTA pair x one output tile of (CTAS * 128) x BN
  const int unit = static_cast<int>(blockIdx.x >> 1);
  const int num_units = static_cast<int>(gridDim.x >> 1);
  constexpr int TILE_M = BLOCK_M * CTAS;
  const int m_tiles = (p.M + TILE_M - 1) / TILE_M;
  const int n_tiles = p.N / BN;
  const int num_tiles = m_tiles * n_tiles;
  // C = A B^T + A2 B2^T: the k-blocks of the second operand pair (LoRA applied: A2 = x A_lora^T, B2 = s B_lora) follow
  // the first pair's through the same ring into the same TMEM accumulator
  const int num_kb1 = p.K / BLOCK_K;
  const int num_kb = num_kb1 + p.K2 / BLOCK_K;
  // SLOTS: the second-pair k-blocks of tile m_blk (projection), or whether tile (m_blk, n_blk) is computed at all (down)
  constexpr uint32_t N_BLOCKS_MASK = (1u << (BN / 64)) - 1u;
  auto slot_kb_mask = [&](int m_blk) -> uint32_t { return (SLOTS && p.K2 > 0) ? tile_slot_mask(p, m_blk, TILE_M) : 0u; };
  auto slot_skip = [&](int m_blk, int n_blk) -> bool {
    return SLOTS && p.K2 == 0 && ((tile_slot_mask(p, m_blk, TILE_M) >> (n_blk * (BN / 64))) & N_BLOCKS_MASK) == 0;
  };

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (p.K2 > 0) {
      tma_prefetch_desc(&tmA2);
      tma_prefetch_desc(&tmB2);
    }
    tma_prefetch_desc(&tmOut);
    if (is_lnprep(EPI)) {
      tma_prefetch_desc(&tmOut2);
      for (int i = 0; i < EPI_WARPS * 8; ++i) mbar_init(&load_bar[i], 1);
    }
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full_bar[s], 1);
      mbar_init(&tmem_empty_bar[s], EPI_WARPS * CTAS);
    }
    fence_mbar_init();
    fence_proxy_async_smem();
  }
  if (warp_idx == 1) {  // the same warp of BOTH CTAs of a pair takes part in a cta_group::2 allocation
    tmem_alloc_pair(tmem_ptr_smem, Cfg::TMEM_COLS);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  cluster_sync_all();   // barriers of both CTAs initialised before anyone signals them
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_ptr_smem);
  // programmatic dependent launch: everything above overlapped the previous kernel's tail; operands, bias, statistics
  // and the residual stream are touched only below
  griddep_wait();

  if (warp_idx == 0) {
    // ===================================================================== TMA producer (every CTA)
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      bool ok = true;
      for (int tile = unit; tile < num_tiles && ok; tile += num_units) {
        const int m_blk = tile / n_tiles, n_blk = tile % n_tiles;
        if (slot_skip(m_blk, n_blk)) continue;
        const int m0 = m_blk * TILE_M + static_cast<int>(cta_rank) * BLOCK_M;
        const int n0 = n_blk * BN + static_cast<int>(cta_rank) * Cfg::B_ROWS;
        uint32_t kb2_rest = slot_kb_mask(m_blk);   // SLOTS: second-pair k-blocks still to load, lowest first
        const int tile_kb = SLOTS && p.K2 > 0 ? num_kb1 + __popc(kb2_rest) : num_kb;
        for (int kb = 0; kb < tile_kb; ++kb) {
          if (!mbar_wait(&empty_bar[stage], phase ^ 1u, p.status, JCB_DEV_TIMEOUT_PRODUCER)) { ok = false; break; }
          uint8_t* sa = ring + stage * Cfg::STAGE_BYTES;
          uint8_t* sb = sa + Cfg::A_BYTES;
          const bool second = kb >= num_kb1;
          const CUtensorMap* ta = second ? &tmA2 : &tmA;
          const CUtensorMap* tb = second ? &tmB2 : &tmB;
          int k0 = (second ? kb - num_kb1 : kb) * BLOCK_K;
          if (SLOTS && second) {
            k0 = (__ffs(static_cast<int>(kb2_rest)) - 1) * BLOCK_K;
            kb2_rest &= kb2_rest - 1u;
          }
          // the leader's barrier collects the bytes of BOTH CTAs; a complete_tx that lands before the
          // leader's expect_tx just drives the transaction count negative for a moment
          if (leader) mbar_arrive_expect_tx(&full_bar[stage], 2 * Cfg::STAGE_BYTES);
          tma_load_2d_pair(sa, ta, &full_bar[stage], k0, m0);
          tma_load_2d_pair(sb, tb, &full_bar[stage], k0, n0);
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp_idx == 1) {
    // ===================================================================== MMA issuer (leader CTA only)
    if (leader && elect_one()) {
      const uint32_t idesc = p.idesc;
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      bool ok = true;
      for (int tile = unit; tile < num_tiles && ok; tile += num_units, ++it) {
        // `it` counts the tiles that use an accumulator stage: the stage and the barrier parities below are per use, so
        // a skipped tile must not advance it (the `++it` of the loop header is undone)
        if (slot_skip(tile / n_tiles, tile % n_tiles)) { --it; continue; }
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        if (!mbar_wait(&tmem_empty_bar[as], aphase ^ 1u, p.status, JCB_DEV_TIMEOUT_MMA)) { ok = false; break; }
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + static_cast<uint32_t>(as * BN);
        const int tile_kb = SLOTS && p.K2 > 0 ? num_kb1 + __popc(slot_kb_mask(tile / n_tiles)) : num_kb;
        for (int kb = 0; kb < tile_kb; ++kb) {
          if (!mbar_wait(&full_bar[stage], phase, p.status, JCB_DEV_TIMEOUT_MMA)) { ok = false; break; }
          tc_fence_after();
          const uint32_t sa = smem_u32(ring + stage * Cfg::STAGE_BYTES);
          const uint64_t da = umma_desc_sw128(sa);
          const uint64_t db = umma_desc_sw128(sa + Cfg::A_BYTES);
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            // +32 B per UMMA_K step inside the 128-B swizzle atom = +2 in the (addr >> 4) field
            umma_bf16_pair(tmem_d, da + static_cast<uint64_t>(2 * k), db + static_cast<uint64_t>(2 * k), idesc,
                           (kb | k) != 0 ? 1u : 0u);
          }
          // smem slot reusable (in both CTAs) once these MMAs have read it
          umma_commit_pair(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        if (ok) umma_commit_pair(&tmem_full_bar[as]);  // accumulator complete -> epilogue warps of both CTAs
      }
    }
  } else {
    // ===================================================================== epilogue (warps 2..5, every CTA)
    const int q = warp_idx & 3;              // TMEM lane quarter this warp may access
    const int ew = warp_idx - 2;             // epilogue warp index
    const int col0 = (ew >> 2) * CW;         // first column of the tile this warp handles
    // Each epilogue warp keeps a private copy of the tile's bias slice: no cross-warp barrier in
    // the epilogue, so a warp that abandons its loop on a pipeline error cannot strand the others.
    float* s_bias = s_bias_all + ew * Cfg::VEC_FLOATS;  // bias (LNFOLD: c[n]) of this warp's columns ...
    float* s_csum = s_bias + CW;                          // ... and, LNFOLD only, the column sums S[n]
    uint64_t* my_lbar = load_bar + ew * 8;
    uint32_t lphase = 0;                                  // LNPREP: parity bit per staging buffer
    const uint32_t empty_addr0 = smem_u32(&tmem_empty_bar[0]) & PEER_BIT_MASK;
    int it = 0;
    bool ok = true;
    for (int tile = unit; tile < num_tiles && ok; tile += num_units, ++it) {
      const int m_blk = tile / n_tiles, n_blk = tile % n_tiles;
      if (slot_skip(m_blk, n_blk)) { --it; continue; }   // as in the MMA issuer: `it` counts processed tiles only
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      __syncwarp();
      for (int i = lane; i < CW; i += 32) {
        s_bias[i] = p.bias ? __ldg(p.bias + n_blk * BN + col0 + i) : 0.0f;
        if (is_lnfold(EPI)) s_csum[i] = __ldg(p.colsum + n_blk * BN + col0 + i);
      }
      __syncwarp();
      const int row0e = m_blk * TILE_M + static_cast<int>(cta_rank) * BLOCK_M + q * 32;   // this warp's 32 rows
      float shift = 0.f;   // LNPREP: what this thread's row is centred by (see GemmDev)
      if (is_lnprep(EPI)) {
        if (p.shift_in != nullptr && row0e + lane < p.M) {
          const long long r = static_cast<long long>(row0e + lane) * p.stats_in_stride;
          const float2* st = reinterpret_cast<const float2*>(p.stats_in) + r * p.stats_slots;
          float su = 0.f;
          for (int i = 0; i < p.stats_slots; ++i) su += __ldg(st + i).x;
          shift = __ldg(p.shift_in + r) + su / static_cast<float>(p.N);
        }
        // the old residual of the first D chunks is requested BEFORE waiting for the accumulator: its latency hides
        // behind the main loop.  Every earlier store of this warp must have released the staging buffers.
        if (lane == 0) {
          bulk_wait_read<0>();
#pragma unroll
          for (int d = 0; d < lnprep_d(EPI); ++d) {
            mbar_arrive_expect_tx(&my_lbar[d], 4096);
            tma_load_2d(staging + ew * WARP_STAGING + d * 4096, &tmOut, &my_lbar[d], n_blk * BN + d * 32, row0e);
          }
        }
        __syncwarp();
      }

      ok = mbar_wait(&tmem_full_bar[as], aphase, p.status, JCB_DEV_TIMEOUT_EPILOGUE);
      ok = __all_sync(0xffffffffu, ok);
      if (!ok) break;
      tc_fence_after();

      const int row0 = m_blk * TILE_M + static_cast<int>(cta_rank) * BLOCK_M + q * 32;  // this warp's 32 rows
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + static_cast<uint32_t>(as * BN + col0);
      if (is_lnprep(EPI)) {
        // Residual epilogue that prepares the next LayerNorm: new = old + acc + bias.  The old residual chunk
        // arrives by TMA load in the swizzled staging buffer (requested D chunks ahead), is updated in place and
        // leaves by TMA store; the same pass emits the bf16 copy the next GEMM consumes as its A operand and this
        // thread's (= this row's) partial sum / sum of squares over the tile's BN columns.
        constexpr int NB = lnprep_nb(EPI), D = lnprep_d(EPI), NH = lnprep_nh(EPI);
        constexpr int NCH = BN / 32;
        uint8_t* my_stage = staging + ew * WARP_STAGING;
        uint8_t* my_half = my_stage + NB * 4096;   // bf16 chunk buffers (64 columns each)
        uint32_t v[2][32];
        tmem_ld_32x32b_x32(taddr, v[0]);
        float rs = 0.f, rq = 0.f;
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          uint32_t(&cur)[32] = v[c & 1];
          constexpr int WAITN = NB - D - 1;
          if (c >= 1) {
            // stores issued up to chunk c - 1 - WAITN have released their buffers: frees the fp32 buffer the next
            // prefetch lands in and the bf16 buffer this chunk (pair) writes
            if (lane == 0) bulk_wait_read<WAITN>();
            __syncwarp();
          }
          if (c + D < NCH && lane == 0) {
            const int nb = (c + D) % NB;
            mbar_arrive_expect_tx(&my_lbar[nb], 4096);
            tma_load_2d(my_stage + nb * 4096, &tmOut, &my_lbar[nb], n_blk * BN + (c + D) * 32, row0);
          }
          float bb[32];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 b4 = *reinterpret_cast<const float4*>(s_bias + c * 32 + 4 * j);
            bb[4 * j] = b4.x; bb[4 * j + 1] = b4.y; bb[4 * j + 2] = b4.z; bb[4 * j + 3] = b4.w;
          }
          tmem_ld_wait();
          if (c + 1 < NCH) {
            tmem_ld_32x32b_x32(taddr + static_cast<uint32_t>((c + 1) * 32), v[(c + 1) & 1]);
          } else {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(empty_addr0 + static_cast<uint32_t>(as * 8));
          }
          const int b = c % NB;
          ok = mbar_wait(&my_lbar[b], (lphase >> b) & 1u, p.status, JCB_DEV_TIMEOUT_EPILOGUE);   // old chunk landed
          lphase ^= 1u << b;
          uint8_t* rowp = my_stage + b * 4096 + lane * 128;
          uint8_t* halfp = my_half + ((c >> 1) % NH) * 4096 + lane * 128;
#pragma unroll
          for (int jj = 0; jj < 4; ++jj) {   // 8 columns = two 16-byte fp32 pieces -> one 16-byte bf16 piece
            float f[8];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const int j = 2 * jj + h;
              float4* piece = reinterpret_cast<float4*>(rowp + ((j ^ (lane & 7)) << 4));
              float4 o = *piece;
              o.x += __uint_as_float(cur[4 * j + 0]) + bb[4 * j + 0];
              o.y += __uint_as_float(cur[4 * j + 1]) + bb[4 * j + 1];
              o.z += __uint_as_float(cur[4 * j + 2]) + bb[4 * j + 2];
              o.w += __uint_as_float(cur[4 * j + 3]) + bb[4 * j + 3];
              *piece = o;
              f[4 * h + 0] = o.x; f[4 * h + 1] = o.y; f[4 * h + 2] = o.z; f[4 * h + 3] = o.w;
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) { f[e] -= shift; rs += f[e]; rq = fmaf(f[e], f[e], rq); }
            uint4 hb;
            hb.x = pack_h2<F16>(f[0], f[1]); hb.y = pack_h2<F16>(f[2], f[3]);
            hb.z = pack_h2<F16>(f[4], f[5]); hb.w = pack_h2<F16>(f[6], f[7]);
            const int hp = (c & 1) * 4 + jj;   // piece of the 128-byte bf16 row (64 columns = two fp32 chunks)
            *reinterpret_cast<uint4*>(halfp + ((hp ^ (lane & 7)) << 4)) = hb;
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_2d(&tmOut, my_stage + b * 4096, n_blk * BN + c * 32, row0);
            if (c & 1) tma_store_2d(&tmOut2, my_half + ((c >> 1) % NH) * 4096, n_blk * BN + (c - 1) * 32, row0);
            bulk_commit();
          }
        }
        ok = __all_sync(0xffffffffu, ok);
        if (row0 + lane < p.M) {
          *reinterpret_cast<float2*>(p.stats + (static_cast<long long>(row0 + lane) * p.stats_slots + n_blk) * 2) =
              make_float2(rs, rq);
          if (n_blk == 0 && p.shift_out != nullptr) p.shift_out[row0 + lane] = shift;
        }
      } else {
        // TMEM -> registers -> (+bias, activation, rounding) -> 128B-swizzled smem chunk of 32 rows x 128 B ->
        // one TMA store (or fp32 reduce-add for the residual epilogues) per chunk: fully coalesced, asynchronous,
        // and the residual stream is never read into the SM.  Rows >= M are clipped by the tensor map.
        constexpr bool OUT_BF16 = out_is_bf16(EPI);
        constexpr bool FOLD = is_lnfold(EPI);
        constexpr bool GELU = EPI == EPI_BIAS_GELU_BF16 || EPI == EPI_LNFOLD_GELU_BF16;
        constexpr int CHUNK_COLS = OUT_BF16 ? 64 : 32;
        constexpr int NCH = CW / CHUNK_COLS;
        uint8_t* my_stage = staging + ew * WARP_STAGING;
        // LayerNorm folded into this GEMM: this thread's row statistics from the producer's partial sums
        float ln_r = 1.f, ln_nmr = 0.f;
        if (FOLD) {
          float su = 0.f, sq = 0.f;
          if (row0 + lane < p.M) {
            const float2* st = reinterpret_cast<const float2*>(p.stats) + static_cast<long long>(row0 + lane) * p.stats_slots;
            for (int i = 0; i < p.stats_slots; ++i) { const float2 t2 = __ldg(st + i); su += t2.x; sq += t2.y; }
          }
          const float inv_k = 1.0f / static_cast<float>(p.K);
          const float mean = su * inv_k;
          const float var = fmaxf(fmaf(sq, inv_k, -mean * mean), 0.f);   // E[x^2] - E[x]^2 (as Jittor computes it), clamped
          ln_r = 1.0f / sqrtf(var + 1e-5f);
          ln_nmr = -mean * ln_r;
        }
        // SLOTS down-projection: this thread's row keeps only the 64-column block of its own view's slot
        int row_slot = -1;
        if (SLOTS && p.K2 == 0 && row0 + lane < p.M) row_slot = __ldg(p.slot_of_view + (row0 + lane) / p.slot_rows);
        const int blk0 = (n_blk * BN + col0) / 64;
        (void)row_slot; (void)blk0;
        const uint64_t r2 = f2_pack(ln_r, ln_r), nmr2 = f2_pack(ln_nmr, ln_nmr);
        const uint64_t k05 = f2_pack(0.5f, 0.5f), k851 = f2_pack(0.851f, 0.851f);
        (void)r2; (void)nmr2; (void)k05; (void)k851;
        // software pipeline: the TMEM load of chunk c+1 is in flight while chunk c is converted; the smem
        // staging holds GROUP chunks so the generic->async proxy fence (MEMBAR + ERRBAR, ~17 % of all
        // stall samples when issued per chunk) and the TMA issue happen once per GROUP chunks
        uint32_t v[2][CHUNK_COLS];
        auto load_chunk = [&](int c, uint32_t (&dst)[CHUNK_COLS]) {
          tmem_ld_32x32b_x32(taddr + static_cast<uint32_t>(c * CHUNK_COLS), *reinterpret_cast<uint32_t(*)[32]>(&dst[0]));
          if (OUT_BF16)
            tmem_ld_32x32b_x32(taddr + static_cast<uint32_t>(c * CHUNK_COLS + 32),
                               *reinterpret_cast<uint32_t(*)[32]>(&dst[CHUNK_COLS - 32]));
        };
        load_chunk(0, v[0]);
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          uint32_t(&cur)[CHUNK_COLS] = v[c & 1];
          // bias of this chunk into registers while the TMEM load is still in flight
          // additive term of every column as packed fp32 pairs: bias, or for the folded LayerNorm c[n] - r mu S[n]
          uint64_t bb2[CHUNK_COLS / 2];
#pragma unroll
          for (int j = 0; j < CHUNK_COLS / 4; ++j) {
            const float4 b4 = *reinterpret_cast<const float4*>(s_bias + c * CHUNK_COLS + 4 * j);
            bb2[2 * j] = f2_pack(b4.x, b4.y);
            bb2[2 * j + 1] = f2_pack(b4.z, b4.w);
            if (FOLD) {
              const float4 s4 = *reinterpret_cast<const float4*>(s_csum + c * CHUNK_COLS + 4 * j);
              bb2[2 * j] = f2_fma(nmr2, f2_pack(s4.x, s4.y), bb2[2 * j]);
              bb2[2 * j + 1] = f2_fma(nmr2, f2_pack(s4.z, s4.w), bb2[2 * j + 1]);
            }
          }
          if (c % GROUP == 0) {
            // the TMA stores of the previous group must have finished READING the staging buffers
            if (lane == 0) bulk_wait_read<0>();
            __syncwarp();
          }
          tmem_ld_wait();  // chunk c is in registers
          if (c + 1 < NCH) {
            load_chunk(c + 1, v[(c + 1) & 1]);
          } else {
            // every TMEM read of this tile has completed: hand the accumulator stage back to the MMA issuer
            // (leader CTA) before the last chunk is even converted
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(empty_addr0 + static_cast<uint32_t>(as * 8));
          }
          uint8_t* rowp = my_stage + (c % GROUP) * 4096 + lane * 128;
#pragma unroll
          for (int j = 0; j < 8; ++j) {  // 16-byte piece j of this thread's 128-byte row, XOR-swizzled by row % 8
            uint4 o;
            if (OUT_BF16) {
              float f[8];
#pragma unroll
              for (int e = 0; e < 4; ++e) {   // two columns per instruction
                const uint64_t a2 = f2_pack(__uint_as_float(cur[8 * j + 2 * e]), __uint_as_float(cur[8 * j + 2 * e + 1]));
                uint64_t x2 = FOLD ? f2_fma(a2, r2, bb2[4 * j + e]) : f2_add(a2, bb2[4 * j + e]);
                if (GELU) {
                  // x * sigmoid(1.702 x)  (reference jclip/model.py:27) = h + h tanh(0.851 x), h = 0.5 x: one MUFU op
                  // per element (tanh.approx, rel. error 2^-11, below the bf16 rounding of the output)
                  const uint64_t h2 = f2_mul(x2, k05);
                  float t0, t1;
                  f2_unpack(f2_mul(x2, k851), t0, t1);
                  // (A/B round 2: tanh.approx.f16x2 -- one MUFU op per two elements at the same 2^-11 relative error -- needs
                  // three conversions per pair around it and ran c_fc at 22.5 instead of 20.7 ms per step: the epilogue's
                  // instruction count, not its MUFU count, is what the power-capped step feels.  The opposite experiment --
                  // folding the 1/2 into the row scale and the staged additive terms, one multiply per element LESS,
                  // bit-identical -- was slower too, 23.3-24.2 vs 22.6 ms on the same box, profiles/r02z_ab_gelu_epilogue.log:
                  // this epilogue's schedule is a local optimum of ptxas, leave it alone)
                  x2 = f2_fma(h2, f2_pack(tanh_approx(t0), tanh_approx(t1)), h2);
                }
                f2_unpack(x2, f[2 * e], f[2 * e + 1]);
              }
              o.x = pack_h2<F16>(f[0], f[1]); o.y = pack_h2<F16>(f[2], f[3]);
              o.z = pack_h2<F16>(f[4], f[5]); o.w = pack_h2<F16>(f[6], f[7]);
              if (SLOTS && p.K2 == 0 && row_slot != blk0 + c) o = make_uint4(0u, 0u, 0u, 0u);   // CHUNK_COLS = 64
            } else {
              float f0, f1, f2, f3;
              f2_unpack(f2_add(f2_pack(__uint_as_float(cur[4 * j + 0]), __uint_as_float(cur[4 * j + 1])), bb2[2 * j]), f0, f1);
              f2_unpack(f2_add(f2_pack(__uint_as_float(cur[4 * j + 2]), __uint_as_float(cur[4 * j + 3])), bb2[2 * j + 1]), f2, f3);
              o.x = __float_as_uint(f0); o.y = __float_as_uint(f1); o.z = __float_as_uint(f2); o.w = __float_as_uint(f3);
            }
            *reinterpret_cast<uint4*>(rowp + ((j ^ (lane & 7)) << 4)) = o;
          }
          if (c % GROUP == GROUP - 1 || c == NCH - 1) {
            fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the TMA (async proxy)
            __syncwarp();
            if (lane == 0) {
              constexpr int G0 = 0;
#pragma unroll
              for (int g = c - (c % GROUP); g <= c; ++g) {
                const uint8_t* src = my_stage + (g % GROUP) * 4096;
                if (EPI == EPI_BIAS_RESID_F32) tma_reduce_add_2d(&tmOut, src, n_blk * BN + col0 + g * CHUNK_COLS, row0);
                else tma_store_2d(&tmOut, src, n_blk * BN + col0 + g * CHUNK_COLS, row0);
              }
              (void)G0;
              bulk_commit();
            }
          }
        }
      }
    }
    if (lane == 0) bulk_wait<0>();  // every TMA store / reduce of this warp has been performed
  }

  tc_fence_before();
  // a CTA of a pair must not retire while its partner can still touch its smem / TMEM / barriers
  cluster_sync_all();
  if (warp_idx == 1) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, Cfg::TMEM_COLS);
  }
}

PFN_cuTensorMapEncodeTiled_v12000 g_encode_tiled = nullptr;
char g_driver_err[256] = {0};

// Encoded tensor maps are pure functions of (base, shape, strides, box, type): the towers launch the same few
// hundred (pointer, shape) combinations every pass, so they are encoded once and looked up afterwards
// (cuTensorMapEncodeTiled costs ~1 us of host time each; 4 per GEMM launch matters for the reference's own call
// pattern of 1 image x 65 views per call, test.py:1692-1705).
struct TmapKey {
  const void* base; uint64_t rows, cols, ld; uint32_t box_rows, box_cols; int dtype;
  bool operator==(const TmapKey& o) const {
    return base == o.base && rows == o.rows && cols == o.cols && ld == o.ld && box_rows == o.box_rows &&
           box_cols == o.box_cols && dtype == o.dtype;
  }
};
struct TmapKeyHash {
  size_t operator()(const TmapKey& k) const {
    uint64_t h = reinterpret_cast<uintptr_t>(k.base) * 0x9E3779B97F4A7C15ull;
    h ^= (k.rows + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2));
    h ^= (k.cols * 1315423911ull + k.ld * 2654435761ull + (h << 6) + (h >> 2));
    h ^= (static_cast<uint64_t>(k.box_rows) << 40) ^ (static_cast<uint64_t>(k.box_cols) << 20) ^ static_cast<uint64_t>(k.dtype);
    return static_cast<size_t>(h);
  }
};
std::mutex g_tmap_mu;
std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> g_tmap_cache;
uint64_t g_tmap_hits = 0, g_tmap_misses = 0;

// 2-D row-major tensor [rows, cols] with leading dimension ld_elems, 128B-swizzled boxes of box_rows x box_cols
bool make_tmap_2d(CUtensorMap* tm, int dtype, const void* base, uint64_t rows, uint64_t cols, uint64_t ld_elems,
                  uint32_t box_rows, uint32_t box_cols) {
  const TmapKey key{base, rows, cols, ld_elems, box_rows, box_cols, dtype};
  {
    std::lock_guard<std::mutex> lock(g_tmap_mu);
    auto it = g_tmap_cache.find(key);
    if (it != g_tmap_cache.end()) { *tm = it->second; ++g_tmap_hits; return true; }
  }
  const uint64_t esz = dtype == TM_F32 ? 4 : 2;
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {ld_elems * esz};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType dt = dtype == TM_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                 : dtype == TM_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  CUresult r = g_encode_tiled(tm, dt, 2, const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return false;
  std::lock_guard<std::mutex> lock(g_tmap_mu);
  if (g_tmap_cache.size() >= 8192) g_tmap_cache.clear();   // workspaces were re-allocated many times: start over
  g_tmap_cache.emplace(key, *tm);
  ++g_tmap_misses;
  return true;
}

template <int BN, int EPI, bool F16, bool SLOTS = false>
cudaError_t launch_cfg(const GemmArgs& a, int* dev_status, int num_sms, cudaStream_t stream) {
  using Cfg = TileCfg<BN, EPI>;
  const int op_dt = a.f16 ? TM_F16 : TM_BF16;
  CUtensorMap tmA, tmB, tmOut;
  if (!make_tmap_2d(&tmA, op_dt, a.A, a.M, a.K, a.lda, BLOCK_M, BLOCK_K)) return cudaErrorInvalidValue;
  if (!make_tmap_2d(&tmB, op_dt, a.B, a.N, a.K, a.ldb, Cfg::B_ROWS, BLOCK_K)) return cudaErrorInvalidValue;
  constexpr bool OUT_BF16 = out_is_bf16(EPI);
  CUtensorMap tmOut2;
  if (!make_tmap_2d(&tmOut, OUT_BF16 ? op_dt : TM_F32, a.out, a.M, a.N, a.ldo, 32, OUT_BF16 ? 64 : 32)) return cudaErrorInvalidValue;
  tmOut2 = tmOut;
  if (is_lnprep(EPI)) {
    if (!a.out2 || !a.stats || a.stats_slots < a.N / BN) return cudaErrorInvalidValue;
    if ((a.shift_in != nullptr) != (a.stats_in != nullptr) || a.stats_in == a.stats) return cudaErrorInvalidValue;
    if (!make_tmap_2d(&tmOut2, op_dt, a.out2, a.M, a.N, a.ldo2, 32, 64)) return cudaErrorInvalidValue;
  }
  if (is_lnfold(EPI) && (!a.stats || !a.colsum || a.stats_slots < 1)) return cudaErrorInvalidValue;
  CUtensorMap tmA2 = tmA, tmB2 = tmB;   // second operand pair (GemmArgs::A2): placeholders when absent
  if (a.K2 > 0) {
    if (!make_tmap_2d(&tmA2, op_dt, a.A2, a.M, a.K2, a.lda2, BLOCK_M, BLOCK_K)) return cudaErrorInvalidValue;
    if (!make_tmap_2d(&tmB2, op_dt, a.B2, a.N, a.K2, a.ldb2, Cfg::B_ROWS, BLOCK_K)) return cudaErrorInvalidValue;
  }
  auto kern = gemm_tcgen05_2cta_kernel<BN, EPI, F16, SLOTS>;
  {
    cudaError_t e = ensure_dynamic_smem(kern, Cfg::SMEM_BYTES);
    if (e != cudaSuccess) return e;
  }
  GemmDev p;
  p.M = a.M; p.N = a.N; p.K = a.K; p.K2 = a.K2;
  p.bias = a.bias; p.out = a.out; p.ldo = a.ldo; p.status = dev_status;
  p.stats = a.stats; p.stats_slots = a.stats_slots; p.colsum = a.colsum;
  p.stats_in = a.stats_in; p.shift_in = a.shift_in; p.shift_out = a.shift_out;
  p.stats_in_stride = a.stats_in_row_stride > 0 ? a.stats_in_row_stride : 1;
  p.idesc = umma_idesc_f32acc(a.f16 != 0, BLOCK_M * CTAS, BN);
  p.slot_of_view = a.slot_of_view; p.slot_rows = a.slot_rows; p.slot_live = a.slot_live;
  const int tile_m = BLOCK_M * CTAS;
  const int tiles = ((a.M + tile_m - 1) / tile_m) * (a.N / BN);
  const int units = num_sms / CTAS;                       // CTA pairs that fit the chip
  const int grid = (tiles < units ? tiles : units) * CTAS;
  {
    cudaError_t e = launch_pdl(kern, dim3(grid), dim3(Cfg::NUM_THREADS), Cfg::SMEM_BYTES, stream, 1, tmA, tmB, tmOut, tmOut2,
                               tmA2, tmB2, p);
    if (e != cudaSuccess) return e;
  }
  return cudaGetLastError();
}

template <int BN>
cudaError_t launch_bn(const GemmArgs& a, int* st, int sms, cudaStream_t s) {
  if (a.slot_of_view) {   // LoRA slots: the QKV projection / down-projection (16-bit out) and out_proj (residual) only
    if (a.epilogue == EPI_BIAS_BF16)
      return a.f16 ? launch_cfg<BN, EPI_BIAS_BF16, true, true>(a, st, sms, s) : launch_cfg<BN, EPI_BIAS_BF16, false, true>(a, st, sms, s);
    if (a.epilogue == EPI_BIAS_RESID_F32 && a.K2 > 0) return launch_cfg<BN, EPI_BIAS_RESID_F32, false, true>(a, st, sms, s);
    return cudaErrorInvalidValue;
  }
#define JCB_CASE16(E) \
  case E: return a.f16 ? launch_cfg<BN, E, true>(a, st, sms, s) : launch_cfg<BN, E, false>(a, st, sms, s)
  switch (a.epilogue) {
    JCB_CASE16(EPI_BIAS_BF16);
    JCB_CASE16(EPI_BIAS_GELU_BF16);
    JCB_CASE16(EPI_LNFOLD_BF16);
    JCB_CASE16(EPI_LNFOLD_GELU_BF16);
    JCB_CASE16(EPI_RESID_LNPREP_SHORT);
    JCB_CASE16(EPI_RESID_LNPREP_LONG);
    case EPI_BIAS_RESID_F32: return launch_cfg<BN, EPI_BIAS_RESID_F32, false>(a, st, sms, s);
    case EPI_F32: return launch_cfg<BN, EPI_F32, false>(a, st, sms, s);
    default: return cudaErrorInvalidValue;
  }
#undef JCB_CASE16
}

}  // namespace

void* gemm_encode_tiled_fn() { return reinterpret_cast<void*>(g_encode_tiled); }

void tmap_cache_stats(uint64_t* hits, uint64_t* misses) {
  std::lock_guard<std::mutex> lock(g_tmap_mu);
  if (hits) *hits = g_tmap_hits;
  if (misses) *misses = g_tmap_misses;
}

const char* gemm_init_driver_api() {
  if (g_encode_tiled) return nullptr;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || fn == nullptr) {
    snprintf(g_driver_err, sizeof(g_driver_err), "cuTensorMapEncodeTiled not available: %s",
             cudaGetErrorString(e));
    return g_driver_err;
  }
  g_encode_tiled = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(fn);
  return nullptr;
}

cudaError_t launch_gemm(const GemmArgs& a, int* dev_status, int num_sms, cudaStream_t stream) {
  if (!g_encode_tiled) return cudaErrorNotReady;
  if (a.M <= 0 || a.N <= 0 || a.K <= 0 || a.K % BLOCK_K != 0 || a.N % 128 != 0) return cudaErrorInvalidValue;
  if ((reinterpret_cast<uintptr_t>(a.A) & 15) || (reinterpret_cast<uintptr_t>(a.B) & 15) || (a.lda % 8) ||
      (a.ldb % 8) || (a.ldo % 8) || (reinterpret_cast<uintptr_t>(a.out) & 15))
    return cudaErrorInvalidValue;
  if (a.K2 < 0 || a.K2 % BLOCK_K != 0) return cudaErrorInvalidValue;
  if (a.K2 > 0 && (!a.A2 || !a.B2 || (reinterpret_cast<uintptr_t>(a.A2) & 15) || (reinterpret_cast<uintptr_t>(a.B2) & 15) ||
                   (a.lda2 % 8) || (a.ldb2 % 8) || a.lda2 < a.K2 || a.ldb2 < a.K2))
    return cudaErrorInvalidValue;
  if (a.slot_of_view && (a.slot_rows < 1 || a.slot_live == 0 || a.slot_live >= (1u << LORA_MAX_SLOTS) ||
                         (a.K2 > 0 && 64 * (32 - __builtin_clz(a.slot_live)) > a.K2) ||
                         (a.K2 == 0 && 64 * (32 - __builtin_clz(a.slot_live)) > a.N)))
    return cudaErrorInvalidValue;
  // BN = 256 whenever N allows it; 128 otherwise (only used by generic/test shapes).  The LoRA-slot down-projection
  // always runs BN = 128: an N tile then covers two slots' 64-column blocks, so a tile whose rows use one slot computes
  // (and skips) in steps of two slots instead of four.
  if (a.N % 256 == 0 && !(a.slot_of_view && a.K2 == 0)) return launch_bn<256>(a, dev_status, num_sms, stream);
  return launch_bn<128>(a, dev_status, num_sms, stream);
}

}  // namespace jcb
