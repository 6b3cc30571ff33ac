// Row-wise, attention and reduction kernels of image-tower LoRA training (the backward pass of encode_image with
// respect to the adapters A and B; host schedule in api.cu, "LoRA training").  The GEMMs of the backward pass run on
// the tcgen05 GEMM (gemm.cu); what is here is the elementwise / per-row / per-head work between them.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <curand_philox4x32_x.h>

#include <cudaTypedefs.h>

#include "kernels.h"
#include "ptx.cuh"

namespace jcb {

void* gemm_encode_tiled_fn();   // gemm.cu
bool make_tmap_heads(CUtensorMap* tm, const void* base, uint64_t n_seq, uint64_t T, uint64_t blocks, int f16);   // attention_tc.cu

namespace {

// 16-bit element of type t (TR_BF16 / TR_F16) or fp32 (TR_F32) at p[i]
__device__ __forceinline__ float ld_any(const void* p, int t, int64_t i) {
  if (t == TR_F32) return static_cast<const float*>(p)[i];
  const uint16_t u = static_cast<const uint16_t*>(p)[i];
  return t == TR_F16 ? __half2float(__ushort_as_half(u)) : __bfloat162float(__ushort_as_bfloat16(u));
}
__device__ __forceinline__ uint16_t to16(float x, bool f16) {
  return f16 ? __half_as_ushort(__float2half_rn(x)) : __bfloat16_as_ushort(__float2bfloat16_rn(x));
}

// Keep decision of the training dropout for element (row, col) of projection `proj` of `layer` at `step`: Philox4x32-10
// (curand_philox4x32_x.h) of the counter (col / 4, row, step, layer * 4 + proj) under the key (seed lo, seed hi); word
// col % 4, top 24 bits, kept iff >= thr24 = floor(rate * 2^24).  The host reproduction in tests/test_lora_train_cpu.py
// computes the same words.
__device__ __forceinline__ bool dropout_keep(const DropoutArgs& d, int proj, int64_t row, int col) {
  const uint4 c = make_uint4(static_cast<unsigned>(col >> 2), static_cast<unsigned>(row), static_cast<unsigned>(d.step),
                             static_cast<unsigned>(d.layer * 4 + proj));
  const uint2 k = make_uint2(static_cast<unsigned>(d.seed), static_cast<unsigned>(d.seed >> 32));
  const uint4 r = curand_Philox4x32_10(c, k);
  const unsigned w = (col & 3) == 0 ? r.x : (col & 3) == 1 ? r.y : (col & 3) == 2 ? r.z : r.w;
  return (w >> 8) >= d.thr24;
}

// xd[m, p W + c] = keep_p(row0 + m, c) ? x[m, c] * inv : 0 for the projections proj0 .. proj0 + npj - 1 (16-bit in and out)
__global__ void dropout_fwd_kernel(const uint16_t* __restrict__ x, int64_t M, int W, int npj, int proj0, DropoutArgs d,
                                   int64_t row0, bool f16, uint16_t* __restrict__ xd) {
  const int64_t n = M * W * npj;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t m = i / (static_cast<int64_t>(W) * npj);
    const int rem = static_cast<int>(i - m * W * npj);
    const int p = rem / W, c = rem - p * W;
    const float v = ld_any(x, f16 ? TR_F16 : TR_BF16, m * W + c);
    xd[i] = to16(dropout_keep(d, proj0 + p, row0 + m, c) ? v * d.inv : 0.f, f16);
  }
}

// dx[m, c] += sum_p keep_p(row0 + m, c) * inv * dxd[m, p W + c]
__global__ void dropout_bwd_add_kernel(const float* __restrict__ dxd, int64_t M, int W, int npj, int proj0, DropoutArgs d,
                                       int64_t row0, float* __restrict__ dx) {
  const int64_t n = M * W;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t m = i / W;
    const int c = static_cast<int>(i - m * W);
    float acc = 0.f;
    for (int p = 0; p < npj; ++p)
      if (dropout_keep(d, proj0 + p, row0 + m, c)) acc += dxd[(m * npj + p) * W + c];
    dx[i] += acc * d.inv;
  }
}

__global__ void dropout_mask_kernel(DropoutArgs d, int proj, int64_t rows, int cols, uint8_t* __restrict__ out) {
  const int64_t n = rows * cols;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = i / cols;
    out[i] = dropout_keep(d, proj, r, static_cast<int>(i - r * cols)) ? 1 : 0;
  }
}

// QuickGELU derivative (jclip/model.py:27, x sigmoid(1.702 x)): dh = dy * (s + 1.702 x s (1 - s)), bf16 out
__global__ void gelu_bwd_kernel(const float* __restrict__ dy, const uint16_t* __restrict__ h, int64_t n, bool h_f16,
                                uint16_t* __restrict__ dh) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float x = ld_any(h, h_f16 ? TR_F16 : TR_BF16, i);
    const float s = 1.f / (1.f + __expf(-1.702f * x));
    dh[i] = to16(dy[i] * (s + 1.702f * x * s * (1.f - s)), false);
  }
}

// LayerNorm backward with frozen gamma / beta, one warp per row: g[r] += rstd (gy - mean(gy) - xhat mean(gy xhat)),
// gy = dy * gamma, statistics recomputed from the fp32 input x (eps 1e-5, biased variance)
__global__ void ln_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy, int64_t rows, int W,
                              const float* __restrict__ gamma, float* __restrict__ g) {
  const int64_t r = blockIdx.x * static_cast<int64_t>(blockDim.x / 32) + threadIdx.x / 32;
  const int lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* xr = x + r * W;
  const float* dr = dy + r * W;
  float s = 0.f;
  for (int c = lane; c < W; c += 32) s += xr[c];
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / W;
  float v = 0.f;
  for (int c = lane; c < W; c += 32) { const float t = xr[c] - mean; v += t * t; }
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  const float rstd = rsqrtf(v / W + 1e-5f);
  float a = 0.f, b = 0.f;
  for (int c = lane; c < W; c += 32) {
    const float gy = dr[c] * gamma[c];
    a += gy;
    b += gy * (xr[c] - mean) * rstd;
  }
  for (int o = 16; o; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
  a /= W;
  b /= W;
  float* gr = g + r * W;
  for (int c = lane; c < W; c += 32) {
    const float xh = (xr[c] - mean) * rstd;
    gr[c] += rstd * (dr[c] * gamma[c] - a - xh * b);
  }
}

// Attention backward of one (view, head), T <= 64, head dim 64, fp32 in shared memory: P = softmax(q k^T / 8) recomputed
// from the taped q|k|v, then dV = P^T dO, dP = dO V^T, dS = P (dP - rowsum(dP P)), dQ = dS K / 8, dK = dS^T Q / 8.
constexpr int AB_T = 64, AB_LD = 65, AB_THREADS = 256;
__global__ void __launch_bounds__(AB_THREADS) attention_bwd_kernel(const uint16_t* __restrict__ qkv, const float* __restrict__ dout,
                                                                   int T, int heads, bool f16, uint16_t* __restrict__ dqkv) {
  extern __shared__ float sm[];
  float* q = sm;
  float* k = q + AB_T * AB_LD;
  float* v = k + AB_T * AB_LD;
  float* dO = v + AB_T * AB_LD;
  float* P = dO + AB_T * AB_LD;
  float* dP = P + AB_T * AB_LD;
  float* Dr = dP + AB_T * AB_LD;   // [AB_T]
  const int h = blockIdx.x % heads;
  const int64_t view = blockIdx.x / heads;
  const int W = heads * 64;
  const int tid = threadIdx.x;
  const int64_t row0 = view * T;
  const int tf = f16 ? TR_F16 : TR_BF16;
  for (int i = tid; i < T * 64; i += AB_THREADS) {
    const int t = i >> 6, d = i & 63;
    const int64_t base = (row0 + t) * 3 * W + h * 64 + d;
    q[t * AB_LD + d] = ld_any(qkv, tf, base);
    k[t * AB_LD + d] = ld_any(qkv, tf, base + W);
    v[t * AB_LD + d] = ld_any(qkv, tf, base + 2 * W);
    dO[t * AB_LD + d] = dout[(row0 + t) * W + h * 64 + d];
  }
  __syncthreads();
  for (int i = tid; i < T * T; i += AB_THREADS) {
    const int a = i / T, b = i - a * T;
    float s = 0.f, dp = 0.f;
#pragma unroll 8
    for (int d = 0; d < 64; ++d) {
      s += q[a * AB_LD + d] * k[b * AB_LD + d];
      dp += dO[a * AB_LD + d] * v[b * AB_LD + d];
    }
    P[a * AB_LD + b] = s * 0.125f;
    dP[a * AB_LD + b] = dp;
  }
  __syncthreads();
  // softmax rows and D_a = sum_b P dP: one warp per row
  const int warp = tid >> 5, lane = tid & 31;
  for (int a = warp; a < T; a += AB_THREADS / 32) {
    float mx = -INFINITY;
    for (int b = lane; b < T; b += 32) mx = fmaxf(mx, P[a * AB_LD + b]);
    for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
    for (int b = lane; b < T; b += 32) {
      const float e = __expf(P[a * AB_LD + b] - mx);
      P[a * AB_LD + b] = e;
      sum += e;
    }
    for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float inv = 1.f / sum;
    float dsum = 0.f;
    for (int b = lane; b < T; b += 32) {
      const float p = P[a * AB_LD + b] * inv;
      P[a * AB_LD + b] = p;
      dsum += p * dP[a * AB_LD + b];
    }
    for (int o = 16; o; o >>= 1) dsum += __shfl_xor_sync(0xffffffffu, dsum, o);
    if (lane == 0) Dr[a] = dsum;
  }
  __syncthreads();
  // dV (needs P), then dS overwrites dP
  for (int i = tid; i < T * 64; i += AB_THREADS) {
    const int b = i >> 6, d = i & 63;
    float acc = 0.f;
    for (int a = 0; a < T; ++a) acc += P[a * AB_LD + b] * dO[a * AB_LD + d];
    dqkv[(row0 + b) * 3 * W + 2 * W + h * 64 + d] = to16(acc, false);
  }
  for (int i = tid; i < T * T; i += AB_THREADS) {
    const int a = i / T, b = i - a * T;
    dP[a * AB_LD + b] = P[a * AB_LD + b] * (dP[a * AB_LD + b] - Dr[a]) * 0.125f;
  }
  __syncthreads();
  for (int i = tid; i < T * 64; i += AB_THREADS) {
    const int t = i >> 6, d = i & 63;
    float aq = 0.f, ak = 0.f;
    for (int j = 0; j < T; ++j) {
      aq += dP[t * AB_LD + j] * k[j * AB_LD + d];
      ak += dP[j * AB_LD + t] * q[j * AB_LD + d];
    }
    dqkv[(row0 + t) * 3 * W + h * 64 + d] = to16(aq, false);
    dqkv[(row0 + t) * 3 * W + W + h * 64 + d] = to16(ak, false);
  }
}

// Attention backward of one (view, head) for 65 <= T <= 256, head dim 64, no mask, on the 5th-generation tensor cores:
// the same contract as attention_bwd_kernel, every product a tcgen05.mma with fp32 accumulators in TMEM.
//
//   CTA = one (view, head), 128 threads; thread = query row = TMEM lane.  Thread 0 issues the TMA copies and the MMAs;
//   the phases below are separated by mbarriers (TMA bytes, MMA commits) and __syncthreads.
//   shared   K, V       resident, ceil(T / 64) swizzled [64 tokens][64] boxes each (the attention_tc.cu layout)   64 KB
//            Q, dO      the current 128-row query tile (dO: bf16, converted from fp32 in shared memory)            32 KB
//            P / dS     [128 queries][256 keys] 16-bit as four swizzled [128][64] sub-tiles; dS overwrites P   64 KB
//            staging    the query tile's fp32 dO (two TMA boxes of [128 tokens][32]), then dQ's bf16 output       32 KB
//   TMEM     dV, dK     [256 keys][64] each, accumulated over the query tiles                          columns 0..255
//            S, dP, dQ  in turn in columns 256..511
//   per query tile qt (one or two):  S = Q K^T -> exact two-pass softmax (row max, then sum) -> P in shared memory;
//            dP = dO V^T, dV += P^T dO -> D = rowsum(P dP), dS = P (dP - D) / 8 in shared memory;
//            dQ = dS K -> TMA store, dK += dS^T Q.  After the last tile dK and dV are stored from TMEM.
//   K is centred (its mean over the T keys subtracted) once it lands: see the comment at that step.
//   P^T and dS^T are the same shared tiles read as MN-major A operands (two 64-key atoms 16 KB apart).  Boxes wholly
//   past T are neither loaded nor multiplied; rows of a tile past T get P = dS = 0 and their outputs are clipped.
//
// Operand types: kind::f16 multiplies operands of one type, and dO and dS are bf16 (as in the backward GEMMs), so an fp16
// tower's Q, K and V tiles are converted to bf16 in shared memory after they land.  Their rounding is then bf16's,
// the same as a bf16 tower's (within the gradient bounds of tests/test_gpu_lora_train_b16.py).
constexpr int BT_TILE = 64 * 64 * 2;                 // one [64 tokens][64] 16-bit box: 8 KB
constexpr int BT_K = 0, BT_V = 4 * BT_TILE, BT_Q = 8 * BT_TILE, BT_DO = 10 * BT_TILE, BT_P = 12 * BT_TILE;
constexpr int BT_P_SUB = 2 * BT_TILE;                // one [128 queries][64 keys] sub-tile of P / dS: 16 KB
constexpr int BT_ST = BT_P + 4 * BT_P_SUB;           // staging: 32 KB
constexpr int BT_BARS = BT_ST + 4 * BT_TILE;
constexpr int BT_KMEAN = BT_BARS + 64;               // [64] fp32 mean key
constexpr int BT_SMEM = BT_KMEAN + 256;              // 196928 B: one CTA per SM
constexpr int BT_THREADS = 128;
constexpr uint32_t BT_DV_COL = 0, BT_DK_COL = 128, BT_S_COL = 256, BT_TMEM_COLS = 512;

struct AbtDev {
  int heads;
  int T;
  int f16;
  int* status;
};

// 8 16-bit values of the tower's type (fp16) -> bf16, in place
__device__ __forceinline__ void f16_to_bf16_x8(uint4* p) {
  uint4 v = *p;
  uint32_t* w = reinterpret_cast<uint32_t*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = unpack_h2<true>(w[i]);
    w[i] = pack_bf16x2(f.x, f.y);
  }
  *p = v;
}

__global__ void __launch_bounds__(BT_THREADS, 1)
attention_bwd_tcgen05_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ CUtensorMap tmDO,
                             const __grid_constant__ CUtensorMap tmOut, const AbtDev p) {
  extern __shared__ __align__(1024) uint8_t bt_smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(bt_smem + BT_BARS);
  uint64_t* kv_full = bars;       // K, V landed
  uint64_t* q_full = bars + 1;    // Q, dO of the query tile landed
  uint64_t* mma_done = bars + 2;  // every MMA issued so far completed
  uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(bars + 3);

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int T = p.T;
  const int h = static_cast<int>(blockIdx.x % p.heads);
  const int seq = static_cast<int>(blockIdx.x / p.heads);
  const int nkb = (T + 63) >> 6;   // 64-key boxes holding valid keys: 2..4
  const int nqt = (T + 127) >> 7;  // 128-row query (and key) tiles: 1 or 2
  const uint32_t sbase = smem_u32(bt_smem);

  if (tid == 0) {
    if ((sbase & 1023u) != 0u) atomicCAS(p.status, 0, JCB_DEV_SMEM_ALIGN);
    tma_prefetch_desc(&tmQKV);
    tma_prefetch_desc(&tmDO);
    tma_prefetch_desc(&tmOut);
    mbar_init(kv_full, 1);
    mbar_init(q_full, 1);
    mbar_init(mma_done, 1);
    fence_mbar_init();
    fence_proxy_async_smem();
  }
  if (warp == 0) {
    tmem_alloc(tmem_ptr_smem, BT_TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_ptr_smem);
  const uint32_t lane_base = tmem_base + (static_cast<uint32_t>(warp * 32) << 16);

  if (tid == 0) {
    mbar_arrive_expect_tx(kv_full, static_cast<uint32_t>(2 * nkb * BT_TILE));
    // coordinates: (d, 64-wide column block of the [T, 3W] row, token, sequence); blocks: q | k | v heads
    for (int b = 0; b < nkb; ++b) {
      tma_load_4d(bt_smem + BT_K + b * BT_TILE, &tmQKV, kv_full, 0, p.heads + h, 64 * b, seq);
      tma_load_4d(bt_smem + BT_V + b * BT_TILE, &tmQKV, kv_full, 0, 2 * p.heads + h, 64 * b, seq);
    }
  }
  // every thread waits; a timeout anywhere ends the work of the whole CTA
  uint32_t mph = 0;
  auto wait_all = [&](uint64_t* bar, uint32_t parity) {
    const bool ok = mbar_wait(bar, parity, p.status, JCB_DEV_TIMEOUT_EPILOGUE);
    return __syncthreads_and(ok) != 0;
  };
  auto commit_wait = [&]() {
    if (tid == 0) umma_commit(mma_done);
    const bool ok = wait_all(mma_done, mph);
    mph ^= 1u;
    tc_fence_after();
    return ok;
  };
  // 16-byte chunk j (8 elements, columns 8j..8j+7) of row r of a swizzled [rows][64] 16-bit tile at `tile`
  auto chunk = [](uint8_t* tile, int r, int j) {
    return reinterpret_cast<uint4*>(tile + (r >> 6) * BT_TILE + (r & 63) * 128 + ((j ^ (r & 7)) << 4));
  };
  const float scale_log2 = 0.125f * 1.4426950408889634f;   // 1/sqrt(64) * log2(e)
  const uint32_t idesc_s = umma_idesc_f32acc(false, 128, 64 * nkb);                           // S, dP
  constexpr uint32_t idesc_q = umma_idesc_f32acc(false, 128, 64, /*b_mn_major=*/true);        // dQ
  constexpr uint32_t idesc_t = umma_idesc_f32acc(false, 128, 64, true, /*a_mn_major=*/true);  // dV, dK
  bool ok = true;

  for (int qt = 0; qt < nqt && ok; ++qt) {
    const int q0 = 128 * qt;
    const int nq = q0 + 64 < T ? 2 : 1;   // Q boxes holding valid rows
    const int r = q0 + tid;               // this thread's query token
    if (tid == 0) {
      bulk_wait_read<0>();   // the previous tile's dQ store has read the staging
      mbar_arrive_expect_tx(q_full, static_cast<uint32_t>(nq * BT_TILE + 4 * BT_TILE));
      for (int b = 0; b < nq; ++b) tma_load_4d(bt_smem + BT_Q + b * BT_TILE, &tmQKV, q_full, 0, h, q0 + 64 * b, seq);
      tma_load_4d(bt_smem + BT_ST, &tmDO, q_full, 0, h, q0, seq);
      tma_load_4d(bt_smem + BT_ST + 2 * BT_TILE, &tmDO, q_full, 32, h, q0, seq);
    }
    if (qt == 0 && !(ok = wait_all(kv_full, 0))) break;
    if (!(ok = wait_all(q_full, static_cast<uint32_t>(qt) & 1u))) break;
    // ---- operands to bf16: fp16 Q (and K, V once), fp32 dO -> the swizzled dO tile
    if (p.f16) {
      for (int i = tid; i < nq * BT_TILE / 16; i += BT_THREADS) f16_to_bf16_x8(reinterpret_cast<uint4*>(bt_smem + BT_Q) + i);
      if (qt == 0)
        for (int i = tid; i < nkb * BT_TILE / 16; i += BT_THREADS) {
          f16_to_bf16_x8(reinterpret_cast<uint4*>(bt_smem + BT_K) + i);
          f16_to_bf16_x8(reinterpret_cast<uint4*>(bt_smem + BT_V) + i);
        }
    }
    if (qt == 0) {
      // K minus its mean over the T keys.  Softmax ignores a vector added to every key (each score of a row moves by
      // the same amount), so P, dP, dS and dK are unchanged; but dQ = dS K no longer carries the mean key times the
      // rounding error of sum_j dS_j (exactly 0 before dS is rounded to bf16), which dominated dQ's error when the
      // keys share a large common component, and S is computed from smaller operands.
      float* kmean = reinterpret_cast<float*>(bt_smem + BT_KMEAN);
      __syncthreads();   // K converted
      if (tid < 64) {
        float acc = 0.f;
        for (int t = 0; t < T; ++t) {
          const uint32_t w = reinterpret_cast<const uint32_t*>(chunk(bt_smem + BT_K, t, tid >> 3))[(tid & 7) >> 1];
          const float2 f = unpack_h2<false>(w);
          acc += (tid & 1) ? f.y : f.x;
        }
        kmean[tid] = acc / static_cast<float>(T);
      }
      __syncthreads();
      for (int i = tid; i < T * 8; i += BT_THREADS) {
        const int t = i >> 3, j = i & 7;
        uint4* cp = chunk(bt_smem + BT_K, t, j);
        const uint4 c = *cp;
        uint32_t w[4] = {c.x, c.y, c.z, c.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 f = unpack_h2<false>(w[e]);
          w[e] = pack_bf16x2(f.x - kmean[8 * j + 2 * e], f.y - kmean[8 * j + 2 * e + 1]);
        }
        *cp = make_uint4(w[0], w[1], w[2], w[3]);
      }
    }
    for (int i = tid; i < 128 * 8; i += BT_THREADS) {
      const int rr = i >> 3, j = i & 7;
      const float4* src = reinterpret_cast<const float4*>(bt_smem + BT_ST + (j >> 2) * 2 * BT_TILE + rr * 128 + (j & 3) * 32);
      const float4 a = src[0], b = src[1];
      *chunk(bt_smem + BT_DO, rr, j) = make_uint4(pack_bf16x2(a.x, a.y), pack_bf16x2(a.z, a.w), pack_bf16x2(b.x, b.y),
                                                  pack_bf16x2(b.z, b.w));
    }
    fence_proxy_async_smem();
    __syncthreads();

    // ---- S = Q K^T
    if (tid == 0) {
      tc_fence_after();
      const uint64_t dq = umma_desc_sw128(sbase + BT_Q), dk = umma_desc_sw128(sbase + BT_K);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        umma_bf16(tmem_base + BT_S_COL, dq + 2 * k, dk + 2 * k, idesc_s, k != 0 ? 1u : 0u);
    }
    if (!(ok = commit_wait())) break;

    // ---- exact softmax of this row: maximum, sum, then P = exp / sum as bf16 into the P sub-tiles (zeros past T)
    {
      const bool valid = r < T;
      float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
      for (int ch = 0; ch < 2 * nkb; ++ch) {
        uint32_t sv[32];
        tmem_ld_32x32b_x32(lane_base + BT_S_COL + static_cast<uint32_t>(ch * 32), sv);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 32; ++c)
          if (ch * 32 + c < T) m4[c & 3] = fmaxf(m4[c & 3], __uint_as_float(sv[c]));
      }
      const float nmx = -fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3])) * scale_log2;
      float s4[4] = {0.f, 0.f, 0.f, 0.f};
      for (int ch = 0; ch < 2 * nkb; ++ch) {
        uint32_t sv[32];
        tmem_ld_32x32b_x32(lane_base + BT_S_COL + static_cast<uint32_t>(ch * 32), sv);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 32; ++c)
          if (ch * 32 + c < T) s4[c & 3] += ex2_approx(fmaf(__uint_as_float(sv[c]), scale_log2, nmx));
      }
      const float inv = 1.f / ((s4[0] + s4[1]) + (s4[2] + s4[3]));
      for (int ch = 0; ch < 4 * nqt; ++ch) {   // 32 keys per chunk, over the key tiles the dV / dK products read
        uint32_t sv[32] = {};
        if (ch < 2 * nkb) {
          tmem_ld_32x32b_x32(lane_base + BT_S_COL + static_cast<uint32_t>(ch * 32), sv);
          tmem_ld_wait();
        }
        uint32_t pv[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) {
          const int k0 = ch * 32 + 2 * c;
          const float p0 = valid && k0 < T ? ex2_approx(fmaf(__uint_as_float(sv[2 * c]), scale_log2, nmx)) * inv : 0.f;
          const float p1 = valid && k0 + 1 < T ? ex2_approx(fmaf(__uint_as_float(sv[2 * c + 1]), scale_log2, nmx)) * inv : 0.f;
          pv[c] = pack_bf16x2(p0, p1);
        }
        uint8_t* sub = bt_smem + BT_P + (ch >> 1) * BT_P_SUB;
#pragma unroll
        for (int j = 0; j < 4; ++j)
          *chunk(sub, tid, (ch & 1) * 4 + j) = make_uint4(pv[4 * j], pv[4 * j + 1], pv[4 * j + 2], pv[4 * j + 3]);
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();

    // ---- dP = dO V^T (over S), dV += P^T dO
    if (tid == 0) {
      tc_fence_after();
      const uint64_t ddo = umma_desc_sw128(sbase + BT_DO), dv = umma_desc_sw128(sbase + BT_V);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        umma_bf16(tmem_base + BT_S_COL, ddo + 2 * k, dv + 2 * k, idesc_s, k != 0 ? 1u : 0u);
      const uint64_t bdo = umma_desc_sw128_mn(sbase + BT_DO);
      for (int kt = 0; kt < nqt; ++kt) {
        const uint64_t apt = umma_desc_sw128_mn(sbase + BT_P + 2 * kt * BT_P_SUB, BT_P_SUB);
        for (int ks = 0; ks < 4 * nq; ++ks)   // 16 query rows per step
          umma_bf16(tmem_base + BT_DV_COL + 64 * kt, apt + ks * (2048 >> 4), bdo + ks * (2048 >> 4), idesc_t,
                    (qt > 0 || ks > 0) ? 1u : 0u);
      }
    }
    if (!(ok = commit_wait())) break;

    // ---- D = rowsum(P dP); dS = P (dP - D) / 8 over P.  D is taken over the stored (bf16) P divided by that P's sum,
    // so that dP - D keeps its relative accuracy when one key holds almost all of a row's weight.
    {
      float d4[4] = {0.f, 0.f, 0.f, 0.f}, s4[4] = {0.f, 0.f, 0.f, 0.f};
      for (int ch = 0; ch < 2 * nkb; ++ch) {
        uint32_t dv[32];
        tmem_ld_32x32b_x32(lane_base + BT_S_COL + static_cast<uint32_t>(ch * 32), dv);
        tmem_ld_wait();
        uint8_t* sub = bt_smem + BT_P + (ch >> 1) * BT_P_SUB;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint4 pc = *chunk(sub, tid, (ch & 1) * 4 + j);
          const uint32_t pw[4] = {pc.x, pc.y, pc.z, pc.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 pf = unpack_h2<false>(pw[e]);
            d4[e] = fmaf(pf.x, __uint_as_float(dv[8 * j + 2 * e]), d4[e]);
            d4[e] = fmaf(pf.y, __uint_as_float(dv[8 * j + 2 * e + 1]), d4[e]);
            s4[e] += pf.x + pf.y;
          }
        }
      }
      const float psum = (s4[0] + s4[1]) + (s4[2] + s4[3]);   // 0 on rows past T
      const float D = psum > 0.f ? ((d4[0] + d4[1]) + (d4[2] + d4[3])) / psum : 0.f;
      for (int ch = 0; ch < 2 * nkb; ++ch) {
        uint32_t dv[32];
        tmem_ld_32x32b_x32(lane_base + BT_S_COL + static_cast<uint32_t>(ch * 32), dv);
        tmem_ld_wait();
        uint8_t* sub = bt_smem + BT_P + (ch >> 1) * BT_P_SUB;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint4* cp = chunk(sub, tid, (ch & 1) * 4 + j);
          const uint4 pc = *cp;
          uint32_t pw[4] = {pc.x, pc.y, pc.z, pc.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 pf = unpack_h2<false>(pw[e]);
            pw[e] = pack_bf16x2(pf.x * (__uint_as_float(dv[8 * j + 2 * e]) - D) * 0.125f,
                                pf.y * (__uint_as_float(dv[8 * j + 2 * e + 1]) - D) * 0.125f);
          }
          *cp = make_uint4(pw[0], pw[1], pw[2], pw[3]);
        }
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();

    // ---- dQ = dS K (over dP), dK += dS^T Q
    if (tid == 0) {
      tc_fence_after();
      const uint64_t bk = umma_desc_sw128_mn(sbase + BT_K);
      for (int ks = 0; ks < 4 * nkb; ++ks)   // 16 keys per step: 32 B within a 64-key sub-tile, then the next sub-tile
        umma_bf16(tmem_base + BT_S_COL, umma_desc_sw128(sbase + BT_P + (ks >> 2) * BT_P_SUB) + 2 * (ks & 3),
                  bk + ks * (2048 >> 4), idesc_q, ks != 0 ? 1u : 0u);
      const uint64_t bq = umma_desc_sw128_mn(sbase + BT_Q);
      for (int kt = 0; kt < nqt; ++kt) {
        const uint64_t ast = umma_desc_sw128_mn(sbase + BT_P + 2 * kt * BT_P_SUB, BT_P_SUB);
        for (int ks = 0; ks < 4 * nq; ++ks)
          umma_bf16(tmem_base + BT_DK_COL + 64 * kt, ast + ks * (2048 >> 4), bq + ks * (2048 >> 4), idesc_t,
                    (qt > 0 || ks > 0) ? 1u : 0u);
      }
    }
    if (!(ok = commit_wait())) break;

    // ---- dQ -> bf16 -> staging -> TMA store (rows past T clipped)
    {
      uint32_t ov[64];
      tmem_ld_32x32b_x32(lane_base + BT_S_COL, *reinterpret_cast<uint32_t(*)[32]>(&ov[0]));
      tmem_ld_32x32b_x32(lane_base + BT_S_COL + 32, *reinterpret_cast<uint32_t(*)[32]>(&ov[32]));
      tmem_ld_wait();
#pragma unroll
      for (int j = 0; j < 8; ++j)
        *chunk(bt_smem + BT_ST, tid, j) =
            make_uint4(pack_bf16x2(__uint_as_float(ov[8 * j]), __uint_as_float(ov[8 * j + 1])),
                       pack_bf16x2(__uint_as_float(ov[8 * j + 2]), __uint_as_float(ov[8 * j + 3])),
                       pack_bf16x2(__uint_as_float(ov[8 * j + 4]), __uint_as_float(ov[8 * j + 5])),
                       pack_bf16x2(__uint_as_float(ov[8 * j + 6]), __uint_as_float(ov[8 * j + 7])));
    }
    fence_proxy_async_smem();
    tc_fence_before();   // the next tile's scores overwrite these columns
    __syncthreads();
    if (tid == 0) {
      for (int b = 0; b < nq; ++b) tma_store_4d(&tmOut, bt_smem + BT_ST + b * BT_TILE, 0, h, q0 + 64 * b, seq);
      bulk_commit();
    }
  }

  // ---- dK, dV of the key tiles -> bf16 -> staging over the (now free) P / dS tile -> TMA store
  if (ok) {
    for (int kt = 0; kt < nqt; ++kt)
      for (int m = 0; m < 2; ++m) {   // m = 0: dK, 1: dV
        uint32_t ov[64];
        const uint32_t col = (m == 0 ? BT_DK_COL : BT_DV_COL) + 64 * kt;
        tmem_ld_32x32b_x32(lane_base + col, *reinterpret_cast<uint32_t(*)[32]>(&ov[0]));
        tmem_ld_32x32b_x32(lane_base + col + 32, *reinterpret_cast<uint32_t(*)[32]>(&ov[32]));
        tmem_ld_wait();
        uint8_t* st = bt_smem + BT_P + (2 * kt + m) * BT_P_SUB;
#pragma unroll
        for (int j = 0; j < 8; ++j)
          *chunk(st, tid, j) = make_uint4(pack_bf16x2(__uint_as_float(ov[8 * j]), __uint_as_float(ov[8 * j + 1])),
                                          pack_bf16x2(__uint_as_float(ov[8 * j + 2]), __uint_as_float(ov[8 * j + 3])),
                                          pack_bf16x2(__uint_as_float(ov[8 * j + 4]), __uint_as_float(ov[8 * j + 5])),
                                          pack_bf16x2(__uint_as_float(ov[8 * j + 6]), __uint_as_float(ov[8 * j + 7])));
      }
    fence_proxy_async_smem();
    __syncthreads();
    if (tid == 0) {
      for (int kt = 0; kt < nqt; ++kt)
        for (int m = 0; m < 2; ++m)
          for (int b = 0; b < 2; ++b)
            if (128 * kt + 64 * b < T)
              tma_store_4d(&tmOut, bt_smem + BT_P + (2 * kt + m) * BT_P_SUB + b * BT_TILE, 0, (m + 1) * p.heads + h,
                           128 * kt + 64 * b, seq);
      bulk_commit();
    }
  }
  if (tid == 0) bulk_wait<0>();

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, BT_TMEM_COLS);
  }
}

// Tail backward of one view (one block): recompute y = ln_post(x0), f = y @ proj; df = dL/df through f / ||f|| when
// normalize; dy = proj df; dx0 = LayerNorm backward (gamma = ln_post weight).  Writes dx0 into row 0 of the view in g.
constexpr int TB_THREADS = 256;
__global__ void __launch_bounds__(TB_THREADS) tail_bwd_kernel(const float* __restrict__ x0, const float* __restrict__ dfeat, int W,
                                                              int E, const float* __restrict__ gam, const float* __restrict__ bet,
                                                              const float* __restrict__ proj, int normalize, int T,
                                                              float* __restrict__ g) {
  extern __shared__ float sm[];
  float* y = sm;          // [W]: xhat, then dy
  float* f = y + W;       // [E]: f, then df
  __shared__ float red[2][TB_THREADS / 32];
  const int64_t v = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* xr = x0 + v * W;
  auto block_sum = [&](float a, int slot) {
    for (int o = 16; o; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    if (lane == 0) red[slot][warp] = a;
    __syncthreads();
    float t = 0.f;
    for (int i = 0; i < TB_THREADS / 32; ++i) t += red[slot][i];
    __syncthreads();
    return t;
  };
  float s = 0.f;
  for (int c = tid; c < W; c += TB_THREADS) s += xr[c];
  const float mean = block_sum(s, 0) / W;
  float q = 0.f;
  for (int c = tid; c < W; c += TB_THREADS) { const float t = xr[c] - mean; q += t * t; }
  const float rstd = rsqrtf(block_sum(q, 1) / W + 1e-5f);
  for (int c = tid; c < W; c += TB_THREADS) y[c] = (xr[c] - mean) * rstd;
  __syncthreads();
  float nrm2 = 0.f;
  for (int e = tid; e < E; e += TB_THREADS) {
    float acc = 0.f;
    for (int c = 0; c < W; ++c) acc += (y[c] * gam[c] + bet[c]) * proj[static_cast<int64_t>(c) * E + e];
    f[e] = acc;
    nrm2 += acc * acc;
  }
  const float norm = sqrtf(block_sum(nrm2, 0));
  float dot = 0.f;
  for (int e = tid; e < E; e += TB_THREADS) dot += f[e] * dfeat[v * E + e];
  dot = block_sum(dot, 1);
  for (int e = tid; e < E; e += TB_THREADS) {
    const float d = dfeat[v * E + e];
    f[e] = normalize ? (d - f[e] * dot / (norm * norm)) / norm : d;
  }
  __syncthreads();
  float a = 0.f, b = 0.f;
  float dyc[8];   // W <= 8 * TB_THREADS
  int n = 0;
  for (int c = tid; c < W; c += TB_THREADS, ++n) {
    float acc = 0.f;
    const float* pr = proj + static_cast<int64_t>(c) * E;
    for (int e = 0; e < E; ++e) acc += pr[e] * f[e];
    const float gy = acc * gam[c];
    dyc[n] = gy;
    a += gy;
    b += gy * y[c];
  }
  a = block_sum(a, 0) / W;
  b = block_sum(b, 1) / W;
  n = 0;
  for (int c = tid; c < W; c += TB_THREADS, ++n) g[v * T * W + c] = rstd * (dyc[n] - a - y[c] * b);
}

// Deterministic split-row X^T Y: partial[chunk, i, j] = sum over rows m of chunk (rows_per_chunk consecutive rows) of
// X[m, i] Y[m, j], i < I, j < J (multiples of 64), fixed summation order.  64 x 64 output tile per block, 4 x 4 per thread.
constexpr int XT_TILE = 64, XT_ROWS = 32;
__global__ void __launch_bounds__(256) xty_partial_kernel(const void* __restrict__ X, int xt, int64_t ldx, const void* __restrict__ Y,
                                                          int yt, int64_t ldy, int64_t M, int I, int J, int64_t rows_per_chunk,
                                                          float* __restrict__ partial) {
  __shared__ float xs[XT_ROWS][XT_TILE + 4];
  __shared__ float ys[XT_ROWS][XT_TILE + 4];
  const int i0 = blockIdx.x * XT_TILE, j0 = blockIdx.y * XT_TILE;
  const int64_t m0 = blockIdx.z * rows_per_chunk;
  const int64_t m1 = min(M, m0 + rows_per_chunk);
  const int tid = threadIdx.x, ti = (tid >> 4) * 4, tj = (tid & 15) * 4;
  float acc[4][4] = {};
  for (int64_t mb = m0; mb < m1; mb += XT_ROWS) {
    for (int e = tid; e < XT_ROWS * XT_TILE; e += 256) {
      const int r = e >> 6, c = e & 63;
      const int64_t m = mb + r;
      const bool in = m < m1;
      xs[r][c] = in ? ld_any(X, xt, m * ldx + i0 + c) : 0.f;
      ys[r][c] = in ? ld_any(Y, yt, m * ldy + j0 + c) : 0.f;
    }
    __syncthreads();
#pragma unroll 4
    for (int r = 0; r < XT_ROWS; ++r) {
      float a[4], b[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) { a[u] = xs[r][ti + u]; b[u] = ys[r][tj + u]; }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int w = 0; w < 4; ++w) acc[u][w] += a[u] * b[w];
    }
    __syncthreads();
  }
  float* out = partial + static_cast<int64_t>(blockIdx.z) * I * J;
#pragma unroll
  for (int u = 0; u < 4; ++u)
#pragma unroll
    for (int w = 0; w < 4; ++w) out[static_cast<int64_t>(i0 + ti + u) * J + j0 + tj + w] = acc[u][w];
}

// acc[e] += sum_{c = 0 .. chunks-1} partial[c, e] in that order
__global__ void reduce_chunks_kernel(const float* __restrict__ partial, int chunks, int64_t n, float* __restrict__ acc) {
  for (int64_t e = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; e < n; e += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    float s = 0.f;
    for (int c = 0; c < chunks; ++c) s += partial[c * n + e];
    acc[e] += s;
  }
}

// out[r, c] = scale * src[(r0 + r) * lds + c0 + c]
__global__ void extract_kernel(const float* __restrict__ src, int64_t lds, int r0, int c0, int rows, int cols, float scale,
                               float* __restrict__ out) {
  const int64_t n = static_cast<int64_t>(rows) * cols;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int r = static_cast<int>(i / cols), c = static_cast<int>(i % cols);
    out[i] = scale * src[(r0 + r) * lds + c0 + c];
  }
}

// dst[c, r] = 16-bit(src[r, c]) for a [rows, cols] fp32 matrix (Wt copies of the backward GEMMs)
__global__ void transpose_cast_kernel(const float* __restrict__ src, int rows, int cols, bool f16, uint16_t* __restrict__ dst) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int k = threadIdx.y; k < 32; k += blockDim.y) {
    const int r = r0 + k, c = c0 + threadIdx.x;
    if (r < rows && c < cols) tile[k][threadIdx.x] = src[static_cast<int64_t>(r) * cols + c];
  }
  __syncthreads();
  for (int k = threadIdx.y; k < 32; k += blockDim.y) {
    const int c = c0 + k, r = r0 + threadIdx.x;
    if (r < rows && c < cols) dst[static_cast<int64_t>(c) * rows + r] = to16(tile[threadIdx.x][k], f16);
  }
}

// The adapter matrices of one projection group (in_proj: q, k, v; or out_proj: o) from fp32 device A_p [r_p, W] and
// B_p [W, r_p].  Element (a, b) of the output of kind `kind`:
//   LP_DN     [128, W]        16-bit: row j0_p + j = A_p[j]                       (the applied-mode down matrix)
//   LP_UP     [n_out, 64]     16-bit: [n0_p + n, j0_p + j] = s_p B_p[n, j]        (the applied-mode up matrix)
//   LP_DN_BLK [128, npj W]    16-bit: [j0_p + j, p W + c] = A_p[j, c]             (down matrix over the dropout copies)
//   LP_DN_T   [npj W, 64]     bf16: the transpose of LP_DN_BLK's first 64 rows
//   LP_UP_T   [128, n_out]    bf16: [j0_p + j, n0_p + n] = s_p B_p[n, j]
__global__ void lora_pack_kernel(LoraGroup g, int kind, int W, int n_out, bool f16, uint16_t* __restrict__ out) {
  int64_t rows, cols;
  switch (kind) {
    case LP_DN: rows = 128; cols = W; break;
    case LP_UP: rows = n_out; cols = 64; break;
    case LP_DN_BLK: rows = 128; cols = static_cast<int64_t>(g.npj) * W; break;
    case LP_DN_T: rows = static_cast<int64_t>(g.npj) * W; cols = 64; break;
    default: rows = 128; cols = n_out; break;
  }
  const bool o16 = (kind == LP_DN_T || kind == LP_UP_T) ? false : f16;
  const int64_t n = rows * cols;
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t a = i / cols, b = i - a * cols;
    // (j, x): the rank index and the other coordinate, by kind
    int64_t j, x;
    if (kind == LP_DN || kind == LP_DN_BLK || kind == LP_UP_T) { j = a; x = b; } else { j = b; x = a; }
    float val = 0.f;
    for (int p = 0; p < g.npj; ++p) {
      if (!g.A[p] || j < g.j0[p] || j >= g.j0[p] + g.r[p]) continue;
      const int jj = static_cast<int>(j - g.j0[p]);
      if (kind == LP_DN) val = g.A[p][jj * static_cast<int64_t>(W) + x];
      else if (kind == LP_DN_BLK || kind == LP_DN_T) {
        if (x >= p * static_cast<int64_t>(W) && x < (p + 1) * static_cast<int64_t>(W)) val = g.A[p][jj * static_cast<int64_t>(W) + x - p * W];
      } else {
        const int64_t nn = x - g.n0[p];
        if (nn >= 0 && nn < W) val = g.s[p] * g.B[p][nn * g.r[p] + jj];
      }
    }
    out[i] = to16(val, o16);
  }
}

unsigned grid_for(int64_t n, int threads = 256) {
  return static_cast<unsigned>(std::min<int64_t>((n + threads - 1) / threads, 148 * 32));
}

}  // namespace

cudaError_t launch_dropout_fwd(const __nv_bfloat16* x, int64_t M, int W, int npj, int proj0, const DropoutArgs& d, int64_t row0,
                               int f16, __nv_bfloat16* xd, cudaStream_t s) {
  if (M <= 0) return cudaSuccess;
  dropout_fwd_kernel<<<grid_for(M * W * npj), 256, 0, s>>>(reinterpret_cast<const uint16_t*>(x), M, W, npj, proj0, d, row0,
                                                           f16 != 0, reinterpret_cast<uint16_t*>(xd));
  return cudaGetLastError();
}
cudaError_t launch_dropout_bwd_add(const float* dxd, int64_t M, int W, int npj, int proj0, const DropoutArgs& d, int64_t row0,
                                   float* dx, cudaStream_t s) {
  if (M <= 0) return cudaSuccess;
  dropout_bwd_add_kernel<<<grid_for(M * W), 256, 0, s>>>(dxd, M, W, npj, proj0, d, row0, dx);
  return cudaGetLastError();
}
cudaError_t launch_dropout_mask(const DropoutArgs& d, int proj, int64_t rows, int cols, uint8_t* out, cudaStream_t s) {
  if (rows <= 0 || cols <= 0) return cudaSuccess;
  dropout_mask_kernel<<<grid_for(rows * cols), 256, 0, s>>>(d, proj, rows, cols, out);
  return cudaGetLastError();
}
cudaError_t launch_gelu_bwd(const float* dy, const __nv_bfloat16* h, int64_t n, int h_f16, __nv_bfloat16* dh, cudaStream_t s) {
  if (n <= 0) return cudaSuccess;
  gelu_bwd_kernel<<<grid_for(n), 256, 0, s>>>(dy, reinterpret_cast<const uint16_t*>(h), n, h_f16 != 0, reinterpret_cast<uint16_t*>(dh));
  return cudaGetLastError();
}
cudaError_t launch_ln_bwd(const float* x, const float* dy, int64_t rows, int W, const float* gamma, float* g, cudaStream_t s) {
  if (rows <= 0) return cudaSuccess;
  ln_bwd_kernel<<<static_cast<unsigned>((rows + 7) / 8), 256, 0, s>>>(x, dy, rows, W, gamma, g);
  return cudaGetLastError();
}
// fp32 dO [n_seq, T, heads, 64] as a 4-D tensor (d, head, token, sequence), boxes of [128 tokens][32] (128-byte rows,
// unswizzled); tokens past T are zero on load
bool make_tmap_dout(CUtensorMap* tm, const float* base, uint64_t n_seq, uint64_t T, uint64_t heads) {
  auto encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(gemm_encode_tiled_fn());
  if (!encode) return false;
  const uint64_t row_bytes = heads * 64 * 4;
  cuuint64_t gdim[4] = {64, heads, T, n_seq};
  cuuint64_t gstride[3] = {64 * 4, row_bytes, T * row_bytes};
  cuuint32_t box[4] = {32, 1, 128, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return encode(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(base), gdim, gstride, box, estr,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

cudaError_t launch_attention_bwd(const __nv_bfloat16* qkv, const float* dout, int64_t n_views, int T, int heads, int f16,
                                 __nv_bfloat16* dqkv, cudaStream_t s, int* dev_status) {
  if (T < 1 || T > 256 || heads < 1) return cudaErrorInvalidValue;
  if (n_views <= 0) return cudaSuccess;
  if (T > AB_T) {
    if (dev_status == nullptr) return cudaErrorInvalidValue;
    if ((reinterpret_cast<uintptr_t>(qkv) | reinterpret_cast<uintptr_t>(dout) | reinterpret_cast<uintptr_t>(dqkv)) & 15)
      return cudaErrorInvalidValue;
    CUtensorMap tmQKV, tmDO, tmOut;
    if (!make_tmap_heads(&tmQKV, qkv, static_cast<uint64_t>(n_views), static_cast<uint64_t>(T), 3ull * heads, f16) ||
        !make_tmap_dout(&tmDO, dout, static_cast<uint64_t>(n_views), static_cast<uint64_t>(T), static_cast<uint64_t>(heads)) ||
        !make_tmap_heads(&tmOut, dqkv, static_cast<uint64_t>(n_views), static_cast<uint64_t>(T), 3ull * heads, 0))
      return cudaErrorInvalidValue;
    cudaError_t e = ensure_dynamic_smem(attention_bwd_tcgen05_kernel, BT_SMEM);
    if (e != cudaSuccess) return e;
    AbtDev p;
    p.heads = heads;
    p.T = T;
    p.f16 = f16 != 0;
    p.status = dev_status;
    attention_bwd_tcgen05_kernel<<<static_cast<unsigned>(n_views * heads), BT_THREADS, BT_SMEM, s>>>(tmQKV, tmDO, tmOut, p);
    return cudaGetLastError();
  }
  const size_t smem = (6 * AB_T * AB_LD + AB_T) * sizeof(float);
  cudaError_t e = ensure_dynamic_smem(attention_bwd_kernel, smem);
  if (e != cudaSuccess) return e;
  attention_bwd_kernel<<<static_cast<unsigned>(n_views * heads), AB_THREADS, smem, s>>>(
      reinterpret_cast<const uint16_t*>(qkv), dout, T, heads, f16 != 0, reinterpret_cast<uint16_t*>(dqkv));
  return cudaGetLastError();
}
cudaError_t launch_tail_bwd(const float* x0, const float* dfeat, int64_t n_views, int W, int E, const float* g, const float* b,
                            const float* proj, int normalize, int T, float* grad, cudaStream_t s) {
  if (W > 8 * TB_THREADS) return cudaErrorInvalidValue;
  if (n_views <= 0) return cudaSuccess;
  tail_bwd_kernel<<<static_cast<unsigned>(n_views), TB_THREADS, (W + E) * sizeof(float), s>>>(x0, dfeat, W, E, g, b, proj, normalize,
                                                                                            T, grad);
  return cudaGetLastError();
}
int64_t xty_chunk_rows(int64_t M) {
  // at most 128 chunks; a multiple of XT_ROWS rows each
  const int64_t r = (M + 127) / 128;
  return std::max<int64_t>(XT_ROWS, (r + XT_ROWS - 1) / XT_ROWS * XT_ROWS);
}
cudaError_t launch_xty_accumulate(const void* X, int xt, int64_t ldx, const void* Y, int yt, int64_t ldy, int64_t M, int I, int J,
                                  float* partial, float* acc, cudaStream_t s) {
  if (I % XT_TILE || J % XT_TILE) return cudaErrorInvalidValue;
  if (M <= 0) return cudaSuccess;
  const int64_t rpc = xty_chunk_rows(M);
  const int chunks = static_cast<int>((M + rpc - 1) / rpc);
  xty_partial_kernel<<<dim3(I / XT_TILE, J / XT_TILE, chunks), 256, 0, s>>>(X, xt, ldx, Y, yt, ldy, M, I, J, rpc, partial);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  reduce_chunks_kernel<<<grid_for(static_cast<int64_t>(I) * J), 256, 0, s>>>(partial, chunks, static_cast<int64_t>(I) * J, acc);
  return cudaGetLastError();
}
cudaError_t launch_extract(const float* src, int64_t lds, int r0, int c0, int rows, int cols, float scale, float* out, cudaStream_t s) {
  if (rows <= 0 || cols <= 0) return cudaSuccess;
  extract_kernel<<<grid_for(static_cast<int64_t>(rows) * cols), 256, 0, s>>>(src, lds, r0, c0, rows, cols, scale, out);
  return cudaGetLastError();
}
cudaError_t launch_transpose_cast(const float* src, int rows, int cols, int f16, __nv_bfloat16* dst, cudaStream_t s) {
  transpose_cast_kernel<<<dim3((cols + 31) / 32, (rows + 31) / 32), dim3(32, 8), 0, s>>>(src, rows, cols, f16 != 0,
                                                                                        reinterpret_cast<uint16_t*>(dst));
  return cudaGetLastError();
}
cudaError_t launch_lora_pack(const LoraGroup& g, int kind, int W, int n_out, int f16, __nv_bfloat16* out, cudaStream_t s) {
  lora_pack_kernel<<<grid_for(static_cast<int64_t>(128) * 4 * W), 256, 0, s>>>(g, kind, W, n_out, f16 != 0, reinterpret_cast<uint16_t*>(out));
  return cudaGetLastError();
}

}  // namespace jcb
