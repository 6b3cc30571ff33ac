// Bandwidth-bound kernels of the image tower: im2col (+ CLIP normalisation), cls/pos + ln_pre + ln_1,
// LayerNorm, the ln_post + projection + L2-norm tail, and the weight-packing helpers.
// All are warp-per-row with 128-bit loads and shuffle reductions; fp32 statistics throughout.
//
// Reference: jclip/model.py:17-21 (LayerNorm), :105-115 (conv1 as patches, cls, pos, ln_pre),
// :121-124 (ln_post, proj), test.py:1301 (tfm_clip), test.py:1706 (L2 normalisation),
// test.py:310-313 (merge_BA).
#include <algorithm>

#include <cstdlib>
#include <cooperative_groups.h>

#include "kernels.h"
#include "ptx.cuh"

namespace jcb {

namespace {

constexpr float LN_EPS = 1e-5f;  // Jittor nn.LayerNorm default

__constant__ float c_clip_mean[3] = {0.48145466f, 0.4578275f, 0.40821073f};
__constant__ float c_clip_std[3] = {0.26862954f, 0.26130258f, 0.27577711f};

// ------------------------------------------------------------------------------------------ im2col
// One block = the K / 8 eight-pixel chunks of a patch row (384 threads for patch 32); a thread keeps its (channel, row,
// column) offset for the whole kernel and walks over patches, UNROLL of them in flight.  Eight pixels per thread for
// every input type: a warp's store is then 512 contiguous bytes (with 16 uint8 pixels per thread each lane wrote two
// 16-byte halves 32 bytes apart -- every store instruction touched 32 half-filled sectors and the kernel sat in the
// LSU queue, ncu: 41 % lg_throttle).
// ToTensor's 1/255 and tfm_clip's (x - mean_c) / std_c are one FMA per pixel, x * a_c + b_c with a_c = 1 / (255 std_c),
// b_c = -mean_c / std_c: for all 3 x 256 possible uint8 inputs the bf16-rounded result equals the reference's
// ((u / 255) - mean) / std evaluated in fp32 (tests/test_host_logic.py::test_u8_normalise_fma_is_exact_in_bf16).
// The first version spent ~600 instructions per thread on 64-bit index divisions and fp32 divisions and ran at
// 1.7 TB/s; this one is a plain streaming kernel.
constexpr int IM2COL_UNROLL = 4;

template <int DT, bool F16>
__global__ void __launch_bounds__(384)
im2col_kernel(const void* __restrict__ images, unsigned n_patches, int R, int P, int G, int apply_norm,
              __nv_bfloat16* __restrict__ patches) {
  griddep_wait();               // programmatic dependent launch (ptx.cuh): nothing global is touched above
  constexpr int EPT = 8;   // 8 pixels per thread for every input type: one fully coalesced 16-byte store per lane
  const int K = 3 * P * P;
  const int col = static_cast<int>(threadIdx.x) * EPT;  // (c, i, j) with j % EPT == 0
  const int c = col / (P * P);
  const int i = (col % (P * P)) / P;
  const int j = col % P;
  const long long thread_off = (static_cast<long long>(c) * R + i) * R + j;   // offset inside a view, patch (0, 0)
  const long long view_elems = 3LL * R * R;
  const int GG = G * G;
  float a = DT == IMG_U8 ? 1.0f / 255.0f : 1.0f, b = 0.0f;
  if (apply_norm) {
    a = 1.0f / ((DT == IMG_U8 ? 255.0f : 1.0f) * c_clip_std[c]);
    b = -c_clip_mean[c] / c_clip_std[c];
  }
  constexpr int NR = DT == IMG_F32 ? 2 : 1;
  auto load = [&](unsigned p, uint4 (&raw)[NR]) {
    const unsigned view = p / GG, pidx = p - view * GG;
    const unsigned py = pidx / G, px = pidx - py * G;
    const long long src = view * view_elems + thread_off + (static_cast<long long>(py) * R + px) * P;
    if (DT == IMG_F32) {
      const uint4* s4 = reinterpret_cast<const uint4*>(static_cast<const float*>(images) + src);
      raw[0] = __ldg(s4);
      raw[NR - 1] = __ldg(s4 + 1);
    } else if (DT == IMG_BF16) {
      raw[0] = __ldg(reinterpret_cast<const uint4*>(static_cast<const __nv_bfloat16*>(images) + src));
    } else {
      const uint2 t = __ldg(reinterpret_cast<const uint2*>(static_cast<const uint8_t*>(images) + src));
      raw[0] = make_uint4(t.x, t.y, 0u, 0u);
    }
  };
  auto emit = [&](unsigned p, const uint4 (&raw)[NR]) {
    float f[EPT];
    if (DT == IMG_F32) {
      const float* v = reinterpret_cast<const float*>(&raw[0]);
#pragma unroll
      for (int e = 0; e < 8; ++e) f[e] = v[e];
    } else if (DT == IMG_BF16) {
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw[0]);
#pragma unroll
      for (int e = 0; e < 4; ++e) { const float2 t = __bfloat1622float2(h[e]); f[2 * e] = t.x; f[2 * e + 1] = t.y; }
    } else {
      const uint32_t* w = reinterpret_cast<const uint32_t*>(&raw[0]);
      // uint8 -> fp32 without the quarter-rate I2F: one PRMT drops the byte into the mantissa of 2^23 (0x4B000000),
      // one FADD removes the 2^23 again -- exact for 0..255
#pragma unroll
      for (int e = 0; e < EPT; ++e)
        f[e] = __uint_as_float(__byte_perm(w[e >> 2], 0x4B000000u, 0x7540u + (e & 3))) - 8388608.0f;
    }
#pragma unroll
    for (int e = 0; e < EPT; ++e) f[e] = fmaf(f[e], a, b);
    uint4* dst = reinterpret_cast<uint4*>(patches + static_cast<long long>(p) * K + col);
#pragma unroll
    for (int h = 0; h < EPT / 8; ++h) {
      uint4 o;
      o.x = pack_h2<F16>(f[8 * h + 0], f[8 * h + 1]); o.y = pack_h2<F16>(f[8 * h + 2], f[8 * h + 3]);
      o.z = pack_h2<F16>(f[8 * h + 4], f[8 * h + 5]); o.w = pack_h2<F16>(f[8 * h + 6], f[8 * h + 7]);
      dst[h] = o;
    }
  };
  // full groups of UNROLL patches: no exit between the loads and their uses, so all UNROLL loads are in flight together
  // (with a tail check inside the group the compiler sank every load to its use: one 16-byte load in flight per thread)
  const unsigned n_full = n_patches / IM2COL_UNROLL * IM2COL_UNROLL;
  for (unsigned p0 = blockIdx.x * IM2COL_UNROLL; p0 < n_full; p0 += gridDim.x * IM2COL_UNROLL) {
    uint4 raw[IM2COL_UNROLL][NR];
#pragma unroll
    for (int u = 0; u < IM2COL_UNROLL; ++u) load(p0 + u, raw[u]);
#pragma unroll
    for (int u = 0; u < IM2COL_UNROLL; ++u) emit(p0 + u, raw[u]);
  }
  for (unsigned p = n_full + blockIdx.x; p < n_patches; p += gridDim.x) {
    uint4 raw[NR];
    load(p, raw);
    emit(p, raw);
  }
}

// ------------------------------------------------------------------------------------------ LayerNorm
template <int NV>
__device__ __forceinline__ void row_stats(const float4 (&v)[NV], int W, float& mean, float& rstd) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  mean = warp_sum(s) / static_cast<float>(W);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    q += (a * a + b * b) + (c * c + d * d);
  }
  const float var = warp_sum(q) / static_cast<float>(W);  // biased variance
  rstd = 1.0f / sqrtf(var + LN_EPS);
}

template <int NV>
__device__ __forceinline__ void normalize_row(float4 (&v)[NV], float mean, float rstd, const float* __restrict__ g,
                                              const float* __restrict__ b, int lane) {
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float4 gg = __ldg(reinterpret_cast<const float4*>(g) + lane + 32 * i);
    const float4 bb = __ldg(reinterpret_cast<const float4*>(b) + lane + 32 * i);
    v[i].x = (v[i].x - mean) * rstd * gg.x + bb.x;
    v[i].y = (v[i].y - mean) * rstd * gg.y + bb.y;
    v[i].z = (v[i].z - mean) * rstd * gg.z + bb.z;
    v[i].w = (v[i].w - mean) * rstd * gg.w + bb.w;
  }
}

template <int NV, bool F16>
__device__ __forceinline__ void store_row_h(const float4 (&v)[NV], __nv_bfloat16* __restrict__ y, int lane) {
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    uint2 o;
    o.x = pack_h2<F16>(v[i].x, v[i].y);
    o.y = pack_h2<F16>(v[i].z, v[i].w);
    reinterpret_cast<uint2*>(y)[lane + 32 * i] = o;
  }
}

constexpr int LN_WARPS = 8;

// what a residual GEMM epilogue with EPI_RESID_LNPREP_* leaves behind, for the first block of a tower:
// y = 16-bit (x - shift), stats[0] = (sum, sum of squares) of the centred copy, stats[1..slots) = 0, and
// shift = the row mean (exact here: the whole row is in registers).  shift == nullptr: uncentred copy (shift 0).
template <int NV, bool F16>
__device__ __forceinline__ void emit_raw_and_stats(float4 (&v)[NV], __nv_bfloat16* __restrict__ y,
                                                   float* __restrict__ st, int slots, float* __restrict__ shift,
                                                   int lane) {
  float mean = 0.f;
  if (shift != nullptr) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i) t += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    mean = warp_sum(t) / static_cast<float>(NV * 128);
  }
  float s = 0.f, q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    v[i].x -= mean; v[i].y -= mean; v[i].z -= mean; v[i].w -= mean;
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    q += (v[i].x * v[i].x + v[i].y * v[i].y) + (v[i].z * v[i].z + v[i].w * v[i].w);
  }
  s = warp_sum(s);
  q = warp_sum(q);
  store_row_h<NV, F16>(v, y, lane);
  if (lane < 2 * slots) st[lane] = lane == 0 ? s : (lane == 1 ? q : 0.f);
  if (shift != nullptr && lane == 0) *shift = mean;
}

template <int NV, bool F16>
__global__ void __launch_bounds__(LN_WARPS * 32)
layernorm_kernel(const float* __restrict__ x, long long rows, const float* __restrict__ g,
                 const float* __restrict__ b, __nv_bfloat16* __restrict__ y) {
  constexpr int W = NV * 128;
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * LN_WARPS + (threadIdx.x >> 5);
  if (row >= rows) return;
  float4 v[NV];
  const float4* xr = reinterpret_cast<const float4*>(x + row * W);
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = xr[lane + 32 * i];
  float mean, rstd;
  row_stats<NV>(v, W, mean, rstd);
  normalize_row<NV>(v, mean, rstd, g, b, lane);
  store_row_h<NV, F16>(v, y + row * W, lane);
}

template <int NV, bool F16>
__global__ void __launch_bounds__(LN_WARPS * 32)
embed_ln_kernel(float* __restrict__ tokens, long long rows, int T, const float* __restrict__ cls,
                const float* __restrict__ pos, const float* __restrict__ vpt, int n_vpt,
                const float* __restrict__ g_pre, const float* __restrict__ b_pre,
                const float* __restrict__ g1, const float* __restrict__ b1, __nv_bfloat16* __restrict__ y,
                float* __restrict__ stats, int stats_slots, const float* __restrict__ patch_out,
                float* __restrict__ shift) {
  griddep_wait();               // programmatic dependent launch (ptx.cuh): nothing global is touched above
  constexpr int W = NV * 128;
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * LN_WARPS + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int t = static_cast<int>(row % T);
  float4 v[NV];
  float4* xr = reinterpret_cast<float4*>(tokens + row * W);
  if (t == 0) {
    // class token: class_embedding + positional_embedding[0]   (jclip/model.py:109-114)
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float4 c = __ldg(reinterpret_cast<const float4*>(cls) + lane + 32 * i);
      const float4 p = __ldg(reinterpret_cast<const float4*>(pos) + lane + 32 * i);
      v[i] = make_float4(c.x + p.x, c.y + p.y, c.z + p.z, c.w + p.w);
    }
  } else if (t >= T - n_vpt) {
    // IVLP / VPT prompt tokens, appended after the positional embedding  (jclip/model1.py:192-196)
#pragma unroll
    for (int i = 0; i < NV; ++i)
      v[i] = __ldg(reinterpret_cast<const float4*>(vpt + static_cast<long long>(t - (T - n_vpt)) * W) + lane + 32 * i);
  } else if (patch_out != nullptr) {
    // patch embedding from the conv1 GEMM's dense output [view * (T - 1 - n_vpt) + t - 1, W] + positional embedding
    const long long prow = (row / T) * (T - 1 - n_vpt) + (t - 1);
    const float4* pr = reinterpret_cast<const float4*>(patch_out + prow * W);
    const float4* pe = reinterpret_cast<const float4*>(pos + static_cast<long long>(t) * W);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float4 a = pr[lane + 32 * i];
      const float4 p = __ldg(pe + lane + 32 * i);
      v[i] = make_float4(a.x + p.x, a.y + p.y, a.z + p.z, a.w + p.w);
    }
  } else {
#pragma unroll
    for (int i = 0; i < NV; ++i) v[i] = xr[lane + 32 * i];  // patch embedding + pos already in place (scatter epilogue)
  }
  float mean, rstd;
  row_stats<NV>(v, W, mean, rstd);
  normalize_row<NV>(v, mean, rstd, g_pre, b_pre, lane);  // ln_pre -> residual stream
#pragma unroll
  for (int i = 0; i < NV; ++i) xr[lane + 32 * i] = v[i];
  if (stats != nullptr) {   // LayerNorm folded into the consuming GEMM: centred 16-bit copy + (sum, sum of squares)
    emit_raw_and_stats<NV, F16>(v, y + row * W, stats + row * stats_slots * 2, stats_slots,
                                shift ? shift + row : nullptr, lane);
    return;
  }
  row_stats<NV>(v, W, mean, rstd);
  normalize_row<NV>(v, mean, rstd, g1, b1, lane);        // layer 0's ln_1
  store_row_h<NV, F16>(v, y + row * W, lane);
}

// ------------------------------------------------------------------------------------------ text front end
template <int NV, bool F16>
__global__ void __launch_bounds__(LN_WARPS * 32)
text_embed_ln_kernel(const long long* __restrict__ ids, long long rows, int T, int vocab,
                     const float* __restrict__ tok_emb, const float* __restrict__ pos, const float* __restrict__ g1,
                     const float* __restrict__ b1, float* __restrict__ tokens, __nv_bfloat16* __restrict__ y,
                     int* __restrict__ eot, float* __restrict__ stats, int stats_slots, float* __restrict__ shift) {
  constexpr int W = NV * 128;
  const int lane = threadIdx.x & 31;
  const long long row = static_cast<long long>(blockIdx.x) * LN_WARPS + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int t = static_cast<int>(row % T);
  long long id = ids[row];
  id = id < 0 ? 0 : (id >= vocab ? vocab - 1 : id);   // out-of-range ids are clamped, never read out of bounds
  float4 v[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float4 e = __ldg(reinterpret_cast<const float4*>(tok_emb + id * W) + lane + 32 * i);
    const float4 p = __ldg(reinterpret_cast<const float4*>(pos + static_cast<long long>(t) * W) + lane + 32 * i);
    v[i] = make_float4(e.x + p.x, e.y + p.y, e.z + p.z, e.w + p.w);
  }
  float4* xr = reinterpret_cast<float4*>(tokens + row * W);
#pragma unroll
  for (int i = 0; i < NV; ++i) xr[lane + 32 * i] = v[i];
  if (stats != nullptr) {
    emit_raw_and_stats<NV, F16>(v, y + row * W, stats + row * stats_slots * 2, stats_slots,
                                shift ? shift + row : nullptr, lane);
  } else {
    float mean, rstd;
    row_stats<NV>(v, W, mean, rstd);
    normalize_row<NV>(v, mean, rstd, g1, b1, lane);
    store_row_h<NV, F16>(v, y + row * W, lane);
  }
  if (t == 0) {  // the warp of a sequence's first token also finds its EOT position: first maximum of the ids
    long long best = -1;
    int best_t = 0;
    for (int j = lane; j < T; j += 32) {
      const long long c = ids[row + j];
      if (c > best) { best = c; best_t = j; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const long long ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int ot = __shfl_xor_sync(0xffffffffu, best_t, o);
      if (ob > best || (ob == best && ot < best_t)) { best = ob; best_t = ot; }
    }
    if (lane == 0) eot[row / T] = best_t;
  }
}

// ------------------------------------------------------------------------------------------ tail
// ln_post(row) @ proj, L2 norm (jclip/model.py:121-124, :211-214; test.py:1706).  TAIL_VIEWS sequences per CTA so that
// proj [W, E] is streamed from L2 once per 16 sequences; warp w owns output columns 64 w + lane and 64 w + 32 + lane.
// The k dimension is summed as TAIL_SPLIT partial sums over consecutive k ranges, added up in range order, and the
// squared norm as one warp-shuffle sum per 64-column slice, slices added in order -- an order that ONE CTA can follow
// (many views: the default form) and that a CLUSTER of TAIL_SPLIT CTAs can follow as well, CTA j taking k range j:
// partial sums travel to the CTA that owns their column slice through distributed shared memory, slice norms to every
// CTA.  Both forms give the same bits.  The cluster form is for few views (one image x 65 views per call, the
// reference's own loop): the 192 dependent L2 round trips of the k loop become 24 (139 -> ~25 us per call).
constexpr int TAIL_VIEWS = 16;
constexpr int TAIL_THREADS = 256;
constexpr int TAIL_SPLIT = 8;     // k ranges = warps per CTA = CTAs per cluster

template <int NV, int E, bool CLUSTER>
__global__ void __launch_bounds__(TAIL_THREADS)
tail_kernel(const float* __restrict__ tokens, long long n_views, int T, const float* __restrict__ g,
            const float* __restrict__ b, const float* __restrict__ proj, int normalize, float* __restrict__ out,
            const int* __restrict__ row_idx) {
  namespace cg = cooperative_groups;
  constexpr int W = NV * 128;
  constexpr int KR = W / TAIL_SPLIT;      // k values per range
  static_assert(E == 64 * (TAIL_THREADS / 32) && TAIL_THREADS / 32 == TAIL_SPLIT && KR % 4 == 0, "tail tiling");
  extern __shared__ __align__(16) float tail_smem[];
  float (*s_x)[W] = reinterpret_cast<float (*)[W]>(tail_smem);                                     // [TAIL_VIEWS][W]
  float (*s_q)[TAIL_VIEWS] = reinterpret_cast<float (*)[TAIL_VIEWS]>(tail_smem + TAIL_VIEWS * W);  // [slice][view]
  // cluster form: partial sums of THIS CTA's column slice from every k range, [range][view][64]
  float (*s_in)[TAIL_VIEWS][64] = reinterpret_cast<float (*)[TAIL_VIEWS][64]>(tail_smem + TAIL_VIEWS * W + TAIL_SPLIT * TAIL_VIEWS);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  griddep_wait();               // programmatic dependent launch (ptx.cuh): nothing global is touched above
  const int crank = CLUSTER ? static_cast<int>(cg::this_cluster().block_rank()) : 0;
  const long long v0 = static_cast<long long>(CLUSTER ? blockIdx.x / TAIL_SPLIT : blockIdx.x) * TAIL_VIEWS;
  for (int vv = warp; vv < TAIL_VIEWS; vv += TAIL_THREADS / 32) {  // ln_post on the CLS row of view v0 + vv  (jclip/model.py:121)
    const long long view = v0 + vv;
    float4 v[NV];
    if (view < n_views) {
      const long long trow = view * T + (row_idx ? row_idx[view] : 0);
      const float4* xr = reinterpret_cast<const float4*>(tokens + trow * W);
#pragma unroll
      for (int i = 0; i < NV; ++i) v[i] = xr[lane + 32 * i];
      float mean, rstd;
      row_stats<NV>(v, W, mean, rstd);
      normalize_row<NV>(v, mean, rstd, g, b, lane);
    } else {
#pragma unroll
      for (int i = 0; i < NV; ++i) v[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int i = 0; i < NV; ++i) reinterpret_cast<float4*>(s_x[vv])[lane + 32 * i] = v[i];
  }
  __syncthreads();
  const int col = 64 * warp + lane;       // this thread's output columns: col, col + 32
  float tot[TAIL_VIEWS][2];
#pragma unroll
  for (int v = 0; v < TAIL_VIEWS; ++v) tot[v][0] = tot[v][1] = 0.f;
  const int j0 = CLUSTER ? crank : 0, j1 = CLUSTER ? crank + 1 : TAIL_SPLIT;
  for (int j = j0; j < j1; ++j) {   // x @ proj  (jclip/model.py:123-124), fp32: one partial sum per k range
    float part[TAIL_VIEWS][2];
#pragma unroll
    for (int v = 0; v < TAIL_VIEWS; ++v) part[v][0] = part[v][1] = 0.f;
    for (int k = j * KR; k < (j + 1) * KR; k += 4) {   // four k per step, x read as float4
      float pw[4][2];
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        pw[kk][0] = __ldg(proj + static_cast<long long>(k + kk) * E + col);
        pw[kk][1] = __ldg(proj + static_cast<long long>(k + kk) * E + col + 32);
      }
#pragma unroll
      for (int v = 0; v < TAIL_VIEWS; ++v) {
        const float4 xv = *reinterpret_cast<const float4*>(&s_x[v][k]);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          part[v][e] = fmaf(xv.x, pw[0][e], part[v][e]);
          part[v][e] = fmaf(xv.y, pw[1][e], part[v][e]);
          part[v][e] = fmaf(xv.z, pw[2][e], part[v][e]);
          part[v][e] = fmaf(xv.w, pw[3][e], part[v][e]);
        }
      }
    }
    if (CLUSTER) {   // to the CTA that owns this warp's column slice (CTA `warp`), slot of k range j
      float (*dst)[TAIL_VIEWS][64] = cg::this_cluster().map_shared_rank(s_in, warp);
#pragma unroll
      for (int v = 0; v < TAIL_VIEWS; ++v) {
        dst[j][v][lane] = part[v][0];
        dst[j][v][lane + 32] = part[v][1];
      }
    } else {
#pragma unroll
      for (int v = 0; v < TAIL_VIEWS; ++v) {
        tot[v][0] = __fadd_rn(tot[v][0], part[v][0]);
        tot[v][1] = __fadd_rn(tot[v][1], part[v][1]);
      }
    }
  }
  if (CLUSTER) {
    cg::cluster_group cluster = cg::this_cluster();
    cluster.sync();
    // this CTA finishes column slice `crank`: warp w takes views w and w + 8, lane l columns l and l + 32 of the slice
    float x[2][2];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int v = warp + 8 * h;
      float t0 = 0.f, t1 = 0.f;
#pragma unroll
      for (int j = 0; j < TAIL_SPLIT; ++j) {
        t0 = __fadd_rn(t0, s_in[j][v][lane]);
        t1 = __fadd_rn(t1, s_in[j][v][lane + 32]);
      }
      x[h][0] = t0; x[h][1] = t1;
      const float q = warp_sum(__fmaf_rn(t1, t1, __fmul_rn(t0, t0)));
      if (lane < TAIL_SPLIT) cluster.map_shared_rank(s_q, lane)[crank][v] = q;   // the slice norm to every CTA
    }
    cluster.sync();
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int v = warp + 8 * h;
      const long long view = v0 + v;
      if (view >= n_views) continue;
      float inv = 1.0f;
      if (normalize) {
        float sq = 0.f;
#pragma unroll
        for (int i = 0; i < TAIL_SPLIT; ++i) sq = __fadd_rn(sq, s_q[i][v]);
        inv = 1.0f / sqrtf(sq);
      }
      out[view * E + 64 * crank + lane] = x[h][0] * inv;
      out[view * E + 64 * crank + lane + 32] = x[h][1] * inv;
    }
    return;
  }
  // f / ||f||_2  (test.py:1706)
#pragma unroll
  for (int v = 0; v < TAIL_VIEWS; ++v) {
    const float q = warp_sum(__fmaf_rn(tot[v][1], tot[v][1], __fmul_rn(tot[v][0], tot[v][0])));
    if (lane == 0) s_q[warp][v] = q;
  }
  __syncthreads();
#pragma unroll
  for (int v = 0; v < TAIL_VIEWS; ++v) {
    const long long view = v0 + v;
    if (view >= n_views) break;
    float inv = 1.0f;
    if (normalize) {
      float sq = 0.f;
#pragma unroll
      for (int i = 0; i < TAIL_SPLIT; ++i) sq = __fadd_rn(sq, s_q[i][v]);
      inv = 1.0f / sqrtf(sq);
    }
    out[view * E + col] = tot[v][0] * inv;
    out[view * E + col + 32] = tot[v][1] * inv;
  }
}

// ------------------------------------------------------------------------------------------ packing
template <bool F16>
__global__ void cast_h_kernel(const float* __restrict__ src, uint16_t* __restrict__ dst, long long n) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = to_h<F16>(src[i]);
}

// dst = bf16(W + scaling * B @ A), fp32 accumulation: the merge the reference's eval path is
// mathematically equal to (test.py:388-398 applies W x + s x (BA)^T un-merged).
template <bool F16>
__global__ void merge_lora_cast_kernel(const float* __restrict__ W, const float* __restrict__ A,
                                       const float* __restrict__ B, int rows, int cols, int r, float scaling,
                                       uint16_t* __restrict__ dst) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(rows) * cols) return;
  const int o = static_cast<int>(i / cols), c = static_cast<int>(i % cols);
  float d = 0.f;
  for (int k = 0; k < r; ++k) d = fmaf(B[o * r + k], A[k * cols + c], d);
  dst[i] = to_h<F16>(W[i] + scaling * d);
}

// in place: W[rows, cols] (fp32) += scaling * B[rows, r] @ A[r, cols]
__global__ void merge_lora_f32_kernel(float* __restrict__ W, const float* __restrict__ A, const float* __restrict__ B,
                                      int rows, int cols, int r, float scaling) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(rows) * cols) return;
  const int o = static_cast<int>(i / cols), c = static_cast<int>(i % cols);
  float d = 0.f;
  for (int k = 0; k < r; ++k) d = fmaf(B[o * r + k], A[k * cols + c], d);
  W[i] += scaling * d;
}

// LayerNorm folded into the consuming GEMM (kernels.h EPI_LNFOLD_*): one warp per output row n of W [N, K]
//   Wf[n, k] = bf16(gamma[k] * W[n, k]);  S[n] = sum_k float(Wf[n, k]);  c[n] = sum_k beta[k] * W[n, k] + bias[n]
// S is the sum of the ROUNDED folded weights, i.e. exactly what the tensor core will multiply the row mean by.
template <bool F16>
__global__ void __launch_bounds__(256)
fold_ln_kernel(const float* __restrict__ W, const float* __restrict__ gamma, const float* __restrict__ beta,
               const float* __restrict__ bias, int N, int K, uint16_t* __restrict__ Wf, float* __restrict__ S,
               float* __restrict__ c) {
  const int lane = threadIdx.x & 31;
  const int n = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (n >= N) return;
  float s = 0.f, cc = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float w = W[static_cast<long long>(n) * K + k];
    const uint16_t wf = to_h<F16>(gamma[k] * w);
    Wf[static_cast<long long>(n) * K + k] = wf;
    s += from_h<F16>(wf);
    cc = fmaf(beta[k], w, cc);
  }
  s = warp_sum(s);
  cc = warp_sum(cc);
  if (lane == 0) { S[n] = s; c[n] = cc + bias[n]; }
}

}  // namespace

cudaError_t launch_merge_lora_f32(float* W, const float* A, const float* B, int rows, int cols, int r, float scaling,
                                  cudaStream_t stream) {
  const long long n = static_cast<long long>(rows) * cols;
  if (n == 0) return cudaSuccess;
  merge_lora_f32_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(W, A, B, rows, cols, r, scaling);
  return cudaGetLastError();
}

cudaError_t launch_fold_ln(const float* W, const float* gamma, const float* beta, const float* bias, int N, int K,
                           __nv_bfloat16* Wf, float* S, float* c, cudaStream_t stream, int f16) {
  if (N == 0) return cudaSuccess;
  uint16_t* dst = reinterpret_cast<uint16_t*>(Wf);
  if (f16) fold_ln_kernel<true><<<static_cast<unsigned>((N + 7) / 8), 256, 0, stream>>>(W, gamma, beta, bias, N, K, dst, S, c);
  else fold_ln_kernel<false><<<static_cast<unsigned>((N + 7) / 8), 256, 0, stream>>>(W, gamma, beta, bias, N, K, dst, S, c);
  return cudaGetLastError();
}

cudaError_t launch_im2col(const void* images, int img_dtype, int64_t n_views, int resolution, int patch,
                          int apply_norm, __nv_bfloat16* patches, cudaStream_t stream, int f16) {
  if (resolution % patch != 0 || patch % 16 != 0) return cudaErrorInvalidValue;
  const int G = resolution / patch;
  const int ept = 8;
  const int threads = 3 * patch * patch / ept;           // one thread per 8 pixels (16 bytes of bf16 output) of a patch row
  if (threads > 384 || threads % 32 != 0) return cudaErrorInvalidValue;   // patch 32: 384 threads
  const int64_t n_patches = n_views * G * G;
  if (n_patches == 0) return cudaSuccess;
  if (n_patches > 0x7fffffffLL) return cudaErrorInvalidValue;
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  }
  const int64_t want = (n_patches + IM2COL_UNROLL - 1) / IM2COL_UNROLL;
  const unsigned grid = static_cast<unsigned>(std::min<int64_t>(want, static_cast<int64_t>(sms) * (1536 / threads) * 2));
  const unsigned np = static_cast<unsigned>(n_patches);
  cudaError_t pdl_err = cudaSuccess;
#define JCB_IM2COL(DT)                                                                                              \
  if (f16) pdl_err = launch_pdl(im2col_kernel<DT, true>, dim3(grid), dim3(threads), 0, stream, 1, images, np, resolution, patch, G, apply_norm, patches); \
  else pdl_err = launch_pdl(im2col_kernel<DT, false>, dim3(grid), dim3(threads), 0, stream, 1, images, np, resolution, patch, G, apply_norm, patches)
  switch (img_dtype) {
    case IMG_F32: JCB_IM2COL(IMG_F32); break;
    case IMG_BF16: JCB_IM2COL(IMG_BF16); break;
    case IMG_U8: JCB_IM2COL(IMG_U8); break;
    default: return cudaErrorInvalidValue;
  }
#undef JCB_IM2COL
  return pdl_err;
}

#define JCB_DISPATCH_NV(W, CALL)               \
  switch ((W) / 128) {                         \
    case 4: { constexpr int NV = 4; CALL; } break; \
    case 6: { constexpr int NV = 6; CALL; } break; \
    case 8: { constexpr int NV = 8; CALL; } break; \
    default: return cudaErrorInvalidValue;     \
  }
// the same with the 16-bit output type as a second compile-time constant F16
#define JCB_DISPATCH_NV_H(W, f16, CALL)                                  \
  if (f16) { constexpr bool F16 = true; JCB_DISPATCH_NV(W, CALL) }       \
  else { constexpr bool F16 = false; JCB_DISPATCH_NV(W, CALL) }

cudaError_t launch_layernorm(const float* x, int64_t rows, int W, const float* g, const float* b,
                             __nv_bfloat16* y, cudaStream_t stream, int f16) {
  if (W % 128 != 0) return cudaErrorInvalidValue;
  if (rows == 0) return cudaSuccess;
  const unsigned grid = static_cast<unsigned>((rows + LN_WARPS - 1) / LN_WARPS);
  JCB_DISPATCH_NV_H(W, f16, (layernorm_kernel<NV, F16><<<grid, LN_WARPS * 32, 0, stream>>>(x, rows, g, b, y)));
  return cudaGetLastError();
}

cudaError_t launch_embed_ln(float* tokens, int64_t n_views, int T, int W, const float* cls, const float* pos,
                            const float* vpt, int n_vpt, const float* g_pre, const float* b_pre, const float* g1,
                            const float* b1, __nv_bfloat16* y, cudaStream_t stream, float* stats, int stats_slots,
                            const float* patch_out, float* shift, int f16) {
  if (W % 128 != 0) return cudaErrorInvalidValue;
  const long long rows = n_views * T;
  if (rows == 0) return cudaSuccess;
  const unsigned grid = static_cast<unsigned>((rows + LN_WARPS - 1) / LN_WARPS);
  cudaError_t e = cudaSuccess;
  JCB_DISPATCH_NV_H(W, f16, (e = launch_pdl(embed_ln_kernel<NV, F16>, dim3(grid), dim3(LN_WARPS * 32), 0, stream, 1,
                                            tokens, rows, T, cls, pos, vpt, n_vpt, g_pre, b_pre, g1, b1, y, stats, stats_slots,
                                            patch_out, shift)));
  return e;
}

cudaError_t launch_tail(const float* tokens, int64_t n_views, int T, int W, const float* g, const float* b,
                        const float* proj, int E, int normalize, float* out, cudaStream_t stream, const int* row_idx) {
  if (W % 128 != 0 || E != 512) return cudaErrorInvalidValue;
  if (n_views == 0) return cudaSuccess;
  const unsigned groups = static_cast<unsigned>((n_views + TAIL_VIEWS - 1) / TAIL_VIEWS);
  // few views: a cluster of TAIL_SPLIT CTAs per 16 views, one k range each (bit-identical, see tail_kernel); many: one
  // CTA per 16 views streams proj once.  JCB_TAIL_CLUSTER=0 / 1 forces one form (tests, A/B).
  const char* env = getenv("JCB_TAIL_CLUSTER");
  const bool clustered = env ? env[0] == '1' : groups * TAIL_SPLIT <= 296;
  const size_t smem = sizeof(float) * (static_cast<size_t>(TAIL_VIEWS) * W + TAIL_SPLIT * TAIL_VIEWS +
                                       (clustered ? TAIL_SPLIT * TAIL_VIEWS * 64 : 0));
  if (!clustered) {
    cudaError_t e = cudaSuccess;
    JCB_DISPATCH_NV(W, (e = ensure_dynamic_smem(tail_kernel<NV, 512, false>, smem)));
    if (e != cudaSuccess) return e;
    const long long nv0 = n_views;
    JCB_DISPATCH_NV(W, (e = launch_pdl(tail_kernel<NV, 512, false>, dim3(groups), dim3(TAIL_THREADS), smem, stream, 1, tokens,
                                       nv0, T, g, b, proj, normalize, out, row_idx)));
    return e;
  }
  const long long nv = n_views;
  cudaError_t e = cudaSuccess;
  JCB_DISPATCH_NV(W, (e = ensure_dynamic_smem(tail_kernel<NV, 512, true>, smem)));
  if (e != cudaSuccess) return e;
  JCB_DISPATCH_NV(W, (e = launch_pdl(tail_kernel<NV, 512, true>, dim3(groups * TAIL_SPLIT), dim3(TAIL_THREADS), smem, stream,
                                     TAIL_SPLIT, tokens, nv, T, g, b, proj, normalize, out, row_idx)));
  return e;
}

cudaError_t launch_text_embed_ln(const long long* ids, int64_t n_seq, int T, int W, int vocab, const float* tok_emb,
                                 const float* pos, const float* g1, const float* b1, float* tokens, __nv_bfloat16* y,
                                 int* eot, cudaStream_t stream, float* stats, int stats_slots, float* shift, int f16) {
  if (W % 128 != 0 || T < 1 || vocab < 1) return cudaErrorInvalidValue;
  const long long rows = n_seq * T;
  if (rows == 0) return cudaSuccess;
  const unsigned grid = static_cast<unsigned>((rows + LN_WARPS - 1) / LN_WARPS);
  JCB_DISPATCH_NV_H(W, f16, (text_embed_ln_kernel<NV, F16><<<grid, LN_WARPS * 32, 0, stream>>>(
                                ids, rows, T, vocab, tok_emb, pos, g1, b1, tokens, y, eot, stats, stats_slots, shift)));
  return cudaGetLastError();
}

cudaError_t launch_cast_bf16(const float* src, __nv_bfloat16* dst, int64_t n, cudaStream_t stream, int f16) {
  if (n == 0) return cudaSuccess;
  uint16_t* d = reinterpret_cast<uint16_t*>(dst);
  if (f16) cast_h_kernel<true><<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(src, d, n);
  else cast_h_kernel<false><<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(src, d, n);
  return cudaGetLastError();
}

cudaError_t launch_merge_lora_cast(const float* W, const float* A, const float* B, int rows, int cols, int r,
                                   float scaling, __nv_bfloat16* dst, cudaStream_t stream, int f16) {
  const long long n = static_cast<long long>(rows) * cols;
  if (n == 0) return cudaSuccess;
  uint16_t* d = reinterpret_cast<uint16_t*>(dst);
  const unsigned grid = static_cast<unsigned>((n + 255) / 256);
  if (f16) merge_lora_cast_kernel<true><<<grid, 256, 0, stream>>>(W, A, B, rows, cols, r, scaling, d);
  else merge_lora_cast_kernel<false><<<grid, 256, 0, stream>>>(W, A, B, rows, cols, r, scaling, d);
  return cudaGetLastError();
}

}  // namespace jcb
