// Attention entry points: launch_attention (every full attention, on the tcgen05 / TMEM kernel of attention_tc.cu)
// and the class-token-only kernel below.  The tcgen05 kernel replaced a round-1 mma.sync kernel (Q, K, V in smem) that
// spent 2/3 of its time in the shared-memory pipe (profiles/r01f): 0.366 vs 0.568 ms per launch of 8320 views on a
// B200 (DESIGN.md section 4).  T <= 128 with the causal mask, T <= 256 without.
//
// Reference: jclip/mha.py:55-83 scaled_dot_product_attention (attn_mask None for the vision tower,
// jclip/model.py:99; dropout 0 in eval), head split jclip/mha.py:351-362 / test.py:584-590.
#include "kernels.h"
#include "ptx.cuh"

namespace jcb {

namespace {

constexpr int HD = 64;       // head dim

// Attention for the class token only: softmax(q_0 K^T / 8) V for query row 0 of every (sequence, head).  Used by
// the opt-in "last block on the class token only" schedule (api.cu): encode_image returns ln_post(x[:, 0, :]) @ proj
// (jclip/model.py:121-124), so in the LAST block nothing but the class-token row of the attention output reaches
// the result.  One warp per (sequence, head): lane j scores keys j and j + 32 (a K row is 128 contiguous bytes),
// P is rounded to bf16 before P V exactly as in the full kernels, lanes own two output columns each.
template <bool F16>
__global__ void __launch_bounds__(256)
attention_cls_kernel(const __nv_bfloat16* __restrict__ qkv, long long n_items, int T, int heads,
                     __nv_bfloat16* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const long long item = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (item >= n_items) return;
  const long long seq = item / heads;
  const int h = static_cast<int>(item % heads);
  const int W = heads * HD;
  const __nv_bfloat16* base = qkv + seq * T * (3LL * W) + h * HD;
  float q[HD];
  {
    const uint4* qp = reinterpret_cast<const uint4*>(base);   // row 0, every lane reads the same 128 B
#pragma unroll
    for (int c = 0; c < HD / 8; ++c) {
      const uint4 v = __ldg(qp + c);
      const uint32_t* hh = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
      for (int e = 0; e < 4; ++e) { const float2 t = unpack_h2<F16>(hh[e]); q[8 * c + 2 * e] = t.x; q[8 * c + 2 * e + 1] = t.y; }
    }
  }
  const float scale_log2 = 0.125f * 1.4426950408889634f;
  float sc[2];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int j = lane + 32 * r;
    float acc = 0.f;
    if (j < T) {
      const uint4* kp = reinterpret_cast<const uint4*>(base + static_cast<long long>(j) * (3 * W) + W);
#pragma unroll
      for (int c = 0; c < HD / 8; ++c) {
        const uint4 v = __ldg(kp + c);
        const uint32_t* hh = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 t = unpack_h2<F16>(hh[e]);
          acc = fmaf(q[8 * c + 2 * e], t.x, acc);
          acc = fmaf(q[8 * c + 2 * e + 1], t.y, acc);
        }
      }
    }
    sc[r] = j < T ? acc * scale_log2 : -INFINITY;
  }
  const float mx = warp_max(fmaxf(sc[0], sc[1]));
  float pr[2];
  pr[0] = exp2f(sc[0] - mx);
  pr[1] = exp2f(sc[1] - mx);
  const float inv = 1.0f / warp_sum(pr[0] + pr[1]);
  pr[0] = from_h<F16>(to_h<F16>(pr[0]));   // P enters P V as a 16-bit operand (as in the tensor-core kernels)
  pr[1] = from_h<F16>(to_h<F16>(pr[1]));
  float o0 = 0.f, o1 = 0.f;
  const __nv_bfloat16* vbase = base + 2 * W + 2 * lane;
  for (int j = 0; j < T; ++j) {
    const float pj = __shfl_sync(0xffffffffu, pr[j >> 5], j & 31);
    const float2 v = unpack_h2<F16>(*reinterpret_cast<const uint32_t*>(vbase + static_cast<long long>(j) * (3 * W)));
    o0 = fmaf(pj, v.x, o0);
    o1 = fmaf(pj, v.y, o1);
  }
  *reinterpret_cast<uint32_t*>(out + seq * W + h * HD + 2 * lane) = pack_h2<F16>(o0 * inv, o1 * inv);
}

}  // namespace

cudaError_t launch_attention_cls(const __nv_bfloat16* qkv, int64_t n_views, int T, int heads, __nv_bfloat16* out,
                                 cudaStream_t stream, int f16) {
  if (T < 1 || T > 64 || heads < 1) return cudaErrorInvalidValue;
  if (n_views == 0) return cudaSuccess;
  const long long items = n_views * heads;
  const unsigned grid = static_cast<unsigned>((items + 7) / 8);
  if (f16) attention_cls_kernel<true><<<grid, 256, 0, stream>>>(qkv, items, T, heads, out);
  else attention_cls_kernel<false><<<grid, 256, 0, stream>>>(qkv, items, T, heads, out);
  return cudaGetLastError();
}

cudaError_t launch_attention(const __nv_bfloat16* qkv, int64_t n_views, int T, int heads, __nv_bfloat16* out,
                             cudaStream_t stream, int causal, int* dev_status, int num_sms, int f16) {
  if (T < 1 || T > 256 || (causal && T > 128) || heads < 1) return cudaErrorInvalidValue;
  if (n_views == 0) return cudaSuccess;
  return launch_attention_tc(qkv, n_views, T, heads, out, stream, dev_status, num_sms, f16, causal);
}

}  // namespace jcb
