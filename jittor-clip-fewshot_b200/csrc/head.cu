// Classification head: cosine logits against the cached text embeddings, Channel_LP (LP++ channel
// re-weighting), logit_normalize, score fusion and top-k -- one CTA per image, one launch per batch.
//
// Reference: Channel_LP test.py:1223-1234; logit_normalize test.py:1304-1308 (global unbiased std,
// per-row mean); fusion test.py:1710-1736; topk test.py:1738 / :1774; ood.py:875-883.
// In the reference every one of these runs on a [1, 403] tensor inside the per-image Python loop, with
// a `.tolist()` host sync per image; batch semantics here are "each image = its own [1, C] call".
#include <cstdlib>
#include <cooperative_groups.h>

#include "kernels.h"
#include "ptx.cuh"

namespace jcb {

namespace {

constexpr int HEAD_THREADS = 256;
constexpr int HEAD_WARPS = HEAD_THREADS / 32;

__device__ __forceinline__ float hblock_sum(float v, float* s_red) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int w = 0; w < HEAD_WARPS; ++w) t += s_red[w];
  return t;
}

// (z - mean(z)) / std_unbiased(z) over one row of C entries, in place   (test.py:1304-1308 with n = 1)
__device__ void normalize_row_inplace(float* z, int C, float* s_red) {
  float s = 0.f;
  for (int c = threadIdx.x; c < C; c += HEAD_THREADS) s += z[c];
  const float mean = hblock_sum(s, s_red) / static_cast<float>(C);
  float q = 0.f;
  for (int c = threadIdx.x; c < C; c += HEAD_THREADS) { const float t = z[c] - mean; q = fmaf(t, t, q); }
  const float var = hblock_sum(q, s_red) / static_cast<float>(C - 1);
  const float stdv = sqrtf(var);
  for (int c = threadIdx.x; c < C; c += HEAD_THREADS) z[c] = (z[c] - mean) / stdv;
  __syncthreads();
}

// Descending top-k with lowest-index tie break; destroys `score` (smem).  Result to out[0..k).
__device__ void topk_block(float* score, int C, int k, int32_t* out, float* s_red, int* s_idx) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int r = 0; r < k; ++r) {
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int c = threadIdx.x; c < C; c += HEAD_THREADS) {
      const float v = score[c];
      if (v > bv || (v == bv && c < bi)) { bv = v; bi = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    __syncthreads();
    if (lane == 0) { s_red[warp] = bv; s_idx[warp] = bi; }
    __syncthreads();
    if (threadIdx.x == 0) {
      float fv = s_red[0];
      int fi = s_idx[0];
      for (int w = 1; w < HEAD_WARPS; ++w)
        if (s_red[w] > fv || (s_red[w] == fv && s_idx[w] < fi)) { fv = s_red[w]; fi = s_idx[w]; }
      if (fi < 0 || fi >= C) fi = 0;  // all -inf / NaN rows: stay in range
      out[r] = fi;
      score[fi] = -INFINITY;
    }
    __syncthreads();
  }
}

// One image = one CTA, or one thread-block CLUSTER of HEAD_CLUSTER CTAs (launch_head decides): the five [C, D] x [D]
// products are split over the cluster's CTAs by class -- every class is still one warp's dot product, summed in the same
// lane order -- and land in the LEADER CTA's shared memory through distributed shared memory; the leader then normalises,
// fuses and ranks exactly as the single CTA does.  So both forms give the same bits; the cluster form turns ~50 dependent
// L2 round trips per warp into ~7 (one image per call, the reference's own loop: 154 -> ~35 us).
constexpr int HEAD_CLUSTER = 8;

__global__ void __launch_bounds__(HEAD_THREADS) head_kernel(const HeadArgs a) {
  extern __shared__ __align__(16) float head_smem[];
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  const int crank = static_cast<int>(cluster.block_rank()), csize = static_cast<int>(cluster.num_blocks());
  griddep_wait();               // programmatic dependent launch (ptx.cuh): nothing global is touched above
  const int C = a.C, D = a.D;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long img = blockIdx.x / csize;
  float* s_pt = head_smem;        // 100 * m_pt          [D]
  float* s_hand = s_pt + D;       // 100 * m_hand        [D]
  float* s_zs = s_hand + D;       // 100 * m_zs          [D]
  float* s_u1 = s_zs + D;         // scale1 * (m_pt + m_hand)/2 + bias1
  float* s_u2 = s_u1 + D;         // scale1 * m_zs + bias1
  float* s_sc = s_u2 + D;         // [SCORE_COUNT][C]
  float* s_l2 = s_sc + SCORE_COUNT * C;  // [C]
  float* s_red = s_l2 + C;        // [32]
  int* s_idx = reinterpret_cast<int*>(s_red + 32);

  for (int d = tid; d < D; d += HEAD_THREADS) {
    const float pt = a.m_pt[img * D + d], hd = a.m_hand[img * D + d], zs = a.m_zs[img * D + d];
    s_pt[d] = 100.0f * pt;   // `100. * image_features_pt @ text.t()`: scale first (test.py:1729-1731)
    s_hand[d] = 100.0f * hd;
    s_zs[d] = 100.0f * zs;
    const float comb = (pt + hd) / 2.0f;                        // :1710
    s_u1[d] = a.scale1[d] * comb + a.bias1[d];                  // :1232
    s_u2[d] = a.scale1[d] * zs + a.bias1[d];
  }
  __syncthreads();
  // where lane 0 leaves a class's five sums: the leader CTA's score arrays (this CTA's own when there is no cluster)
  float* r_sc = csize > 1 ? cluster.map_shared_rank(s_sc, 0) : s_sc;
  float* r_l2 = csize > 1 ? cluster.map_shared_rank(s_l2, 0) : s_l2;
  float* lg = s_sc + SCORE_LOGITS * C;
  float* cs = s_sc + SCORE_CS * C;
  float* cs1 = s_sc + SCORE_CS1 * C;
  float* cs2 = s_sc + SCORE_CS2 * C;
  float* cs3 = s_sc + SCORE_CS3 * C;
  float* cs4 = s_sc + SCORE_CS4 * C;
  float* cs5 = s_sc + SCORE_CS5 * C;
  // one warp per class, rows of [C, D] read coalesced.  D = 512 with 16-byte aligned banks (every real call): all
  // sixteen 16-byte loads of a class are issued before the first FMA -- the scalar loop below kept one L2 round trip
  // per 32 columns on the critical path (0.7 ms per 128 images, profiles/r01u_bench_n1.json)
  const bool vec = D == 512 && a.vec_ok;
  for (int c = crank * HEAD_WARPS + warp; c < C; c += HEAD_WARPS * csize) {
    const float* w = a.fc_w + static_cast<long long>(c) * D;
    const float* tp = a.T_pt + static_cast<long long>(c) * D;
    const float* th = a.T_hand + static_cast<long long>(c) * D;
    const float* tz = a.T_zs + static_cast<long long>(c) * D;
    float z1 = 0.f, z2 = 0.f, d0 = 0.f, d1 = 0.f, d3 = 0.f;
    if (vec) {
      float4 vw[4], vp[4], vh[4], vz[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i4 = lane + 32 * q;
        vw[q] = __ldg(reinterpret_cast<const float4*>(w) + i4);
        vp[q] = __ldg(reinterpret_cast<const float4*>(tp) + i4);
        vh[q] = __ldg(reinterpret_cast<const float4*>(th) + i4);
        vz[q] = __ldg(reinterpret_cast<const float4*>(tz) + i4);
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int i4 = lane + 32 * q;
        const float4 u1 = reinterpret_cast<const float4*>(s_u1)[i4], u2 = reinterpret_cast<const float4*>(s_u2)[i4];
        const float4 sh = reinterpret_cast<const float4*>(s_hand)[i4], sp = reinterpret_cast<const float4*>(s_pt)[i4];
        const float4 sz = reinterpret_cast<const float4*>(s_zs)[i4];
        z1 = fmaf(u1.x, vw[q].x, z1); z1 = fmaf(u1.y, vw[q].y, z1); z1 = fmaf(u1.z, vw[q].z, z1); z1 = fmaf(u1.w, vw[q].w, z1);
        z2 = fmaf(u2.x, vw[q].x, z2); z2 = fmaf(u2.y, vw[q].y, z2); z2 = fmaf(u2.z, vw[q].z, z2); z2 = fmaf(u2.w, vw[q].w, z2);
        d0 = fmaf(sh.x, vh[q].x, d0); d0 = fmaf(sh.y, vh[q].y, d0); d0 = fmaf(sh.z, vh[q].z, d0); d0 = fmaf(sh.w, vh[q].w, d0);
        d1 = fmaf(sp.x, vp[q].x, d1); d1 = fmaf(sp.y, vp[q].y, d1); d1 = fmaf(sp.z, vp[q].z, d1); d1 = fmaf(sp.w, vp[q].w, d1);
        d3 = fmaf(sz.x, vz[q].x, d3); d3 = fmaf(sz.y, vz[q].y, d3); d3 = fmaf(sz.z, vz[q].z, d3); d3 = fmaf(sz.w, vz[q].w, d3);
      }
    } else {
      for (int d = lane; d < D; d += 32) {
        const float ww = __ldg(w + d);
        z1 = fmaf(s_u1[d], ww, z1);
        z2 = fmaf(s_u2[d], ww, z2);
        d0 = fmaf(s_hand[d], __ldg(th + d), d0);
        d1 = fmaf(s_pt[d], __ldg(tp + d), d1);
        d3 = fmaf(s_zs[d], __ldg(tz + d), d3);
      }
    }
    z1 = warp_sum(z1); z2 = warp_sum(z2); d0 = warp_sum(d0); d1 = warp_sum(d1); d3 = warp_sum(d3);
    if (lane == 0) {
      const float b = a.fc_b[c];
      r_sc[SCORE_LOGITS * C + c] = z1 + b;   // logits1 (pre-normalisation)      :1715
      r_l2[c] = z2 + b;                      // logits2                          :1716
      r_sc[SCORE_CS * C + c] = d0;           // cosine_similarity                :1729
      r_sc[SCORE_CS1 * C + c] = d1;          // cosine_similarity1               :1730
      r_sc[SCORE_CS3 * C + c] = d3;          // cosine_similarity3               :1731
    }
  }
  if (csize > 1) {
    cluster.sync();          // every CTA's sums are in the leader's shared memory (release / acquire at cluster scope)
    if (crank != 0) return;  // nobody reads the other CTAs' shared memory: they may leave
  } else {
    __syncthreads();
  }
  normalize_row_inplace(lg, C, s_red);                           // :1717
  normalize_row_inplace(s_l2, C, s_red);                         // :1718
  for (int c = tid; c < C; c += HEAD_THREADS) lg[c] = (lg[c] + s_l2[c]) / 2.0f;  // :1721
  __syncthreads();
  normalize_row_inplace(lg, C, s_red);                           // :1722
  for (int c = tid; c < C; c += HEAD_THREADS) {
    const float c2 = (cs[c] + cs1[c]) / 2.0f;                    // :1733
    cs2[c] = c2;
    const float c4 = (c2 + cs3[c]) / 2.0f;                       // :1734
    cs4[c] = c4;
    cs5[c] = c4 + 0.5f * lg[c];                                  // :1735
  }
  __syncthreads();
  if (a.out_all)
    for (int i = tid; i < SCORE_COUNT * C; i += HEAD_THREADS) a.out_all[img * SCORE_COUNT * C + i] = s_sc[i];
  float* ranked = s_sc + a.rank_by * C;
  if (a.out_scores)
    for (int c = tid; c < C; c += HEAD_THREADS) a.out_scores[img * C + c] = ranked[c];
  __syncthreads();
  topk_block(ranked, C, a.k, a.out_topk + img * a.k, s_red, s_idx);   // :1738
}

// scores = scale * f @ T^T, top-k  (evaluate_new test.py:1770-1774; OOD argmax ood.py:875-877 with k = 1)
__global__ void __launch_bounds__(HEAD_THREADS)
cosine_topk_kernel(const float* __restrict__ feats, const float* __restrict__ text, int C, int D, float scale, int k,
                   int32_t* __restrict__ out_topk, float* __restrict__ out_scores) {
  extern __shared__ __align__(16) float head_smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long img = blockIdx.x;
  float* s_f = head_smem;   // [D]
  float* s_s = s_f + D;     // [C]
  float* s_red = s_s + C;
  int* s_idx = reinterpret_cast<int*>(s_red + 32);
  for (int d = tid; d < D; d += HEAD_THREADS) s_f[d] = scale * feats[img * D + d];
  __syncthreads();
  for (int c = warp; c < C; c += HEAD_WARPS) {
    const float* t = text + static_cast<long long>(c) * D;
    float s = 0.f;
    for (int d = lane; d < D; d += 32) s = fmaf(s_f[d], __ldg(t + d), s);
    s = warp_sum(s);
    if (lane == 0) s_s[c] = s;
  }
  __syncthreads();
  if (out_scores)
    for (int c = tid; c < C; c += HEAD_THREADS) out_scores[img * C + c] = s_s[c];
  __syncthreads();
  if (out_topk) topk_block(s_s, C, k, out_topk + img * k, s_red, s_idx);
}

// out[n, C] = (scale1 * f + bias1) @ W^T + b      (Channel_LP.execute, test.py:1229-1234)
__global__ void __launch_bounds__(HEAD_THREADS)
channel_lp_kernel(const float* __restrict__ feats, int C, int D, const float* __restrict__ scale1,
                  const float* __restrict__ bias1, const float* __restrict__ fc_w, const float* __restrict__ fc_b,
                  float* __restrict__ out) {
  extern __shared__ __align__(16) float head_smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long row = blockIdx.x;
  float* s_u = head_smem;
  for (int d = tid; d < D; d += HEAD_THREADS) s_u[d] = scale1[d] * feats[row * D + d] + bias1[d];
  __syncthreads();
  for (int c = warp; c < C; c += HEAD_WARPS) {
    const float* w = fc_w + static_cast<long long>(c) * D;
    float s = 0.f;
    for (int d = lane; d < D; d += 32) s = fmaf(s_u[d], __ldg(w + d), s);
    s = warp_sum(s);
    if (lane == 0) out[row * C + c] = s + fc_b[c];
  }
}

// logit_normalize on an [n, C] tensor with the reference's exact semantics: ONE global unbiased std
// over all n*C entries, per-row mean (test.py:1304-1308).  Single CTA (n is 1 at every call site).
__global__ void __launch_bounds__(HEAD_THREADS)
logit_normalize_kernel(const float* __restrict__ in, long long n, int C, float* __restrict__ out) {
  __shared__ float s_red[32];
  const long long total = n * C;
  float s = 0.f;
  for (long long i = threadIdx.x; i < total; i += HEAD_THREADS) s += in[i];
  const float gmean = hblock_sum(s, s_red) / static_cast<float>(total);
  float q = 0.f;
  for (long long i = threadIdx.x; i < total; i += HEAD_THREADS) { const float t = in[i] - gmean; q = fmaf(t, t, q); }
  const float stdv = sqrtf(hblock_sum(q, s_red) / static_cast<float>(total - 1));
  for (long long r = 0; r < n; ++r) {
    float rs = 0.f;
    for (int c = threadIdx.x; c < C; c += HEAD_THREADS) rs += in[r * C + c];
    const float rmean = hblock_sum(rs, s_red) / static_cast<float>(C);
    for (int c = threadIdx.x; c < C; c += HEAD_THREADS) out[r * C + c] = (in[r * C + c] - rmean) / stdv;
  }
}

// clip_classifier (test.py:920-940): per class, mean of the (already unit-norm) template embeddings, re-normalised.
// emb [n, D], offsets [C + 1] (templates of class c are rows offsets[c] .. offsets[c+1]), out [C, D].
__global__ void __launch_bounds__(HEAD_THREADS)
class_mean_kernel(const float* __restrict__ emb, const int* __restrict__ offsets, int D, float* __restrict__ out) {
  __shared__ float s_red[32];
  const int c = blockIdx.x;
  const int lo = offsets[c], hi = offsets[c + 1];
  const float inv_n = 1.0f / static_cast<float>(hi - lo);
  float q = 0.f;
  for (int d = threadIdx.x; d < D; d += HEAD_THREADS) {
    float s = 0.f;
    for (int r = lo; r < hi; ++r) s += emb[static_cast<long long>(r) * D + d];
    s *= inv_n;
    out[static_cast<long long>(c) * D + d] = s;
    q = fmaf(s, s, q);
  }
  const float inv = 1.0f / sqrtf(hblock_sum(q, s_red));
  for (int d = threadIdx.x; d < D; d += HEAD_THREADS) out[static_cast<long long>(c) * D + d] *= inv;
}

}  // namespace

cudaError_t launch_class_mean(const float* emb, const int* offsets, int C, int D, float* out, cudaStream_t stream) {
  if (C == 0) return cudaSuccess;
  class_mean_kernel<<<static_cast<unsigned>(C), HEAD_THREADS, 0, stream>>>(emb, offsets, D, out);
  return cudaGetLastError();
}

cudaError_t launch_head(const HeadArgs& a, cudaStream_t stream) {
  if (a.k < 1 || a.k > 8 || a.k > a.C || a.rank_by < 0 || a.rank_by >= SCORE_COUNT || a.C < 2 || a.D < 1)
    return cudaErrorInvalidValue;
  if (a.I == 0) return cudaSuccess;
  const size_t smem = sizeof(float) * (5 * a.D + (SCORE_COUNT + 1) * a.C + 32) + sizeof(int) * 32;
  if (smem > 200 * 1024) return cudaErrorInvalidValue;
  {
    cudaError_t e = ensure_dynamic_smem(head_kernel, smem);
    if (e != cudaSuccess) return e;
  }
  HeadArgs b = a;
  b.vec_ok = ((reinterpret_cast<uintptr_t>(a.T_pt) | reinterpret_cast<uintptr_t>(a.T_hand) |
               reinterpret_cast<uintptr_t>(a.T_zs) | reinterpret_cast<uintptr_t>(a.fc_w)) & 15) == 0;
  // few images: a cluster of CTAs per image (bit-identical, see head_kernel); many: the images fill the chip already.
  // JCB_HEAD_CLUSTER=0 / 1 forces one form (tests, A/B).
  const char* env = getenv("JCB_HEAD_CLUSTER");
  const bool clustered = env ? env[0] == '1' : (a.I <= 512 && a.C >= 2 * HEAD_WARPS * HEAD_CLUSTER);
  if (!clustered) return launch_pdl(head_kernel, dim3(static_cast<unsigned>(a.I)), dim3(HEAD_THREADS), smem, stream, 1, b);
  return launch_pdl(head_kernel, dim3(static_cast<unsigned>(a.I) * HEAD_CLUSTER), dim3(HEAD_THREADS), smem, stream,
                    HEAD_CLUSTER, b);
}


cudaError_t launch_cosine_topk(const float* feats, const float* text, int64_t n, int C, int D, float scale, int k,
                               int32_t* out_topk, float* out_scores, cudaStream_t stream) {
  if (out_topk && (k < 1 || k > C)) return cudaErrorInvalidValue;
  if (n == 0) return cudaSuccess;
  const size_t smem = sizeof(float) * (D + C + 32) + sizeof(int) * 32;
  if (smem > 48 * 1024) return cudaErrorInvalidValue;
  cosine_topk_kernel<<<static_cast<unsigned>(n), HEAD_THREADS, smem, stream>>>(feats, text, C, D, scale, k, out_topk,
                                                                             out_scores);
  return cudaGetLastError();
}

cudaError_t launch_channel_lp(const float* feats, int64_t n, int C, int D, const float* scale1, const float* bias1,
                              const float* fc_w, const float* fc_b, float* out, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  const size_t smem = sizeof(float) * D;
  if (smem > 48 * 1024) return cudaErrorInvalidValue;
  channel_lp_kernel<<<static_cast<unsigned>(n), HEAD_THREADS, smem, stream>>>(feats, C, D, scale1, bias1, fc_w, fc_b,
                                                                            out);
  return cudaGetLastError();
}

cudaError_t launch_logit_normalize(const float* in, int64_t n, int C, float* out, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  if (n * C < 2) return cudaErrorInvalidValue;
  logit_normalize_kernel<<<1, HEAD_THREADS, 0, stream>>>(in, n, C, out);
  return cudaGetLastError();
}

}  // namespace jcb
