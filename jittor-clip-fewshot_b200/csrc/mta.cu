// MTA (MeanShift for Test-time Augmentation) mode seeking: the whole solver for one image in ONE CTA.
//
// The reference (test.py:1391-1461, twin ood.py:751-820) runs ~100 tiny Jittor kernels and up to 50
// device->host syncs (`if jt.norm(...) < th`) per image.  Here each image is one thread block: view
// embeddings, the affinity matrix and all iteration state live in shared memory, the data-dependent
// early exits are block-uniform branches, and a batch of images is a single launch.
//
//   logits = 100 * X T                                     test.py:1393
//   D = cdist(X, X); bandwidth_i from the k nearest         test.py:1403-1408   (D^2 clamped >= 0, k >= 1)
//   A = softmax(logits) softmax(logits)^T                   test.py:1411
//   5 x { y <- softmax((rho + 4 A y) / 0.2)  (<= 5 its)     test.py:1426-1438
//         m <- normalise(sum rho_i y_i x_i)  (<= 5 its) }   test.py:1443-1453
//
// X [V, D] unit rows (row 0 = un-augmented view), T given as [D, C] (the orientation the reference
// passes: `text_features.t()`), so class-parallel threads read it coalesced.

#include "kernels.h"
#include "ptx.cuh"

namespace jcb {

namespace {

constexpr int MTA_THREADS = 256;
constexpr int MTA_WARPS = MTA_THREADS / 32;
constexpr int VB = 8;  // views per register block in the logits GEMM

struct MtaDev {
  MtaSet sets[MTA_MAX_SETS];  // blockIdx.y selects (feats [I,V,D], text [D,C], out_mode [I,D], out_logits)
  long long I;
  int V, C, D, ldA, k;
  MtaParams p;
  const float* P;       // [n_sets, I*V, C] row-softmaxed logits from mta_probs_kernel (nullptr: compute here)
  float* scratch;       // per image: region R (max(V*C, V*D)) + A (V*ldA), only used when !in_smem
  long long scratch_stride;
  int in_smem;
  int ldx, ldp;         // fast kernel: padded row strides of X and P in shared memory
  // large view counts (the problem does not fit in shared memory): affinity and bandwidths come from the batched
  // pre-pass kernels (mta_gram_big_kernel, mta_bw_big_kernel); this kernel is then only the iterative solver
  const float* A_pre;   // [n_sets * I, V, ldA] or nullptr
  const float* bw_pre;  // [n_sets * I, V] or nullptr
  // fast kernel: text banks that share ONE feature tensor (prompt-tuned and hand-crafted text on the same tower; all
  // three in the single-tower pipeline) are solved by the same CTA: the view embeddings are brought on chip, multiplied
  // into their Gram matrix and rank-selected for the bandwidths once per image instead of once per bank
  int n_groups, max_group;   // max_group = the largest group_count: affinity slots in shared memory
  int group_count[MTA_MAX_SETS];
  int group_sets[MTA_MAX_SETS][MTA_MAX_SETS];
  MtaDebug dbg;              // set 0's bandwidths, final y and affinity (jcb_mta_debug); all nullptr otherwise
};

template <int NW>
__device__ __forceinline__ float block_sum(float v, float* s_red) {
  v = warp_sum(v);
  __syncthreads();  // protect s_red from the previous use
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int w = 0; w < NW; ++w) t += s_red[w];
  return t;
}
template <int NW>
__device__ __forceinline__ float block_max(float v, float* s_red) {
  v = warp_max(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = -INFINITY;
#pragma unroll
  for (int w = 0; w < NW; ++w) t = fmaxf(t, s_red[w]);
  return t;
}
template <int NW>
__device__ __forceinline__ void density_step(const float* __restrict__ X, const float* s_mode, const float* s_bw,
                                             float* s_dens, int V, int D) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = warp; i < V; i += NW) {
    float q = 0.f;
    for (int d = lane; d < D; d += 32) {
      const float t = X[i * D + d] - s_mode[d];
      q = fmaf(t, t, q);
    }
    q = warp_sum(q);
    if (lane == 0) {
      const float dist = sqrtf(q);  // jt.norm(...), then dist**2 as the reference does
      const float bw = s_bw[i];
      s_dens[i] = expf(-(dist * dist) / (2.0f * bw * bw));
    }
  }
  __syncthreads();
}
// the solver state of image `img` for jcb_mta_debug, written by threads t0, t0 + nt, ...
__device__ __forceinline__ void mta_write_debug(const MtaDebug& g, long long img, int V, const float* s_bw, const float* s_y,
                                                const float* A, int ldA, int t0, int nt) {
  if (g.bw)
    for (int i = t0; i < V; i += nt) g.bw[img * V + i] = s_bw[i];
  if (g.y)
    for (int i = t0; i < V; i += nt) g.y[img * V + i] = s_y[i];
  if (g.affinity)
    for (int idx = t0; idx < V * V; idx += nt) {
      const int i = idx / V, j = idx - i * V;
      g.affinity[img * V * V + idx] = A[static_cast<long long>(i) * ldA + j];
    }
}


// ---------------------------------------------------------------------------------------------------
// P = softmax_rows(100 * X T / temperature) for every view of every image of every (feats, text) set:
// one smem-tiled fp32 SIMT GEMM over all rows at once instead of each image's CTA streaming the text
// bank from L2 (which was ~half of the solver's time).  fp32 on purpose: the logits are O(10..100) and
// feed a softmax whose output defines the affinity matrix; bf16 tensor-core inputs would move the
// modes by ~1e-3, far outside the parity tolerance.
//   CTA = 64 rows x all C classes (C <= 416), 256 threads: warp w owns rows 8w..8w+7, lane l owns
//   classes l, l+32, ... (13 per lane); K is consumed in chunks of 32 staged by cp.async, two stages.
constexpr int PB_ROWS = 64, PB_KC = 32, PB_NC = 13, PB_CPAD = PB_NC * 32;  // 416 >= 403
constexpr int PB_XS = PB_ROWS * PB_KC;                                      // floats per X stage
constexpr int PB_TS = PB_KC * PB_CPAD;                                      // floats per T stage
constexpr int PB_SMEM = 2 * (PB_XS + PB_TS) * 4;                            // 122880 B

struct ProbsDev {
  MtaSet sets[MTA_MAX_SETS];
  long long rows;   // I * V
  int C, D;
  float scale;
  float* P;         // [n_sets, rows, C]
};

__global__ void __launch_bounds__(256, 1) mta_probs_kernel(const ProbsDev a) {
  extern __shared__ __align__(16) float pb_smem[];
  float* Xs = pb_smem;                 // [2][PB_ROWS][PB_KC]
  float* Ts = pb_smem + 2 * PB_XS;     // [2][PB_KC][PB_CPAD]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const MtaSet& set = a.sets[blockIdx.y];
  const long long row0 = static_cast<long long>(blockIdx.x) * PB_ROWS;
  const float* __restrict__ X = set.feats;
  const float* __restrict__ T = set.text;
  const int C = a.C, D = a.D;

  // columns >= C of the T stages are never written by cp.async: zero them once
  for (int i = tid; i < 2 * PB_TS; i += 256) {
    const int c = i % PB_CPAD;
    if (c >= C) Ts[i] = 0.f;
  }
  auto load_stage = [&](int stage, int k0) {
    // X: 64 rows x 32 k = 512 x 16-byte pieces; rows past the end re-read the last valid row
    for (int i = tid; i < PB_ROWS * (PB_KC / 4); i += 256) {
      const int r = i / (PB_KC / 4), p4 = i % (PB_KC / 4);
      long long gr = row0 + r;
      if (gr >= a.rows) gr = a.rows - 1;
      cp_async_16(smem_u32(Xs + stage * PB_XS + r * PB_KC + p4 * 4), X + gr * D + k0 + p4 * 4);
    }
    // T: 32 k x C classes, 4-byte pieces (row stride C = 403 floats is not 16-byte aligned)
    for (int i = tid; i < PB_KC * C; i += 256) {
      const int k = i / C, c = i % C;
      asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(Ts + stage * PB_TS + k * PB_CPAD + c)),
                   "l"(T + static_cast<long long>(k0 + k) * C + c)
                   : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };

  float acc[8][PB_NC];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < PB_NC; ++j) acc[i][j] = 0.f;

  const int nk = D / PB_KC;
  load_stage(0, 0);
  for (int kc = 0; kc < nk; ++kc) {
    if (kc + 1 < nk) {
      load_stage((kc + 1) & 1, (kc + 1) * PB_KC);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    const float* xs = Xs + (kc & 1) * PB_XS + warp * 8 * PB_KC;
    const float* ts = Ts + (kc & 1) * PB_TS + lane;
#pragma unroll 4
    for (int k = 0; k < PB_KC; ++k) {
      float t[PB_NC], x[8];
#pragma unroll
      for (int j = 0; j < PB_NC; ++j) t[j] = ts[k * PB_CPAD + 32 * j];
#pragma unroll
      for (int i = 0; i < 8; ++i) x[i] = xs[i * PB_KC + k];  // warp-uniform address: broadcast
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < PB_NC; ++j) acc[i][j] = fmaf(x[i], t[j], acc[i][j]);
    }
    __syncthreads();
  }
  // row softmax (test.py:1411 `(logits/temperature).softmax(1)`), one warp per row
  float* Pout = a.P + static_cast<long long>(blockIdx.y) * a.rows * C;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const long long gr = row0 + warp * 8 + i;
    float mx = -INFINITY;
#pragma unroll
    for (int j = 0; j < PB_NC; ++j) {
      acc[i][j] *= a.scale;
      if (lane + 32 * j < C) mx = fmaxf(mx, acc[i][j]);
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < PB_NC; ++j) {
      const float e = (lane + 32 * j < C) ? expf(acc[i][j] - mx) : 0.f;
      acc[i][j] = e;
      sum += e;
    }
    sum = warp_sum(sum);
    const float inv = 1.0f / sum;
    if (gr < a.rows) {
#pragma unroll
      for (int j = 0; j < PB_NC; ++j)
        if (lane + 32 * j < C) Pout[gr * C + lane + 32 * j] = acc[i][j] * inv;
    }
  }
}

// ---------------------------------------------------------------------------------------------------
// The same probabilities on the tensor cores (round 2): logits = 100 X T is a [rows, 512] x [512, 403] contraction per
// text bank that must keep fp32 accuracy (bf16 logits move the modes by 1e-3).  Every fp32 value is split into three
// bf16 limbs, x = x1 + x2 + x3 (24 significand bits, fp32's exponent range -- no underflow of the small limbs, which is
// what rules fp16 limbs out), and the six limb products of weight >= 2^-16,
//     x.t ~= x3 t1 + x2 t2 + x1 t3 + x2 t1 + x1 t2 + x1 t1        (dropped: <= 2^-24 relative),
// are ONE bf16 GEMM with the limbs concatenated along K:  A' = [X3 X2 X1 X2 X1 X1],  B' = [T1 T2 T3 T1 T2 T1].  The
// smallest products come first: every MMA step adds to the accumulator at the accumulator's precision, and adding the
// small limbs onto the finished x1 t1 sum (the order [X1 X1 X1 X2 X2 X3]) rounded six times as many steps at full
// magnitude -- affinities ~2e-5 from the float64 reference, against ~5e-6 on the fp32 SIMT path (B200, 1000 W);
// K' = 6 D = 3072 -- the tower's own tcgen05 kernel (gemm.cu, fp32 accumulation in TMEM, fp32 output), 26 GFLOP per bank
// instead of 8.6 GFLOP of fp32 SIMT FMAs at a third of the SIMT peak.  A row softmax kernel finishes.
__device__ __forceinline__ void split3(float x, uint16_t (&l)[3]) {
  const __nv_bfloat16 a = __float2bfloat16_rn(x);
  const float r1 = x - __bfloat162float(a);                     // exact
  const __nv_bfloat16 b = __float2bfloat16_rn(r1);
  const float r2 = r1 - __bfloat162float(b);                    // exact
  const __nv_bfloat16 c = __float2bfloat16_rn(r2);
  l[0] = __bfloat16_as_ushort(a); l[1] = __bfloat16_as_ushort(b); l[2] = __bfloat16_as_ushort(c);
}
// X [rows, D] fp32 -> A' [rows, 6 D] bf16, blocks (3, 2, 1, 2, 1, 1)
__global__ void __launch_bounds__(256) mta_split_x_kernel(const float* __restrict__ X, long long rows, int D,
                                                          uint16_t* __restrict__ out) {
  griddep_wait();               // programmatic dependent launch (ptx.cuh): nothing global is touched above
  const long long i = static_cast<long long>(blockIdx.x) * 256 + threadIdx.x;
  if (i >= rows * D) return;
  const long long r = i / D;
  const int d = static_cast<int>(i - r * D);
  uint16_t l[3];
  split3(X[i], l);
  uint16_t* o = out + r * 6 * D + d;
  o[0] = l[2]; o[D] = l[1]; o[2 * D] = l[0]; o[3 * D] = l[1]; o[4 * D] = l[0]; o[5 * D] = l[0];
}
// T^T [D, C] fp32 (the orientation solve_mta receives) -> B' [CP, 6 D] bf16, blocks (1, 2, 3, 1, 2, 1); rows >= C zero
__global__ void __launch_bounds__(256) mta_split_t_kernel(const float* __restrict__ Tt, int C, int CP, int D,
                                                          uint16_t* __restrict__ out) {
  griddep_wait();               // programmatic dependent launch (ptx.cuh): nothing global is touched above
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i >= CP * D) return;
  const int d = i / CP, c = i - d * CP;          // threads along c: coalesced reads of Tt
  uint16_t l[3] = {0, 0, 0};
  if (c < C) split3(Tt[static_cast<long long>(d) * C + c], l);
  uint16_t* o = out + static_cast<long long>(c) * 6 * D + d;
  o[0] = l[0]; o[D] = l[1]; o[2 * D] = l[2]; o[3 * D] = l[0]; o[4 * D] = l[1]; o[5 * D] = l[0];
}
// P[r, :] = softmax(scale * L[r, 0:C]) (test.py:1411), one warp per row; L has leading dimension CP
__global__ void __launch_bounds__(256) mta_softmax_rows_kernel(const float* __restrict__ L, long long rows, int C, int CP,
                                                               float scale, float* __restrict__ P) {
  griddep_wait();               // programmatic dependent launch (ptx.cuh): nothing global is touched above
  const int lane = threadIdx.x & 31;
  const long long r = static_cast<long long>(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (r >= rows) return;
  const float* l = L + r * CP;
  float v[16];
  float mx = -INFINITY;
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const int c = lane + 32 * j;
    v[j] = c < C ? l[c] * scale : -INFINITY;
    mx = fmaxf(mx, v[j]);
  }
  mx = warp_max(mx);
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    v[j] = (lane + 32 * j < C) ? expf(v[j] - mx) : 0.f;
    sum += v[j];
  }
  sum = warp_sum(sum);
  const float inv = 1.0f / sum;
#pragma unroll
  for (int j = 0; j < 16; ++j)
    if (lane + 32 * j < C) P[r * C + lane + 32 * j] = v[j] * inv;
}
constexpr int TCP_CP = 512;   // class count padded to the GEMM's N granularity (C <= 512)

// ---------------------------------------------------------------------------------------------------
// Large view counts (V = 513 in the reference's test.py: 512 crops + the centre view).  One CTA per (image, bank) cannot
// hold the problem on chip, and doing its two V x V x {C, D} Gram matrices and the V^3 rank select inside that one CTA
// took 76 ms per 16 images (3 banks) -- 48 CTAs on 148 SMs.  Those three pieces are batched over ALL problems here:
//   mta_gram_big_kernel   G = M M^T per problem, fp32, 64 x 64 tiles of the upper triangle (mirrored on store); M = P
//                         (affinity, test.py:1411) or M = X (dot products for cdist, test.py:1314-1318)
//   mta_bw_big_kernel     one warp per (problem, view): distances from the Gram row, rank select, bandwidth (:1403-1408)
// and mta_kernel below runs only the iterations, reading the affinity from global memory (L2 resident).
constexpr int GB_TILE = 64, GB_KC = 16;

struct GramBigDev {
  MtaSet sets[MTA_MAX_SETS];
  long long I;
  int V, K, ld, ldg, from_feats;   // from_feats: M = sets[set].feats + img * V * ld, else M = P + problem * V * ld
  const float* P;
  float* G;                        // [n_sets * I, V, ldg]
};

__global__ void __launch_bounds__(256) mta_gram_big_kernel(const GramBigDev a) {
  __shared__ float As[GB_KC][GB_TILE + 4];   // As[k][i]: k-major so that a thread's 4 rows are one LDS.128
  __shared__ float Bs[GB_KC][GB_TILE + 4];
  const int nt = (a.V + GB_TILE - 1) / GB_TILE;
  // blockIdx.x enumerates the upper-triangle tile pairs (ti <= tj)
  int ti = 0, rem = blockIdx.x;
  while (rem >= nt - ti) { rem -= nt - ti; ++ti; }
  const int tj = ti + rem;
  const long long problem = blockIdx.y;
  const int set = static_cast<int>(problem / a.I);
  const long long img = problem % a.I;
  const float* __restrict__ M = a.from_feats ? a.sets[set].feats + img * a.V * a.ld : a.P + problem * a.V * a.ld;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  float acc[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;
  for (int k0 = 0; k0 < a.K; k0 += GB_KC) {
    // 64 rows x 16 k per operand tile: thread t loads row t / 4, k-quad t % 4 (4 consecutive k of one row)
    {
      const int r = tid >> 2, kq = (tid & 3) * 4;
#pragma unroll
      for (int op = 0; op < 2; ++op) {
        const int row = (op == 0 ? ti : tj) * GB_TILE + r;
        float v[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int k = k0 + kq + e;
          v[e] = (row < a.V && k < a.K) ? __ldg(M + static_cast<long long>(row) * a.ld + k) : 0.f;
        }
        float (*dst)[GB_TILE + 4] = op == 0 ? As : Bs;
#pragma unroll
        for (int e = 0; e < 4; ++e) dst[kq + e][r] = v[e];
      }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < GB_KC; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[k][4 * ty]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[k][4 * tx]);
      const float ar[4] = {av.x, av.y, av.z, av.w}, br[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(ar[r], br[c], acc[r][c]);
    }
    __syncthreads();
  }
  float* G = a.G + problem * a.V * a.ldg;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int i = ti * GB_TILE + 4 * ty + r;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int j = tj * GB_TILE + 4 * tx + c;
      if (i < a.V && j < a.V) {
        G[static_cast<long long>(i) * a.ldg + j] = acc[r][c];
        if (ti != tj) G[static_cast<long long>(j) * a.ldg + i] = acc[r][c];
      }
    }
  }
}

struct BwBigDev {
  const float* G;      // [problems, V, ldg] Gram of X
  float* bw;           // [problems, V]
  int V, ldg, k;
};

__global__ void __launch_bounds__(256) mta_bw_big_kernel(const BwBigDev a) {
  extern __shared__ __align__(16) float bw_smem[];
  const int V = a.V;
  float* s_sq = bw_smem;                 // [V] ||x_j||^2 = the Gram diagonal (same summation as the dots)
  float* s_rows = bw_smem + V;           // [8][V] one distance row per warp
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long problem = blockIdx.y;
  const float* __restrict__ G = a.G + problem * V * a.ldg;
  for (int j = tid; j < V; j += 256) s_sq[j] = __ldg(G + static_cast<long long>(j) * a.ldg + j);
  __syncthreads();
  const int i = blockIdx.x * 8 + warp;
  if (i >= V) return;
  float* my_row = s_rows + warp * V;
  const float sqi = s_sq[i];
  for (int j = lane; j < V; j += 32) {
    const float d2 = sqi - 2.0f * __ldg(G + static_cast<long long>(i) * a.ldg + j) + s_sq[j];
    my_row[j] = fabsf(sqrtf(fmaxf(d2, 0.0f)));   // never -0: the bisection below orders bit patterns
  }
  __syncwarp();
  // Mean of the squared k smallest distances, skipping rank 0 (test.py:1404-1408: sorted_dist[:, 1:k+1]).  Counting
  // every element's rank is V^2 compares per row (V^3 per problem: 135 M at V = 513); instead find the value t of rank
  // k by bisection on the bit pattern (distances are >= 0, so their uint32 images order like the floats): ranks 0..k
  // are the elements below t plus (k + 1 - #below) copies of t, and rank 0 is the row minimum -- equal values are
  // interchangeable in a sum of squares, so the index tie-break of the sort does not matter.
  const int kk = a.k < V - 1 ? a.k : V - 1;          // rank of the threshold element (0-based)
  uint32_t lo = 0u, hi = 0x7f800000u;                 // invariant: #(d <= lo - 1) <= kk < #(d <= hi)
  while (lo < hi) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    int cnt = 0;
    for (int j = lane; j < V; j += 32) cnt += __float_as_uint(my_row[j]) <= mid ? 1 : 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (cnt > kk) hi = mid; else lo = mid + 1;
  }
  const float t = __uint_as_float(lo);                // the (kk + 1)-th smallest distance
  float below = 0.f, mn = INFINITY;
  int n_below = 0;
  for (int j = lane; j < V; j += 32) {
    const float dj = my_row[j];
    mn = fminf(mn, dj);
    if (dj < t) { below = fmaf(dj, dj, below); ++n_below; }
  }
  below = warp_sum(below);
  mn = -warp_max(-mn);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n_below += __shfl_xor_sync(0xffffffffu, n_below, o);
  const float acc = below + static_cast<float>(kk + 1 - n_below) * t * t - mn * mn;
  if (lane == 0) a.bw[problem * V + i] = sqrtf(0.5f * (acc / static_cast<float>(a.k)));
}

// NT threads per CTA: 256 for problems held in shared memory, 1024 for the large-V solver (every pass streams X or the
// affinity from L2: four times the warps, four times the loads in flight)
template <int NT>
__global__ void __launch_bounds__(NT, 1) mta_kernel(const MtaDev a) {
  constexpr int NW = NT / 32;
  extern __shared__ __align__(16) float mta_smem[];
  const int V = a.V, C = a.C, D = a.D, ldA = a.ldA;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long img = blockIdx.x;
  const MtaSet& set = a.sets[blockIdx.y];
  const long long problem = static_cast<long long>(blockIdx.y) * a.I + img;
  const float* __restrict__ Xg = set.feats + img * V * D;
  const float* __restrict__ Tt = set.text;

  // small state (always in smem)
  float* s_mode = mta_smem;           // [D]
  float* s_new = s_mode + D;          // [D]
  float* s_bw = s_new + D;            // [V]
  float* s_y = s_bw + V;              // [V]
  float* s_dens = s_y + V;            // [V]
  float* s_z = s_dens + V;            // [V]
  float* s_sq = s_z + V;              // [V]
  float* s_red = s_sq + V;            // [32]
  float* s_rows = s_red + 32;         // [NW][V] one distance row per warp
  float* big = s_rows + 8 * V;   // layout of small_state_bytes(); s_rows is only used by the NT = 256 path
  big = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(big) + 15) & ~static_cast<uintptr_t>(15));
  // region R (probabilities, later the view embeddings) and the V x V matrix
  const long long r_elems = static_cast<long long>(V) * (C > D ? C : D);
  const bool pre = a.A_pre != nullptr;   // affinity + bandwidths precomputed (large V): only the solver runs here
  float* R = a.in_smem ? big : (pre ? nullptr : a.scratch + problem * a.scratch_stride);
  const float* A = pre ? a.A_pre + problem * static_cast<long long>(V) * ldA
                       : (a.in_smem ? big + ((r_elems + 3) & ~3LL) : a.scratch + problem * a.scratch_stride + ((r_elems + 3) & ~3LL));
  float* Aw = const_cast<float*>(A);     // written only when !pre
  const float* X = Xg;
  if (pre) {
    for (int i = tid; i < V; i += NT) s_bw[i] = __ldg(a.bw_pre + problem * V + i);
  } else {
  if (a.P != nullptr) {
    // ---- 1+2. probabilities were computed for the whole batch by mta_probs_kernel: bring this problem's
    //           V x C block on chip (or use it in place when the problem does not fit in shared memory)
    const float* Pg = a.P + (static_cast<long long>(blockIdx.y) * a.I + img) * V * C;
    for (int i = tid; i < V * C; i += NT) R[i] = __ldg(Pg + i);
    __syncthreads();
  } else {
    // ---- 1. logits = 100 * X T / temperature -> R[v*C + c]      (test.py:1393)
    {
      const float scale = 100.0f / a.p.temperature;
      for (int c0 = 0; c0 < C; c0 += NT) {
        const int c = c0 + tid;
        const int cc = c < C ? c : C - 1;
        for (int v0 = 0; v0 < V; v0 += VB) {
          float acc[VB];
  #pragma unroll
          for (int j = 0; j < VB; ++j) acc[j] = 0.f;
          for (int d = 0; d < D; d += 4) {
            float t[4];
  #pragma unroll
            for (int e = 0; e < 4; ++e) t[e] = __ldg(Tt + static_cast<long long>(d + e) * C + cc);
  #pragma unroll
            for (int j = 0; j < VB; ++j) {
              const int v = v0 + j < V ? v0 + j : V - 1;
              const float4 x = __ldg(reinterpret_cast<const float4*>(Xg + v * D + d));  // warp-uniform address
              acc[j] = fmaf(x.x, t[0], acc[j]);
              acc[j] = fmaf(x.y, t[1], acc[j]);
              acc[j] = fmaf(x.z, t[2], acc[j]);
              acc[j] = fmaf(x.w, t[3], acc[j]);
            }
          }
          if (c < C) {
  #pragma unroll
            for (int j = 0; j < VB; ++j)
              if (v0 + j < V) R[(v0 + j) * C + c] = acc[j] * scale;
          }
        }
      }
    }
    __syncthreads();
    // ---- 2. row softmax in place
    for (int v = warp; v < V; v += NW) {
      float mx = -INFINITY;
      for (int c = lane; c < C; c += 32) mx = fmaxf(mx, R[v * C + c]);
      mx = warp_max(mx);
      float s = 0.f;
      for (int c = lane; c < C; c += 32) {
        const float e = expf(R[v * C + c] - mx);
        R[v * C + c] = e;
        s += e;
      }
      s = warp_sum(s);
      const float inv = 1.0f / s;
      for (int c = lane; c < C; c += 32) R[v * C + c] *= inv;
    }
    __syncthreads();
  }
  // ---- 3. affinity A = P P^T                                    (test.py:1411)
  for (int idx = tid; idx < V * V; idx += NT) {
    const int i = idx / V, j = idx % V;
    float s = 0.f;
    for (int c = 0; c < C; ++c) s = fmaf(R[i * C + c], R[j * C + c], s);
    Aw[i * ldA + j] = s;
  }
  __syncthreads();
  // ---- 4. bring the view embeddings on chip (region R is free now)
  if (a.in_smem) {
    for (int i = tid; i < V * D / 4; i += NT)
      reinterpret_cast<float4*>(R)[i] = __ldg(reinterpret_cast<const float4*>(Xg) + i);
    X = R;
  } else {
    X = Xg;
  }
  __syncthreads();
  // ---- 5. pairwise distances and per-view bandwidth             (test.py:1314-1318, :1403-1408)
  for (int i = warp; i < V; i += NW) {
    float q = 0.f;
    for (int d = lane; d < D; d += 32) q = fmaf(X[i * D + d], X[i * D + d], q);
    q = warp_sum(q);
    if (lane == 0) s_sq[i] = q;
  }
  __syncthreads();
  {
    float* my_row = s_rows + warp * V;
    for (int i = warp; i < V; i += NW) {
      for (int j = 0; j < V; ++j) {
        float dot = 0.f;
        for (int d = lane; d < D; d += 32) dot = fmaf(X[i * D + d], X[j * D + d], dot);
        dot = warp_sum(dot);
        if (lane == 0) {
          const float d2 = s_sq[i] - 2.0f * dot + s_sq[j];
          my_row[j] = sqrtf(fmaxf(d2, 0.0f));
        }
      }
      __syncwarp();
      // mean of the squared k smallest distances, skipping rank 0 (the point itself)
      float acc = 0.f;
      for (int j = lane; j < V; j += 32) {
        const float dj = my_row[j];
        int rank = 0;
        for (int l = 0; l < V; ++l) {
          const float dl = my_row[l];
          rank += (dl < dj || (dl == dj && l < j)) ? 1 : 0;
        }
        if (rank >= 1 && rank <= a.k) acc += dj * dj;
      }
      acc = warp_sum(acc);
      if (lane == 0) s_bw[i] = sqrtf(0.5f * (acc / static_cast<float>(a.k)));
      __syncwarp();
    }
  }
  }  // !pre
  __syncthreads();
  // ---- 6. initialise: y uniform, mode = un-augmented view        (test.py:1414-1418)
  for (int i = tid; i < V; i += NT) s_y[i] = 1.0f / static_cast<float>(V);
  for (int d = tid; d < D; d += NT) s_mode[d] = X[d];
  __syncthreads();

  const float inv_lambda_y = 1.0f / a.p.lambda_y;
  for (int outer = 0; outer < a.p.max_iter; ++outer) {            // test.py:1424, :1455-1457
    density_step<NW>(X, s_mode, s_bw, s_dens, V, D);                   // :1426
    for (int it = 1;; ++it) {                                      // inlierness loop :1430-1438
      float zmax = -INFINITY;
      if (pre) {
        // A lives in global memory (L2): one warp per row, lanes along the row (coalesced)
        for (int i = warp; i < V; i += NW) {
          const float* Ar = A + static_cast<long long>(i) * ldA;
          float s = 0.f;
          for (int j = lane; j < V; j += 32) s = fmaf(__ldg(Ar + j), s_y[j], s);
          s = warp_sum(s);
          if (lane == 0) s_z[i] = inv_lambda_y * (s_dens[i] + a.p.lambda_q * s);
        }
        __syncthreads();
        for (int i = tid; i < V; i += NT) zmax = fmaxf(zmax, s_z[i]);
      } else {
        for (int i = tid; i < V; i += NT) {
          float s = 0.f;
          for (int j = 0; j < V; ++j) s = fmaf(A[i * ldA + j], s_y[j], s);
          const float z = inv_lambda_y * (s_dens[i] + a.p.lambda_q * s);
          s_z[i] = z;
          zmax = fmaxf(zmax, z);
        }
      }
      zmax = block_max<NW>(zmax, s_red);
      float zs = 0.f;
      for (int i = tid; i < V; i += NT) {
        const float e = expf(s_z[i] - zmax);
        s_z[i] = e;
        zs += e;
      }
      zs = block_sum<NW>(zs, s_red);
      const float inv = 1.0f / zs;
      float diff = 0.f;
      for (int i = tid; i < V; i += NT) {
        const float yn = s_z[i] * inv;
        const float t = s_y[i] - yn;
        diff = fmaf(t, t, diff);
        s_z[i] = yn;
      }
      diff = block_sum<NW>(diff, s_red);
      // all threads finished reading s_y inside the A*y products before block_max's barrier
      for (int i = tid; i < V; i += NT) s_y[i] = s_z[i];
      __syncthreads();
      if (sqrtf(diff) < a.p.th || it >= a.p.max_iter) break;       // :1436
    }
    for (int it = 1;; ++it) {                                      // mode loop :1443-1453
      density_step<NW>(X, s_mode, s_bw, s_dens, V, D);                 // :1446
      float wsum = 0.f;
      for (int i = tid; i < V; i += NT) {
        const float w = s_dens[i] * s_y[i];                        // :1447
        s_z[i] = w;
        wsum += w;
      }
      wsum = block_sum<NW>(wsum, s_red);
      float nrm = 0.f;
      for (int d = tid; d < D; d += NT) {
        float s = 0.f;
        for (int i = 0; i < V; ++i) s = fmaf(s_z[i], X[i * D + d], s);
        s = s / wsum;                                              // :1448
        s_new[d] = s;
        nrm = fmaf(s, s, nrm);
      }
      nrm = block_sum<NW>(nrm, s_red);
      const float inv = 1.0f / sqrtf(nrm);                         // :1449
      float diff = 0.f;
      for (int d = tid; d < D; d += NT) {
        const float m = s_new[d] * inv;
        const float t = s_mode[d] - m;
        diff = fmaf(t, t, diff);
        s_new[d] = m;
      }
      diff = block_sum<NW>(diff, s_red);
      for (int d = tid; d < D; d += NT) s_mode[d] = s_new[d];
      __syncthreads();
      if (sqrtf(diff) < a.p.th || it >= a.p.max_iter) break;       // :1452
    }
  }

  // ---- 7. outputs: mode (test.py:1461) and optionally 100 * mode @ T (ood.py:819)
  for (int d = tid; d < D; d += NT) set.out_mode[img * D + d] = s_mode[d];
  if (set.out_logits) {
    for (int c = tid; c < C; c += NT) {
      float s = 0.f;
      for (int d = 0; d < D; ++d) s = fmaf(s_mode[d], __ldg(Tt + static_cast<long long>(d) * C + c), s);
      set.out_logits[img * C + c] = s * 100.0f;
    }
  }
  if (blockIdx.y == 0) mta_write_debug(a.dbg, img, V, s_bw, s_y, A, ldA, tid, NT);
}

constexpr size_t MTA_SMEM_LIMIT = 220 * 1024;

// ---------------------------------------------------------------------------------------------------
// Fast solver for problems that fit in shared memory (V <~ 95 at D = 512, C = 403): 512 threads, the two V x V
// Gram matrices (P P^T and X X^T) as register-tiled fp32 products instead of one warp-shuffle dot per pair, the
// mode vector in registers during the density passes, two block barriers per inlierness iteration.
// Measured on B200 at V = 65 (ncu, profiles/r01l_*): the first kernel spent 65 % of its 1.0 M cycles per problem
// in the per-pair dots of the set-up and ran 8 warps per SM.
constexpr int MF_THREADS = 512;

// row stride (floats) >= n: a multiple of 4 (16-byte rows) whose quarter is odd, so 8 consecutive rows read as
// float4 at the same column hit 8 different 4-bank groups
__host__ __device__ inline int mf_pad(int n) {
  int ld = (n + 3) & ~3;
  if (((ld >> 2) & 1) == 0) ld += 4;
  return ld;
}

// G[i * ldg + j] = sum_k M[i * ld + k] M[j * ld + k] for i, j < V, k < 4 * K4 (columns past the logical width are
// zero).  One thread = one 4 x 4 tile of the upper triangle; tile t of a dimension owns rows t, t + nt, t + 2 nt,
// t + 3 nt so that neighbouring threads (neighbouring column tiles) read neighbouring rows: conflict-free LDS.128,
// and the row tile they share is a broadcast.
template <int NT>
__device__ void mf_gram(const float* __restrict__ M, int ld, int K4, int V, float* __restrict__ G, int ldg) {
  const int nt = (V + 3) >> 2;
  const int npairs = nt * (nt + 1) / 2;
  for (int p = threadIdx.x; p < npairs; p += NT) {
    int ta = 0, rem = p;
    while (rem >= nt - ta) { rem -= nt - ta; ++ta; }
    const int tb = ta + rem;
    const float4* pa[4];
    const float4* pb[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int ia = ta + nt * r, ib = tb + nt * r;
      pa[r] = reinterpret_cast<const float4*>(M + static_cast<long long>(ia < V ? ia : V - 1) * ld);
      pb[r] = reinterpret_cast<const float4*>(M + static_cast<long long>(ib < V ? ib : V - 1) * ld);
    }
    float acc[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;
#pragma unroll 2
    for (int k = 0; k < K4; ++k) {
      float4 xa[4], xb[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) { xa[r] = pa[r][k]; xb[r] = pb[r][k]; }
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          acc[r][c] = fmaf(xa[r].x, xb[c].x, acc[r][c]);
          acc[r][c] = fmaf(xa[r].y, xb[c].y, acc[r][c]);
          acc[r][c] = fmaf(xa[r].z, xb[c].z, acc[r][c]);
          acc[r][c] = fmaf(xa[r].w, xb[c].w, acc[r][c]);
        }
    }
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int i = ta + nt * r, j = tb + nt * c;
        if (i < V && j < V) {
          G[i * ldg + j] = acc[r][c];
          G[j * ldg + i] = acc[r][c];
        }
      }
  }
}

// ---- the iterations of ONE bank, run by a group of GW warps (all warps of the CTA, or a third of them when the CTA's
// banks iterate side by side).  Every sum is taken in an order that depends on (V, D) only, never on GW: the density of
// a view by 16 lanes, a row of A y by one thread, the mode update as MF_IQ partial sums over fixed view ranges per
// 128-column slot.  So a bank gives the same bits whether it has the CTA to itself (few images per call) or shares it.
constexpr int MF_IQ = 4;
__host__ __device__ inline int mf_iq(int V) { return V >= 16 ? MF_IQ : 1; }
// floats of one bank's iteration state: mode [D], partial sums [iq, D] (the first D double as the new mode), y, density,
// density * y, z [V rounded up to 4], reduction slots [32]
__host__ __device__ inline int mf_state_floats(int V, int D) { return D + mf_iq(V) * D + 4 * ((V + 3) & ~3) + 32; }

__device__ __forceinline__ void mf_bar(int id, int nthreads) {
  if (nthreads == 32) __syncwarp();
  else asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// gaussian_kernel(mode, bandwidth, X)  (test.py:1310-1313): 16 lanes per view, two views per warp pass, the mode in
// registers.  out[i] = density_i, or density_i * y_i (test.py:1447) for the mode loop
template <bool WITH_Y, int MAXQ>
__device__ __forceinline__ void mf_density_q(const float* __restrict__ X, int ldx, const float* s_mode, const float* s_bw,
                                           const float* s_y, float* s_out, int V, int D, int gw, int GW) {
  const int lane = threadIdx.x & 31, sub = lane & 15, half = lane >> 4;
  const int nq = D >> 6;  // float4 per lane, D % 64 == 0; MAXQ = 0: any D, the mode is re-read from shared memory
  float4 m[MAXQ > 0 ? MAXQ : 1];
#pragma unroll
  for (int q = 0; q < MAXQ; ++q)
    if (q < nq) m[q] = *reinterpret_cast<const float4*>(s_mode + 64 * q + 4 * sub);
  for (int p = gw; 2 * p < V; p += GW) {
    const int i = 2 * p + half;
    const float* xr = X + (i < V ? i : V - 1) * ldx + 4 * sub;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    if (MAXQ > 0) {
#pragma unroll
      for (int q = 0; q < MAXQ; ++q)
        if (q < nq) {
          const float4 x = *reinterpret_cast<const float4*>(xr + 64 * q);
          float t = x.x - m[q].x; a0 = fmaf(t, t, a0);
          t = x.y - m[q].y; a1 = fmaf(t, t, a1);
          t = x.z - m[q].z; a2 = fmaf(t, t, a2);
          t = x.w - m[q].w; a3 = fmaf(t, t, a3);
        }
    } else {
#pragma unroll 4
      for (int q = 0; q < nq; ++q) {
        const float4 x = *reinterpret_cast<const float4*>(xr + 64 * q);
        const float4 mm = *reinterpret_cast<const float4*>(s_mode + 64 * q + 4 * sub);
        float t = x.x - mm.x; a0 = fmaf(t, t, a0);
        t = x.y - mm.y; a1 = fmaf(t, t, a1);
        t = x.z - mm.z; a2 = fmaf(t, t, a2);
        t = x.w - mm.w; a3 = fmaf(t, t, a3);
      }
    }
    float acc = (a0 + a1) + (a2 + a3);
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (sub == 0 && i < V) {
      const float dist = sqrtf(acc);  // jt.norm(...), then dist**2 as the reference does
      const float bw = s_bw[i];
      const float dens = expf(-(dist * dist) / (2.0f * bw * bw));
      s_out[i] = WITH_Y ? dens * s_y[i] : dens;
    }
  }
}

template <bool WITH_Y>
__device__ __forceinline__ void mf_density(const float* __restrict__ X, int ldx, const float* s_mode, const float* s_bw,
                                           const float* s_y, float* s_out, int V, int D, int gw, int GW) {
  if (D <= 512) mf_density_q<WITH_Y, 8>(X, ldx, s_mode, s_bw, s_y, s_out, V, D, gw, GW);   // (CLIP ViT-B: 512)
  else mf_density_q<WITH_Y, 0>(X, ldx, s_mode, s_bw, s_y, s_out, V, D, gw, GW);
}

__device__ __forceinline__ void mf_solve_bank(const MtaDev& a, int si, long long img, const float* __restrict__ X,
                              const float* __restrict__ A, const float* s_bw, float* st, int gw, int GW, int bar_id) {
  const MtaSet& set = a.sets[si];
  const int V = a.V, C = a.C, D = a.D, ldA = a.ldA, ldx = a.ldx;
  const int lane = threadIdx.x & 31, gt = gw * 32 + lane, GT = GW * 32;
  const int vp = (V + 3) & ~3, iq_n = mf_iq(V), nds = D >> 7;
  float* s_mode = st;                  // [D]
  float* s_part = s_mode + D;          // [iq_n, D]; row 0 becomes the new mode
  float* s_y = s_part + iq_n * D;      // [vp]
  float* s_dens = s_y + vp;            // [vp]
  float* s_w = s_dens + vp;            // [vp]
  float* s_z = s_w + vp;               // [vp]
  float* s_red = s_z + vp;             // [32]
  const float inv_lambda_y = 1.0f / a.p.lambda_y, lambda_q = a.p.lambda_q, th = a.p.th;
  const int max_iter = a.p.max_iter;

  mf_bar(bar_id, GT);   // (banks one after another: the previous bank's mode has been written out)
  // ---- 6. initialise: y uniform, mode = un-augmented view        (test.py:1414-1418)
  for (int i = gt; i < vp; i += GT) s_y[i] = i < V ? 1.0f / static_cast<float>(V) : 0.f;
  for (int d = gt; d < D; d += GT) s_mode[d] = X[d];
  mf_bar(bar_id, GT);

  for (int outer = 0; outer < max_iter; ++outer) {                 // test.py:1424, :1455-1457
    mf_density<false>(X, ldx, s_mode, s_bw, s_y, s_dens, V, D, gw, GW);   // :1426
    mf_bar(bar_id, GT);
    for (int it = 1;; ++it) {                                       // inlierness loop :1430-1438
      for (int i = gt; i < V; i += GT) {                            // z = (rho + lambda_q A y) / lambda_y, a row per thread
        const float* ar = A + i * ldA;
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
        int j = 0;
        for (; j + 4 <= V; j += 4) {
          const float4 y4 = *reinterpret_cast<const float4*>(s_y + j);
          s0 = fmaf(ar[j], y4.x, s0);
          s1 = fmaf(ar[j + 1], y4.y, s1);
          s2 = fmaf(ar[j + 2], y4.z, s2);
          s3 = fmaf(ar[j + 3], y4.w, s3);
        }
        for (; j < V; ++j) s0 = fmaf(ar[j], s_y[j], s0);
        s_z[i] = inv_lambda_y * (s_dens[i] + lambda_q * ((s0 + s1) + (s2 + s3)));
      }
      mf_bar(bar_id, GT);
      if (gw == 0) {                                                // y <- softmax(z), ||y_old - y||
        float mx = -INFINITY;
        for (int i = lane; i < V; i += 32) mx = fmaxf(mx, s_z[i]);
        mx = warp_max(mx);
        float zs = 0.f;
        for (int i = lane; i < V; i += 32) {
          const float e = expf(s_z[i] - mx);
          s_z[i] = e;
          zs += e;
        }
        zs = warp_sum(zs);
        const float inv = 1.0f / zs;
        float diff = 0.f;
        for (int i = lane; i < V; i += 32) {
          const float yn = s_z[i] * inv;
          const float t = s_y[i] - yn;
          diff = fmaf(t, t, diff);
          s_y[i] = yn;
        }
        diff = warp_sum(diff);
        if (lane == 0) s_red[31] = diff;
      }
      mf_bar(bar_id, GT);
      if (sqrtf(s_red[31]) < th || it >= max_iter) break;          // :1436
    }
    const int q4 = (V + iq_n - 1) / iq_n;
    for (int it = 1;; ++it) {                                       // mode loop :1443-1453
      mf_density<true>(X, ldx, s_mode, s_bw, s_y, s_w, V, D, gw, GW);     // :1446-1447: w = density * y
      mf_bar(bar_id, GT);
      // sum_i w_i x_i (:1448) as iq_n partial sums over fixed view ranges, one warp per (range, 128-column slot)
      for (int u = gw; u < nds * iq_n; u += GW) {
        const int ds = u % nds, qi = u / nds;
        const int i0 = qi * q4, i1 = (i0 + q4 < V) ? i0 + q4 : V;
        const float* xc = X + 128 * ds + 4 * lane;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
        for (int i = i0; i < i1; ++i) {
          const float w = s_w[i];
          const float4 x = *reinterpret_cast<const float4*>(xc + i * ldx);
          acc.x = fmaf(w, x.x, acc.x);
          acc.y = fmaf(w, x.y, acc.y);
          acc.z = fmaf(w, x.z, acc.z);
          acc.w = fmaf(w, x.w, acc.w);
        }
        *reinterpret_cast<float4*>(s_part + qi * D + 128 * ds + 4 * lane) = acc;
      }
      mf_bar(bar_id, GT);
      for (int ds = gw; ds < nds; ds += GW) {                       // / sum_i w_i, and the slot's share of ||.||^2
        float wsum = 0.f;
        for (int i = lane; i < V; i += 32) wsum += s_w[i];
        wsum = warp_sum(wsum);
        float* pc = s_part + 128 * ds + 4 * lane;
        float4 s = *reinterpret_cast<const float4*>(pc);
        for (int qi = 1; qi < iq_n; ++qi) {
          const float4 t = *reinterpret_cast<const float4*>(pc + qi * D);
          s.x += t.x; s.y += t.y; s.z += t.z; s.w += t.w;
        }
        s.x = s.x / wsum; s.y = s.y / wsum; s.z = s.z / wsum; s.w = s.w / wsum;   // :1448
        *reinterpret_cast<float4*>(pc) = s;
        float nrm = fmaf(s.x, s.x, fmaf(s.y, s.y, fmaf(s.z, s.z, s.w * s.w)));
        nrm = warp_sum(nrm);
        if (lane == 0) s_red[ds] = nrm;
      }
      mf_bar(bar_id, GT);
      float nrm = 0.f;
      for (int ds = 0; ds < nds; ++ds) nrm += s_red[ds];
      const float inv = 1.0f / sqrtf(nrm);                          // :1449
      for (int ds = gw; ds < nds; ds += GW) {
        const int d = 128 * ds + 4 * lane;
        float4 mnew = *reinterpret_cast<const float4*>(s_part + d);
        const float4 mold = *reinterpret_cast<const float4*>(s_mode + d);
        mnew.x *= inv; mnew.y *= inv; mnew.z *= inv; mnew.w *= inv;
        float t = mold.x - mnew.x, diff = t * t;
        t = mold.y - mnew.y; diff = fmaf(t, t, diff);
        t = mold.z - mnew.z; diff = fmaf(t, t, diff);
        t = mold.w - mnew.w; diff = fmaf(t, t, diff);
        *reinterpret_cast<float4*>(s_mode + d) = mnew;
        diff = warp_sum(diff);
        if (lane == 0) s_red[8 + ds] = diff;
      }
      mf_bar(bar_id, GT);
      float diff = 0.f;
      for (int ds = 0; ds < nds; ++ds) diff += s_red[8 + ds];
      if (sqrtf(diff) < th || it >= max_iter) break;                // :1452
    }
  }

  // ---- 7. outputs: mode (test.py:1461) and optionally 100 * mode @ T (ood.py:819)
  for (int d = gt; d < D; d += GT) set.out_mode[img * D + d] = s_mode[d];
  if (set.out_logits) {
    const float* __restrict__ Tt = set.text;
    for (int c = gt; c < C; c += GT) {
      float s2 = 0.f;
      for (int d = 0; d < D; ++d) s2 = fmaf(s_mode[d], __ldg(Tt + static_cast<long long>(d) * C + c), s2);
      set.out_logits[img * C + c] = s2 * 100.0f;
    }
  }
  if (si == 0) mta_write_debug(a.dbg, img, V, s_bw, s_y, A, ldA, gt, GT);
}

// NT = 512 threads and one CTA per SM for the headline view counts (V = 65: 215 KB of shared memory with three banks);
// NT = 128 and up to four CTAs per SM for V <= 32, where a problem is a few KB and 512 threads mostly wait at barriers
// (N = 1 and N = 16 crops: thousands of tiny problems per step).
// NT = 32 / 64: one or two warps per problem for the smallest view counts (V = 2 at N = 1 crop: 12 480 problems per step
// whose ~50 iterations are pure barrier latency with four warps; with one warp a barrier is free and 16 problems share
// an SM).
// With NT = 512 the banks of a CTA iterate SIDE BY SIDE, each on NW / nb warps with its own named barrier and state: the
// iterations are latency- and barrier-bound (a few hundred instructions between barriers), so three independent
// instruction streams fill the issue slots one stream leaves empty.
template <int NT>
__global__ void __launch_bounds__(NT, NT == 512 ? 1 : (NT == 128 ? 4 : (NT == 64 ? 8 : 16))) mta_fast_kernel(const MtaDev a) {
  constexpr int NW = NT / 32;
  extern __shared__ __align__(16) float mta_smem[];
  griddep_wait();               // programmatic dependent launch (ptx.cuh): nothing global is touched above
  const int V = a.V, C = a.C, D = a.D, ldA = a.ldA, ldx = a.ldx, ldp = a.ldp;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long img = blockIdx.x;
  const int group = blockIdx.y;
  const int nb = a.group_count[group];                   // banks solved by this CTA (they share the feature tensor)
  const float* __restrict__ Xg = a.sets[a.group_sets[group][0]].feats + img * V * D;

  const int vp = (V + 3) & ~3;
  float* s_bw = mta_smem;             // [vp]
  float* s_sq = s_bw + vp;            // [vp]
  float* R = s_sq + vp;                                  // P [V, ldp] of one bank at a time, later X [V, ldx]
  const int r_elems = V * (ldp > ldx ? ldp : ldx);
  const int a_elems = (V * ldA + 3) & ~3;
  float* A_all = R + r_elems;                            // affinities [nb][V, ldA]
  float* U = A_all + a.max_group * a_elems;              // Gram of X, then the pairwise distances [V, ldA]; afterwards
  float* Dm = U;                                         // the iteration state of the banks

  for (int b = 0; b < nb; ++b) {
    // ---- 1+2. this problem's V x C block of softmax(100 X T), zero padded to ldp columns
    const int si = a.group_sets[group][b];
    const float* Pg = a.P + (static_cast<long long>(si) * a.I + img) * V * C;
    for (int i = tid; i < V * ldp; i += NT) {
      const int v = i / ldp, c = i - v * ldp;
      R[i] = c < C ? __ldg(Pg + v * C + c) : 0.f;
    }
    __syncthreads();
    // ---- 3. affinity A = P P^T                                    (test.py:1411)
    mf_gram<NT>(R, ldp, ldp >> 2, V, A_all + b * a_elems, ldA);
    __syncthreads();
  }
  // ---- 4. the view embeddings replace P on chip
  for (int i = tid; i < V * (D >> 2); i += NT) {
    const int v = i / (D >> 2), c4 = i - v * (D >> 2);
    *reinterpret_cast<float4*>(R + v * ldx + 4 * c4) = __ldg(reinterpret_cast<const float4*>(Xg + v * D) + c4);
  }
  __syncthreads();
  const float* X = R;
  // ---- 5. pairwise distances and per-view bandwidth             (test.py:1314-1318, :1403-1408)
  mf_gram<NT>(X, ldx, D >> 2, V, Dm, ldA);
  __syncthreads();
  for (int i = tid; i < V; i += NT) s_sq[i] = Dm[i * ldA + i];   // ||x_i||^2, same summation as the dots
  __syncthreads();
  for (int idx = tid; idx < V * V; idx += NT) {
    const int i = idx / V, j = idx - i * V;
    const float d2 = s_sq[i] - 2.0f * Dm[i * ldA + j] + s_sq[j];
    Dm[i * ldA + j] = sqrtf(fmaxf(d2, 0.0f));
  }
  __syncthreads();
  for (int i = warp; i < V; i += NW) {
    // mean of the squared k smallest distances, skipping rank 0 (the point itself)
    const float* my_row = Dm + i * ldA;
    float acc = 0.f;
    for (int j = lane; j < V; j += 32) {
      const float dj = my_row[j];
      int rank = 0;
      for (int l = 0; l < V; ++l) {
        const float dl = my_row[l];
        rank += (dl < dj || (dl == dj && l < j)) ? 1 : 0;
      }
      if (rank >= 1 && rank <= a.k) acc += dj * dj;
    }
    acc = warp_sum(acc);
    if (lane == 0) s_bw[i] = sqrtf(0.5f * (acc / static_cast<float>(a.k)));
  }
  __syncthreads();   // s_bw is complete; the distances are dead, their memory becomes the banks' state

  int b0 = 0, b1 = nb, gw = warp, GW = NW, bar = 0;
  float* st = U;
  if (NT == 512 && nb > 1) {         // side by side: bank b on warps [b GW, (b + 1) GW), barrier 1 + b, its own state
    GW = NW / nb;
    b0 = warp / GW;
    if (b0 >= nb) return;            // spare warp (16 = 3 x 5 + 1)
    b1 = b0 + 1;
    gw = warp - b0 * GW;
    bar = 1 + b0;
    st = U + b0 * mf_state_floats(V, D);
  }
  for (int b = b0; b < b1; ++b)
    mf_solve_bank(a, a.group_sets[group][b], img, X, A_all + b * a_elems, s_bw, st, gw, GW, bar);
}

// banks whose iteration state is live at the same time: the 512-thread kernel (V > 32) iterates its banks side by side
static int mf_states(int V, int banks) { return V > 32 ? banks : 1; }
size_t mf_smem_bytes(int V, int C, int D, int banks = 1) {
  const int ldx = mf_pad(D), ldp = mf_pad(C), ldA = V | 1, vp = (V + 3) & ~3;
  const size_t a_elems = (static_cast<size_t>(V) * ldA + 3) & ~static_cast<size_t>(3);
  // bandwidths + squared norms, the P / X region, one affinity per bank the CTA solves, and the region that first holds
  // the distance matrix and then the banks' iteration state
  const size_t state = static_cast<size_t>(mf_states(V, banks)) * mf_state_floats(V, D);
  const size_t bigf = static_cast<size_t>(V) * (ldp > ldx ? ldp : ldx) + banks * a_elems + (a_elems > state ? a_elems : state);
  return (2 * vp + bigf) * sizeof(float) + 16;
}


size_t small_state_bytes(int V, int D) { return sizeof(float) * (2 * D + (5 + MTA_WARPS) * V + 32) + 16; }
long long big_elems(int V, int C, int D, int ldA) {
  const long long r = static_cast<long long>(V) * (C > D ? C : D);
  return ((r + 3) & ~3LL) + static_cast<long long>(V) * ldA;
}

}  // namespace

static bool mta_fits_smem(int V, int C, int D) {
  return small_state_bytes(V, D) + static_cast<size_t>(big_elems(V, C, D, V | 1)) * sizeof(float) <= MTA_SMEM_LIMIT;
}

static bool mta_use_probs_kernel(int C, int D) { return C <= PB_CPAD && D % PB_KC == 0; }

// floats per problem of the large-V path: affinity [V, ldA] + Gram of X [V, ldA] + bandwidths [V]
static long long big_pre_elems(int V, int ldA) {
  const long long m = (static_cast<long long>(V) * ldA + 3) & ~3LL;
  return 2 * m + ((V + 3) & ~3);
}
static bool mta_fast_fits(int V, int C, int D) {
  return mta_use_probs_kernel(C, D) && D % 128 == 0 && mf_smem_bytes(V, C, D) <= MTA_SMEM_LIMIT;
}

// bytes of the tensor-core probabilities path for `rows` view rows per bank and `n_sets` banks: A' limbs (one copy per
// distinct feature tensor, at most n_sets), B' limbs and the fp32 logits
static size_t tcp_bytes(size_t n_sets, size_t rows, int D) {
  auto up = [](size_t x) { return (x + 255) / 256 * 256; };
  return n_sets * (up(rows * 6 * D * 2) + up(static_cast<size_t>(TCP_CP) * 6 * D * 2) + up(rows * TCP_CP * 4));
}
static bool mta_tc_probs_possible(int C, int D) { return C <= TCP_CP && C <= 512 && D % 64 == 0 && D >= 64; }

size_t mta_scratch_bytes(int64_t n_problems, int V, int C, int D) {
  size_t b = 0;
  if (mta_use_probs_kernel(C, D)) b += (static_cast<size_t>(n_problems) * V * C * sizeof(float) + 255) / 256 * 256;
  // (n_problems = n_sets * images: n_sets banks of n_problems / n_sets * V rows each = n_problems * V rows in total)
  if (mta_use_probs_kernel(C, D) && mta_tc_probs_possible(C, D)) b += tcp_bytes(1, static_cast<size_t>(n_problems) * V, D) + 3 * 4 * 256 + tcp_bytes(MTA_MAX_SETS, 0, D);
  if (!mta_fast_fits(V, C, D) && !mta_fits_smem(V, C, D)) {
    const long long be = big_elems(V, C, D, V | 1), bp = big_pre_elems(V, V | 1);
    b += static_cast<size_t>(n_problems) * static_cast<size_t>(be > bp ? be : bp) * sizeof(float);
  }
  return b;
}

bool mta_shape_supported(int V, int C, int D) {
  return V >= 1 && V <= 2048                    // small state must stay well inside shared memory
         && C >= 1 && D >= 32 && D % 32 == 0 && D <= 1024;
}

cudaError_t launch_mta(const MtaSet* sets, int n_sets, int64_t I, int V, int C, int D, const MtaParams& p,
                       float* scratch, cudaStream_t stream, int* dev_status, int num_sms, const MtaDebug* debug) {
  if (!mta_shape_supported(V, C, D)) return cudaErrorInvalidValue;
  if (n_sets < 1 || n_sets > MTA_MAX_SETS) return cudaErrorInvalidValue;
  if (I == 0) return cudaSuccess;
  MtaDev a;
  a.dbg = debug ? *debug : MtaDebug{nullptr, nullptr, nullptr};
  for (int s = 0; s < n_sets; ++s) a.sets[s] = sets[s];
  for (int s = n_sets; s < MTA_MAX_SETS; ++s) a.sets[s] = sets[0];
  a.I = I; a.V = V; a.C = C; a.D = D;
  a.ldA = V | 1;  // odd row stride: conflict-free column walks
  // int(0.3 * (V - 1)) in double precision, exactly as the Python expression (test.py:1405)
  int k = static_cast<int>(p.k_frac * static_cast<double>(V - 1));
  a.k = k < 1 ? 1 : k;
  a.p = p;
  const size_t small = small_state_bytes(V, D);
  const long long be = big_elems(V, C, D, a.ldA);
  a.in_smem = mta_fits_smem(V, C, D) ? 1 : 0;
  a.P = nullptr;
  a.A_pre = nullptr;
  a.bw_pre = nullptr;
  if (mta_use_probs_kernel(C, D)) {
    if (scratch == nullptr) return cudaErrorInvalidValue;
    const size_t p_bytes = (static_cast<size_t>(n_sets) * I * V * C * sizeof(float) + 255) / 256 * 256;
    const long long rows = static_cast<long long>(I) * V;
    // taken at EVERY batch size: a row's probabilities must not depend on how many other rows share the launch (the
    // path's pass-size and batch-split invariance is bit-exact); at one image the three extra launches per bank cost ~40 us
    if (mta_tc_probs_possible(C, D)) {
      auto up = [](size_t x) { return (x + 255) / 256 * 256; };
      uint8_t* w = reinterpret_cast<uint8_t*>(scratch) + p_bytes;     // behind P; sized by mta_scratch_bytes
      const size_t a_b = up(static_cast<size_t>(rows) * 6 * D * 2), b_b = up(static_cast<size_t>(TCP_CP) * 6 * D * 2);
      const size_t l_b = up(static_cast<size_t>(rows) * TCP_CP * 4);
      const float* split_of[MTA_MAX_SETS];
      uint16_t* a_of[MTA_MAX_SETS];
      int n_split = 0;
      for (int s2 = 0; s2 < n_sets; ++s2) {
        // banks that share a feature tensor (prompt-tuned and hand-crafted text on the same tower) share its limbs
        uint16_t* ap = nullptr;
        for (int q = 0; q < n_split; ++q)
          if (split_of[q] == sets[s2].feats) ap = a_of[q];
        if (!ap) {
          ap = reinterpret_cast<uint16_t*>(w);
          w += a_b;
          split_of[n_split] = sets[s2].feats;
          a_of[n_split++] = ap;
          const long long n = rows * D;
          if (cudaError_t e = launch_pdl(mta_split_x_kernel, dim3(static_cast<unsigned>((n + 255) / 256)), dim3(256), 0, stream, 1,
                                         sets[s2].feats, rows, D, ap)) return e;
        }
        uint16_t* bp = reinterpret_cast<uint16_t*>(w);
        w += b_b;
        float* lg = reinterpret_cast<float*>(w);
        w += l_b;
        if (cudaError_t e = launch_pdl(mta_split_t_kernel, dim3((TCP_CP * D + 255) / 256), dim3(256), 0, stream, 1, sets[s2].text, C,
                                       TCP_CP, D, bp)) return e;
        GemmArgs g;
        g.A = reinterpret_cast<const __nv_bfloat16*>(ap); g.B = reinterpret_cast<const __nv_bfloat16*>(bp);
        g.lda = 6 * D; g.ldb = 6 * D; g.M = static_cast<int>(rows); g.N = TCP_CP; g.K = 6 * D;
        g.bias = nullptr; g.epilogue = EPI_F32; g.out = lg; g.ldo = TCP_CP; g.f16 = 0;
        cudaError_t e = launch_gemm(g, dev_status, num_sms, stream);
        if (e != cudaSuccess) return e;
        if ((e = launch_pdl(mta_softmax_rows_kernel, dim3(static_cast<unsigned>((rows + 7) / 8)), dim3(256), 0, stream, 1, lg, rows, C,
                            TCP_CP, 100.0f / p.temperature, scratch + static_cast<long long>(s2) * rows * C)) != cudaSuccess) return e;
      }
      cudaError_t e = cudaGetLastError();
      if (e != cudaSuccess) return e;
    } else {
      ProbsDev pd;
      for (int s2 = 0; s2 < MTA_MAX_SETS; ++s2) pd.sets[s2] = a.sets[s2];
      pd.rows = rows;
      pd.C = C; pd.D = D; pd.scale = 100.0f / p.temperature; pd.P = scratch;
      {
        cudaError_t e = ensure_dynamic_smem(mta_probs_kernel, PB_SMEM);
        if (e != cudaSuccess) return e;
      }
      dim3 pgrid(static_cast<unsigned>((pd.rows + PB_ROWS - 1) / PB_ROWS), static_cast<unsigned>(n_sets));
      mta_probs_kernel<<<pgrid, 256, PB_SMEM, stream>>>(pd);
      cudaError_t e = cudaGetLastError();
      if (e != cudaSuccess) return e;
    }
    a.P = scratch;
    scratch = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(scratch) + p_bytes +
                                       (mta_tc_probs_possible(C, D) ? tcp_bytes(static_cast<size_t>(n_sets), static_cast<size_t>(rows), D) : 0));
  }
  if (mta_fast_fits(V, C, D)) {
    a.ldx = mf_pad(D);
    a.ldp = mf_pad(C);
    a.in_smem = 1;
    a.scratch = nullptr;
    a.scratch_stride = 0;
    a.n_groups = 0;
    for (int s2 = 0; s2 < n_sets; ++s2) {
      int g = -1;
      for (int q = 0; q < a.n_groups; ++q)
        if (sets[a.group_sets[q][0]].feats == sets[s2].feats) g = q;
      if (g < 0) { g = a.n_groups++; a.group_count[g] = 0; }
      a.group_sets[g][a.group_count[g]++] = s2;
    }
    a.max_group = 1;
    for (int q = 0; q < a.n_groups; ++q) a.max_group = a.group_count[q] > a.max_group ? a.group_count[q] : a.max_group;
    // Sharing pays when there are more problems than SMs (a wave of one-bank CTAs would not fit anyway); with a handful
    // of images (the reference's one-image-per-call loop) three CTAs in parallel beat one CTA doing three solves in a
    // row.  Either way a bank's arithmetic is the same instruction sequence: the results are bit-identical.
    if (mf_smem_bytes(V, C, D, a.max_group) > MTA_SMEM_LIMIT || I * n_sets <= num_sms) {   // (or no room for several affinities: V > 65)
      a.n_groups = n_sets;
      a.max_group = 1;
      for (int s2 = 0; s2 < n_sets; ++s2) { a.group_count[s2] = 1; a.group_sets[s2][0] = s2; }
    }
    dim3 fgrid(static_cast<unsigned>(I), static_cast<unsigned>(a.n_groups));
    const size_t fsmem = mf_smem_bytes(V, C, D, a.max_group);
    if (V <= 32) {
      // threads per CTA by view count, as measured at N = 1 and N = 16 crops (profiles/r02q_mta_small_v_thread_count.log)
      const int nt = V <= 4 ? 32 : (V <= 12 ? 64 : 128);
      cudaError_t e = cudaSuccess;
      if (nt == 32) {
        if ((e = ensure_dynamic_smem(mta_fast_kernel<32>, fsmem)) != cudaSuccess) return e;
        if ((e = launch_pdl(mta_fast_kernel<32>, fgrid, dim3(32), fsmem, stream, 1, a)) != cudaSuccess) return e;
      } else if (nt == 64) {
        if ((e = ensure_dynamic_smem(mta_fast_kernel<64>, fsmem)) != cudaSuccess) return e;
        if ((e = launch_pdl(mta_fast_kernel<64>, fgrid, dim3(64), fsmem, stream, 1, a)) != cudaSuccess) return e;
      } else {
        if ((e = ensure_dynamic_smem(mta_fast_kernel<128>, fsmem)) != cudaSuccess) return e;
        if ((e = launch_pdl(mta_fast_kernel<128>, fgrid, dim3(128), fsmem, stream, 1, a)) != cudaSuccess) return e;
      }
    } else {
      // (A/B this round: the same solver with 128 threads per CTA takes 2.3x as long per bank -- 3.25 vs 1.61 ms per step
      // un-grouped -- so running the banks of a CTA concurrently on 128-thread groups would gain < 25 % of the iterations)
      cudaError_t e = ensure_dynamic_smem(mta_fast_kernel<MF_THREADS>, MTA_SMEM_LIMIT);
      if (e != cudaSuccess) return e;
      if ((e = launch_pdl(mta_fast_kernel<MF_THREADS>, fgrid, dim3(MF_THREADS), fsmem, stream, 1, a)) != cudaSuccess) return e;
    }
    return cudaGetLastError();
  }
  if (!a.in_smem && scratch == nullptr) return cudaErrorInvalidValue;
  a.scratch = scratch;
  a.scratch_stride = be;
  if (!a.in_smem && a.P != nullptr) {
    // large V: affinity, distances and bandwidths batched over all problems, then one solver CTA per problem
    const long long n_prob = static_cast<long long>(n_sets) * I;
    const long long m = (static_cast<long long>(V) * a.ldA + 3) & ~3LL;
    float* A_all = scratch;
    float* G_all = scratch + n_prob * m;
    float* bw_all = scratch + 2 * n_prob * m;
    if (n_prob > 65535) return cudaErrorInvalidValue;
    const int nt = (V + GB_TILE - 1) / GB_TILE;
    GramBigDev g;
    for (int s2 = 0; s2 < MTA_MAX_SETS; ++s2) g.sets[s2] = a.sets[s2];
    g.I = I; g.V = V; g.ldg = a.ldA; g.P = a.P;
    dim3 ggrid(static_cast<unsigned>(nt * (nt + 1) / 2), static_cast<unsigned>(n_prob));
    g.K = C; g.ld = C; g.from_feats = 0; g.G = A_all;
    mta_gram_big_kernel<<<ggrid, 256, 0, stream>>>(g);
    g.K = D; g.ld = D; g.from_feats = 1; g.G = G_all;
    mta_gram_big_kernel<<<ggrid, 256, 0, stream>>>(g);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    BwBigDev b;
    b.G = G_all; b.bw = bw_all; b.V = V; b.ldg = a.ldA; b.k = a.k;
    const size_t bw_smem = sizeof(float) * static_cast<size_t>(9) * V;
    e = ensure_dynamic_smem(mta_bw_big_kernel, bw_smem);
    if (e != cudaSuccess) return e;
    dim3 bgrid(static_cast<unsigned>((V + 7) / 8), static_cast<unsigned>(n_prob));
    mta_bw_big_kernel<<<bgrid, 256, bw_smem, stream>>>(b);
    e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    a.A_pre = A_all;
    a.bw_pre = bw_all;
    a.scratch = nullptr;
    a.scratch_stride = 0;
  }
  const size_t smem = a.in_smem ? small + static_cast<size_t>(be) * sizeof(float) : small;
  dim3 grid(static_cast<unsigned>(I), static_cast<unsigned>(n_sets));
  if (a.A_pre != nullptr) {
    cudaError_t e = ensure_dynamic_smem(mta_kernel<1024>, smem);
    if (e != cudaSuccess) return e;
    mta_kernel<1024><<<grid, 1024, smem, stream>>>(a);
  } else {
    cudaError_t e = ensure_dynamic_smem(mta_kernel<MTA_THREADS>, MTA_SMEM_LIMIT);
    if (e != cudaSuccess) return e;
    mta_kernel<MTA_THREADS><<<grid, MTA_THREADS, smem, stream>>>(a);
  }
  return cudaGetLastError();
}

}  // namespace jcb
