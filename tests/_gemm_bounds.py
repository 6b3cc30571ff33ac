"""Error bounds of the tcgen05 GEMM (csrc/gemm.cu) and its fused epilogues, derived from the operation, shared by
test_gpu_gemm_edges.py (the kernel against float64) and test_gemm_bounds_cpu.py (the bounds have power).

u = 2^-24 (fp32 unit roundoff).  P = |A| |B|^T (+ |A2| |B2|^T), computed in float64.  ref = the epilogue's operation in
float64 on the kernel's own 16-bit operands (and, for the LayerNorm fold, on its own fp32 row scale r and -r mu, see
ln_scale).  Per output element the fp32 part of the bound is e = KAPPA u P (the tensor core's fp32 accumulation, in
whatever order) + 4 u Q, where Q sums the magnitudes the epilogue's fp32 adds / multiplies act on: at most two
roundings of at most u Q each, doubled so that a correct fp32 epilogue stays 3 x inside (test_gemm_bounds_cpu.py):

  EPI_F32            Q = P + |bias|                        fl(acc + bias)
  EPI_BIAS_RESID_F32 Q = P + |bias| + |old|                fl(old + fl(acc + bias)), the reduce-add of the TMA store
  EPI_BIAS_16        Q = P + |bias|                        then + half an ulp of |ref| + e (round to nearest; fp16
                                                           saturates, cvt.rn.satfinite)
  EPI_LNFOLD_16      y = r acc + (-r mu) S + c with the epilogue's own fp32 r and -r mu (ln_scale):
                     e = KAPPA u r P + 4 u (r P + r |mu| |S| + |c|)    (the 4 u also covers r, -r mu one ulp off)
  GELU forms         x = the above before the activation, e_x its e:  e = 1.1 e_x + (2^-10 + 2 u) |x|  + half an ulp.
                     1.1 bounds |d quickgelu / dx|.  tanh.approx.f32 has relative error <= 2^-10.987 and the epilogue
                     multiplies it by h = x / 2, i.e. <= 2^-11.987 |x|; 2^-10 |x| is 4 x that (2^-11 |x| would leave
                     only 2 x).  For x << 0 the output is ~x e^{1.702 x}, far below 2^-10 |x|: there the bound is the
                     tanh error, not an ulp of the output, and says so.
  EPI_RESID_LNPREP_* residual: as EPI_BIAS_RESID_F32
                     shift_out = shift_in + sum(stats_in[., :, 0]) / N:  (slots + 2) u (|shift_in| + sum |.| / N)
                     copy = round16(fl(x - shift)) from the kernel's own x and shift:  u |d| + half an ulp of |d|
                     stats[m, n / BN] = fp32 sums of fl(x - shift) over the BN columns of the tile, sequentially:
                     (BN + 1) u sum |d|  and  (BN + 4) u sum d^2

Rounding direction: half an ulp is what round-to-nearest is allowed, so a 16-bit output rounded the wrong way is
caught only up to 2x by the element bound.  rounding_bias() is the second check: over the elements whose fp32 part
e is below 1/4 ulp, the mean of (out - ref) sign(ref) / ulp(ref) is ~0 for round-to-nearest and -1/2 for truncation.
The accumulation itself does not lean: its mean normalised error (C - ref) / (u P) measured within +-0.006.

KAPPA is set from cuBLAS on the same operands (torch.mm on fp16 / bf16 tensors with an fp32 output and the
reduced-precision reductions disallowed, against float64).  Its worst normalised error |C - ref| / (u P) grows with K,
roughly as sqrt(K): 1.8 / 2.8 (bf16 / fp16) at K = 64, 4.4 / 6.1 at K = 768, 10.4 / 11.4 at K = 3072 (M = 513,
N = 3072), measured on an NVIDIA B200 at its 1000 W power limit.  The kernel's EPI_F32 output was bit-identical to
cuBLAS's at every one of those shapes.  KAPPA = 46, 4 x the worst (11.44), is one constant for every K, so it is
loosest at small K; test_gpu_gemm_edges.py::test_kappa_covers_cublas keeps it at least 2 x cuBLAS's error.
"""
import torch

U = 2.0 ** -24
KAPPA = 46.0
TANH_REL = 2.0 ** -10     # of |x|: 4 x the worst tanh.approx error times h = x / 2
GELU_SLOPE = 1.1            # max |d/dx x sigmoid(1.702 x)| = 1.0998
LN_EPS = 1e-5
RN_BIAS_TOL = 0.05          # |mean signed error| in ulps; truncation gives 0.5
RN_BIAS_MAX_E = 1.0 / 4     # elements whose fp32 part e is below this many ulps enter rounding_bias
RN_BIAS_MIN_COUNT = 4096

# (mantissa bits with the hidden one, exponent of the smallest normal)
_FMT = {torch.bfloat16: (8, -126), torch.float16: (11, -14)}
F16_MAX = 65504.0

EPILOGUES = ("BIAS_16", "BIAS_GELU_16", "BIAS_RESID_F32", "F32", "LNFOLD_16", "LNFOLD_GELU_16",
             "RESID_LNPREP_SHORT", "RESID_LNPREP_LONG")


def out16(epi):
    return epi in ("BIAS_16", "BIAS_GELU_16", "LNFOLD_16", "LNFOLD_GELU_16")


def is_gelu(epi):
    return epi in ("BIAS_GELU_16", "LNFOLD_GELU_16")


def is_fold(epi):
    return epi in ("LNFOLD_16", "LNFOLD_GELU_16")


def is_lnprep(epi):
    return epi in ("RESID_LNPREP_SHORT", "RESID_LNPREP_LONG")


def ulp(x, dtype):
    """ulp of the 16-bit format at |x| (float64 in, float64 out; 0 at x == 0)."""
    p, emin = _FMT[dtype]
    x = x.abs()
    _, e = torch.frexp(x)                     # x = m 2^e, m in [0.5, 1): floor(log2 x) = e - 1
    u = torch.ldexp(torch.ones_like(x), (e - p).clamp(min=emin + 1 - p))
    return torch.where(x > 0, u, torch.zeros_like(x))


def half_ulp(x, dtype):
    return 0.5 * ulp(x, dtype)


def qgelu(x):
    return x * torch.sigmoid(1.702 * x)       # reference jclip/model.py:27


def round16(y, dtype):
    """the epilogue's conversion: round to nearest; fp16 saturates at +-65504 (cvt.rn.satfinite)"""
    if dtype == torch.float16:
        y = y.clamp(-F16_MAX, F16_MAX)
    return y.to(dtype)


def abs_prod(A, B):
    return A.double().abs() @ B.double().abs().t()


def ln_scale(stats, K):
    """(r, -r mu) as the LNFOLD epilogue computes them in fp32 from the producer's partial sums stats [M, slots, 2]:
    su, sq summed over the slots in order, mean = su (1/K), var = max(fma(sq, 1/K, -mean^2), 0), r = 1 / sqrt(var + 1e-5).
    (The fma is formed in float64 and rounded once: exact but for a double rounding, which the 4 u term of
    the bound covers.)"""
    st = stats.float()
    su = st[:, 0, 0].clone()
    sq = st[:, 0, 1].clone()
    for i in range(1, st.shape[1]):
        su = su + st[:, i, 0]
        sq = sq + st[:, i, 1]
    inv_k = torch.tensor(1.0 / K, dtype=torch.float32, device=st.device)
    mean = su * inv_k
    var = (sq.double() * inv_k.double() - (mean * mean).double()).float().clamp(min=0.0)
    r = 1.0 / torch.sqrt(var + LN_EPS)
    return r, -mean * r


def row_stats(A):
    """(sum, sum of squares) per 256 columns of a 16-bit copy [M, K], in fp32: the LNFOLD consumer's stats input"""
    Af = A.float()
    return torch.stack([torch.stack([Af[:, k:k + 256].sum(-1), (Af[:, k:k + 256] ** 2).sum(-1)], -1)
                        for k in range(0, A.shape[1], 256)], 1)


def expect(epi, dtype, A, B, bias=None, old=None, stats=None, colsum=None, A2=None, B2=None):
    """(ref, e, x): the float64 result of epilogue `epi` on the kernel's operands, the fp32 part of its bound, and the
    pre-activation x (GELU forms; else None).  The full bound of a 16-bit output is e + half_ulp(|ref| + e)."""
    acc = A.double() @ B.double().t()
    P = abs_prod(A, B)
    if A2 is not None:
        acc = acc + A2.double() @ B2.double().t()
        P = P + abs_prod(A2, B2)
    b = bias.double() if bias is not None else torch.zeros(B.shape[0], dtype=torch.float64, device=A.device)
    if is_fold(epi):
        r, nmr = ln_scale(stats, A.shape[1])
        r, nmr = r.double()[:, None], nmr.double()[:, None]
        S = colsum.double()
        x = r * acc + nmr * S + b
        e = KAPPA * U * r * P + 4 * U * (r * P + nmr.abs() * S.abs() + b.abs())
    elif epi == "BIAS_RESID_F32" or is_lnprep(epi):
        x = old.double() + acc + b
        e = KAPPA * U * P + 4 * U * (P + b.abs() + old.double().abs())
    else:
        x = acc + b
        e = KAPPA * U * P + 4 * U * (P + b.abs())
    if is_gelu(epi):
        return qgelu(x), GELU_SLOPE * e + (TANH_REL + 2 * U) * x.abs(), x
    return x, e, None


def bound16(ref, e, dtype):
    return e + half_ulp(ref.abs() + e, dtype)


def excess(out, ref, bound):
    """max |out - ref| / bound (inf where out is not finite): <= 1 passes."""
    d = (out.double() - ref).abs()
    d = torch.where(torch.isfinite(d), d, torch.full_like(d, float("inf")))
    ratio = torch.where(d == 0, torch.zeros_like(d), d / bound)
    return float(ratio.max()) if d.numel() else 0.0


def rounding_bias(out, ref, e, dtype):
    """mean of (out - ref) sign(ref) / ulp(ref) over elements whose fp32 part e is below RN_BIAS_MAX_E ulp; None when
    fewer than RN_BIAS_MIN_COUNT elements qualify."""
    u16 = ulp(ref, dtype)
    keep = (u16 > 0) & (e < RN_BIAS_MAX_E * u16)
    if dtype == torch.float16:
        keep &= ref.abs() < F16_MAX
    if int(keep.sum()) < RN_BIAS_MIN_COUNT:
        return None
    s = ((out.double() - ref) * torch.sign(ref) / u16)[keep]
    return float(s.mean())


def shift_expect(stats_in, shift_in, N):
    """(shift, bound) of the LNPREP producer's shift_out rows: shift_in + sum(stats_in[:, :, 0]) / N."""
    su = stats_in[:, :, 0].double()
    slots = stats_in.shape[1]
    ref = shift_in.double() + su.sum(-1) / N
    return ref, (slots + 2) * U * (shift_in.double().abs() + su.abs().sum(-1) / N)


def copy_expect(x, shift, dtype):
    """(ref, bound) of the LNPREP 16-bit copy from the kernel's own residual x [M, N] and shift [M]."""
    d = x.double() - shift.double()[:, None]
    return d, U * d.abs() + half_ulp(d.abs() * (1 + U), dtype)


def stats_expect(x, shift, BN):
    """(sum, sumsq, bound_sum, bound_sumsq) per BN block [M, N / BN] from the kernel's own residual and shift."""
    d = x.double() - shift.double()[:, None]
    M, N = d.shape
    blk = d.view(M, N // BN, BN)
    return (blk.sum(-1), (blk * blk).sum(-1), (BN + 1) * U * blk.abs().sum(-1), (BN + 4) * U * (blk * blk).sum(-1))
