"""CPU: the GEMM bounds of _gemm_bounds.py (used by test_gpu_gemm_edges.py) have power.  An fp32 emulation of the
kernel's arithmetic (csrc/gemm.cu: fp32 accumulation one UMMA_K = 16 step at a time, the epilogues' fp32 operations
and 16-bit conversions, tanh.approx at its documented worst relative error 2^-10.987) is compared with the float64
reference at a few small shapes:

  - the correct emulation stays at least 3 x inside every bound's fp32 part, and within the full bound (half an ulp is
    exactly what round-to-nearest may use, so the rounded output has no 3 x margin there; its rounding is held by
    the rounding-bias check instead, which the correct emulation meets with 3 x to spare);
  - each plausible mistake below, substituted for the correct step, moves the result by at least 3 x its bound (the
    element bound, or for the rounding direction the rounding-bias check; the element bound sees a wrong rounding
    direction only up to 2 x, held here at 1.5 x).
"""
import math

import pytest
import torch

import _gemm_bounds as gb

MISTAKES = ("drop_last_kblock", "drop_last_kblock2", "bias_shift", "truncate16", "bf16_partial", "erf_gelu",
            "ln_wrong_slot", "ln_no_clamp", "swap_halves", "stats_slot_per_256")
TANH_APPROX_REL = 2.0 ** -10.987


def _f32(x):
    return x.to(torch.float32)


def _fma(a, b, c):
    """fp32 fused multiply-add: exact in float64 but for a double rounding"""
    return (a.double() * b.double() + c.double()).float()


def _acc(A, B, A2=None, B2=None, mistake=None):
    M, N = A.shape[0], B.shape[0]
    pairs = [(A[:, k:k + 64], B[:, k:k + 64]) for k in range(0, A.shape[1], 64)]
    if mistake == "drop_last_kblock":
        pairs = pairs[:-1]
    if A2 is not None:
        p2 = [(A2[:, k:k + 64], B2[:, k:k + 64]) for k in range(0, A2.shape[1], 64)]
        pairs += p2[:-1] if mistake == "drop_last_kblock2" else p2
    acc = torch.zeros(M, N, dtype=torch.float32)
    for a, b in pairs:
        for k in range(0, 64, 16):
            acc = acc + a[:, k:k + 16].float() @ b[:, k:k + 16].float().t()
        if mistake == "bf16_partial":
            acc = acc.bfloat16().float()
    if mistake == "swap_halves":
        perm = torch.arange(M)
        full = (M // 256) * 256
        perm[:full] = perm[:full] ^ 128
        acc = acc[perm]
    return acc


def _round16(y, dtype, mistake=None):
    t = gb.round16(y, dtype)
    if mistake == "truncate16":
        bits = t.view(torch.int16)
        t = torch.where(t.float().abs() > y.abs(), bits - 1, bits).view(dtype)
    return t


def _gelu32(x, mistake=None):
    if mistake == "erf_gelu":
        return _f32(0.5 * x.double() * (1 + torch.erf(x.double() / math.sqrt(2))))
    h = x * 0.5
    t = x * torch.tensor(0.851, dtype=torch.float32)
    sign = 1.0 - 2.0 * (torch.arange(x.numel()).view(x.shape) % 2)
    th = _f32(torch.tanh(t.double()) * (1 + TANH_APPROX_REL * sign))
    return _fma(h, th, h)


def _ln_scale(stats, K, mistake=None):
    if mistake == "ln_wrong_slot":
        stats = stats[:, :1]
    if mistake != "ln_no_clamp":
        return gb.ln_scale(stats, K)
    st = stats.float()
    su, sq = st[:, 0, 0].clone(), st[:, 0, 1].clone()
    for i in range(1, st.shape[1]):
        su, sq = su + st[:, i, 0], sq + st[:, i, 1]
    inv_k = torch.tensor(1.0 / K, dtype=torch.float32)
    mean = su * inv_k
    var = (sq.double() * inv_k.double() - (mean * mean).double()).float()
    r = 1.0 / torch.sqrt(var + gb.LN_EPS)
    return r, -mean * r


def emulate(epi, dtype, A, B, bias=None, old=None, stats=None, colsum=None, A2=None, B2=None, stats_in=None,
            shift_in=None, mistake=None):
    """(pre, out, extra): the kernel's fp32 result before the 16-bit conversion, its output, and for LNPREP a dict of
    copy / stats / shift"""
    N = B.shape[0]
    acc = _acc(A, B, A2, B2, mistake)
    b = bias.float() if bias is not None else torch.zeros(N)
    if mistake == "bias_shift":           # one column off inside each 32-column chunk
        n = torch.arange(N)
        b = b[(n // 32) * 32 + (n % 32 + 1) % 32]
    if gb.is_fold(epi):
        r, nmr = _ln_scale(stats, A.shape[1], mistake)
        bb = _fma(nmr[:, None], colsum.float()[None], b[None])
        x = _fma(acc, r[:, None], bb)
    elif epi == "BIAS_RESID_F32" or gb.is_lnprep(epi):
        x = old.float() + (acc + b)
    else:
        x = acc + b
    if gb.is_gelu(epi):
        x = _gelu32(x, mistake)
    if gb.out16(epi):
        return x, _round16(x, dtype, mistake), None
    if not gb.is_lnprep(epi):
        return x, x, None
    M = x.shape[0]
    shift = torch.zeros(M)
    if stats_in is not None:
        su = stats_in[:, 0, 0].float().clone()
        for i in range(1, stats_in.shape[1]):
            su = su + stats_in[:, i, 0].float()
        shift = shift_in.float() + su / torch.tensor(float(N))
    f = x - shift[:, None]
    BN = 256 if N % 256 == 0 else 128
    nb = N // BN
    st = torch.zeros(M, nb, 2)
    for j in range(nb):
        rs, rq = torch.zeros(M), torch.zeros(M)
        for c in range(BN):
            v = f[:, j * BN + c]
            rs, rq = rs + v, _fma(v, v, rq)
        slot = j * BN // 256 if mistake == "stats_slot_per_256" else j
        st[:, slot, 0], st[:, slot, 1] = rs, rq
    return x, x, {"copy": _round16(f, dtype, mistake), "stats": st, "shift": shift, "BN": BN}


def _inputs(epi, dtype, M, N, K, K2=0, seed=0, degenerate=False):
    g = torch.Generator().manual_seed(seed)
    new = lambda *s: torch.randn(*s, generator=g)
    kw = {}
    if gb.is_fold(epi):
        A = (new(M, K) + 0.3 * new(M, 1)).to(dtype)
        if degenerate:                    # every third row constant: var = 0 up to rounding, or below it
            A[::3] = new(M, 1)[::3].to(dtype).expand(-1, K)
        st = gb.row_stats(A)
        if degenerate:
            st[1::6, :, 1] *= 1 - 2.0 ** -10       # sq a hair short of K a^2 on some rows (var < 0 before the clamp)
            st[2::6, :, 1] = 0.0                  # and far short on others
        kw.update(stats=st)
    else:
        A = new(M, K).to(dtype)
    B = (new(N, K) * K ** -0.5).to(dtype)
    kw["bias"] = 0.5 * new(N)
    if gb.is_gelu(epi):
        kw["bias"] = kw["bias"] + torch.linspace(-6, 6, N)
    if gb.is_fold(epi):
        kw["colsum"] = B.float().sum(1) + 0.05 * new(N)
    if K2:
        kw.update(A2=(0.5 * new(M, K2)).to(dtype), B2=(new(N, K2) * K2 ** -0.5).to(dtype))
    if epi == "BIAS_RESID_F32" or gb.is_lnprep(epi):
        kw["old"] = 2 * new(M, N) + new(M, 1)
    lnprep = {}
    if gb.is_lnprep(epi):
        slots = N // (256 if N % 256 == 0 else 128)
        lnprep = dict(stats_in=torch.stack([16 * new(M, slots), 256 + 10 * new(M, slots).abs()], -1), shift_in=new(M))
    return A, B, kw, lnprep


def _ratios(epi, dtype, A, B, kw, lnprep, mistake=None):
    """{check: (worst error / bound of the emulation, kind)} for one emulated call; kind 'element' or 'bias'"""
    ref, e, _ = gb.expect(epi, dtype, A, B, **kw)
    ekw = dict(kw)
    pre, out, extra = emulate(epi, dtype, A, B, **ekw, **lnprep, mistake=mistake)
    res = {}
    if gb.out16(epi):
        res["fp32 part"] = gb.excess(pre, ref, e)
        res["element"] = gb.excess(out, ref, gb.bound16(ref, e, dtype))
        rb = gb.rounding_bias(out, ref, e, dtype)
        if rb is not None and not gb.is_gelu(epi):
            res["rounding bias"] = abs(rb) / gb.RN_BIAS_TOL
    else:
        res["element"] = gb.excess(out, ref, e)
    if extra is not None:
        if lnprep:
            want, b = gb.shift_expect(lnprep["stats_in"], lnprep["shift_in"], B.shape[0])
            res["shift"] = gb.excess(extra["shift"], want, b)
        d, b = gb.copy_expect(out, extra["shift"], dtype)
        res["copy"] = gb.excess(extra["copy"], d, b)
        rb = gb.rounding_bias(extra["copy"], d, gb.U * d.abs(), dtype)
        if rb is not None:
            res["copy rounding bias"] = abs(rb) / gb.RN_BIAS_TOL
        s1, s2, b1, b2 = gb.stats_expect(out, extra["shift"], extra["BN"])
        res["stats"] = max(gb.excess(extra["stats"][..., 0], s1, b1), gb.excess(extra["stats"][..., 1], s2, b2))
    return res


OPS = [torch.bfloat16, torch.float16]
IDS = ["bf16", "f16"]
SHAPES = [(300, 384, 320, 0), (512, 256, 768, 128)]


@pytest.mark.parametrize("op", OPS, ids=IDS)
@pytest.mark.parametrize("epi", gb.EPILOGUES)
def test_correct_emulation_inside_bounds(epi, op):
    """the fp32 part of every bound is >= 3 x the correct emulation's error; rounded outputs stay within the bound"""
    for i, (M, N, K, K2) in enumerate(SHAPES):
        if gb.is_fold(epi) or gb.is_lnprep(epi):
            K2 = 0
        A, B, kw, lnprep = _inputs(epi, op, M, N, K, K2, seed=i, degenerate=gb.is_fold(epi))
        for check, v in _ratios(epi, op, A, B, kw, lnprep).items():
            limit = 1.0 if check in ("element", "copy") and (gb.out16(epi) or check == "copy") else 1 / 3
            print(f"{epi} {check}: {v:.3f}")
            assert v <= limit, (epi, check, (M, N, K, K2), v)


# mistake -> [(epilogue, operand type, check that must see it, power it must reach)]
POWER = {
    "drop_last_kblock": [(e, t, "element", 3) for e in gb.EPILOGUES for t in OPS],
    "drop_last_kblock2": [(e, t, "element", 3) for e in ("BIAS_16", "BIAS_RESID_F32", "F32") for t in OPS],
    "bias_shift": [(e, t, "element", 3) for e in gb.EPILOGUES for t in OPS],
    "truncate16": [(e, t, c, p) for e in ("BIAS_16", "LNFOLD_16") for t in OPS
                   for c, p in (("rounding bias", 3), ("element", 1.5))] +
                  [(e, t, c, p) for e in ("RESID_LNPREP_SHORT",) for t in OPS
                   for c, p in (("copy rounding bias", 3), ("copy", 1.5))],
    "bf16_partial": [(e, t, "element", 3) for e in ("F32", "BIAS_RESID_F32", "RESID_LNPREP_LONG") for t in OPS] +
                    [("BIAS_16", torch.float16, "element", 3)],
    "erf_gelu": [(e, t, "element", 3) for e in ("BIAS_GELU_16", "LNFOLD_GELU_16") for t in OPS],
    "ln_wrong_slot": [(e, t, "element", 3) for e in ("LNFOLD_16", "LNFOLD_GELU_16") for t in OPS],
    "ln_no_clamp": [(e, t, "element", 3) for e in ("LNFOLD_16", "LNFOLD_GELU_16") for t in OPS],
    "swap_halves": [(e, t, "element", 3) for e in gb.EPILOGUES for t in OPS],
    "stats_slot_per_256": [("RESID_LNPREP_SHORT", t, "stats", 3) for t in OPS],
}


@pytest.mark.parametrize("mistake", MISTAKES)
def test_mistakes_exceed_bounds(mistake):
    """each mistake moves its result by >= `power` x the bound of the check that must see it"""
    weak = []
    for epi, op, check, power in POWER[mistake]:
        N = 384 if mistake == "stats_slot_per_256" else 256
        M, K, K2 = 512, 768, 128 if mistake == "drop_last_kblock2" else 0
        A, B, kw, lnprep = _inputs(epi, op, M, N, K, K2, seed=7, degenerate=gb.is_fold(epi))
        v = _ratios(epi, op, A, B, kw, lnprep, mistake).get(check, 0.0)
        print(f"{mistake} {epi} {op}: {check} {v:.2f}")
        if not v >= power:
            weak.append((epi, str(op), check, v))
    assert not weak, weak
