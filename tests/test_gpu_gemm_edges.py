"""GPU: the persistent CTA-pair tcgen05 GEMM (csrc/gemm.cu) through jcb_gemm at tile edges, at bench-scale tile
counts and with every fused epilogue, against float64 on the kernel's own 16-bit operands.  The bounds are derived
from the operation in _gemm_bounds.py (stated there once); test_gemm_bounds_cpu.py shows they have power.

  matrix       every epilogue x {bf16, fp16}: M in {1, 2, 127, 128, 129, 255, 256, 257, 511, 513} (the 128-row halves
               and 256-row tiles of a CTA pair), N in {128, 384} (BN = 128) and {256, 768, 2304, 3072} (BN = 256),
               K in {64, 320, 384, 768, 3072} (one k-block, about one ring of stages, the tower's K), paired so that
               every value of every axis meets every epilogue; bias = None in some cases of each; ldo = N or N + 64.
  second pair  K2 in {64, 128, 192} (C = A B^T + A2 B2^T) with ragged M, both BN forms.
  LNPREP       stats [m, n / BN] per BN block (BN = 128 gives N / 128 slots), shift_out, the centred 16-bit copy;
               stats_in_row_stride > 1 with ldo = T W, as the class-token-only last block calls it.
  LNFOLD       rows whose statistics give var <= 0 (constant rows, the clamp): the result is c[n], never NaN.
  GELU         pre-activations spanning [-20, 20].
  bench scale  M = 416,000 (128 images x 65 views x 50 tokens) at each tower shape with its epilogue: each CTA pair
               runs dozens of tiles through its ring and both TMEM accumulator stages.  Sampled rows against float64;
               row ranges at offsets that are not multiples of 128 bit-identical to a separate small call.
  guards       every output is [M + 67, ldo] filled with a sentinel (NaN for plain stores; a finite value where the
               epilogue reads what is there: the reduce-add and LNPREP residual); rows >= M and columns in [N, ldo)
               keep it bit for bit, as do stats / shift_out rows >= M, stats slots >= N / BN and the copy's rows >= M.
"""
import random

import pytest
import torch

import _gemm_bounds as gb

pytestmark = pytest.mark.gpu

OPS = [torch.bfloat16, torch.float16]
IDS = ["bf16", "f16"]
MS = [1, 2, 127, 128, 129, 255, 256, 257, 511, 513]
NS = [128, 384, 256, 768, 2304, 3072]
KS = [64, 320, 384, 768, 3072]
PAD_ROWS = 67
RESID_SENTINEL = 7.25
worst = {}      # (check, dtype) -> worst measured error / bound, printed at the end of the module


def _note(name, dtype, v):
    k = (name, IDS[OPS.index(dtype)])
    worst[k] = max(worst.get(k, 0.0), v)


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    for (name, op), v in sorted(worst.items()):
        print(f"gemm edges: worst error / bound  {name:34s} {op:5s} {v:.3f}")


def _bits(t):
    return t.view({torch.float32: torch.int32, torch.float16: torch.int16, torch.bfloat16: torch.int16}[t.dtype])


def _assert_untouched(buf, fill, what):
    """every element of `buf` still holds `fill`, bit for bit (NaN included)"""
    if buf.numel():
        ref = torch.full_like(buf, fill)
        assert torch.equal(_bits(buf), _bits(ref)), f"{what}: written past its extent"


def _guarded(M, N, ldo, dtype, fill, dev):
    return torch.full((M + PAD_ROWS, ldo), fill, dtype=dtype, device=dev)


def _check_guards(out, M, N, fill, what):
    _assert_untouched(out[M:], fill, f"{what} rows >= M")
    _assert_untouched(out[:M, N:], fill, f"{what} columns in [N, ldo)")


def _bn(N):
    return 256 if N % 256 == 0 else 128


def _check16(name, dtype, out, ref, e, gelu=False):
    b = gb.bound16(ref, e, dtype)
    ex = gb.excess(out, ref, b)
    _note(name, dtype, ex)
    assert ex <= 1.0, f"{name}: error {ex:.3f} x its bound"
    rb = gb.rounding_bias(out, ref, e, dtype)
    if rb is not None and not gelu:     # tanh.approx may lean either way; the element bound holds it
        assert abs(rb) <= gb.RN_BIAS_TOL, f"{name}: mean signed error {rb:+.3f} ulp (round to nearest: ~0)"


def _check32(name, dtype, out, ref, e):
    ex = gb.excess(out, ref, e)
    _note(name, dtype, ex)
    assert ex <= 1.0, f"{name}: error {ex:.3f} x its bound"


def _lnfold_inputs(M, N, K, dtype, g, dev):
    """a centred 16-bit copy with a small per-row offset, its (sum, sumsq) per 256 columns, S and c"""
    A = (torch.randn(M, K, generator=g) + 0.3 * torch.randn(M, 1, generator=g)).to(dtype).to(dev)
    return A, gb.row_stats(A)


def _run(jb, dev, epi, dtype, M, N, K, ldo, with_bias, seed, K2=0, lda2_pad=0, stats_in=True, extra_slot=False):
    """one jcb_gemm call on guarded outputs; checks the result against float64 and the guards"""
    C = jb._capi
    g = torch.Generator().manual_seed(seed)
    new = lambda *s: torch.randn(*s, generator=g)
    if gb.is_fold(epi):
        A, st = _lnfold_inputs(M, N, K, dtype, g, dev)
    else:
        A = new(M, K).to(dtype).to(dev)
    B = (new(N, K) * K ** -0.5).to(dtype).to(dev)
    bias = (0.5 * new(N)).to(dev) if with_bias else None
    kw = {}
    A2 = B2 = None
    if K2:
        A2f = (0.5 * new(M, K2 + lda2_pad)).to(dtype).to(dev)
        A2 = A2f[:, :K2]
        B2 = (new(N, K2) * K2 ** -0.5).to(dtype).to(dev)
        kw.update(A2=A2, B2=B2, K2=K2)
    if gb.is_fold(epi):
        S = (B.float().sum(1) + 0.05 * new(N).to(dev))
        kw.update(stats=st, colsum=S)
    resid_like = epi == "BIAS_RESID_F32" or gb.is_lnprep(epi)
    if resid_like:
        out = _guarded(M, N, ldo, torch.float32, RESID_SENTINEL, dev)
        old = (2 * new(M, N) + new(M, 1)).to(dev)
        out[:M, :N] = old
    else:
        out = _guarded(M, N, ldo, dtype if gb.out16(epi) else torch.float32, float("nan"), dev)
        old = None
    if gb.is_lnprep(epi):
        BN = _bn(N)
        slots = N // BN + (1 if extra_slot else 0)
        copy = _guarded(M, N, N, dtype, float("nan"), dev)
        stats = torch.full((M + PAD_ROWS, slots, 2), float("nan"), device=dev)
        kw.update(stats=stats, out2=copy)
        if stats_in:
            st_in = torch.stack([16 * new(M, slots), 256 + 10 * new(M, slots).abs()], -1).to(dev)
            sh_in = new(M).to(dev)
            shift = torch.full((M + PAD_ROWS,), float("nan"), device=dev)
            kw.update(stats_in=st_in, shift_in=sh_in, shift_out=shift)
    jb.blocks.gemm(A, B, out, getattr(C, "EPI_" + epi), bias=bias, ldo=ldo, **kw)

    ref, e, _ = gb.expect(epi, dtype, A, B, bias=bias, old=old, stats=kw.get("stats") if gb.is_fold(epi) else None,
                          colsum=kw.get("colsum"), A2=A2, B2=B2)
    y = out[:M, :N]
    if gb.out16(epi):
        _check16(epi, dtype, y, ref, e, gb.is_gelu(epi))
    else:
        _check32(epi, dtype, y, ref, e)
    if epi == "F32" and bias is None:     # the accumulation alone, in units of u P: what KAPPA has to cover (not a check)
        _note("F32 error / (u P), for KAPPA", dtype, gb.excess(y, ref, gb.U * gb.abs_prod(A, B) + 1e-30))
    _check_guards(out, M, N, RESID_SENTINEL if resid_like else float("nan"), "out")
    if gb.is_lnprep(epi):
        _check_lnprep(epi, dtype, y, kw, M, N, BN, slots)


def _check_lnprep(epi, dtype, x, kw, M, N, BN, slots, stride=1):
    """shift_out, the centred copy and the per-BN-block statistics of a LNPREP call whose new residual is x [M, N]"""
    if "stats_in" in kw:
        shift = kw["shift_out"][:M]
        want, b = gb.shift_expect(kw["stats_in"][::stride][:M], kw["shift_in"][::stride][:M], N)
        _check32("LNPREP shift_out", dtype, shift, want, b)
        _assert_untouched(kw["shift_out"][M:], float("nan"), "shift_out rows >= M")
    else:
        shift = torch.zeros(M, device=x.device)
    copy = kw["out2"]
    d, b = gb.copy_expect(x, shift, dtype)
    ex = gb.excess(copy[:M], d, b)
    _note("LNPREP copy", dtype, ex)
    assert ex <= 1.0, f"{epi} copy: error {ex:.3f} x its bound"
    rb = gb.rounding_bias(copy[:M], d, gb.U * d.abs(), dtype)
    assert rb is None or abs(rb) <= gb.RN_BIAS_TOL, f"{epi} copy: mean signed error {rb:+.3f} ulp"
    _assert_untouched(copy[M:], float("nan"), "copy rows >= M")
    st = kw["stats"]
    s1, s2, b1, b2 = gb.stats_expect(x, shift, BN)
    nb = N // BN
    _check32("LNPREP stats sum", dtype, st[:M, :nb, 0], s1, b1)
    _check32("LNPREP stats sumsq", dtype, st[:M, :nb, 1], s2, b2)
    _assert_untouched(st[M:], float("nan"), "stats rows >= M")
    _assert_untouched(st[:M, nb:], float("nan"), "stats slots >= N / BN")


def _matrix():
    cases = []
    for ei, epi in enumerate(gb.EPILOGUES):
        for i, M in enumerate(MS):
            N, K = NS[(i + ei) % len(NS)], KS[(i + 2 * ei) % len(KS)]
            ldo = N + 64 if (i + ei) % 2 else N
            with_bias = (i + ei) % 4 != 0
            opts = {}
            if gb.is_lnprep(epi):
                opts = dict(stats_in=i % 5 != 4, extra_slot=i % 3 == 1)
            cases.append(pytest.param(epi, M, N, K, ldo, with_bias, opts,
                                      id=f"{epi}-M{M}-N{N}-K{K}-ldo{ldo}" + ("" if with_bias else "-nobias")))
    return cases


@pytest.mark.parametrize("op", OPS, ids=IDS)
@pytest.mark.parametrize("epi,M,N,K,ldo,with_bias,opts", _matrix())
def test_epilogue_matrix(jb, cuda_dev, epi, M, N, K, ldo, with_bias, opts, op):
    _run(jb, cuda_dev, epi, op, M, N, K, ldo, with_bias, seed=M * 31 + N * 7 + K + len(epi), **opts)


def _k2_matrix():
    cases = []
    for epi in ("BIAS_16", "BIAS_RESID_F32", "F32"):
        for i in range(6):
            K2, N = (64, 128, 192)[i % 3], (384, 768)[i % 2]
            M, K = (1, 129, 255, 257, 513)[i % 5], (64, 768)[(i // 2) % 2]
            cases.append(pytest.param(epi, M, N, K, K2, i % 2, id=f"{epi}-M{M}-N{N}-K{K}-K2_{K2}" + ("-lda2pad" if i % 2 else "")))
    return cases


@pytest.mark.parametrize("op", OPS, ids=IDS)
@pytest.mark.parametrize("epi,M,N,K,K2,pad", _k2_matrix())
def test_second_operand_pair(jb, cuda_dev, epi, M, N, K, K2, pad, op):
    _run(jb, cuda_dev, epi, op, M, N, K, N + 64 * pad, True, seed=M + N + K2, K2=K2, lda2_pad=64 * pad)


@pytest.mark.parametrize("op", OPS, ids=IDS)
@pytest.mark.parametrize("epi", ["RESID_LNPREP_SHORT", "RESID_LNPREP_LONG"])
@pytest.mark.parametrize("n_views", [1, 129, 257])
def test_lnprep_class_token_rows(jb, cuda_dev, epi, n_views, op):
    """The class-token-only last block: M = views, the residual addressed as [views, T W] (ldo = T W, row v = class
    token of view v), stats_in / shift_in read at row v T.  The other tokens' columns are left untouched."""
    C = jb._capi
    d = cuda_dev
    T, W = 50, 768
    K = 768 if epi.endswith("SHORT") else 3072
    g = torch.Generator().manual_seed(n_views + K)
    new = lambda *s: torch.randn(*s, generator=g)
    M, N, ldo = n_views, W, T * W
    slots = N // 256
    A = new(M, K).to(op).to(d)
    B = (new(N, K) * K ** -0.5).to(op).to(d)
    bias = (0.5 * new(N)).to(d)
    tokens = (2 * new(M * T, W)).to(d)
    before = tokens.clone()
    view = tokens.view(M, ldo)
    old = view[:, :N].clone()
    st_in = torch.stack([16 * new(M * T, slots), 256 + 10 * new(M * T, slots).abs()], -1).to(d)
    sh_in = new(M * T).to(d)
    copy = _guarded(M, N, N, op, float("nan"), d)
    stats = torch.full((M + PAD_ROWS, slots, 2), float("nan"), device=d)
    shift = torch.full((M + PAD_ROWS,), float("nan"), device=d)
    kw = dict(stats=stats, out2=copy, stats_in=st_in, shift_in=sh_in, shift_out=shift)
    jb.blocks.gemm(A, B, view, getattr(C, "EPI_" + epi), bias=bias, ldo=ldo, stats_in_row_stride=T, **kw)
    ref, e, _ = gb.expect(epi, op, A, B, bias=bias, old=old)
    x = view[:, :N]
    _check32(epi, op, x, ref, e)
    assert torch.equal(view[:, N:], before.view(M, ldo)[:, N:]), "tokens other than the class token were written"
    _check_lnprep(epi, op, x, kw, M, N, 256, slots, stride=T)


@pytest.mark.parametrize("op", OPS, ids=IDS)
@pytest.mark.parametrize("epi", ["LNFOLD_16", "LNFOLD_GELU_16"])
def test_lnfold_degenerate_rows(jb, cuda_dev, epi, op):
    """Constant rows: the statistics give var = 0 up to rounding, var < 0 (sq a hair short of K a^2) or var = -a^2
    (sq = 0): the epilogue clamps var at 0, and r (acc - mu S) cancels to 0, so the output is c[n] up to the bound
    (quickgelu(c[n]) for the GELU form).  Without the clamp the last rows would be NaN."""
    C = jb._capi
    d = cuda_dev
    M, N, K = 260, 768, 768
    g = torch.Generator().manual_seed(17)
    a = torch.randn(M, generator=g).to(op).float()
    a[::13] = 0.0
    A = a[:, None].expand(M, K).to(op).contiguous().to(d)
    B = (torch.randn(N, K, generator=g) * K ** -0.5).to(op).to(d)
    S = B.double().sum(1).float()
    c = (0.5 * torch.randn(N, generator=g)).to(d)
    slots = K // 256
    st = torch.zeros(M, slots, 2)
    su, sq = K * a, K * a * a
    kind = torch.arange(M) % 3
    sq = torch.where(kind == 1, sq * (1 - 2.0 ** -10), torch.where(kind == 2, torch.zeros_like(sq), sq))
    st[:, 0, 0], st[:, 0, 1] = su / slots, sq / slots
    st[:, 1:, 0], st[:, 1:, 1] = (su / slots)[:, None], (sq / slots)[:, None]
    st = st.to(d)
    out = _guarded(M, N, N, op, float("nan"), d)
    jb.blocks.gemm(A, B, out, getattr(C, "EPI_" + epi), bias=c, stats=st, colsum=S)
    y = out[:M]
    assert torch.isfinite(y.float()).all()
    ref, e, _ = gb.expect(epi, op, A, B, bias=c, stats=st, colsum=S)
    _check16(epi + " var<=0", op, y, ref, e, gb.is_gelu(epi))
    want = gb.qgelu(c.double()) if gb.is_gelu(epi) else c.double()
    assert (ref - want[None]).abs().max() <= 1e-3 * want.abs().max()    # the reference itself is c[n]
    _check_guards(out, M, N, float("nan"), "out")


@pytest.mark.parametrize("op", OPS, ids=IDS)
@pytest.mark.parametrize("epi,N", [("BIAS_GELU_16", 2304), ("BIAS_GELU_16", 384), ("LNFOLD_GELU_16", 3072),
                                   ("LNFOLD_GELU_16", 128)])
def test_gelu_wide_range(jb, cuda_dev, epi, N, op):
    """pre-activations spanning [-20, 20]: bias (or c) sweeps the range across the columns"""
    C = jb._capi
    d = cuda_dev
    M, K = 257, 768
    g = torch.Generator().manual_seed(N)
    bias = torch.linspace(-20, 20, N).to(d)
    B = (torch.randn(N, K, generator=g) * K ** -0.5).to(op).to(d)
    kw = {}
    if gb.is_fold(epi):
        A, st = _lnfold_inputs(M, N, K, op, g, d)
        kw = dict(stats=st, colsum=B.float().sum(1))
    else:
        A = torch.randn(M, K, generator=g).to(op).to(d)
    out = _guarded(M, N, N, op, float("nan"), d)
    jb.blocks.gemm(A, B, out, getattr(C, "EPI_" + epi), bias=bias, **kw)
    ref, e, x = gb.expect(epi, op, A, B, bias=bias, **kw)
    assert x.min() < -19 and x.max() > 19
    _check16(epi + " [-20, 20]", op, out[:M], ref, e, True)
    _check_guards(out, M, N, float("nan"), "out")


# ---------------------------------------------------------------------------------------------- bench-scale tile counts
BENCH_M = 128 * 65 * 50
TOWER = [("qkv", 2304, 768, "LNFOLD_16"), ("out_proj", 768, 768, "RESID_LNPREP_SHORT"),
         ("c_fc", 3072, 768, "LNFOLD_GELU_16"), ("c_proj", 768, 3072, "RESID_LNPREP_LONG"), ("conv1", 768, 3072, "F32")]


def _sample_rows(M, seed):
    m_tiles = (M + 255) // 256
    rows = {t * 256 + o for t in (0, m_tiles // 2, m_tiles - 1) for o in (0, 127, 128, 255)}
    rng = random.Random(seed)
    rows |= {rng.randrange(M) for _ in range(300)}
    return torch.tensor(sorted(r for r in rows if r < M))


def _split_ranges(M):
    return [(37, 300), (M // 2 + 77, 389), (M - 301, 301)]


@pytest.mark.parametrize("op", OPS, ids=IDS)
@pytest.mark.parametrize("name,N,K,epi", TOWER, ids=[t[0] for t in TOWER])
def test_bench_scale(jb, cuda_dev, name, N, K, epi, op):
    C = jb._capi
    d = cuda_dev
    M = BENCH_M
    g = torch.Generator(device=d).manual_seed(N + K)
    gc = torch.Generator().manual_seed(N * K)
    A = torch.randn(M, K, device=d, generator=g)
    if gb.is_fold(epi):
        A += 0.3 * torch.randn(M, 1, device=d, generator=g)
    A = A.to(op)
    B = (torch.randn(N, K, generator=gc) * K ** -0.5).to(op).to(d)
    bias = None if epi == "F32" else (0.5 * torch.randn(N, generator=gc)).to(d)   # conv1 has no bias
    kw, old = {}, None
    if gb.is_fold(epi):
        kw["stats"] = gb.row_stats(A)
        kw["colsum"] = B.float().sum(1) + 0.05 * torch.randn(N, generator=gc).to(d)
    resid_like = gb.is_lnprep(epi)
    if resid_like:
        out = 2 * torch.randn(M, N, device=d, generator=g)
        slots = N // 256
        kw.update(out2=torch.empty(M, N, dtype=op, device=d), stats=torch.empty(M, slots, 2, device=d),
                  stats_in=torch.stack([16 * torch.randn(M, slots, device=d, generator=g),
                                        256 + 10 * torch.randn(M, slots, device=d, generator=g).abs()], -1),
                  shift_in=torch.randn(M, device=d, generator=g), shift_out=torch.empty(M, device=d))
    else:
        out = torch.empty(M, N, dtype=op if gb.out16(epi) else torch.float32, device=d)
    rows = _sample_rows(M, N + K).to(d)
    splits = _split_ranges(M)
    if resid_like:
        old = out[rows].clone()
        split_old = [out[r0:r0 + n].clone() for r0, n in splits]
    jb.blocks.gemm(A, B, out, getattr(C, "EPI_" + epi), bias=bias, **kw)

    # sampled rows against float64
    sub = lambda t: t[rows] if t is not None else None
    ref, e, _ = gb.expect(epi, op, sub(A), B, bias=bias, old=old, stats=sub(kw.get("stats")) if gb.is_fold(epi) else None,
                          colsum=kw.get("colsum"))
    if gb.out16(epi):
        _check16(f"bench {name}", op, out[rows], ref, e, gb.is_gelu(epi))
    else:
        _check32(f"bench {name}", op, out[rows], ref, e)
    if resid_like:
        kws = {k: sub(v) for k, v in kw.items() if k != "colsum"}
        _check_lnprep(epi, op, out[rows], kws, len(rows), N, 256, N // 256)

    # split invariance: rows [r0, r0 + n) of the big call == the same rows computed alone
    for j, (r0, n) in enumerate(splits):
        r1 = r0 + n
        kws = {}
        if gb.is_fold(epi):
            kws = dict(stats=kw["stats"][r0:r1].contiguous(), colsum=kw["colsum"])
        if resid_like:
            small = split_old[j]
            kws = dict(out2=torch.empty(n, N, dtype=op, device=d), stats=torch.empty(n, N // 256, 2, device=d),
                       stats_in=kw["stats_in"][r0:r1].contiguous(), shift_in=kw["shift_in"][r0:r1].contiguous(),
                       shift_out=torch.empty(n, device=d))
        else:
            small = torch.empty(n, N, dtype=out.dtype, device=d)
        jb.blocks.gemm(A[r0:r1], B, small, getattr(C, "EPI_" + epi), bias=bias, **kws)
        assert torch.equal(_bits(small), _bits(out[r0:r1])), f"rows [{r0}, {r1}) differ from the full call"
        if resid_like:
            for k in ("out2", "stats", "shift_out"):
                assert torch.equal(_bits(kws[k]), _bits(kw[k][r0:r1])), f"{k} rows [{r0}, {r1}) differ"


# ------------------------------------------------------------------------------------------------- calibration of KAPPA
@pytest.mark.parametrize("op", OPS, ids=IDS)
def test_kappa_covers_cublas(jb, cuda_dev, op):
    """KAPPA is at least 2 x cuBLAS's worst normalised accumulation error |C - ref| / (u |A| |B|^T) on operands of
    the shapes above (fp32 output, reduced-precision reductions disallowed).  It was set at ~4 x (_gemm_bounds.py)."""
    torch.backends.cuda.matmul.allow_fp16_reduced_precision_reduction = False
    torch.backends.cuda.matmul.allow_bf16_reduced_precision_reduction = False
    d = cuda_dev
    g = torch.Generator().manual_seed(3)
    w = 0.0
    for M, N, K in [(513, 3072, 3072), (513, 768, 768), (257, 2304, 768), (129, 384, 320), (511, 256, 64),
                    (513, 768, 3072)]:
        A = torch.randn(M, K, generator=g).to(op).to(d)
        B = (torch.randn(N, K, generator=g) * K ** -0.5).to(op).to(d)
        Cm = torch.mm(A, B.t(), out_dtype=torch.float32)
        ref = A.double() @ B.double().t()
        w = max(w, float(((Cm.double() - ref).abs() / (gb.U * gb.abs_prod(A, B))).max()))
    print(f"cuBLAS worst normalised error {IDS[OPS.index(op)]}: {w:.3f} (KAPPA {gb.KAPPA})")
    assert gb.KAPPA >= 2 * w
