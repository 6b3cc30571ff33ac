"""Python handles of the library's building-block entry points (include/jclip_b200.h, "building blocks"): the GEMM
with its fused epilogues, the LayerNorm-fold weight preparation, LayerNorm, attention and im2col on caller-owned
device tensors.  The towers never go through here (they are scheduled inside the library, csrc/api.cu); the parity
tests and tools/bench_kernel.py do, so that each kernel is held to its reference op in isolation
(reference jclip/model.py:17-21, :38-39, :59-62, :105-108; jclip/mha.py:55-83, :129-146, :461).
"""
import torch

from . import _capi
from ._capi import byref, check
from .runtime import get_context, ptr


def operand_code(dtype):
    if dtype == torch.float16:
        return _capi.OPERAND_F16
    if dtype == torch.bfloat16:
        return _capi.OPERAND_BF16
    raise TypeError(f"16-bit operands must be torch.float16 or torch.bfloat16, got {dtype}")


def _ctx(t):
    ctx = get_context(t.device)
    ctx.bind_current_stream()
    return ctx


def gemm(A, B, out, epilogue, bias=None, ldo=None, stats=None, colsum=None, out2=None, stats_in=None, shift_in=None,
         shift_out=None, stats_in_row_stride=1, sync=True, A2=None, B2=None, K2=None):
    """out (+)= A[M,K] @ B[N,K]^T (+ A2[:, :K2] @ B2[:, :K2]^T, accumulated in the same tile) with the fused epilogue
    `epilogue` (_capi.EPI_*)."""
    ctx = _ctx(A)
    g = _capi.GemmArgs()
    g.A_dev, g.B_dev = A.data_ptr(), B.data_ptr()
    g.M, g.K = A.shape
    g.N = B.shape[0]
    g.operand_type = operand_code(A.dtype)
    g.bias_dev = bias.data_ptr() if bias is not None else None
    g.epilogue = int(epilogue)
    g.out_dev = out.data_ptr()
    g.ldo = int(ldo) if ldo is not None else g.N
    if stats is not None:
        g.stats_dev = stats.data_ptr()
        g.stats_slots = stats.shape[1]
    g.colsum_dev = colsum.data_ptr() if colsum is not None else None
    g.out2_dev = out2.data_ptr() if out2 is not None else None
    g.stats_in_dev = stats_in.data_ptr() if stats_in is not None else None
    g.shift_in_dev = shift_in.data_ptr() if shift_in is not None else None
    g.shift_out_dev = shift_out.data_ptr() if shift_out is not None else None
    g.stats_in_row_stride = int(stats_in_row_stride)
    if A2 is not None:
        g.A2_dev, g.B2_dev = A2.data_ptr(), B2.data_ptr()
        g.K2 = int(K2) if K2 is not None else A2.shape[1]
        g.lda2, g.ldb2 = A2.stride(0), B2.stride(0)
    check(ctx.lib.jcb_gemm(ctx.handle, byref(g)), ctx.handle)
    if sync:
        ctx.sync()


def fold_ln(W, gamma, beta, bias, dtype):
    """(Wf [N,K] `dtype`, S [N], c [N]) of a LayerNorm-folded linear layer: LN(x) W^T + b = r (x Wf^T) - r mu S + c."""
    ctx = _ctx(W)
    N, K = W.shape
    Wf = torch.empty(N, K, dtype=dtype, device=W.device)
    S = torch.empty(N, dtype=torch.float32, device=W.device)
    c = torch.empty(N, dtype=torch.float32, device=W.device)
    check(ctx.lib.jcb_fold_ln(ctx.handle, ptr(W), ptr(gamma), ptr(beta), ptr(bias), N, K, operand_code(dtype), ptr(Wf),
                              ptr(S), ptr(c)), ctx.handle)
    ctx.sync()
    return Wf, S, c


def layernorm(x, gamma, beta, out):
    ctx = _ctx(x)
    check(ctx.lib.jcb_layernorm(ctx.handle, ptr(x), x.shape[0], x.shape[1], ptr(gamma), ptr(beta), operand_code(out.dtype),
                                ptr(out)), ctx.handle)
    ctx.sync()


def attention(qkv, n_views, tokens, heads, out, causal=False, sync=True):
    ctx = _ctx(qkv)
    check(ctx.lib.jcb_attention(ctx.handle, ptr(qkv), n_views, tokens, heads, int(bool(causal)), operand_code(qkv.dtype),
                                ptr(out)), ctx.handle)
    if sync:
        ctx.sync()


def mta_debug(feats, text, params=None):
    """jcb_mta_debug on feats [I, V, D] fp32 and text [D, C] fp32 (CUDA): the modes [I, D] and logits [I, C] of jcb_mta
    with the solver's state -- bandwidths [I, V], final inlierness weights y [I, V], affinity [I, V, V].  `params`: dict
    of jcb_mta_params fields to override (others keep the reference's constants)."""
    ctx = _ctx(feats)
    I, V, D = feats.shape
    C = text.shape[1]
    p = _capi.MtaParams()
    ctx.lib.jcb_mta_default_params(byref(p))
    for k, v in (params or {}).items():
        setattr(p, k, v)
    new = lambda *shape: torch.empty(shape, dtype=torch.float32, device=feats.device)
    out = {"mode": new(I, D), "logits": new(I, C), "bw": new(I, V), "y": new(I, V), "affinity": new(I, V, V)}
    check(ctx.lib.jcb_mta_debug(ctx.handle, ptr(feats), ptr(text), I, V, C, D, byref(p),
                                *(ptr(out[k]) for k in ("mode", "logits", "bw", "y", "affinity"))), ctx.handle)
    ctx.sync()
    return out


def im2col(images, resolution, patch, apply_clip_norm, out):
    from .runtime import img_dtype_code
    ctx = _ctx(images)
    check(ctx.lib.jcb_im2col(ctx.handle, ptr(images), img_dtype_code(images), images.shape[0], resolution, patch,
                             int(bool(apply_clip_norm)), operand_code(out.dtype), ptr(out)), ctx.handle)
    ctx.sync()
