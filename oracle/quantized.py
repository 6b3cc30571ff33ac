"""Oracle with operand rounding: the fp32 tower of oracle/vit.py with the GEMM operands rounded to bf16 or
fp16 at exactly the points where the CUDA schedule rounds them (the folded schedule).  TEST INFRASTRUCTURE ONLY.

Purpose: attribute the end-to-end logit deviation of the tensor-core path (VERDICT r01 "what's weak" 1) without
GPU time.  Accumulation stays fp32 (as in TMEM); only what the kernels store as 16-bit operands is rounded:

  patches (im2col output) and conv1 weight                                            csrc/rowwise.cu im2col_kernel
  the raw copy of the residual stream the LayerNorm-folded GEMMs consume               csrc/gemm.cu EPI_RESID_LNPREP_*
  the gamma-folded in_proj / c_fc weights (LoRA merged in fp32 first), out_proj, c_proj csrc/rowwise.cu fold_ln
  q | k | v, the un-normalised softmax numerator P, the attention output, the MLP hidden  csrc/attention_tc.cu, gemm.cu

`act` / `wgt` select the rounding of activations and of weights independently ("f32" = none), which separates
the systematic part of the error (weights: identical for every view) from the per-view part (activations).
Follows jclip/model.py:59-62, :104-126 and test.py:388-398 like oracle/vit.py.
"""
import math

import torch

from .vit import _t, clip_normalize, merge_lora_into_state_dict

_DT = {"bf16": torch.bfloat16, "f16": torch.float16}


def _q(x, kind):
    if kind == "f32":
        return x
    return x.to(_DT[kind]).to(torch.float32)


@torch.no_grad()
def vit_encode_image_rounded(sd, images, lora=None, scaling=0.5, apply_clip_norm=True, normalize=True,
                             act="bf16", wgt="bf16", fold=True, centre=True, kinds=None, layer_kind=None,
                             lora_mode="merged"):
    """kinds: optional per-tensor-class overrides of `act` / `wgt`, e.g. {"hidden": "bf16"}; classes: patch, conv_w,
    ln1_copy, qkv_w, qkv, p, attn, out_w, ln2_copy, fc_w, hidden, proj_w (per-class attribution of the deviation).
    layer_kind: optional callable block index -> operand type of EVERY 16-bit tensor of that block (overrides act / wgt /
    kinds inside the blocks; per-layer attribution).
    fold: LayerNorm folded into the consuming GEMM (the folded schedule) instead of a rounded stand-alone LayerNorm.
    centre: the 16-bit copy of the residual row is x - shift, shift = the row's mean at the previous LayerNorm point
    (what the EPI_RESID_LNPREP_* epilogues write since round 2); False = the round-1 raw copy.
    lora_mode: "merged" (W + s B A in fp32, then rounded: api.cu Packer) or "applied" (jcb_ctx_set_lora_mode: base weights
    rounded un-merged, U = x [A_q; A_k; A_v]^T rounded to 16 bits, the projection accumulates U (s B)^T with s B rounded;
    stand-alone LayerNorm schedule, i.e. fold is ignored; test.py:388-398)."""
    x = _t(images)
    if apply_clip_norm:
        x = clip_normalize(x)
    rows = None
    applied = bool(lora) and lora_mode == "applied"
    if applied:
        fold = False
    elif lora:
        sd = merge_lora_into_state_dict(sd, lora, scaling)    # fp32 merge, then rounding (api.cu Packer)
    g = lambda k: _t(sd[k])
    conv_w = g("visual.conv1.weight")
    width, _, P, _ = conv_w.shape
    H = width // 64
    L = len([k for k in sd if k.startswith("visual.") and k.endswith(".attn.in_proj_weight")])
    eps = 1e-5

    kinds = dict(kinds or {})
    A = lambda name: kinds.get(name, act)      # activation classes
    Wk = lambda name: kinds.get(name, wgt)     # weight classes
    x = torch.nn.functional.conv2d(_q(x, A("patch")), _q(conv_w, Wk("conv_w")), bias=None, stride=P)
    x = x.reshape(x.shape[0], x.shape[1], -1).permute(0, 2, 1)
    cls = g("visual.class_embedding").view(1, 1, -1).expand(x.shape[0], 1, -1)
    x = torch.cat([cls, x], dim=1) + g("visual.positional_embedding")
    if "visual.VPT" in sd:
        x = torch.cat([x, g("visual.VPT").unsqueeze(0).expand(x.shape[0], -1, -1)], dim=1)

    def ln_stats(t):
        mean = t.mean(-1, keepdim=True)
        var = (t * t).mean(-1, keepdim=True) - mean * mean      # E[x^2] - E[x]^2 as the epilogue computes it
        return mean, 1.0 / torch.sqrt(var.clamp_min(0) + eps)

    state = {"shift": None}

    def ln_linear(t, gam, bet, W, b, a_kind, w_kind):
        """LN(t) @ W^T + b the way the folded GEMM computes it (or, fold=False, a rounded stand-alone LN)."""
        if not fold:
            mean, r = ln_stats(t)
            return _q((t - mean) * r * gam + bet, a_kind) @ _q(W, w_kind).t() + b
        Wf = _q(W * gam, w_kind)
        S = Wf.sum(-1)
        c = W @ bet + b
        if centre:
            shift = state["shift"] if state["shift"] is not None else t.mean(-1, keepdim=True)   # embed kernel: exact mean
            tc = t - shift
            state["shift"] = t.mean(-1, keepdim=True)          # = shift + mean of the centred copy: the next point's shift
        else:
            tc = t
        mean, r = ln_stats(tc)
        return r * (_q(tc, a_kind) @ Wf.t()) - r * mean * S + c

    mean, r = ln_stats(x)
    x = (x - mean) * r * g("visual.ln_pre.weight") + g("visual.ln_pre.bias")
    B, S_, W = x.shape
    base_A, base_W = A, Wk
    for i in range(L):
        if layer_kind is not None:
            A = Wk = (lambda name, k=layer_kind(i): k)
        else:
            A, Wk = base_A, base_W
        p = f"visual.transformer.resblocks.{i}."
        qkv = ln_linear(x, g(p + "ln_1.weight"), g(p + "ln_1.bias"), g(p + "attn.in_proj_weight"),
                        g(p + "attn.in_proj_bias"), A("ln1_copy"), Wk("qkv_w"))
        if applied:   # + U (s B)^T accumulated in the same fp32 tile; U = ln_1(x) A^T stored as a 16-bit operand
            mean1, r1 = ln_stats(x)
            u_in = _q((x - mean1) * r1 * g(p + "ln_1.weight") + g(p + "ln_1.bias"), A("ln1_copy"))
            delta = torch.zeros_like(qkv)
            for j, name in enumerate(("q_proj", "k_proj", "v_proj")):
                if name in lora[i]:
                    La, Lb = _t(lora[i][name][0]), _t(lora[i][name][1])
                    U = _q(u_in @ _q(La, Wk("qkv_w")).t(), A("qkv"))
                    delta[..., j * W:(j + 1) * W] = U @ _q(scaling * Lb, Wk("qkv_w")).t()
            qkv = qkv + delta
        qkv = _q(qkv, A("qkv"))
        q, k, v = (t.view(B, S_, H, 64).permute(0, 2, 1, 3) for t in qkv.split(W, dim=-1))
        s = (q @ k.transpose(-2, -1)) * (1.0 / math.sqrt(64))
        pnum = torch.exp(s - s.max(-1, keepdim=True).values)
        o = (_q(pnum, A("p")) @ v) / pnum.sum(-1, keepdim=True)     # P rounded, row sum in fp32
        o = _q(o.permute(0, 2, 1, 3).reshape(B, S_, W), A("attn"))
        x = x + o @ _q(g(p + "attn.out_proj.weight"), Wk("out_w")).t() + g(p + "attn.out_proj.bias")
        if applied and "proj" in lora[i]:
            La, Lb = _t(lora[i]["proj"][0]), _t(lora[i]["proj"][1])
            x = x + _q(o @ _q(La, Wk("out_w")).t(), A("attn")) @ _q(scaling * Lb, Wk("out_w")).t()
        h = ln_linear(x, g(p + "ln_2.weight"), g(p + "ln_2.bias"), g(p + "mlp.c_fc.weight"), g(p + "mlp.c_fc.bias"),
                      A("ln2_copy"), Wk("fc_w"))
        h = _q(h * torch.sigmoid(1.702 * h), A("hidden"))
        x = x + h @ _q(g(p + "mlp.c_proj.weight"), Wk("proj_w")).t() + g(p + "mlp.c_proj.bias")
    c0 = x[:, 0, :]
    mean, r = c0.mean(-1, keepdim=True), None
    var = ((c0 - mean) ** 2).mean(-1, keepdim=True)
    f = (c0 - mean) / torch.sqrt(var + eps) * g("visual.ln_post.weight") + g("visual.ln_post.bias")
    f = f @ g("visual.proj")
    if normalize:
        f = f / f.norm(dim=-1, keepdim=True)
    return f
