"""GPU: the ViT-B/16 image tower (patch 16, 197 tokens; 201 with the four IVLP prompt tokens) and the long form of the
tcgen05 attention kernel it runs on (attention_tc.cu attention_tcgen05_long_kernel: 129 <= T <= 256, no mask), for
both 16-bit operand types.

Tolerances are the ones the ViT-B/32 files use:
  attention kernel : P is rounded to 16 bits before P V: 1e-2 (bf16) / 2e-3 (fp16) absolute + one ulp of the
                     reference (test_gpu_kernels.py), against torch fp32 on the same 16-bit operands
  tower            : embedding and token cosine >= 0.99999 (fp16) / 0.9995 (bf16) against the fp32 oracle
                     (test_gpu_tower.py, test_gpu_lnfold.py)
  pipeline         : logits within 1e-2 and top-5 agreement >= 99.5 % (fp16), 0.10 and 99 % / 97 % (bf16)
                     (test_gpu_fullsize.py::test_end_to_end_agreement_with_fp32_oracle)
The CPU file test_vit_b16_cpu.py shows that the attention tolerance is far below what the likely indexing mistakes of
the long kernel move the result by.
"""
import math
import os
import pickle
import re
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

OPS = [torch.bfloat16, torch.float16]
ULP = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}
ATOL = {torch.bfloat16: 1e-2, torch.float16: 2e-3}
IDS = ["bf16", "f16"]
COS_FLOOR = {"bf16": 0.9995, "f16": 0.99999}
GUARD_ROWS = 67


def _attention_ref(qkv, n_views, T, H, causal):
    d = 64
    x = qkv.float().view(n_views, T, 3, H, d)
    q, k, v = (x[:, :, i].permute(0, 2, 1, 3) for i in range(3))
    s = q @ k.transpose(-2, -1) / math.sqrt(d)                                # jclip/mha.py:55-83
    if causal:                                                                # jclip/model.py:189-193 build_attention_mask
        s = s + torch.triu(torch.full((T, T), float("-inf"), device=s.device), 1)
    return (torch.softmax(s, dim=-1) @ v).permute(0, 2, 1, 3).reshape(n_views * T, H * d)


def _run_attention(jb, qkv, n_seq, T, H):
    """The kernel's output, written into a NaN-filled buffer with an untouched guard region after it."""
    W = H * 64
    buf = torch.full((n_seq * T + GUARD_ROWS, W), float("nan"), dtype=qkv.dtype, device=qkv.device)
    jb.blocks.attention(qkv, n_seq, T, H, buf[:n_seq * T])
    assert torch.isnan(buf[n_seq * T:].float()).all(), "the kernel wrote past its output"
    out = buf[:n_seq * T]
    assert torch.isfinite(out.float()).all()
    return out


def _check(out, ref, op):
    err = (out.float() - ref).abs()
    assert (err <= ATOL[op] + ULP[op] * ref.abs()).all(), float(err.max())


# every T the long kernel distinguishes (one Q box of tile 1 and three K / V boxes up to 192, four above; partial and
# full last boxes), head counts 12 (ViT-B/16), 8, 3 and 1; n_seq up to 1500 so that each of the 296 persistent CTAs
# runs about 120 items
LONG_SHAPES = [(1, 129, 12), (40, 129, 1), (3, 160, 8), (5, 192, 3), (2, 193, 1), (1500, 197, 12), (11, 197, 3),
               (700, 201, 12), (4, 255, 8), (9, 256, 12), (300, 256, 3), (1, 256, 1)]


@pytest.mark.parametrize("op", OPS, ids=IDS)
@pytest.mark.parametrize("n_seq,T,H", LONG_SHAPES)
def test_long_attention_matches_fp32(jb, cuda_dev, n_seq, T, H, op):
    g = torch.Generator().manual_seed(n_seq * 1000 + T * 10 + H)
    qkv = (torch.randn(n_seq * T, 3 * H * 64, generator=g) * 1.2).to(op).to(cuda_dev)
    out = _run_attention(jb, qkv, n_seq, T, H)
    _check(out, _attention_ref(qkv, n_seq, T, H, False), op)


def _hard_inputs(kind, n_seq, T, H, g):
    x = torch.randn(n_seq, T, 3, H, 64, generator=g)
    if kind == "large":                  # q and k x 4: scores with a spread of ~16 (in units of the softmax's exponent)
        x[:, :, :2] *= 4.0               # (v stays at unit scale: the absolute tolerance is in units of v)
    elif kind == "dominant":             # key T - 1 (in the last key box) takes almost all of every row's weight
        u = torch.sign(torch.randn(64, generator=g))
        x[:, :, 0] = 0.3 * x[:, :, 0] + u
        x[:, :, 1] *= 0.3
        x[:, T - 1, 1] = 2.0 * u
        x[:, T - 1, 2] = 3.0 + x[:, T - 1, 2]
    elif kind == "equal":                # every key of a (sequence, head) is the same row: uniform weights
        x[:, :, 1] = x[:, :1, 1]
    return x.reshape(n_seq * T, 3 * H * 64)


@pytest.mark.parametrize("op", OPS, ids=IDS)
@pytest.mark.parametrize("kind", ["large", "dominant", "equal"])
@pytest.mark.parametrize("n_seq,T,H", [(64, 197, 12), (8, 160, 8), (5, 256, 3)])
def test_long_attention_hard_inputs(jb, cuda_dev, kind, n_seq, T, H, op):
    """Peaked rows (large scores), one key that takes almost all the weight (in the last key box) and rows of equal
    scores.  The error of P rounded to 16 bits scales with |v|: with v x 4 as well, bf16 reached 0.04-0.06 absolute on a
    B200 (fp16 stayed within its bar), which is why only q and k are scaled for the large-score case."""
    g =torch.Generator().manual_seed(T + H)
    qkv = _hard_inputs(kind, n_seq, T, H, g).to(op).to(cuda_dev)
    out = _run_attention(jb, qkv, n_seq, T, H)
    ref = _attention_ref(qkv, n_seq, T, H, False)
    _check(out, ref, op)
    if kind == "dominant":               # the inputs do what they claim
        v_last = qkv.float().view(n_seq, T, 3, H, 64)[:, T - 1, 2]          # [n_seq, H, 64]
        assert (ref.view(n_seq, T, H, 64) - v_last[:, None]).abs().max() < 0.05
    if kind == "equal":
        v_mean = qkv.float().view(n_seq, T, 3, H, 64)[:, :, 2].mean(1)     # [n_seq, H, 64]
        assert (ref.view(n_seq, T, H, 64) - v_mean[:, None]).abs().max() < 1e-4


ROUTES = [(64, 12, "attention_tcgen05_kernel<0,{},0>"), (50, 12, "attention_tcgen05_kernel<50,{},0>"),
          (128, 12, "attention_tcgen05_kernel<0,{},1>"), (129, 12, "attention_tcgen05_long_kernel<{}>"),
          (256, 12, "attention_tcgen05_long_kernel<{}>"), (197, 3, "attention_tcgen05_long_kernel<{}>")]


def test_routes_launch_the_expected_kernels(jb, cuda_dev):
    """T <= 128 keeps today's instantiations (two heads per tile at T <= 64, one head per tile up to 128); 129 and 256
    tokens run the long kernel.  All twelve launches are recorded in ONE profiler step and matched to the kernels by
    their start order: every launch must show up exactly once, under the expected name.

    The recorded step follows a warm-up step of the same launches (the profiler's schedule: tracing on, results
    discarded).  Without it the first launches of a session can go unrecorded: on a B200 the first two of these twelve
    (both T = 64) were missing from the list while the other ten came in order."""
    from torch.profiler import ProfilerActivity, profile, schedule
    cases = []
    for T, H, want in ROUTES:
        for op in OPS:
            qkv = torch.randn(4 * T, 3 * H * 64, device=cuda_dev).to(op)
            out = torch.empty(4 * T, H * 64, dtype=op, device=cuda_dev)
            jb.blocks.attention(qkv, 4, T, H, out)          # modules loaded and tensor maps encoded before the session
            cases.append((T, H, qkv, out, want.format("true" if op == torch.float16 else "false")))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA], schedule=schedule(wait=0, warmup=1, active=1, repeat=1)) as prof:
        for step in range(2):                               # 0: warm-up, 1: recorded
            for T, H, qkv, out, _ in cases:
                out.fill_(float("nan"))
                jb.blocks.attention(qkv, 4, T, H, out)
            torch.cuda.synchronize()
            prof.step()
    # every recorded launch ran: a missing name below is the profiler's, not a kernel that did not run
    assert all(torch.isfinite(c[3].float()).all() for c in cases)
    launched = []
    for e in prof.events():
        m = re.search(r"(attention_tcgen05_(?:long_)?kernel<[^>]*>)", e.name)
        if m and e.device_type == torch.autograd.DeviceType.CUDA:
            launched.append((e.time_range.start, m.group(1).replace(" ", "")))
    got = [name for _, name in sorted(launched)]
    want = [c[4] for c in cases]
    assert got == want, list(zip([(c[0], c[1]) for c in cases], want, got + [None] * (len(want) - len(got))))


@pytest.mark.parametrize("T,causal", [(129, True), (256, True), (257, False), (257, True)])
def test_unsupported_attention_is_rejected(jb, cuda_dev, T, causal):
    H = 2
    qkv = torch.zeros(T, 3 * H * 64, dtype=torch.float16, device=cuda_dev)
    out = torch.full((T, H * 64), float("nan"), dtype=torch.float16, device=cuda_dev)
    with pytest.raises(jb.JcbError) as e:
        jb.blocks.attention(qkv, 1, T, H, out, causal=causal)
    assert e.value.code == jb._capi.JCB_E_INVALID, str(e.value)
    assert torch.isnan(out.float()).all()


def test_tower_of_257_tokens_is_rejected(jb, cuda_dev):
    sd = jb.synth.make_vit_state_dict(seed=0, layers=1, patch=16, resolution=256)      # 16 x 16 + 1 = 257 tokens
    model = jb.jclip.build_model(sd)
    with pytest.raises(jb.JcbError, match=r"tokens=257 \(max 256\)") as e:
        model.encode_image(torch.zeros(1, 3, 256, 256, device=cuda_dev))
    assert e.value.code == jb._capi.JCB_E_INVALID


# ------------------------------------------------------------------------------------------------ tower vs oracle
def _cos(a, b):
    a, b = a.double(), b.double()
    return (a * b).sum(-1) / (a.norm(dim=-1) * b.norm(dim=-1))


def _set_lora(layers, lora):
    for i, layer in enumerate(layers):
        for name, (A, B) in lora[i].items():
            getattr(layer, name).w_lora_A.data = A
            getattr(layer, name).w_lora_B.data = B


def _lora_args(position="all"):
    return types.SimpleNamespace(encoder="vision", position=position, params=["q", "k", "v"], r=4, alpha=1,
                                 dropout_rate=0.25, backbone="ViT-B/16")


_oracle_cache = {}


def _tower_case(jb, case):
    """(state dict, LoRA or None, model, images [n, 3, 224, 224] in [0, 1], oracle embeddings, oracle tokens), built
    once per case: the oracle's cost does not depend on the operand type."""
    if case in _oracle_cache:
        return _oracle_cache[case]
    from oracle import vit_encode_image
    from oracle.vit import layer_norm
    vpt = 4 if case == "ivlp" else 0
    sd = jb.synth.make_vit_state_dict(seed=16, patch=16, vpt_tokens=vpt, trained_like="both" if case == "trained" else False)
    if vpt:
        sd["visual.VPT"] = sd["visual.VPT"] * 25.0          # make the prompt tokens count (0.5 instead of 0.02 std)
        model = jb.jclip.build_model(sd, dict(jb.clip.IVLP_DESIGN))
    else:
        model = jb.jclip.build_model(sd)
    lora = None
    if case in ("lora", "ivlp"):
        layers = jb.apply_lora(_lora_args(), model)
        lora = jb.synth.make_lora(seed=17, b_std=0.3)
        _set_lora(layers, lora)
    imgs = jb.synth.make_views(18, 1, 3).reshape(3, 3, 224, 224)
    torch.set_num_threads(os.cpu_count() or 1)
    ref_tok = vit_encode_image(sd, imgs, lora=lora, scaling=0.5, apply_clip_norm=True, return_tokens=True)
    t = lambda k: torch.from_numpy(np.asarray(sd[k]))
    ref = layer_norm(ref_tok[:, 0, :], t("visual.ln_post.weight"), t("visual.ln_post.bias")) @ t("visual.proj")
    ref = ref / ref.norm(dim=-1, keepdim=True)                # the oracle's tail (oracle/vit.py), on the same tokens
    _oracle_cache[case] = (sd, lora, model, imgs, ref, ref_tok)
    return _oracle_cache[case]


@pytest.mark.parametrize("op", ["f16", "bf16"])
@pytest.mark.parametrize("case,mode", [("zero_shot", "merged"), ("trained", "merged"), ("lora", "merged"),
                                       ("lora", "applied"), ("ivlp", "merged"), ("ivlp", "applied")])
def test_tower_matches_oracle(jb, cuda_dev, case, mode, op):
    """Embeddings and the residual stream of every token after the last block against the fp32 oracle."""
    sd, lora, model, imgs, ref, ref_tok = _tower_case(jb, case)
    T = 201 if case == "ivlp" else 197
    assert model.visual.patch_size == 16 and model.visual.input_resolution == 224 and model.visual.heads == 12
    ctx = jb.get_context(cuda_dev)
    prev_op, prev_mode = ctx.operand_type, ctx.lora_mode
    x = torch.from_numpy(imgs).to(cuda_dev)
    try:
        ctx.set_operand_type(op)
        ctx.set_lora_mode(mode)
        out = model.visual(x, apply_clip_norm=True, normalize=True).cpu()
        tok = model.visual.debug_tokens(x, apply_clip_norm=True).cpu()
    finally:
        ctx.set_operand_type(prev_op)
        ctx.set_lora_mode(prev_mode)
    assert tok.shape == ref_tok.shape == (3, T, 768)
    cos_e, cos_t = _cos(out, ref).min().item(), _cos(tok.reshape(-1, 768), ref_tok.reshape(-1, 768)).min().item()
    print(f"{case} {mode} {op}: embedding cosine {cos_e:.8f}, token cosine {cos_t:.8f}")
    assert cos_e >= COS_FLOOR[op], cos_e
    assert cos_t >= COS_FLOOR[op], cos_t


def test_pass_split_and_host_input(jb, cuda_dev):
    """The default pass bound gives a 197-token tower 16384 * 64 / 197 = 5322 views; a small bound splits the call into
    several passes with bit-identical results, and host input equals device input."""
    sd, lora, model, _, _, _ = _tower_case(jb, "lora")
    x = jb.synth.make_views_torch(19, 1, 23, cuda_dev)[0]                     # [23, 3, 224, 224]
    ctx = jb.get_context(cuda_dev)
    prev = ctx.chunk_views, ctx.host_chunk_views
    ctx.set_chunk_views(16384)                                                # the library's default
    try:
        one = model.visual(x, apply_clip_norm=True, normalize=True).cpu()
        ctx.set_chunk_views(24)                                               # 24 * 64 / 197 = 7 views: 4 passes
        split = model.visual(x, apply_clip_norm=True, normalize=True).cpu()
        ctx.set_host_chunk_views(20)                                          # 20 * 64 / 197 = 6 views per host pass
        host = model.visual(x.cpu().pin_memory(), apply_clip_norm=True, normalize=True)
    finally:
        ctx.set_chunk_views(prev[0])
        ctx.set_host_chunk_views(prev[1])
    assert torch.equal(split, one)
    assert not host.is_cuda and torch.equal(host, one)


def test_cls_only_option_has_no_effect(jb, cuda_dev):
    """The class-token-only last block applies to towers of up to 64 tokens; on ViT-B/16 the option changes nothing."""
    sd, lora, model, _, _, _ = _tower_case(jb, "lora")
    x = jb.synth.make_views_torch(20, 1, 9, cuda_dev)[0]
    ctx = jb.get_context(cuda_dev)
    off = model.visual(x, apply_clip_norm=True, normalize=True).cpu()
    try:
        ctx.set_cls_only_last_block(True)
        on = model.visual(x, apply_clip_norm=True, normalize=True).cpu()
    finally:
        ctx.set_cls_only_last_block(False)
    assert torch.equal(on, off)


# ------------------------------------------------------------------------------------------------ whole pipeline
E2E_BOUNDS = {"f16": {"dlogit": 1e-2, "cs1": 0.995, "cs5": 0.995}, "bf16": {"dlogit": 0.10, "cs1": 0.99, "cs5": 0.97}}


@pytest.fixture(scope="module")
def b16_pipeline(jb):
    """LoRA ViT-B/16 tower, its fp32 oracle embeddings for 6 images x 9 views and 1 image x 65 views (119 oracle views),
    random text banks and head."""
    from oracle import vit_encode_image
    torch.set_num_threads(os.cpu_count() or 1)
    sd = jb.synth.make_vit_state_dict(seed=21, patch=16)
    model = jb.jclip.build_model(sd)
    layers = jb.apply_lora(_lora_args(), model)
    lora = jb.synth.make_lora(seed=22, b_std=0.05)
    _set_lora(layers, lora)
    sd_t = {k: torch.from_numpy(v) for k, v in sd.items()}
    data = {}
    for I, V in [(6, 9), (1, 65)]:
        imgs = jb.synth.make_views(23, I, V)
        feats = torch.stack([vit_encode_image(sd_t, imgs[i], lora=lora, scaling=0.5, apply_clip_norm=True, normalize=True)
                             for i in range(I)])
        data[(I, V)] = (imgs, feats)
    Ts = [torch.from_numpy(jb.synth.make_text_features(seed=30 + i)) for i in range(3)]
    lp_np = jb.synth.make_head(2, Ts[2].numpy())
    return model, data, Ts, lp_np


@pytest.mark.parametrize("op", ["f16", "bf16"])
def test_pipeline_matches_oracle(jb, cuda_dev, b16_pipeline, op):
    """HotPath.evaluate_base on the ViT-B/16 tower against oracle tower -> oracle MTA x3 -> oracle head."""
    from oracle import pipeline_image
    model, data, Ts, lp_np = b16_pipeline
    lp_t = tuple(torch.from_numpy(a) for a in lp_np)
    lp = jb.Channel_LP()
    lp.scale1.data, lp.bias1.data, lp.fc.weight.data, lp.fc.bias.data = lp_np
    ctx = jb.get_context(cuda_dev)
    prev = ctx.operand_type
    res = []
    try:
        ctx.set_operand_type(op)
        for (I, V), (imgs, ref_feats) in data.items():
            for rank_by in ("cs5", "cs1"):
                hp = jb.HotPath(model, jb.TextBank(Ts[0], Ts[1], Ts[2], cuda_dev), lp, rank_by=rank_by)
                topk, feats, scores = hp.evaluate_base(torch.from_numpy(imgs).to(cuda_dev), return_feats=True,
                                                       return_scores=True)
                topk, feats, scores = topk.cpu(), feats.cpu(), scores.cpu()
                agree, cos_min, dlogit = 0, 1.0, 0.0
                for i in range(I):
                    f = ref_feats[i]
                    cos_min = min(cos_min, float(_cos(feats[i], f).min()))
                    t5, sc, _ = pipeline_image(f, f, Ts[0], Ts[1], Ts[2], lp_t, score=rank_by)
                    dlogit = max(dlogit, float((scores[i] - sc[rank_by][0]).abs().max()))
                    agree += len(set(t5.tolist()) & set(topk[i].tolist()))
                res.append({"images": I, "views": V, "rank_by": rank_by, "min_embedding_cosine": cos_min,
                            "max_abs_logit_diff": dlogit, "top5_label_agreement": agree / (5 * I)})
    finally:
        ctx.set_operand_type(prev)
    print(op, res)
    b = E2E_BOUNDS[op]
    for r in res:
        assert r["min_embedding_cosine"] >= 0.999, res
        assert r["max_abs_logit_diff"] <= b["dlogit"], res
        assert r["top5_label_agreement"] >= b[r["rank_by"]], res


def _img(rng, h, w):
    return (rng.random((h, w, 3)) * 255).astype(np.uint8)


def test_clip_load_and_image_stream(jb, cuda_dev, tmp_path):
    """A ViT-B/16 checkpoint through clip.load, encode_image against the oracle, and the image stream with views generated
    as patch-16 patch matrices (TTAViews(emit="patches", patch=16)) equal to evaluate_base on uint8 views."""
    from oracle import vit_encode_image
    sd = jb.synth.make_vit_state_dict(seed=24, layers=2, patch=16)
    p = tmp_path / "ViT-B-16.pkl"
    with open(p, "wb") as f:
        pickle.dump(sd, f, protocol=4)
    model = jb.clip.load(str(p))[0]
    assert model.visual.patch_size == 16
    imgs = jb.synth.make_views(25, 1, 2).reshape(2, 3, 224, 224)
    out = model.encode_image(torch.from_numpy(jb.synth.clip_normalize(imgs)).to(cuda_dev)).cpu()
    ref = vit_encode_image(sd, jb.synth.clip_normalize(imgs))
    assert _cos(out, ref).min() >= COS_FLOOR[jb.get_context(cuda_dev).operand_type]
    rng = np.random.default_rng(26)
    batches = [[_img(rng, 300 + 7 * i, 400 - 5 * i) for i in range(n)] for n in (3, 2, 1)]
    Ts = [torch.from_numpy(jb.synth.make_text_features(seed=10 + i)) for i in range(3)]
    lp = jb.Channel_LP()
    lp.scale1.data, lp.bias1.data, lp.fc.weight.data, lp.fc.bias.data = jb.synth.make_head(2, Ts[2].numpy())
    hp = jb.HotPath(model, jb.TextBank(Ts[0], Ts[1], Ts[2], cuda_dev), lp, rank_by="cs5")
    gen = jb.TTAViews(n_crops=6, seed=2)
    want = [hp.evaluate_base(gen(b)).cpu() for b in batches]
    gen = jb.TTAViews(n_crops=6, seed=2, emit="patches", patch=16)
    patches = gen(batches[0])
    assert patches.shape == (3, 7, 196, 768)
    gen = jb.TTAViews(n_crops=6, seed=2, emit="patches", patch=16)
    streamed = list(hp.evaluate_image_stream(iter(batches), gen))
    assert len(streamed) == len(want)
    assert all(torch.equal(g, w) for g, w in zip(streamed, want))
