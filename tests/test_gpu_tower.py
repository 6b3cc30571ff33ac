"""GPU parity of `encode_image` (CLIP ViT-B/32 image tower, LoRA on q/k/v/o) against the fp32 CPU
oracle, through the reference-facing Python API (`build_model`, `apply_lora`, `model.encode_image`).

Tolerances (north_star): embedding cosine similarity >= 0.999 against the fp32 oracle.  The GEMM
operands are bf16 (fp32 accumulate, fp32 residual stream / LayerNorm / softmax), so element-wise
differences of the unnormalised 512-d embedding are bounded here at 3 % of its RMS, and the
measured cosine is asserted at >= 0.9995 (tighter than the north-star bound).
"""
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _args(params=("q", "k", "v"), encoder="vision"):
    return types.SimpleNamespace(encoder=encoder, position="all", params=list(params), r=4, alpha=1,
                                 dropout_rate=0.25, backbone="ViT-B/32")


def _cos(a, b):
    a, b = a.double(), b.double()
    return (a * b).sum(-1) / (a.norm(dim=-1) * b.norm(dim=-1))


@pytest.fixture(scope="module")
def tower(jb):
    sd = jb.synth.make_vit_state_dict(seed=0)
    return sd, jb.jclip.build_model(sd)


def test_encode_image_zero_shot_matches_oracle(jb, cuda_dev, tower):
    from oracle import vit_encode_image
    sd, model = tower
    imgs = jb.synth.clip_normalize(jb.synth.make_views(3, 2, 4).reshape(8, 3, 224, 224))
    ref = vit_encode_image(sd, imgs)
    out = model.encode_image(torch.from_numpy(imgs).to(cuda_dev)).cpu()
    assert out.shape == (8, 512) and out.dtype == torch.float32
    cos = _cos(out, ref)
    assert cos.min() >= 0.9995, cos
    rms = ref.pow(2).mean().sqrt()
    assert (out - ref).abs().max() <= 0.03 * rms


def test_tokens_before_ln_post(jb, cuda_dev, tower):
    """Residual stream after 12 blocks, every token (not only CLS): catches attention / layout bugs the
    CLS-only embedding could hide."""
    from oracle import vit_encode_image
    sd, model = tower
    imgs = jb.synth.clip_normalize(jb.synth.make_views(4, 1, 3).reshape(3, 3, 224, 224))
    ref = vit_encode_image(sd, imgs, return_tokens=True)
    out = model.visual.debug_tokens(torch.from_numpy(imgs).to(cuda_dev)).cpu()
    assert out.shape == ref.shape == (3, 50, 768)
    cos = _cos(out.reshape(-1, 768), ref.reshape(-1, 768))
    assert cos.min() >= 0.9995, cos.min()


@pytest.mark.parametrize("params", [("q", "k", "v"), ("q", "v"), ("q", "k", "v", "o")])
def test_encode_image_lora_matches_oracle(jb, cuda_dev, params):
    """LoRA applied un-merged in the oracle (reference eval path, test.py:388-398) vs merged in fp32
    then cast to bf16 on the device."""
    from oracle import vit_encode_image
    sd = jb.synth.make_vit_state_dict(seed=1)
    model = jb.jclip.build_model(sd)
    layers = jb.apply_lora(_args(params), model)
    assert len(layers) == 12
    lora = jb.synth.make_lora(seed=7, params=[p for p in params], b_std=0.3)
    for i, layer in enumerate(layers):
        for name, (A, B) in lora[i].items():
            getattr(layer, name).w_lora_A.data = A
            getattr(layer, name).w_lora_B.data = B
    imgs = jb.synth.make_views(5, 1, 6).reshape(6, 3, 224, 224)
    ref = vit_encode_image(sd, imgs, lora=lora, scaling=0.5, apply_clip_norm=True, normalize=True)
    ref0 = vit_encode_image(sd, imgs, lora=None, apply_clip_norm=True, normalize=True)
    x = torch.from_numpy(imgs).to(cuda_dev)
    out = model.visual(x, apply_clip_norm=True, normalize=True).cpu()
    cos = _cos(out, ref)
    assert cos.min() >= 0.9995, cos
    assert (out.norm(dim=-1) - 1).abs().max() < 1e-5
    # the adapters must actually matter for this test to mean anything
    assert _cos(ref, ref0).min() < 0.9999
    assert (_cos(out, ref) > _cos(out, ref0)).all()


def test_ivlp_vpt_tower_matches_oracle(jb, cuda_dev):
    """54-token IVLP / VPT tower (`clip1.load_vlp`, jclip/model1.py:161-196) with LoRA on q,k,v: what test.py's
    primary `clip_model` is (test.py:1855)."""
    from oracle import vit_encode_image
    sd = jb.synth.make_vit_state_dict(seed=3, vpt_tokens=4)
    sd["visual.VPT"] = sd["visual.VPT"] * 25.0          # make the prompt tokens count (0.5 instead of 0.02 std)
    model = jb.jclip.build_model(sd, dict(jb.clip.IVLP_DESIGN))
    assert model.visual.n_ctx == 4
    layers = jb.apply_lora(_args(), model)
    lora = jb.synth.make_lora(seed=8, b_std=0.3)
    for i, layer in enumerate(layers):
        for name, (A, B) in lora[i].items():
            getattr(layer, name).w_lora_A.data = A
            getattr(layer, name).w_lora_B.data = B
    imgs = jb.synth.make_views(13, 1, 5).reshape(5, 3, 224, 224)
    x = torch.from_numpy(imgs).to(cuda_dev)
    ref_tok = vit_encode_image(sd, imgs, lora=lora, scaling=0.5, apply_clip_norm=True, return_tokens=True)
    tok = model.visual.debug_tokens(x, apply_clip_norm=True).cpu()
    assert tok.shape == ref_tok.shape == (5, 54, 768)
    assert _cos(tok.reshape(-1, 768), ref_tok.reshape(-1, 768)).min() >= 0.9995
    ref = vit_encode_image(sd, imgs, lora=lora, scaling=0.5, apply_clip_norm=True, normalize=True)
    out = model.visual(x, apply_clip_norm=True, normalize=True).cpu()
    assert _cos(out, ref).min() >= 0.9995
    sd0 = {k: v for k, v in sd.items() if k != "visual.VPT"}
    ref0 = vit_encode_image(sd0, imgs, lora=lora, scaling=0.5, apply_clip_norm=True, normalize=True)
    assert _cos(ref, ref0).min() < 0.9999 and (_cos(out, ref) > _cos(out, ref0)).all()


def test_lora_update_refreshes_packed_weights(jb, cuda_dev, tower):
    sd, _ = tower
    model = jb.jclip.build_model(sd)
    layers = jb.apply_lora(_args(), model)
    x = torch.from_numpy(jb.synth.make_views(6, 1, 2).reshape(2, 3, 224, 224)).to(cuda_dev)
    f0 = model.visual(x, apply_clip_norm=True, normalize=True).clone()      # B = 0 -> no-op adapters
    rng = np.random.default_rng(0)
    # apply_lora draws A from an unseeded generator (as the reference's kaiming_uniform_ does): pin it, and make B large
    # enough that the effect of ONE adapter on the unit-norm embedding is far above rounding (it was marginal at 0.05)
    layers[3].q_proj.w_lora_A.data = rng.uniform(-768 ** -0.5, 768 ** -0.5, (4, 768)).astype(np.float32)
    f0 = model.visual(x, apply_clip_norm=True, normalize=True).clone()      # still a no-op: B = 0
    layers[3].q_proj.w_lora_B.data = (0.5 * rng.standard_normal((768, 4))).astype(np.float32)
    f1 = model.visual(x, apply_clip_norm=True, normalize=True)
    assert (f0 - f1).abs().max() > 1e-4
    layers[3].q_proj.w_lora_B.data = np.zeros((768, 4), np.float32)
    f2 = model.visual(x, apply_clip_norm=True, normalize=True)
    assert torch.equal(f0, f2)


@pytest.mark.parametrize("dtype", ["u8", "bf16"])
def test_image_dtypes(jb, cuda_dev, tower, dtype):
    from oracle import vit_encode_image
    sd, model = tower
    img = jb.synth.make_views(7, 1, 3).reshape(3, 3, 224, 224)
    if dtype == "u8":
        q = np.round(img * 255).astype(np.uint8)
        ref_in, x = q.astype(np.float32) / 255.0, torch.from_numpy(q)
    else:
        x = torch.from_numpy(img).to(torch.bfloat16)
        ref_in = x.float().numpy()
    ref = vit_encode_image(sd, ref_in, apply_clip_norm=True, normalize=True)
    out = model.visual(x.to(cuda_dev), apply_clip_norm=True, normalize=True).cpu()
    assert _cos(out, ref).min() >= 0.9995


def test_host_entry_point_and_chunking(jb, cuda_dev, tower):
    """jcb_encode_image_host (pinned host in, host out, chunks double-buffered on a copy stream) must
    equal the device-resident call bit for bit, for a view count that is not a multiple of the chunk."""
    sd, model = tower
    img = jb.synth.make_views(8, 1, 23).reshape(23, 3, 224, 224)
    dev_out = model.visual(torch.from_numpy(img).to(cuda_dev), apply_clip_norm=True, normalize=True).cpu()
    ctx = jb.get_context(cuda_dev)
    ctx.set_chunk_views(5)
    try:
        host_out = model.visual(torch.from_numpy(img).pin_memory(), apply_clip_norm=True, normalize=True)
        np_out = model.visual(img, apply_clip_norm=True, normalize=True)
    finally:
        ctx.set_chunk_views(16384)
    assert not host_out.is_cuda and isinstance(np_out, np.ndarray)
    assert torch.equal(host_out, dev_out)
    assert np.array_equal(np_out, dev_out.numpy())


def test_dlpack_entry_point(jb, cuda_dev, tower):
    sd, model = tower
    x = torch.from_numpy(jb.synth.make_views(9, 1, 4).reshape(4, 3, 224, 224)).to(cuda_dev)
    ref = model.visual(x, apply_clip_norm=True, normalize=True)
    out = torch.zeros(4, 512, device=cuda_dev)
    model.visual.execute_dlpack(x, out, apply_clip_norm=True, normalize=True)
    torch.cuda.synchronize()
    assert torch.equal(out, ref)


def test_empty_and_bad_inputs(jb, cuda_dev, tower):
    sd, model = tower
    out = model.encode_image(torch.zeros(0, 3, 224, 224, device=cuda_dev))
    assert out.shape == (0, 512)
    with pytest.raises(ValueError):
        model.encode_image(torch.zeros(2, 3, 200, 224, device=cuda_dev))
    with pytest.raises(TypeError):
        model.encode_image(torch.zeros(2, 3, 224, 224, dtype=torch.int32, device=cuda_dev))


def test_lora_pickle_round_trip(jb, cuda_dev, tmp_path):
    """The LoRA pickle layout (SURVEY.md Appendix D): round-trip through save_lora / load_lora with
    encoder='both' (text layers first, vision layers 12..23), then encode."""
    sd = jb.synth.make_vit_state_dict(seed=2, text_layers=12)
    model = jb.jclip.build_model(sd)
    args = _args(encoder="both")
    layers = jb.apply_lora(args, model)
    assert len(layers) == 24
    rng = np.random.default_rng(3)
    for layer in layers:
        for name in ("q_proj", "k_proj", "v_proj"):
            lin = getattr(layer, name)
            lin.w_lora_B.data = (0.01 * rng.standard_normal(lin.w_lora_B.shape)).astype(np.float32)
    args.filename = "t"
    path = jb.save_lora(args, 0, layers, save_dir=str(tmp_path))
    x = torch.from_numpy(jb.synth.make_views(10, 1, 2).reshape(2, 3, 224, 224)).to(cuda_dev)
    f_a = model.visual(x, apply_clip_norm=True, normalize=True).clone()
    model2 = jb.jclip.build_model(sd)
    layers2 = jb.apply_lora(args, model2)
    jb.load_lora(args, layers2, path)
    f_b = model2.visual(x, apply_clip_norm=True, normalize=True)
    assert torch.equal(f_a, f_b)


@pytest.mark.parametrize("vpt", [0, 4])
def test_cls_only_last_block_matches_full_schedule(jb, cuda_dev, vpt):
    """Opt-in schedule (jcb_ctx_set_cls_only_last_block): the last block on the class-token rows only.  Same
    embeddings as the full schedule to rounding (one attention row summed in another order), same distance to the
    fp32 oracle; 50- and 54-token towers; batch sizes around the 256-row GEMM tile."""
    from oracle import vit_encode_image
    sd = jb.synth.make_vit_state_dict(seed=2, vpt_tokens=vpt)
    design = dict(jb.clip.IVLP_DESIGN) if vpt else None
    model = jb.jclip.build_model(sd, design) if design else jb.jclip.build_model(sd)
    layers = jb.apply_lora(_args(), model)
    lora = jb.synth.make_lora(seed=9, b_std=0.3)
    for i, layer in enumerate(layers):
        for name, (A, B) in lora[i].items():
            getattr(layer, name).w_lora_A.data = A
            getattr(layer, name).w_lora_B.data = B
    ctx = jb.get_context(cuda_dev)
    imgs = jb.synth.make_views(6, 1, 7).reshape(7, 3, 224, 224)
    ref = vit_encode_image(sd, imgs, lora=lora, scaling=0.5, apply_clip_norm=True, normalize=True)
    big = torch.from_numpy(jb.synth.make_views(7, 3, 87).reshape(261, 3, 224, 224)).to(cuda_dev)
    x = torch.from_numpy(imgs).to(cuda_dev)
    try:
        full, full_big = model.visual(x, apply_clip_norm=True, normalize=True).cpu(), model.visual(big, apply_clip_norm=True, normalize=True).cpu()
        ctx.set_cls_only_last_block(True)
        fast, fast_big = model.visual(x, apply_clip_norm=True, normalize=True).cpu(), model.visual(big, apply_clip_norm=True, normalize=True).cpu()
    finally:
        ctx.set_cls_only_last_block(False)
    assert _cos(fast, ref).min() >= 0.9995
    assert _cos(fast, full).min() >= 0.99999 and (fast - full).abs().max() <= 2e-3
    assert _cos(fast_big, full_big).min() >= 0.99999 and (fast_big - full_big).abs().max() <= 2e-3
    assert torch.equal(model.visual(x, apply_clip_norm=True, normalize=True).cpu(), full)     # switched off again


def _shipped_lora_pickle(tmp_path):
    """The reference's trained adapters (lora_weights1/lora_weights.pkl) rebuilt in the reference's pickle layout
    (save_lora, test.py:642-684) from the numeric fixture tests/golden/lora_weights1_arrays.npz
    (oracle/make_golden_lora.py; stored as float16, widened back to the checkpoint's float32 here)."""
    import json
    import os
    import pickle
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "lora_weights1_arrays.npz"))
    meta = json.loads(bytes(z["metadata_json"]).decode())
    weights = {}
    for key in z.files:
        if key == "metadata_json":
            continue
        layer, proj, name = key.split("/")
        weights.setdefault(layer, {}).setdefault(proj, {})[name] = z[key].astype(np.float32)
    path = tmp_path / "lora_weights.pkl"
    with open(path, "wb") as f:
        pickle.dump({"weights": weights, "metadata": meta}, f)
    return str(path), meta, weights


@pytest.mark.parametrize("op", ["f16", "bf16"])
def test_shipped_trained_lora_through_load_lora(jb, cuda_dev, tmp_path, op):
    """The only real weight artefact of the reference: trained rank-4 adapters on q, k, v of all 24 blocks
    (encoder='both': layer_0..11 = text tower, layer_12..23 = vision tower; SURVEY.md F5, Appendix D), loaded through
    `load_lora` exactly as test.py:1800-1803 does and run through BOTH towers against the fp32 oracle, which applies
    them un-merged (test.py:388-398)."""
    from oracle import text_encode, vit_encode_image
    path, meta, weights = _shipped_lora_pickle(tmp_path)
    assert meta == {"r": 4, "alpha": 1, "encoder": "both", "params": ["q", "k", "v"], "position": "all"}
    sd = jb.synth.make_vit_state_dict(seed=2, text_layers=12)
    model = jb.jclip.build_model(sd)
    args = _args(encoder="both")
    layers = jb.apply_lora(args, model)
    assert len(layers) == 24
    jb.load_lora(args, layers, path)
    assert np.array_equal(layers[12].q_proj.w_lora_A.data, weights["layer_12"]["q_proj"]["w_lora_A"])
    assert layers[0].q_proj.w_lora_B.data.shape == (512, 4) and layers[23].v_proj.w_lora_B.data.shape == (768, 4)
    # a mismatching metadata field is refused as in the reference (test.py:702-717)
    with pytest.raises(ValueError):
        jb.load_lora(_args(params=("q", "v"), encoder="both"), layers, path)
    lora_v = {i: {p: (weights[f"layer_{12 + i}"][p]["w_lora_A"], weights[f"layer_{12 + i}"][p]["w_lora_B"])
                  for p in ("q_proj", "k_proj", "v_proj")} for i in range(12)}
    lora_t = {i: {p: (weights[f"layer_{i}"][p]["w_lora_A"], weights[f"layer_{i}"][p]["w_lora_B"])
                  for p in ("q_proj", "k_proj", "v_proj")} for i in range(12)}
    imgs = jb.synth.make_views(12, 1, 6).reshape(6, 3, 224, 224)
    tok = jb.synth.make_tokens(9, 7, vocab=64)
    ref = vit_encode_image(sd, imgs, lora=lora_v, scaling=0.5, apply_clip_norm=True, normalize=True)
    ref0 = vit_encode_image(sd, imgs, lora=None, apply_clip_norm=True, normalize=True)
    reft = text_encode(sd, tok, lora=lora_t, scaling=0.5, normalize=True)
    ctx = jb.get_context(cuda_dev)
    prev = ctx.operand_type
    try:
        ctx.set_operand_type(op)
        out = model.visual(torch.from_numpy(imgs).to(cuda_dev), apply_clip_norm=True, normalize=True).cpu()
        outt = model.encode_text(torch.from_numpy(tok).to(cuda_dev), normalize=True).cpu()
    finally:
        ctx.set_operand_type(prev)
    floor = 0.9995 if op == "bf16" else 0.99999
    assert _cos(out, ref).min() >= floor, _cos(out, ref).min()
    assert _cos(outt, reft).min() >= floor, _cos(outt, reft).min()
    # What the adapters do at their trained magnitudes (on these random-init base weights): 1 - cos = 1.7e-6 between the
    # embeddings with and without them.  fp16 operands resolve that ten times over (1 - cos = 4e-8 vs the oracle); bf16
    # operands (3e-6) do not -- their rounding is larger than the whole LoRA effect.
    if op == "f16":
        assert (1 - _cos(ref0, ref)).min() > 10 * (1 - _cos(out, ref)).max()
