"""LoRA slots: several adapter sets on one image tower, chosen per view (`visual(x, slot_of_view=...)`,
`jcb_encode_image_slots`) or per image (`HotPath.evaluate_base(..., slot_of_image=...)`, `jcb_pipeline_slots`).

The contract is bit-identity: a view encoded with slot g inside a mixed batch is `torch.equal` to the same view
encoded by a tower that carries only slot g, in applied mode.  The single-slot towers here are packed through the
C-ABI (`jcb_vit_clear_lora` / `jcb_vit_set_lora` / `jcb_vit_finalize`), so a slot's adapters can have any ranks.
Slot patterns: one slot per image (V views of T tokens: slot changes inside 256-row GEMM tiles at image boundaries)
and one slot per view (every tile holds several slots: the worst case).
"""
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

CODES = {"q": 0, "k": 1, "v": 2, "o": 3}
NAMES = {"q": "q_proj", "k": "k_proj", "v": "v_proj", "o": "proj"}


@pytest.fixture
def applied(jb, cuda_dev):
    ctx = jb.get_context(cuda_dev)
    assert ctx.lora_mode == "merged"
    prev = ctx.operand_type
    ctx.set_lora_mode("applied")
    yield ctx
    ctx.set_lora_mode("merged")
    ctx.set_operand_type(prev)


def _slot(seed, layers, ranks, width=768, b_std=0.1, skip_layers=()):
    """{layer: {proj: (A [r, W], B [W, r], scaling)}}, ranks = {proj: r}; no adapter at all on `skip_layers`."""
    rng = np.random.default_rng(seed)
    bound = 1.0 / np.sqrt(width)
    out = {}
    for i in range(layers):
        if i in skip_layers:
            continue
        out[i] = {}
        for p, r in ranks.items():
            A = rng.uniform(-bound, bound, size=(r, width)).astype(np.float32)
            B = (rng.standard_normal((width, r)) * b_std).astype(np.float32)
            out[i][p] = (A, B, float(1.0 / np.sqrt(r)))
    return out


def _multi_model(jb, sd, slots, backbone):
    """Slot 0 through apply_lora (uniform rank, like the reference), slots 1.. through set_lora_slots."""
    model = jb.jclip.build_model(sd)
    s0 = slots[0]
    params = [p for p in "qkvo" if p in next(iter(s0.values()))]
    r = next(iter(s0.values()))[params[0]][0].shape[0]
    args = types.SimpleNamespace(encoder="vision", position="all", params=params, r=r, alpha=1, dropout_rate=0.0,
                                 backbone=backbone)
    for i, layer in enumerate(jb.apply_lora(args, model)):
        for p, (A, B, _) in s0[i].items():
            getattr(layer, NAMES[p]).w_lora_A.data = A
            getattr(layer, NAMES[p]).w_lora_B.data = B
    model.visual.set_lora_slots(slots[1:])
    return model


def _pack_single(jb, ctx, model, slot, dev):
    """Re-pack `model`'s tower (no adapters of its own) with `slot` as its only adapter set."""
    _, vit = model.visual._engine(dev)
    lib = ctx.lib
    jb._capi.check(lib.jcb_vit_clear_lora(vit), ctx.handle)
    for i, projs in slot.items():
        for p, (A, B, s) in projs.items():
            jb._capi.check(lib.jcb_vit_set_lora(vit, i, CODES[p], A.ctypes.data, B.ctypes.data, A.shape[0], s), ctx.handle)
    jb._capi.check(lib.jcb_vit_finalize(vit), ctx.handle)
    assert lib.jcb_vit_lora_slots(vit) == 1


TOWERS = {   # name: (state-dict kwargs, backbone, images, views per image); tokens 50 / 54 / 197
    "b32": (dict(layers=2), "ViT-B/32", 7, 5),
    "ivlp": (dict(layers=2, vpt_tokens=4), "ViT-B/32", 6, 5),
    "b16": (dict(layers=2, patch=16), "ViT-B/16", 4, 3),
}
CASES = [   # tower, slots as (ranks, skipped layers)
    ("b32", [({"q": 4, "k": 4, "v": 4}, ())] * 2),
    ("b32", [({"q": 16, "k": 16, "v": 16, "o": 16}, ()), ({"q": 4, "k": 4, "v": 4, "o": 4}, ()),
             ({"q": 20, "k": 20, "v": 24, "o": 64}, ())]),                    # slot 2: q, k, v ranks sum to 64
    ("ivlp", [({"q": 4, "k": 4, "v": 4, "o": 4}, ()), ({"q": 16, "k": 16, "v": 16}, ()), ({"o": 16}, (1,))]),
    ("b16", [({"q": 16, "k": 16, "v": 16}, ())] * 5 + [({"q": 4, "k": 4, "v": 4}, (0,))] + [({"q": 4, "v": 4}, ())] * 2),
    ("b32", [({"q": 4, "k": 4, "v": 4, "o": 4}, ())] * 3 + [({"q": 16, "k": 16, "v": 16, "o": 16}, (1,))] * 5),
]


@pytest.mark.parametrize("op", ["f16", "bf16"])
@pytest.mark.parametrize("case", range(len(CASES)), ids=lambda c: f"{CASES[c][0]}-G{len(CASES[c][1])}-{c}")
def test_mixed_slots_bit_identical_to_single_slot_towers(jb, cuda_dev, applied, case, op):
    ctx = applied
    ctx.set_operand_type(op)
    tower, slot_specs = CASES[case]
    sd_kw, backbone, I, V = TOWERS[tower]
    sd = jb.synth.make_vit_state_dict(seed=30 + case, **sd_kw)
    if "visual.VPT" in sd:
        sd["visual.VPT"] = sd["visual.VPT"] * 25.0
    layers = sd_kw["layers"]
    G = len(slot_specs)
    slots = [_slot(100 * case + g, layers, ranks, skip_layers=skip) for g, (ranks, skip) in enumerate(slot_specs)]
    model = _multi_model(jb, sd, slots, backbone)
    assert model.visual.lora_slots == G
    R = model.visual.input_resolution
    imgs = torch.from_numpy(jb.synth.make_views(case, I, V, resolution=R).reshape(I * V, 3, R, R)).to(cuda_dev)
    per_image = np.repeat(np.arange(I) % G, V)                   # slot changes at image boundaries inside tiles
    per_view = (np.arange(I * V) * 5 + 1) % G                    # a different slot at every view
    patterns = {"image": per_image, "view": per_view}
    outs = {k: model.visual(imgs, apply_clip_norm=True, normalize=True, slot_of_view=s) for k, s in patterns.items()}
    plain = model.visual(imgs, apply_clip_norm=True, normalize=True)           # no slot array: slot 0
    assert ctx.lib.jcb_vit_lora_slots(model.visual._vit) == G
    ref_model = jb.jclip.build_model(sd)
    refs = []
    for g in range(G):
        _pack_single(jb, ctx, ref_model, slots[g], cuda_dev)
        refs.append(ref_model.visual(imgs, apply_clip_norm=True, normalize=True))
    for name, s in patterns.items():
        for g in range(G):
            rows = torch.from_numpy(np.nonzero(s == g)[0]).to(cuda_dev)
            if len(rows):
                assert torch.equal(outs[name][rows], refs[g][rows]), (name, g, (outs[name][rows] - refs[g][rows]).abs().max())
    assert torch.equal(plain, refs[0])
    # the slots matter: different adapter sets give different embeddings of the same view
    for g in range(1, G):
        assert (refs[g] - refs[0]).abs().max() > 1e-3


@pytest.mark.parametrize("op", ["f16", "bf16"])
def test_many_tiles_per_cta_pair_with_skipped_tiles(jb, cuda_dev, applied, op):
    """512 views of 50 tokens = 100 GEMM tiles of 256 rows: every CTA pair of the persistent GEMMs runs several tiles, and
    the down-projection skips the N tiles (two slots each) that hold no slot of a tile's rows -- for G = 8 most of them,
    for G = 3 those of a slot that has no adapter on a projection of some layer.  A skipped tile uses no accumulator
    stage, so the tiles after it must still run on the right stage and barrier phase."""
    ctx = applied
    ctx.set_operand_type(op)
    sd = jb.synth.make_vit_state_dict(seed=80, layers=2)
    I, V = 64, 8
    imgs = torch.from_numpy(jb.synth.make_views(8, I, V).reshape(I * V, 3, 224, 224)).to(cuda_dev)
    qkvo = {"q": 4, "k": 4, "v": 4, "o": 4}
    cases = {
        8: [_slot(800 + g, 2, qkvo, skip_layers=(0,) if g == 5 else ()) for g in range(8)],
        3: [_slot(830, 2, qkvo), _slot(831, 2, {"q": 4, "k": 4, "v": 4}), _slot(832, 2, qkvo, skip_layers=(1,))],
    }
    ref_model = jb.jclip.build_model(sd)
    for G, slots in cases.items():
        model = _multi_model(jb, sd, slots, "ViT-B/32")
        patterns = {"image": np.repeat((np.arange(I) * 3) % G, V), "view": np.arange(I * V) % G}
        outs = {k: model.visual(imgs, apply_clip_norm=True, normalize=True, slot_of_view=sl) for k, sl in patterns.items()}
        for g in range(G):
            _pack_single(jb, ctx, ref_model, slots[g], cuda_dev)
            ref = ref_model.visual(imgs, apply_clip_norm=True, normalize=True)
            for name, sl in patterns.items():
                rows = torch.from_numpy(np.nonzero(sl == g)[0]).to(cuda_dev)
                assert torch.equal(outs[name][rows], ref[rows]), (G, name, g, (outs[name][rows] - ref[rows]).abs().max())
        model.visual.release()


def test_registered_slots_without_adapters_count(jb, cuda_dev, applied):
    """An empty adapter set is a slot too: set_lora_slots([A, {}]) is a tower of three slots, slot 2 = no adapters."""
    ctx = applied
    sd = jb.synth.make_vit_state_dict(seed=90, layers=2)
    slots = [_slot(90, 2, {"q": 4, "k": 4, "v": 4}), _slot(91, 2, {"q": 4, "k": 4, "v": 4})]
    model = _multi_model(jb, sd, slots, "ViT-B/32")
    model.visual.set_lora_slots([slots[1], {}])
    x = torch.from_numpy(jb.synth.make_views(9, 2, 3).reshape(6, 3, 224, 224)).to(cuda_dev)
    out = model.visual(x, apply_clip_norm=True, slot_of_view=[2, 0, 1, 2, 2, 0])
    assert model.visual.lora_slots == 3 == ctx.lib.jcb_vit_lora_slots(model.visual._vit)
    plain = jb.jclip.build_model(sd).visual(x, apply_clip_norm=True)         # applied mode, no adapters
    idx = torch.tensor([0, 3, 4], device=cuda_dev)
    assert torch.equal(out[idx], plain[idx])
    model.visual.set_lora_slots([{}] * 7)
    assert model.visual(x, slot_of_view=[7] * 6).shape == (6, 512)
    assert ctx.lib.jcb_vit_lora_slots(model.visual._vit) == 8
    ctx.set_lora_mode("merged")                                                # eight slots: applied mode only
    with pytest.raises(RuntimeError, match="applied"):
        model.visual(x)
    ctx.set_lora_mode("applied")
    vit = model.visual._vit
    for bad in (0, 9):
        assert ctx.lib.jcb_vit_set_lora_slot_count(vit, bad) == jb._capi.JCB_E_INVALID


def test_one_slot_tower_with_a_slot_array_is_the_plain_call(jb, cuda_dev, applied):
    sd = jb.synth.make_vit_state_dict(seed=41, layers=2)
    slot = _slot(41, 2, {"q": 4, "k": 4, "v": 4})
    model = _multi_model(jb, sd, [slot], "ViT-B/32")
    x = torch.from_numpy(jb.synth.make_views(3, 2, 3).reshape(6, 3, 224, 224)).to(cuda_dev)
    a = model.visual(x, apply_clip_norm=True, slot_of_view=[0] * 6)
    b = model.visual(x, apply_clip_norm=True)
    assert torch.equal(a, b)
    # host images: copied to the device, same result, returned on the host
    c = model.visual(x.cpu(), apply_clip_norm=True, slot_of_view=np.zeros(6, np.int32))
    assert not c.is_cuda and torch.equal(c, b.cpu())


def _hot_path(jb, model, dev):
    texts = [torch.from_numpy(jb.synth.make_text_features(seed=10 + i)) for i in range(3)]
    lp_np = jb.synth.make_head(2, texts[2].numpy())
    lp = jb.Channel_LP()
    lp.scale1.data, lp.bias1.data, lp.fc.weight.data, lp.fc.bias.data = lp_np
    return jb.HotPath(model, jb.TextBank(*texts, dev), lp, rank_by="cs5")


@pytest.mark.parametrize("op", ["f16", "bf16"])
def test_pipeline_slot_of_image_matches_per_slot_runs(jb, cuda_dev, applied, op):
    ctx = applied
    ctx.set_operand_type(op)
    sd = jb.synth.make_vit_state_dict(seed=50, layers=2)
    slots = [_slot(50 + g, 2, {"q": 8, "k": 8, "v": 8, "o": 8}, b_std=0.3) for g in range(3)]
    model = _multi_model(jb, sd, slots, "ViT-B/32")
    I, V = 7, 9
    imgs = torch.from_numpy(jb.synth.make_views(5, I, V)).to(cuda_dev)
    soi = np.array([2, 0, 0, 1, 2, 1, 0], np.int32)
    hp = _hot_path(jb, model, cuda_dev)
    top, feats, scores = hp.evaluate_base(imgs, return_feats=True, return_scores=True, slot_of_image=soi)
    ref_model = jb.jclip.build_model(sd)
    hp_ref = _hot_path(jb, ref_model, cuda_dev)
    for g in range(3):
        _pack_single(jb, ctx, ref_model, slots[g], cuda_dev)
        t_g, f_g, s_g = hp_ref.evaluate_base(imgs, return_feats=True, return_scores=True)
        idx = torch.from_numpy(np.nonzero(soi == g)[0]).to(cuda_dev)
        assert torch.equal(feats[idx], f_g[idx])
        assert torch.equal(scores[idx], s_g[idx])
        assert torch.equal(top[idx], t_g[idx])
    assert len({tuple(scores[i].tolist()[:4]) for i in range(I)}) == I
    # the stream form: (images, slot_of_image) pairs, two batches in flight; host top-k of each batch
    batches = [(imgs, soi), (imgs[:4], soi[:4][::-1].copy()), (imgs[2:], soi[2:])]
    got = list(hp.evaluate_stream(batches, depth=2))
    for (b_imgs, b_soi), t in zip(batches, got):
        want = hp.evaluate_base(b_imgs, slot_of_image=b_soi)
        assert torch.equal(t, want.cpu())
    assert torch.equal(got[0], top.cpu())


@pytest.mark.parametrize("op", ["f16", "bf16"])
def test_slot_against_oracle_unmerged(jb, cuda_dev, applied, op):
    """One slot of a three-slot tower against the fp32 oracle's un-merged form (the same bounds as one adapter set)."""
    from oracle import vit_encode_image
    ctx = applied
    ctx.set_operand_type(op)
    sd = jb.synth.make_vit_state_dict(seed=1)
    slots = [_slot(60 + g, 12, {"q": 4, "k": 4, "v": 4}, b_std=0.3) for g in range(3)]
    model = _multi_model(jb, sd, slots, "ViT-B/32")
    imgs = jb.synth.make_views(5, 2, 3).reshape(6, 3, 224, 224)
    s = np.array([2, 0, 2, 1, 2, 2], np.int32)
    out = model.visual(torch.from_numpy(imgs).to(cuda_dev), apply_clip_norm=True, normalize=True, slot_of_view=s).cpu()
    lora = {i: {NAMES[p]: (A, B) for p, (A, B, _) in d.items()} for i, d in slots[2].items()}
    ref = vit_encode_image(sd, imgs[s == 2], lora=lora, scaling=0.5, apply_clip_norm=True, normalize=True)
    ref0 = vit_encode_image(sd, imgs[s == 2], lora=None, apply_clip_norm=True, normalize=True)
    o2 = out[torch.from_numpy(s == 2)].double()
    cos = (o2 * ref.double()).sum(-1) / (o2.norm(dim=-1) * ref.double().norm(dim=-1))
    cos0 = (ref0.double() * ref.double()).sum(-1) / (ref0.double().norm(dim=-1) * ref.double().norm(dim=-1))
    assert cos.min() >= (0.99999 if op == "f16" else 0.9995), cos
    assert cos0.min() < 0.9999                                  # the adapters matter


# ---- rejections: before anything is launched, the output untouched -------------------------------------------------
def _three_slot_model(jb, cuda_dev):
    sd = jb.synth.make_vit_state_dict(seed=70, layers=1)
    slots = [_slot(70 + g, 1, {"q": 4, "k": 4, "v": 4}) for g in range(3)]
    return _multi_model(jb, sd, slots, "ViT-B/32"), slots


def test_merged_mode_with_several_slots_is_rejected(jb, cuda_dev, applied):
    model, _ = _three_slot_model(jb, cuda_dev)
    applied.set_lora_mode("merged")
    x = torch.zeros(2, 3, 224, 224, device=cuda_dev)
    with pytest.raises(RuntimeError, match="applied"):
        model.visual(x)
    model.visual.set_lora_slots([])                              # one slot: merged mode packs it
    assert model.visual(x).shape == (2, 512)


def test_bad_slot_arrays_are_rejected_before_launch(jb, cuda_dev, applied):
    ctx = applied
    model, _ = _three_slot_model(jb, cuda_dev)
    x = torch.zeros(4, 3, 224, 224, device=cuda_dev)
    model.visual(x)                                              # packed
    vit, lib = model.visual._vit, ctx.lib
    out = torch.full((4, 512), float("nan"), device=cuda_dev)
    n0 = ctx.launch_count
    for bad in ([0, 1, 3, 0], [0, -1, 0, 0], None):
        arr = None if bad is None else np.array(bad, np.int32)
        rc = lib.jcb_encode_image_slots(vit, x.data_ptr(), jb._capi.IMG_F32, 4, None if arr is None else arr.ctypes.data,
                                        1, 1, out.data_ptr())
        assert rc == jb._capi.JCB_E_INVALID
    torch.cuda.synchronize()
    assert ctx.launch_count == n0 and torch.isnan(out).all()
    with pytest.raises(RuntimeError, match="out of range"):
        model.visual(x, slot_of_view=[0, 1, 2, 3])
    # the pipeline: per-image slots out of range, or a NULL array
    hp = _hot_path(jb, model, cuda_dev)
    imgs = torch.zeros(2, 3, 3, 224, 224, device=cuda_dev)
    topk = torch.full((2, 5), -7, dtype=torch.int32, device=cuda_dev)
    a = hp._args(imgs, 2, 3, False, topk, None, None, cuda_dev)
    ticket = jb._capi.c_int64(-1)
    for arr in (np.array([0, 5], np.int32), None):
        p = None if arr is None else arr.ctypes.data
        assert lib.jcb_pipeline_slots(vit, None, jb._capi.byref(a), p) == jb._capi.JCB_E_INVALID
        assert lib.jcb_pipeline_submit_slots(vit, None, jb._capi.byref(a), p, jb._capi.byref(ticket)) == jb._capi.JCB_E_INVALID
    torch.cuda.synchronize()
    assert ctx.launch_count == n0 and (topk == -7).all() and ticket.value == -1
    with pytest.raises(RuntimeError, match="out of range"):
        hp.evaluate_base(imgs, slot_of_image=[0, 3])


def test_more_than_eight_slots_and_ranks_over_64_are_rejected(jb, cuda_dev, applied):
    ctx = applied
    model, slots = _three_slot_model(jb, cuda_dev)
    with pytest.raises(ValueError, match="at most 8"):
        model.visual.set_lora_slots([slots[1]] * 8)
    x = torch.zeros(1, 3, 224, 224, device=cuda_dev)
    model.visual(x)
    vit = model.visual._vit
    A, B, s = slots[1][0]["q"]
    assert ctx.lib.jcb_vit_set_lora_slot(vit, 8, 0, 0, A.ctypes.data, B.ctypes.data, 4, s) == jb._capi.JCB_E_INVALID
    assert ctx.lib.jcb_vit_set_lora_slot(vit, -1, 0, 0, A.ctypes.data, B.ctypes.data, 4, s) == jb._capi.JCB_E_INVALID
    assert ctx.lib.jcb_vit_lora_slots(vit) == 3
    for ranks in ({"q": 32, "k": 32, "v": 8}, {"o": 65}):        # q + k + v = 72 > 64; r(o) = 65 > 64
        model.visual.set_lora_slots([slots[1], _slot(7, 1, ranks)])
        with pytest.raises(RuntimeError, match="ranks"):
            model.visual(x)
    model.visual.set_lora_slots([slots[1], _slot(7, 1, {"q": 32, "k": 32})])   # exactly 64
    assert model.visual(x, slot_of_view=[2]).shape == (1, 512)
