"""CPU: what `VisionTransformer.set_lora_slots` accepts -- reference-layout LoRA pickles and {layer: {proj: (A, B)}}
dicts -- and the checks that happen before anything reaches the library."""
import math
import types

import numpy as np
import pytest


def _args(params, r, position="all", encoder="vision"):
    return types.SimpleNamespace(encoder=encoder, position=position, params=list(params), r=r, alpha=2,
                                 dropout_rate=0.0, backbone="ViT-B/32", filename="slot")


def test_pickle_slot_maps_layers_and_scaling(jb, tmp_path):
    sd = jb.synth.make_vit_state_dict(seed=0, layers=12)
    model = jb.jclip.build_model(sd)
    args = _args(("q", "v", "o"), r=4, position="up")               # blocks 8..11
    layers = jb.apply_lora(args, model)
    rng = np.random.default_rng(0)
    for layer in layers:
        for name in ("q_proj", "v_proj", "proj"):
            getattr(layer, name).w_lora_B.data = rng.standard_normal((768, 4)).astype(np.float32)
    path = jb.save_lora(args, 1, layers, save_dir=str(tmp_path))
    slot = jb.lora.slot_adapters(path, 12, 768)
    assert sorted(slot) == [8, 9, 10, 11]
    for i, block in enumerate(range(8, 12)):
        assert sorted(slot[block]) == [0, 2, 3]                    # q, v, o
        A, B, r, s = slot[block][2]
        assert r == 4 and s == pytest.approx(2 / math.sqrt(4))     # metadata alpha / sqrt(r), test.py:288-289
        assert np.array_equal(A, layers[i].v_proj.w_lora_A.data) and np.array_equal(B, layers[i].v_proj.w_lora_B.data)


def test_dict_slot_and_its_checks(jb):
    rng = np.random.default_rng(1)
    A, B = rng.standard_normal((8, 768)).astype(np.float32), rng.standard_normal((768, 8)).astype(np.float32)
    slot = jb.lora.slot_adapters({3: {"q": (A, B), "o": (A[:2], B[:, :2], 0.25)}}, 12, 768, alpha=4.0)
    assert slot[3][0][2:] == (8, pytest.approx(4.0 / math.sqrt(8))) and slot[3][3][2:] == (2, 0.25)
    with pytest.raises(ValueError, match="projection"):
        jb.lora.slot_adapters({0: {"x": (A, B)}}, 12, 768)
    with pytest.raises(ValueError, match="block"):
        jb.lora.slot_adapters({12: {"q": (A, B)}}, 12, 768)
    with pytest.raises(ValueError, match="expected"):
        jb.lora.slot_adapters({0: {"q": (A, A)}}, 12, 768)
    with pytest.raises(FileNotFoundError):
        jb.lora.slot_adapters("/nonexistent/slot.pkl", 12, 768)


def test_text_only_pickle_and_too_many_slots_are_rejected(jb, tmp_path):
    sd = jb.synth.make_vit_state_dict(seed=0, layers=2, text_layers=12)
    model = jb.jclip.build_model(sd)
    args = _args(("q",), r=2, encoder="text")
    path = jb.save_lora(args, 1, jb.apply_lora(args, model), save_dir=str(tmp_path))
    with pytest.raises(ValueError, match="image-tower"):
        model.visual.set_lora_slots([path])
    with pytest.raises(ValueError, match="at most 8"):
        model.visual.set_lora_slots([{}] * 8)
    model.visual.set_lora_slots([{}] * 7)
    assert model.visual.lora_slots == 8


def test_slot_array_shape_is_checked(jb):
    from jclip_b200.jclip.model import slot_array
    assert slot_array([0, 2, 1], 3, "s").dtype == np.int32
    with pytest.raises(ValueError, match="3 slot indices"):
        slot_array([0, 1], 3, "slot_of_view")
