"""CPU: host logic of image-tower LoRA training -- the Philox4x32-10 reproduction of the device dropout masks, the mask's
keep rate and independence across projections, the C-ABI declarations and the trainer's argument checks."""
import numpy as np
import pytest
import torch


def test_philox_known_answers(jb):
    """Random123's known-answer vectors for Philox4x32-10 (the generator of curand_philox4x32_x.h)."""
    P = jb.train.philox4x32_10
    cases = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
             ((0xFFFFFFFF,) * 4, (0xFFFFFFFF, 0xFFFFFFFF), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
             ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
              (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for c, k, want in cases:
        assert tuple(int(x) for x in P(*c, *k)) == want


@pytest.mark.parametrize("rate", [0.0, 0.1, 0.25, 0.5])
def test_mask_keep_rate(jb, rate):
    m = jb.train.dropout_mask_host(12345, 7, 3, 1, 500, 768, rate)
    assert m.dtype == np.uint8 and m.shape == (500, 768)
    if rate == 0.0:
        assert m.all()
    else:
        assert abs(m.mean() - (1 - rate)) < 0.005


def test_masks_are_independent(jb):
    """q, k and v of one block see different masks of the same input; so do blocks, steps and seeds."""
    base = jb.train.dropout_mask_host(1, 0, 0, 0, 64, 768, 0.25)
    for args in [(1, 0, 0, 1), (1, 0, 0, 2), (1, 0, 0, 3), (1, 0, 1, 0), (1, 1, 0, 0), (2, 0, 0, 0)]:
        other = jb.train.dropout_mask_host(*args, 64, 768, 0.25)
        agree = (other == base).mean()
        assert 0.55 < agree < 0.70      # independent masks of keep rate 0.75 agree on 0.75^2 + 0.25^2 = 0.625


def test_mask_is_a_function_of_row_and_column(jb):
    """The row index is global within a call, so a mask does not depend on how views are split into passes."""
    full = jb.train.dropout_mask_host(9, 4, 2, 0, 300, 768, 0.25)
    assert np.array_equal(full[:120], jb.train.dropout_mask_host(9, 4, 2, 0, 120, 768, 0.25))


def test_training_entry_points_are_bound(jb):
    for name in ("jcb_vit_train_set_lora", "jcb_vit_train_forward", "jcb_vit_train_forward_dlpack", "jcb_vit_train_backward",
                 "jcb_tape_release", "jcb_lora_dropout_mask"):
        assert name in jb._capi.PROTOTYPES


def test_trainer_rejects_layers_without_adapters(jb):
    import types
    sd = jb.synth.make_vit_state_dict(seed=0, layers=1)
    model = jb.jclip.build_model(sd)
    args = types.SimpleNamespace(encoder="vision", position="all", params=["q"], r=0, alpha=1, dropout_rate=0.25,
                                 backbone="ViT-B/32")
    layers = jb.apply_lora(args, model)
    if torch.cuda.is_available():
        with pytest.raises(ValueError, match="no adapter"):
            jb.LoraTrainer(model, layers)
    else:
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            jb.LoraTrainer(model, layers)
