"""CPU: the host side of ViT-B/16 (patch 16, 14 x 14 grid, 197 tokens) and the power of the long attention kernel's
tolerance (tests/test_gpu_vit_b16.py)."""
import types

import pytest
import torch

from test_gpu_vit_b16 import ATOL, LONG_SHAPES, OPS, ULP, _attention_ref


def test_build_model_infers_vit_b16(jb):
    sd = jb.synth.make_vit_state_dict(seed=0, patch=16)
    model = jb.jclip.build_model(sd)
    v = model.visual
    assert (v.patch_size, v.input_resolution, v.heads, v.width) == (16, 224, 12, 768)
    assert v.positional_embedding.shape[0] == 197 == (224 // 16) ** 2 + 1
    args = types.SimpleNamespace(encoder="vision", position="top", params=["q", "k", "v"], r=4, alpha=1,
                                 dropout_rate=0.25, backbone="ViT-B/16")
    layers = jb.apply_lora(args, model)
    blocks = model.visual.transformer.resblocks
    assert len(layers) == 1 and layers[0] is blocks[11].attn
    assert [i for i, b in enumerate(blocks) if getattr(b.attn, "is_lora", False)] == [11]


def _mutants(qkv, n, T, H):
    """The fp32 reference with each of three indexing mistakes a 256-key, two-query-tile kernel can make."""
    d, nkb = 64, (T + 63) // 64
    x = qkv.float().view(n, T, 3, H, d)
    q, k, v = (x[:, :, i].permute(0, 2, 1, 3) for i in range(3))          # [n, H, T, 64]
    s = q @ k.transpose(-2, -1) / 8.0
    heads = lambda o: o.permute(0, 2, 1, 3).reshape(n * T, H * d)
    # 1. the last key box is not loaded / not multiplied: keys 64 (nkb - 1) .. T - 1 missing
    kk = 64 * (nkb - 1)
    drop = heads(torch.softmax(s[..., :kk], -1) @ v[:, :, :kk])
    # 2. the zero-filled keys T .. 64 nkb - 1 (score 0, value 0) enter the softmax (where the last box has more than one)
    pad = 64 * nkb - T
    sp = torch.cat([s, s.new_zeros(*s.shape[:-1], pad)], -1)
    vp = torch.cat([v, v.new_zeros(n, H, pad, d)], 2)
    padded = heads(torch.softmax(sp, -1) @ vp) if pad > 1 else None
    # 3. query tile 1 computed from tile 0's query rows
    o = torch.softmax(s, -1) @ v
    o1 = o.clone()
    o1[:, :, 128:] = o[:, :, :T - 128]
    return {"last key box dropped": drop, "padding keys in the softmax": padded, "tile 0 queries in tile 1": heads(o1)}


@pytest.mark.parametrize("op", OPS, ids=["bf16", "f16"])
def test_tolerances_have_power(op):
    """On the kernel test's inputs (every shape up to 300 sequences, same seeds), each mistake moves the fp32 reference
    by at least 3x the attention tolerance (1e-2 / 2e-3 absolute + one ulp) at some element of every shape.  The padding
    mistake is measured on the five shapes with 32 to 63 zero-filled keys; T = 255 has a single one, which moves the
    reference by only 0.1x (bf16) / 0.7x (fp16) of the tolerance, and runs the same masking code as the others.

    Measured smallest margins (max |mutant - ref| / tolerance over a shape, smallest over the shapes):
      bf16: last key box dropped 34.7x, padding keys in the softmax 6.2x, tile 0 queries in tile 1 93x
      fp16: last key box dropped 175x, padding keys in the softmax 34x, tile 0 queries in tile 1 484x
    """
    worst = {}
    for n, T, H in LONG_SHAPES:
        if n > 300:
            continue
        g = torch.Generator().manual_seed(n * 1000 + T * 10 + H)
        qkv = (torch.randn(n * T, 3 * H * 64, generator=g) * 1.2).to(op)
        ref = _attention_ref(qkv, n, T, H, False)
        tol = ATOL[op] + ULP[op] * ref.abs()
        for name, mut in _mutants(qkv, n, T, H).items():
            if mut is None:
                continue
            r = float(((mut - ref).abs() / tol).max())
            worst[name] = min(worst.get(name, float("inf")), r)
    print(op, {k: round(v, 1) for k, v in worst.items()})
    assert all(r >= 3.0 for r in worst.values()), worst
