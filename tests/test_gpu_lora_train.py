"""GPU: image-tower LoRA training (`LoraTrainer`, jcb_vit_train_*): dL/dA and dL/dB of the device backward pass against
torch autograd through a fp32 CPU restatement of the tower (oracle/vit.py's layer_norm / quick_gelu and the
VisionTransformer.execute order of oracle.vit.vit_encode_image, with A and B as leaf tensors and the LoRA branch
input dropped out by the host reproduction of the device masks).

Bounds: per adapter tensor, cosine >= 0.999 and relative L2 error <= 2e-2 (16-bit forward operands, bf16 backward
operands, fp32 accumulation).  The bound has power: dropping the LoRA term of the input gradients, or the ln_2
backward, moves the reference gradients by many times it (test_bound_has_power).
"""
import os
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

COS_MIN, REL_MAX = 0.999, 2e-2
_PROJ = (("q_proj", 0), ("k_proj", 1), ("v_proj", 2), ("proj", 3))


def _args(params=("q", "k", "v"), r=4, position="all", rate=0.0):
    return types.SimpleNamespace(encoder="vision", position=position, params=list(params), r=r, alpha=1,
                                 dropout_rate=rate, backbone="ViT-B/32", filename="lora_weights")


def _model(jb, layers=2, vpt=0, params=("q", "k", "v"), r=4, position="all", rate=0.0, seed=3):
    sd = jb.synth.make_vit_state_dict(seed=seed, layers=layers, vpt_tokens=vpt)
    if vpt:
        sd["visual.VPT"] = sd["visual.VPT"] * 25.0
        model = jb.jclip.build_model(sd, dict(jb.clip.IVLP_DESIGN))
    else:
        model = jb.jclip.build_model(sd)
    if layers < 12 and position != "all":
        raise ValueError("position tables index 12 blocks")
    lora_layers = jb.apply_lora(_args(params, r, position, rate), model)
    rng = np.random.default_rng(seed + 100)
    for attn in lora_layers:
        for name, _ in _PROJ:
            lin = getattr(attn, name)
            if lin.lora_enabled:
                lin.w_lora_A.data = (rng.standard_normal(lin.w_lora_A.shape) * 0.05).astype(np.float32)
                lin.w_lora_B.data = (rng.standard_normal(lin.w_lora_B.shape) * 0.05).astype(np.float32)
    return sd, model, lora_layers


def _views(n, seed=5):
    return torch.from_numpy(jb_views(n, seed))


def jb_views(n, seed):
    import jclip_b200
    v = jclip_b200.synth.make_views(seed, 1, n)
    return jclip_b200.synth.clip_normalize(v.reshape(n, 3, 224, 224)).astype(np.float32)


def ref_features(sd, images, adapters, normalize, masks=None, rate=0.0, cut_lora_dx=False, cut_ln2=False):
    """VisionTransformer.execute in fp32 with the applied LoRA branch s B (A dropout(x)) (reference test.py:388-398);
    adapters {(block, code): (A, B, s)}; masks {(block, code): [n * T, W] keep mask} or None.
    cut_lora_dx / cut_ln2: the two ablations of test_bound_has_power."""
    from oracle.vit import layer_norm, quick_gelu
    g = lambda k: torch.from_numpy(np.asarray(sd[k], np.float32))
    x = images
    conv_w = g("visual.conv1.weight")
    W = conv_w.shape[0]
    P = conv_w.shape[-1]
    heads = W // 64
    L = len([k for k in sd if k.startswith("visual.") and k.endswith(".attn.in_proj_weight")])
    x = torch.nn.functional.conv2d(x, conv_w, stride=P)
    x = x.reshape(x.shape[0], W, -1).permute(0, 2, 1)
    x = torch.cat([g("visual.class_embedding").view(1, 1, -1).expand(x.shape[0], 1, -1), x], 1) + g("visual.positional_embedding")
    if "visual.VPT" in sd:
        x = torch.cat([x, g("visual.VPT").unsqueeze(0).expand(x.shape[0], -1, -1)], 1)
    x = layer_norm(x, g("visual.ln_pre.weight"), g("visual.ln_pre.bias"))
    n, T, _ = x.shape

    def lora(h, blk, code):
        if (blk, code) not in adapters:
            return 0.0
        A, B, s = adapters[(blk, code)]
        hi = h.detach() if cut_lora_dx else h
        if masks is not None:
            hi = hi * masks[(blk, code)].view(n, T, W) / (1.0 - rate)
        return (hi @ A.t()) @ B.t() * s

    for i in range(L):
        p = f"visual.transformer.resblocks.{i}."
        h = layer_norm(x, g(p + "ln_1.weight"), g(p + "ln_1.bias"))
        w_in, b_in = g(p + "attn.in_proj_weight"), g(p + "attn.in_proj_bias")
        q = h @ w_in[:W].t() + b_in[:W] + lora(h, i, 0)
        k = h @ w_in[W:2 * W].t() + b_in[W:2 * W] + lora(h, i, 1)
        v = h @ w_in[2 * W:].t() + b_in[2 * W:] + lora(h, i, 2)
        sh = lambda t: t.view(n, T, heads, 64).permute(0, 2, 1, 3)
        att = torch.softmax(sh(q) @ sh(k).transpose(-2, -1) / 8.0, -1)
        o = (att @ sh(v)).permute(0, 2, 1, 3).reshape(n, T, W)
        x = x + o @ g(p + "attn.out_proj.weight").t() + g(p + "attn.out_proj.bias") + lora(o, i, 3)
        xin = x.detach() if cut_ln2 else x
        h = layer_norm(xin, g(p + "ln_2.weight"), g(p + "ln_2.bias"))
        h = quick_gelu(h @ g(p + "mlp.c_fc.weight").t() + g(p + "mlp.c_fc.bias"))
        mlp = h @ g(p + "mlp.c_proj.weight").t() + g(p + "mlp.c_proj.bias")
        x = (x + mlp) if not cut_ln2 else (x + mlp + 0.0 * xin)
    f = layer_norm(x[:, 0, :], g("visual.ln_post.weight"), g("visual.ln_post.bias")) @ g("visual.proj")
    return f / f.norm(dim=-1, keepdim=True) if normalize else f


def _ref_grads(jb, sd, trainer, images, dfeat, normalize, rate=0.0, step=0, **cut):
    adapters, leaves = {}, []
    for (blk, code), k in trainer._slots.items():
        A = trainer._params[2 * k].detach().cpu().clone().requires_grad_(True)
        B = trainer._params[2 * k + 1].detach().cpu().clone().requires_grad_(True)
        adapters[(blk, code)] = (A, B, float(trainer._lins[k].scaling))
        leaves += [A, B]
    masks = None
    if rate > 0:
        n, T = images.shape[0], _tokens(trainer)
        masks = {key: torch.from_numpy(jb.train.dropout_mask_host(trainer.seed, step, key[0], key[1], n * T,
                                                                  trainer.visual.width, rate).astype(np.float32))
                 for key in adapters}
    torch.set_num_threads(os.cpu_count() or 1)
    f = ref_features(sd, images, adapters, normalize, masks=masks, rate=rate, **cut)
    (f * dfeat).sum().backward()
    return f.detach(), [t.grad for t in leaves]


def _tokens(trainer):
    v = trainer.visual
    return (v.input_resolution // v.patch_size) ** 2 + 1 + v.n_ctx


def _dev_grads(trainer, images_dev, dfeat):
    for p in trainer.parameters():
        p.grad = None
    f = trainer(images_dev)
    f.backward(dfeat.to(images_dev.device))
    return f.detach().cpu(), [p.grad.detach().cpu() for p in trainer.parameters()]


def _compare(dev, ref, what=""):
    for i, (a, b) in enumerate(zip(dev, ref)):
        a, b = a.double().flatten(), b.double().flatten()
        cos = float(a @ b / (a.norm() * b.norm()))
        rel = float((a - b).norm() / b.norm())
        assert cos >= COS_MIN and rel <= REL_MAX, f"{what} tensor {i}: cos {cos:.6f} rel {rel:.4f}"


CASES = [  # layers, vpt, params, r, position, views, normalize
    (2, 0, ("q", "k", "v"), 4, "all", 1, True),
    (2, 0, ("q", "k", "v", "o"), 16, "all", 7, False),
    (2, 4, ("q", "k", "v", "o"), 4, "all", 130, True),
    (2, 4, ("q", "k", "v"), 16, "all", 7, False),
    (12, 0, ("q", "k", "v", "o"), 4, "all", 1, True),
    (12, 4, ("q", "k", "v"), 16, "up", 7, True),
]


@pytest.fixture
def applied_ctx(jb, cuda_dev):
    ctx = jb.get_context(cuda_dev)
    prev = ctx.lora_mode
    yield ctx
    ctx.set_lora_mode(prev)


@pytest.mark.parametrize("operands", ["f16", "bf16"])
@pytest.mark.parametrize("layers,vpt,params,r,position,n,normalize", CASES)
def test_gradient_parity(jb, cuda_dev, applied_ctx, operands, layers, vpt, params, r, position, n, normalize):
    applied_ctx.set_operand_type(operands)
    try:
        sd, model, lora_layers = _model(jb, layers, vpt, params, r, position)
        trainer = jb.LoraTrainer(model, lora_layers, seed=1, normalize=normalize)
        images = _views(n)
        dfeat = torch.randn(n, 512, generator=torch.Generator().manual_seed(n + layers))
        f_dev, g_dev = _dev_grads(trainer, images.to(cuda_dev), dfeat)
        f_ref, g_ref = _ref_grads(jb, sd, trainer, images, dfeat, normalize)
        assert torch.nn.functional.cosine_similarity(f_dev.double(), f_ref.double()).min() > 0.999
        _compare(g_dev, g_ref, f"{layers} blocks {params} r={r} {position} n={n}")
    finally:
        applied_ctx.set_operand_type("f16")


def test_ref_restatement_is_the_oracle(jb):
    """The differentiable restatement equals oracle.vit.vit_encode_image on the same adapters (no dropout)."""
    from oracle import vit_encode_image
    sd, model, lora_layers = _model(jb, 2, 0, ("q", "k", "v", "o"), 4)
    images = _views(2)
    lora, adapters = {}, {}
    for i, attn in enumerate(lora_layers):
        lora[i] = {}
        for name, code in _PROJ:
            lin = getattr(attn, name)
            lora[i][name] = (lin.w_lora_A.data, lin.w_lora_B.data)
            adapters[(i, code)] = (torch.from_numpy(lin.w_lora_A.data), torch.from_numpy(lin.w_lora_B.data), lin.scaling)
    want = vit_encode_image(sd, images, lora=lora, scaling=lora_layers[0].q_proj.scaling, normalize=True)
    with torch.no_grad():
        got = ref_features(sd, images, adapters, True)
    assert torch.allclose(got, want, atol=1e-5)


def test_bound_has_power(jb, cuda_dev, applied_ctx):
    """Without the LoRA term of the input gradients, or without the ln_2 backward, the reference gradients move by far
    more than the bound: a device backward missing either piece would fail test_gradient_parity."""
    sd, model, lora_layers = _model(jb, 2, 0, ("q", "k", "v", "o"), 16)
    trainer = jb.LoraTrainer(model, lora_layers, seed=1)
    images = _views(3)
    dfeat = torch.randn(3, 512, generator=torch.Generator().manual_seed(9))
    _, full = _ref_grads(jb, sd, trainer, images, dfeat, True)
    for cut in ({"cut_lora_dx": True}, {"cut_ln2": True}):
        _, ablated = _ref_grads(jb, sd, trainer, images, dfeat, True, **cut)
        worst = max(float((a - b).norm() / b.norm()) for a, b in zip(ablated, full))
        assert worst > 5 * REL_MAX, (cut, worst)


def test_dropout_mask_matches_host(jb, cuda_dev):
    for seed, step, layer, proj, rate in [(0, 0, 0, 0, 0.25), (2 ** 40 + 7, 123, 11, 3, 0.5), (99, 5, 4, 1, 0.1)]:
        dev = jb.train.dropout_mask(seed, step, layer, proj, 130 * 50, 768, rate, device=cuda_dev).cpu().numpy()
        host = jb.train.dropout_mask_host(seed, step, layer, proj, 130 * 50, 768, rate)
        assert np.array_equal(dev, host)
        assert abs(dev.mean() - (1 - rate)) < 0.01
    a = jb.train.dropout_mask(1, 0, 0, 0, 64, 768, 0.25, device=cuda_dev)
    b = jb.train.dropout_mask(1, 0, 0, 1, 64, 768, 0.25, device=cuda_dev)
    assert not torch.equal(a, b)          # q and k see different masks of the same input


def test_dropout_gradients(jb, cuda_dev, applied_ctx):
    """Training dropout 0.25: the device gradients against the reference run with the host-reproduced masks, for
    two steps (different masks)."""
    sd, model, lora_layers = _model(jb, 2, 0, ("q", "k", "v", "o"), 8, rate=0.25)
    trainer = jb.LoraTrainer(model, lora_layers, seed=77)
    assert trainer.dropout_rate == 0.25
    images = _views(7)
    for step in range(2):
        dfeat = torch.randn(7, 512, generator=torch.Generator().manual_seed(step))
        assert trainer.step == step
        _, g_dev = _dev_grads(trainer, images.to(cuda_dev), dfeat)
        _, g_ref = _ref_grads(jb, sd, trainer, images, dfeat, True, rate=0.25, step=step)
        _compare(g_dev, g_ref, f"dropout step {step}")


def test_eval_is_encode_image(jb, cuda_dev, applied_ctx):
    sd, model, lora_layers = _model(jb, 2, 4, ("q", "k", "v", "o"), 4, rate=0.25)
    trainer = jb.LoraTrainer(model, lora_layers, seed=1)
    images = _views(9).to(cuda_dev)
    f_eval = trainer.eval()(images)
    f_enc = model.visual(images, normalize=True)
    assert torch.equal(f_eval, f_enc)
    # training mode with rate 0 runs the same tower (to rounding: the LoRA down-projection is one GEMM over the three
    # dropout copies there)
    trainer.dropout_rate = 0.0
    f_train = trainer.train()(images).detach()
    assert torch.nn.functional.cosine_similarity(f_train, f_enc).min() > 0.99999


def test_determinism_and_pass_split(jb, cuda_dev, applied_ctx):
    sd, model, lora_layers = _model(jb, 2, 0, ("q", "k", "v", "o"), 4, rate=0.25)
    images = _views(130).to(cuda_dev)
    dfeat = torch.randn(130, 512, generator=torch.Generator().manual_seed(3))
    runs = []
    for _ in range(2):
        trainer = jb.LoraTrainer(model, lora_layers, seed=5)
        runs.append(_dev_grads(trainer, images, dfeat)[1])
    for a, b in zip(*runs):
        assert torch.equal(a, b)
    applied_ctx.set_chunk_views(40)           # 4 forward passes of 32-33 views instead of one
    try:
        trainer = jb.LoraTrainer(model, lora_layers, seed=5)
        split = _dev_grads(trainer, images, dfeat)[1]
    finally:
        applied_ctx.set_chunk_views(16384)
    for a, b in zip(split, runs[0]):
        assert float((a - b).norm() / b.norm()) < 1e-2


def _fewshot_data(n_classes=8, shots=4, seed=0):
    g = torch.Generator().manual_seed(seed)
    images = torch.from_numpy(jb_views(n_classes * shots, seed + 11))
    labels = torch.arange(n_classes).repeat_interleave(shots)
    text = torch.nn.functional.normalize(torch.randn(n_classes, 512, generator=g), dim=-1)
    return images, labels, text


def _loop(params, forward, images, labels, text, steps=30, lr=2e-3):
    opt = torch.optim.AdamW(params, lr=lr, weight_decay=1e-2)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, steps)
    losses = []
    for _ in range(steps):
        f = forward(images)
        loss = torch.nn.functional.cross_entropy(100 * f @ text.T.to(f.device), labels.to(f.device))
        opt.zero_grad()
        loss.backward()
        opt.step()
        sched.step()
        losses.append(loss.item())
    return losses


def test_training_loop(jb, cuda_dev, applied_ctx, tmp_path):
    """30 AdamW steps of the reference recipe (100 f T^T logits, cross-entropy, cosine schedule) on seeded synthetic
    few-shot data without dropout: the loss decreases and each step's loss stays within 0.05 (relative) of the same loop
    with torch autograd over the fp32 restatement.  The pickle the trainer saves reloads (load_lora) to the same eval
    features."""
    sd, model, lora_layers = _model(jb, 2, 0, ("q", "k", "v"), 4)
    images, labels, text = _fewshot_data()
    trainer = jb.LoraTrainer(model, lora_layers, seed=0)
    dev_losses = _loop(trainer.parameters(), trainer, images.to(cuda_dev), labels, text)
    # reference run from the same initial adapters
    sd2, model2, lora_layers2 = _model(jb, 2, 0, ("q", "k", "v"), 4)
    ref_ad = {}
    for i, attn in enumerate(lora_layers2):
        for name, code in _PROJ:
            lin = getattr(attn, name)
            if lin.lora_enabled:
                ref_ad[(i, code)] = (torch.from_numpy(lin.w_lora_A.data.copy()).requires_grad_(True),
                                     torch.from_numpy(lin.w_lora_B.data.copy()).requires_grad_(True), lin.scaling)
    torch.set_num_threads(os.cpu_count() or 1)
    ref_params = [t for a in ref_ad.values() for t in a[:2]]
    ref_losses = _loop(ref_params, lambda x: ref_features(sd2, x, ref_ad, True), images, labels, text)
    assert dev_losses[-1] < 0.7 * dev_losses[0]
    for a, b in zip(dev_losses, ref_losses):
        assert abs(a - b) <= 0.05 * abs(b) + 1e-3, (dev_losses, ref_losses)
    # save -> load_lora -> the same eval features
    args = _args(("q", "k", "v"), 4)
    path = trainer.save(args, 30, lora_layers, save_dir=str(tmp_path))
    f_trained = trainer.eval()(images.to(cuda_dev))
    sd3, model3, lora_layers3 = _model(jb, 2, 0, ("q", "k", "v"), 4, seed=3)
    jb.load_lora(args, lora_layers3, path)
    f_loaded = model3.visual(images.to(cuda_dev), normalize=True)
    assert torch.equal(f_trained, f_loaded)


def test_rejections(jb, cuda_dev, applied_ctx):
    from ctypes import byref, c_void_p
    lib = jb.load_library()
    out = torch.full((2, 512), 7.0, device=cuda_dev)
    images = _views(2).to(cuda_dev)

    def forward_rc(model):
        ctx, vit = model.visual._engine(cuda_dev)
        ctx.bind_current_stream()
        tape = c_void_p()
        return lib.jcb_vit_train_forward(vit, c_void_p(images.data_ptr()), 0, 2, 0, 1, 0.0, 0, 0, c_void_p(out.data_ptr()),
                                         byref(tape)), tape

    # a 197-token tower (ViT-B/16)
    sd = jb.synth.make_vit_state_dict(seed=1, layers=1, patch=16)
    m16 = jb.jclip.build_model(sd)
    jb.apply_lora(types.SimpleNamespace(**{**vars(_args()), "backbone": "ViT-B/16"}), m16)
    rc, tape = forward_rc(m16)
    assert rc == jb._capi.JCB_E_INVALID and not tape.value
    # several slots (applied mode, so that the tower packs)
    applied_ctx.set_lora_mode("applied")
    sd, model, lora_layers = _model(jb, 2)
    model.visual.set_lora_slots([{0: {"q": (np.ones((4, 768), np.float32), np.ones((768, 4), np.float32))}}])
    rc, tape = forward_rc(model)
    assert rc == jb._capi.JCB_E_INVALID and not tape.value
    model.visual.set_lora_slots([])
    # no adapter
    sd0 = jb.synth.make_vit_state_dict(seed=1, layers=2)
    m0 = jb.jclip.build_model(sd0)
    rc, tape = forward_rc(m0)
    assert rc == jb._capi.JCB_E_INVALID
    # ranks over 64 (q, k, v of r = 32 each): the applied-mode tower cannot be packed, training refuses it too
    sd, model, lora_layers = _model(jb, 2, r=32)
    with pytest.raises(jb.JcbError):
        jb.LoraTrainer(model, lora_layers)(images)
    # an unfinalized tower
    vit = c_void_p()
    ctx = jb.get_context(cuda_dev)
    cfg = jb._capi.VitConfig(2, 768, 32, 224, 512, 0)
    assert lib.jcb_vit_create(ctx.handle, byref(cfg), byref(vit)) == 0
    tape = c_void_p()
    assert lib.jcb_vit_train_forward(vit, c_void_p(images.data_ptr()), 0, 2, 0, 1, 0.0, 0, 0, c_void_p(out.data_ptr()),
                                     byref(tape)) == jb._capi.JCB_E_INVALID
    lib.jcb_vit_destroy(vit)
    torch.cuda.synchronize()
    assert (out == 7.0).all()                # outputs untouched
