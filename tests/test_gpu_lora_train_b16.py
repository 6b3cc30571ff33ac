"""GPU: LoRA training on ViT-B/16 image towers (197 tokens, 201 with IVLP prompts).

The attention backward of 65 <= T <= 256 tokens runs on attention_bwd_tcgen05_kernel (csrc/train.cu); T <= 64 keeps
attention_bwd_kernel.  The kernel is checked alone against torch fp32 autograd of softmax(q k^T / 8) v, per gradient
(dq, dk, dv) with cosine >= 0.999 and relative L2 error <= 2e-2 (bf16 P, dO and dS, bf16 output, fp32 accumulation;
an fp16 tower's q, k, v are rounded to bf16 in the kernel).  The bound has power: dropping the D = rowsum(P dP) term,
or the 1/8 of dS, moves the reference far beyond it.  The tower's dA and dB are checked against the fp32 restatement
of tests/test_gpu_lora_train.py within that file's bounds.
"""
import types

import numpy as np
import pytest
import torch

from test_gpu_lora_train import _compare, _dev_grads, _ref_grads, jb_views, ref_features

pytestmark = pytest.mark.gpu

COS_MIN, REL_MAX = 0.999, 2e-2
_PROJ = (("q_proj", 0), ("k_proj", 1), ("v_proj", 2), ("proj", 3))
OPS = [torch.float16, torch.bfloat16]


# ------------------------------------------------------------------------------------------------ the kernel alone
def _inputs(kind, n, T, H, g):
    """q | k | v [n T, 3 64 H] fp32 and dO [n T, 64 H]; v carries a mean so that the D term of dS matters."""
    q, k, v = (torch.randn(n, T, H, 64, generator=g) for _ in range(3))
    v = v + 1.0
    if kind == "peaked":          # scores / 8 with a standard deviation of about 3
        q = q * 3.0
    elif kind == "dominant":      # one key takes most of every query's weight
        u = torch.nn.functional.normalize(torch.randn(n, 1, H, 64, generator=g), dim=-1)
        q = q + 4.0 * u
        k[:, T // 2] = 16.0 * u[:, 0]
    elif kind == "equal":         # every score equal: P uniform
        q = torch.zeros_like(q)
    qkv = torch.stack([q, k, v], 2).reshape(n * T, 3 * H * 64)
    dout = torch.randn(n * T, H * 64, generator=g)
    return qkv, dout


def _ref(qkv, dout, n, T, H, drop_d=False, no_scale=False):
    """torch fp32 autograd of softmax(q k^T / 8) v; drop_d / no_scale: the two ablations of the bound's power test."""
    x = qkv.double().view(n, T, 3, H, 64).permute(2, 0, 3, 1, 4)
    q, k, v = (t.clone().requires_grad_(True) for t in x)
    do = dout.double().view(n, T, H, 64).permute(0, 2, 1, 3)
    if not (drop_d or no_scale):
        o = torch.softmax(q @ k.transpose(-1, -2) / 8.0, -1) @ v
        o.backward(do)
        grads = [q.grad, k.grad, v.grad]
    else:
        q, k, v = (t.detach() for t in (q, k, v))
        P = torch.softmax(q @ k.transpose(-1, -2) / 8.0, -1)
        dP = do @ v.transpose(-1, -2)
        D = 0.0 if drop_d else (P * dP).sum(-1, keepdim=True)
        dS = P * (dP - D) / (1.0 if no_scale else 8.0)
        grads = [dS @ k, dS.transpose(-1, -2) @ q, P.transpose(-1, -2) @ do]
    return torch.stack(grads, 2).permute(0, 3, 2, 1, 4).reshape(n * T, 3 * H * 64)


def _errors(got, ref, W):
    out = []
    for i in range(3):
        a, b = got[:, i * W:(i + 1) * W].double().flatten(), ref[:, i * W:(i + 1) * W].double().flatten()
        out.append((float(a @ b / (a.norm() * b.norm())), float((a - b).norm() / b.norm())))
    return out


def _run(jb, cuda_dev, qkv16, dout, n, T, H, guard=64):
    """dqkv from the device into a NaN-filled buffer with `guard` NaN rows past it; returns (dqkv, guard rows)."""
    buf = torch.full((n * T + guard, 3 * H * 64), float("nan"), dtype=torch.bfloat16, device=cuda_dev)
    jb.blocks.attention_bwd(qkv16.to(cuda_dev), dout.to(cuda_dev), n, T, H, buf)
    return buf[:n * T].float().cpu(), buf[n * T:].float().cpu()


@pytest.mark.parametrize("op", OPS, ids=["f16", "bf16"])
@pytest.mark.parametrize("T,H,n", [(65, 12, 40), (96, 4, 300), (127, 12, 24), (128, 4, 100), (129, 12, 24),
                                   (197, 12, 125), (201, 4, 60), (255, 12, 8), (256, 4, 1500)])
def test_kernel_matches_autograd(jb, cuda_dev, op, T, H, n):
    g = torch.Generator().manual_seed(T * 31 + H)
    qkv, dout = _inputs("random", n, T, H, g)
    qkv16 = qkv.to(op)
    got, guard = _run(jb, cuda_dev, qkv16, dout, n, T, H)
    assert torch.isnan(guard).all()                       # nothing written past the output
    assert torch.isfinite(got).all()                      # every output element written
    ref = _ref(qkv16.float(), dout, n, T, H)
    for what, (cos, rel) in zip("qkv", _errors(got, ref, 64 * H)):
        assert cos >= COS_MIN and rel <= REL_MAX, f"d{what}: cos {cos:.6f} rel {rel:.4f}"


@pytest.mark.parametrize("op", OPS, ids=["f16", "bf16"])
@pytest.mark.parametrize("kind", ["peaked", "dominant", "equal"])
def test_kernel_hard_inputs(jb, cuda_dev, op, kind):
    n, T, H = 16, 197, 12
    g = torch.Generator().manual_seed(7)
    qkv, dout = _inputs(kind, n, T, H, g)
    qkv16 = qkv.to(op)
    got, guard = _run(jb, cuda_dev, qkv16, dout, n, T, H)
    assert torch.isnan(guard).all() and torch.isfinite(got).all()
    ref = _ref(qkv16.float(), dout, n, T, H)
    W = 64 * H
    errs = _errors(got, ref, W)
    if kind == "equal":           # q = 0: dk is exactly zero (every score has the same derivative sum), compare dq, dv
        assert got[:, W:2 * W].abs().max() < 1e-6
        errs = [errs[0], errs[2]]
    for cos, rel in errs:
        assert cos >= COS_MIN and rel <= REL_MAX, (kind, errs)
    P = torch.softmax(qkv16.float().view(n, T, 3, H, 64)[:, :, 0].transpose(1, 2) @
                      qkv16.float().view(n, T, 3, H, 64)[:, :, 1].permute(0, 2, 3, 1) / 8.0, -1)
    if kind == "peaked":          # the inputs do what they claim
        assert P.max(-1).values.mean() > 0.3       # uniform: 1 / 197
    if kind == "dominant":
        assert P[..., T // 2].mean() > 0.75


def test_kernel_bound_has_power():
    """Without the D term, or with dS missing its 1/8, the reference moves by many times the bound."""
    n, T, H = 8, 197, 4
    qkv, dout = _inputs("random", n, T, H, torch.Generator().manual_seed(1))
    full = _ref(qkv, dout, n, T, H)
    W = 64 * H
    for cut in ({"drop_d": True}, {"no_scale": True}):
        ablated = _ref(qkv, dout, n, T, H, **cut)
        rel_dq = _errors(ablated, full, W)[0][1]
        assert rel_dq > 5 * REL_MAX, (cut, rel_dq)


# The routing check profiles in a child process.  Opened in the pytest process after this file's other GPU work, a torch
# profiler session (with or without a warm-up schedule) left every later session of that process missing its first
# kernels, which broke the profiler-based route checks of test_gpu_mta_routes that run after this file.
_ROUTES_SCRIPT = r"""
import json, re, sys
sys.path.insert(0, sys.argv[1])
import torch
from torch.profiler import ProfilerActivity, profile
import jclip_b200 as jb
dev = torch.device("cuda", 0)
cases = []
for T in (50, 64, 65, 197, 256):
    qkv = torch.randn(4 * T, 3 * 12 * 64, device=dev).half()
    dout = torch.randn(4 * T, 12 * 64, device=dev)
    dqkv = torch.empty(4 * T, 3 * 12 * 64, dtype=torch.bfloat16, device=dev)
    jb.blocks.attention_bwd(qkv, dout, 4, T, 12, dqkv)
    cases.append((T, qkv, dout, dqkv))
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(2):                                  # 0: warm-up, 1: checked
        for T, qkv, dout, dqkv in cases:
            dqkv.fill_(float("nan"))
            jb.blocks.attention_bwd(qkv, dout, 4, T, 12, dqkv, sync=False)
        torch.cuda.synchronize()
launched = []
for e in prof.events():
    m = re.search(r"(attention_bwd_(?:tcgen05_)?kernel)", e.name)
    if m and e.device_type == torch.autograd.DeviceType.CUDA:
        launched.append((e.time_range.start, m.group(1)))
print(json.dumps({"finite": all(bool(torch.isfinite(c[3].float()).all()) for c in cases),
                  "names": [name for _, name in sorted(launched)]}))
"""


def test_kernel_routes(jb, cuda_dev):
    """T <= 64 runs attention_bwd_kernel, 65 <= T <= 256 the tcgen05 kernel.  One profiler session (in a child
    process, see above) records a warm-up pass and then the checked pass of the same launches: the first launches of a
    session can go unrecorded, and those belong to the warm-up pass."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-c", _ROUTES_SCRIPT, root], capture_output=True, text=True, timeout=600, cwd=root)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    got = json.loads(r.stdout.strip().splitlines()[-1])
    want = ["attention_bwd_kernel"] * 2 + ["attention_bwd_tcgen05_kernel"] * 3
    # every launch of the checked pass ran: a missing name below is the profiler's, not a kernel that did not run
    assert got["finite"]
    assert len(got["names"]) >= len(want) and got["names"][-len(want):] == want, got["names"]


@pytest.mark.parametrize("T", [0, 257])
def test_kernel_rejects_out_of_range(jb, cuda_dev, T):
    rows = max(T, 1)
    qkv = torch.zeros(rows, 3 * 64, dtype=torch.float16, device=cuda_dev)
    dout = torch.zeros(rows, 64, device=cuda_dev)
    dqkv = torch.full((rows, 3 * 64), float("nan"), dtype=torch.bfloat16, device=cuda_dev)
    with pytest.raises(jb.JcbError) as e:
        jb.blocks.attention_bwd(qkv, dout, 1, T, 1, dqkv)
    assert e.value.code == jb._capi.JCB_E_INVALID
    assert torch.isnan(dqkv.float()).all()


# ------------------------------------------------------------------------------------------------ the tower
def _args(params=("q", "k", "v"), r=4, position="all", rate=0.0):
    return types.SimpleNamespace(encoder="vision", position=position, params=list(params), r=r, alpha=1,
                                 dropout_rate=rate, backbone="ViT-B/16", filename="lora_weights")


def _model(jb, layers=2, vpt=0, params=("q", "k", "v"), r=4, position="all", rate=0.0, seed=3):
    sd = jb.synth.make_vit_state_dict(seed=seed, layers=layers, vpt_tokens=vpt, patch=16)
    if vpt:
        sd["visual.VPT"] = sd["visual.VPT"] * 25.0
        model = jb.jclip.build_model(sd, dict(jb.clip.IVLP_DESIGN))
    else:
        model = jb.jclip.build_model(sd)
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


@pytest.fixture
def applied_ctx(jb, cuda_dev):
    ctx = jb.get_context(cuda_dev)
    prev, prev_chunk = ctx.lora_mode, ctx.chunk_views
    yield ctx
    ctx.set_lora_mode(prev)
    ctx.set_chunk_views(prev_chunk)
    ctx.set_operand_type("f16")


CASES = [  # layers, vpt, params, r, position, views, normalize, chunk_views (None: the default)
    (2, 0, ("q", "k", "v"), 4, "all", 1, True, None),
    (2, 0, ("q", "k", "v", "o"), 16, "all", 7, False, None),
    (2, 4, ("q", "k", "v", "o"), 4, "all", 30, True, 40),      # 12 views per pass: three forward and backward passes
    (2, 4, ("q", "k", "v"), 16, "all", 7, False, None),
    (12, 0, ("q", "k", "v", "o"), 4, "all", 1, True, None),
    (12, 4, ("q", "k", "v"), 16, "up", 7, True, None),
]


@pytest.mark.parametrize("operands", ["f16", "bf16"])
@pytest.mark.parametrize("layers,vpt,params,r,position,n,normalize,chunk", CASES)
def test_gradient_parity(jb, cuda_dev, applied_ctx, operands, layers, vpt, params, r, position, n, normalize, chunk):
    applied_ctx.set_operand_type(operands)
    if chunk:
        applied_ctx.set_chunk_views(chunk)
    sd, model, lora_layers = _model(jb, layers, vpt, params, r, position)
    trainer = jb.LoraTrainer(model, lora_layers, seed=1, normalize=normalize)
    images = _views(n)
    dfeat = torch.randn(n, 512, generator=torch.Generator().manual_seed(n + layers))
    f_dev, g_dev = _dev_grads(trainer, images.to(cuda_dev), dfeat)
    f_ref, g_ref = _ref_grads(jb, sd, trainer, images, dfeat, normalize)
    assert torch.nn.functional.cosine_similarity(f_dev.double(), f_ref.double()).min() > 0.999
    _compare(g_dev, g_ref, f"ViT-B/16 {layers} blocks vpt={vpt} {params} r={r} {position} n={n}")


@pytest.mark.parametrize("operands", ["f16", "bf16"])
def test_dropout_gradients(jb, cuda_dev, applied_ctx, operands):
    applied_ctx.set_operand_type(operands)
    sd, model, lora_layers = _model(jb, 2, 0, ("q", "k", "v", "o"), 8, rate=0.25)
    trainer = jb.LoraTrainer(model, lora_layers, seed=77)
    images = _views(7)
    for step in range(2):
        dfeat = torch.randn(7, 512, generator=torch.Generator().manual_seed(step))
        _, g_dev = _dev_grads(trainer, images.to(cuda_dev), dfeat)
        _, g_ref = _ref_grads(jb, sd, trainer, images, dfeat, True, rate=0.25, step=step)
        _compare(g_dev, g_ref, f"ViT-B/16 dropout step {step}")


def test_determinism_and_pass_split(jb, cuda_dev, applied_ctx):
    """The same inputs give the same bits, with one pass and with several; the two splits agree to rounding."""
    sd, model, lora_layers = _model(jb, 2, 0, ("q", "k", "v", "o"), 4, rate=0.25)
    images = _views(30).to(cuda_dev)
    dfeat = torch.randn(30, 512, generator=torch.Generator().manual_seed(3))

    def grads():
        return _dev_grads(jb.LoraTrainer(model, lora_layers, seed=5), images, dfeat)[1]

    one = grads()
    assert all(torch.equal(a, b) for a, b in zip(one, grads()))
    applied_ctx.set_chunk_views(40)           # 12 views per pass at 197 tokens: three passes
    split = grads()
    assert all(torch.equal(a, b) for a, b in zip(split, grads()))
    for a, b in zip(split, one):
        assert float((a - b).norm() / b.norm()) < 1e-2


def test_eval_is_encode_image(jb, cuda_dev, applied_ctx):
    sd, model, lora_layers = _model(jb, 2, 4, ("q", "k", "v", "o"), 4, rate=0.25)
    trainer = jb.LoraTrainer(model, lora_layers, seed=1)
    images = _views(9).to(cuda_dev)
    assert torch.equal(trainer.eval()(images), model.visual(images, normalize=True))


def test_training_loop_and_pickle(jb, cuda_dev, applied_ctx, tmp_path):
    """12 AdamW steps (100 f T^T logits, cross-entropy, cosine schedule) on seeded few-shot data: the loss decreases and
    tracks the same loop through the fp32 restatement; the saved pickle reloads (load_lora, backbone ViT-B/16) to the
    same eval features."""
    from test_gpu_lora_train import _fewshot_data, _loop
    sd, model, lora_layers = _model(jb, 2, 0, ("q", "k", "v"), 4)
    images, labels, text = _fewshot_data(n_classes=6, shots=3)
    trainer = jb.LoraTrainer(model, lora_layers, seed=0)
    dev_losses = _loop(trainer.parameters(), trainer, images.to(cuda_dev), labels, text, steps=12)
    sd2, model2, lora_layers2 = _model(jb, 2, 0, ("q", "k", "v"), 4)
    ref_ad = {}
    for i, attn in enumerate(lora_layers2):
        for name, code in _PROJ:
            lin = getattr(attn, name)
            if lin.lora_enabled:
                ref_ad[(i, code)] = (torch.from_numpy(lin.w_lora_A.data.copy()).requires_grad_(True),
                                     torch.from_numpy(lin.w_lora_B.data.copy()).requires_grad_(True), lin.scaling)
    ref_params = [t for a in ref_ad.values() for t in a[:2]]
    ref_losses = _loop(ref_params, lambda x: ref_features(sd2, x, ref_ad, True), images, labels, text, steps=12)
    assert dev_losses[-1] < 0.8 * dev_losses[0]
    for a, b in zip(dev_losses, ref_losses):
        assert abs(a - b) <= 0.05 * abs(b) + 1e-3, (dev_losses, ref_losses)
    args = _args(("q", "k", "v"), 4)
    path = trainer.save(args, 12, lora_layers, save_dir=str(tmp_path))
    f_trained = trainer.eval()(images.to(cuda_dev))
    sd3, model3, lora_layers3 = _model(jb, 2, 0, ("q", "k", "v"), 4, seed=3)
    jb.load_lora(args, lora_layers3, path)
    assert torch.equal(f_trained, model3.visual(images.to(cuda_dev), normalize=True))


def test_merged_mode_is_rejected(jb, cuda_dev, applied_ctx):
    from ctypes import byref, c_void_p
    lib = jb.load_library()
    applied_ctx.set_lora_mode("merged")
    sd, model, lora_layers = _model(jb, 1)
    images = _views(2).to(cuda_dev)
    out = torch.full((2, 512), 7.0, device=cuda_dev)
    ctx, vit = model.visual._engine(cuda_dev)
    ctx.bind_current_stream()
    tape = c_void_p()
    rc = lib.jcb_vit_train_forward(vit, c_void_p(images.data_ptr()), 0, 2, 0, 1, 0.0, 0, 0, c_void_p(out.data_ptr()),
                                   byref(tape))
    assert rc == jb._capi.JCB_E_INVALID and not tape.value
    torch.cuda.synchronize()
    assert (out == 7.0).all()
