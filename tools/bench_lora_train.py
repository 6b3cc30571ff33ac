#!/usr/bin/env python
"""Image-tower LoRA training: steps per second and images per second of the device forward + backward.
    python tools/bench_lora_train.py --out DIR [--steps K] [--warmup W] [--views N] [--backbone ViT-B/32|ViT-B/16]
Writes DIR/bench_lora_train.json and prints it.  The line carries the card's name, power limit and maximum SM clock,
read with nvidia-smi (a query) in the same run.

A step is the reference's training step (lora_train_vlp.py:921-1024) on N = 256 images x 1 view (fp32 device input,
already CLIP-normalised) through a 12-layer ViT-B/32 tower, fp16 forward operands: `LoraTrainer` forward with dropout
0.25, cross-entropy of 100 f T^T logits against 100 fixed classes, backward, AdamW.  LoRA on q, k, v of all blocks with
r = 2 (the reference's train.sh setting).  Forward and backward ms per step from CUDA events around each half over
`steps` steps after `warmup`; then one profiled step (jcb_ctx_profile) gives the backward kernel classes' shares.
--backbone ViT-B/16 runs the same step on a patch-16 tower (197 tokens) and writes bench_lora_train_vit_b16.json;
it also times the attention backward alone (attention_bwd_tcgen05_kernel) at T = 197, 12 heads, over one backward
pass's worth of sequences (332 views), as ms and algorithmic TFLOP/s (10 T^2 64 FLOP per sequence and head).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import jclip_b200 as jb  # noqa: E402


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True, check=True)
    name, power, clock = (s.strip() for s in r.stdout.strip().splitlines()[1].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def attention_bwd_alone(dev, n=332, T=197, H=12, reps=50):
    g = torch.Generator(device=dev).manual_seed(0)
    qkv = torch.randn(n * T, 3 * H * 64, generator=g, device=dev).half()
    dout = torch.randn(n * T, H * 64, generator=g, device=dev)
    dqkv = torch.empty(n * T, 3 * H * 64, dtype=torch.bfloat16, device=dev)
    for _ in range(3):
        jb.blocks.attention_bwd(qkv, dout, n, T, H, dqkv)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        jb.blocks.attention_bwd(qkv, dout, n, T, H, dqkv, sync=False)
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / reps
    return {"views": n, "tokens": T, "heads": H, "ms": round(ms, 4),
            "algorithmic_tflops": round(10.0 * T * T * 64 * n * H / (ms * 1e-3) / 1e12, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--views", type=int, default=256)
    ap.add_argument("--backbone", default="ViT-B/32", choices=["ViT-B/32", "ViT-B/16"])
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    info = card()
    patch = 16 if a.backbone == "ViT-B/16" else 32
    sd = jb.synth.make_vit_state_dict(seed=0, patch=patch)
    model = jb.jclip.build_model(sd)
    args = argparse.Namespace(encoder="vision", position="all", params=["q", "k", "v"], r=2, alpha=1, dropout_rate=0.25,
                              backbone=a.backbone)
    layers = jb.apply_lora(args, model)
    trainer = jb.LoraTrainer(model, layers, seed=0)
    opt = torch.optim.AdamW(trainer.parameters(), lr=2e-4)
    g = torch.Generator().manual_seed(0)
    views = torch.from_numpy(jb.synth.clip_normalize(jb.synth.make_views(1, 1, a.views).reshape(a.views, 3, 224, 224))).to(dev)
    text = torch.nn.functional.normalize(torch.randn(100, 512, generator=g), dim=-1).to(dev)
    labels = torch.randint(0, 100, (a.views,), generator=g).to(dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]

    def step(timed):
        if timed:
            ev[0].record()
        f = trainer(views)
        loss = torch.nn.functional.cross_entropy(100 * f @ text.T, labels)
        if timed:
            ev[1].record()
        opt.zero_grad()
        loss.backward()
        opt.step()
        if timed:
            ev[2].record()
            torch.cuda.synchronize()
            return ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])
        return None

    for _ in range(a.warmup):
        step(False)
    torch.cuda.synchronize()
    fw, bw = [], []
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(a.steps):
        step(False)
    t1.record()
    torch.cuda.synchronize()
    total_ms = t0.elapsed_time(t1) / a.steps
    for _ in range(a.steps):
        f_ms, b_ms = step(True)
        fw.append(f_ms)
        bw.append(b_ms)
    ctx = jb.get_context(dev)
    ctx.profile_start()
    step(False)
    prof = ctx.profile_stop()
    bwd = {k: v for k, v in prof.items() if k in ("bwd_gemm", "bwd_attention", "bwd_rowwise", "lora_grad")}
    bwd_ms = sum(v["ms"] for v in bwd.values())
    out = dict(info, what=f"LoRA training step, {a.backbone} 12 layers, q/k/v r=2 all blocks, dropout 0.25, fp16 forward",
               views=a.views, steps=a.steps, ms_per_step=round(total_ms, 3), steps_per_s=round(1000 / total_ms, 2),
               images_per_s=round(a.views * 1000 / total_ms, 1),
               forward_ms_median=round(float(np.median(fw)), 3), backward_ms_median=round(float(np.median(bw)), 3),
               backward_kernel_ms_profiled={k: round(v["ms"], 3) for k, v in bwd.items()},
               backward_kernel_share={k: round(v["ms"] / bwd_ms, 3) for k, v in bwd.items()},
               profiled_classes_ms={k: round(v["ms"], 3) for k, v in prof.items()})
    if patch == 16:
        out["attention_bwd_alone"] = attention_bwd_alone(dev)
    os.makedirs(a.out, exist_ok=True)
    name = "bench_lora_train.json" if patch == 32 else "bench_lora_train_vit_b16.json"
    with open(os.path.join(a.out, name), "w") as fh:
        json.dump(out, fh, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
