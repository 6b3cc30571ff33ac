#!/usr/bin/env python
"""LoRA slots: ms per step of the image tower with G adapter sets chosen per view, against one adapter set.
    python tools/bench_lora_slots.py --out DIR [--steps K] [--warmup W] [--rounds R]
Writes DIR/bench_lora_slots.jsonl (one JSON object per line) and prints the same lines.  Every line carries the card's
name, power limit and maximum SM clock, read with nvidia-smi (a query) in the same run.

A step is encode_image over 32 images x 65 views (2080 views, uint8 device input, CLIP normalisation fused) on a 12-layer
ViT-B/32 tower in applied LoRA mode, fp16 operands, every slot with q, k, v, o adapters of rank 16 on all blocks.
  G = 1         : the tower with one adapter set, plain call (today's applied mode)
  G = 2, 4, 6, 8: "image" = slot i % G for every view of image i (image-contiguous: 65 x 50 token rows per image, so
                  most 256-row GEMM tiles hold one slot); "view" = slot v % G for view v (every tile holds min(G, 6)
                  slots: the worst case)
ms per step from CUDA events over `steps` steps after `warmup`, without the profiler; the configurations are measured in
turn and the whole sequence is repeated `rounds` times (spread = the rounds' range).  Then one profiled step per
configuration gives ms per kernel class for the QKV, out_proj and down-projection (gemm_lora) GEMMs.
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

I, V = 32, 65


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True, check=True)
    name, power, clock = (s.strip() for s in r.stdout.strip().splitlines()[1].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def slot_dict(seed, layers=12, width=768, r=16):
    rng = np.random.default_rng(seed)
    bound = 1.0 / np.sqrt(width)
    return {i: {p: (rng.uniform(-bound, bound, (r, width)).astype(np.float32),
                    (rng.standard_normal((width, r)) * 0.02).astype(np.float32)) for p in "qkvo"}
            for i in range(layers)}


def make_model(G, dev):
    sd = jb.synth.make_vit_state_dict(seed=0)
    model = jb.jclip.build_model(sd)
    args = argparse.Namespace(encoder="vision", position="all", params=["q", "k", "v", "o"], r=16, alpha=1,
                              dropout_rate=0.0, backbone="ViT-B/32")
    s0 = slot_dict(100)
    names = {"q": "q_proj", "k": "k_proj", "v": "v_proj", "o": "proj"}
    for i, layer in enumerate(jb.apply_lora(args, model)):
        for p, (A, B) in s0[i].items():
            getattr(layer, names[p]).w_lora_A.data = A
            getattr(layer, names[p]).w_lora_B.data = B
    model.visual.set_lora_slots([slot_dict(100 + g) for g in range(1, G)])
    model.visual._engine(dev)
    return model


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=2)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    dev = torch.device("cuda", 0)
    info = card()
    ctx = jb.get_context(dev)
    ctx.set_operand_type("f16")
    ctx.set_lora_mode("applied")
    imgs = (torch.rand(I * V, 3, 224, 224, device=dev) * 255).to(torch.uint8)
    out = torch.empty(I * V, 512, device=dev)
    vit_of = {G: make_model(G, dev) for G in (1, 2, 4, 6, 8)}
    configs = [("1", 1, None)]
    for G in (2, 4, 6, 8):
        configs.append((f"{G}-image", G, np.repeat(np.arange(I) % G, V).astype(np.int32)))
        configs.append((f"{G}-view", G, (np.arange(I * V) % G).astype(np.int32)))

    def step_fn(G, slots):
        vit = vit_of[G].visual._vit
        if slots is None:
            return lambda: jb._capi.check(ctx.lib.jcb_encode_image(vit, imgs.data_ptr(), jb._capi.IMG_U8, I * V, 1, 1,
                                                                    out.data_ptr()), ctx.handle)
        p = slots.ctypes.data
        return lambda: jb._capi.check(ctx.lib.jcb_encode_image_slots(vit, imgs.data_ptr(), jb._capi.IMG_U8, I * V, p, 1, 1,
                                                                      out.data_ptr()), ctx.handle)

    ctx.bind_current_stream()
    times = {name: [] for name, _, _ in configs}
    for _ in range(a.rounds):
        for name, G, slots in configs:
            fn = step_fn(G, slots)
            for _ in range(a.warmup):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / a.steps)
    lines = []
    base = min(times["1"])
    for name, G, slots in configs:
        fn = step_fn(G, slots)
        ctx.profile_start()
        fn()
        prof = ctx.profile_stop()
        per_class = {k: round(prof[k]["ms"], 3) for k in ("gemm_qkv", "gemm_out", "gemm_lora") if k in prof}
        line = dict(info, bench="lora_slots", config=name, slots=G, images=I, views=V, operands="f16",
                    ms_per_step=[round(t, 3) for t in times[name]], best_ms=round(min(times[name]), 3),
                    vs_one_slot=round(min(times[name]) / base, 4), profiled_ms=per_class)
        lines.append(line)
        print(json.dumps(line), flush=True)
    with open(os.path.join(a.out, "bench_lora_slots.jsonl"), "w") as f:
        for line in lines:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
