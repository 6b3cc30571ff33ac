#!/usr/bin/env python
"""ViT-B/16 measurements: the long attention kernel alone and the whole pipeline on a ViT-B/16 tower.
    python tools/bench_vit_b16.py --out DIR [--steps K] [--warmup W]
Writes DIR/bench_vit_b16.jsonl (one JSON object per line) and prints the same lines.  Every line carries the card's
name, power limit and maximum SM clock, read with nvidia-smi (a query) in the same run.

Lines:
  attention : T = 197, 12 heads, 2048 sequences (1.9 GB of q|k|v, larger than L2) on the long kernel, and T = 50 on the
              two-heads-per-tile kernel at the same bytes (8192 sequences); CUDA events over >= 20 launches after
              warm-up.  GB/s counts 8 B per element of [T, W] (bf16/fp16 q|k|v read + output written, as
              tools/bench_kernel.py does); TFLOP/s counts 4 T^2 64 per (sequence, head) (algorithmic) and, for the long
              kernel, the 256 x 256 tile it executes (4 * 256 * 256 * 64).
  pipeline  : HotPath.evaluate_base on a 12-layer ViT-B/16 tower with LoRA on q, k, v: 32 images x 65 views per step,
              uint8 device input, fp16 operands (409,760 token rows per pass).  ms per step from CUDA events without the
              profiler, then one profiled step for ms per kernel class (jcb_ctx_profile) and attention's share.
              TFLOP/s from 35.13 GFLOP per view (ViT-B/16 at 224 px: 33.46 block GEMMs, 0.23 conv1, 1.43 attention).
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import jclip_b200 as jb  # noqa: E402

GFLOP_PER_VIEW = 35.13


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                       capture_output=True, text=True, check=True)
    print(r.stdout.strip())
    name, power, clock = (s.strip() for s in r.stdout.strip().splitlines()[1].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def time_ms(fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def attention_line(dev, n, T, H, iters):
    W = H * 64
    qkv = torch.randn(n * T, 3 * W, device=dev).to(torch.float16)
    out = torch.empty(n * T, W, dtype=torch.float16, device=dev)
    ms = time_ms(lambda: jb.blocks.attention(qkv, n, T, H, out, sync=False), iters)
    flops = 4.0 * T * T * 64 * n * H
    line = {"what": "attention", "T": T, "heads": H, "sequences": n, "operands": "f16", "launches": iters,
            "qkv_gb": qkv.numel() * 2 / 1e9, "ms": ms, "gb_per_s": 8.0 * n * T * W / ms / 1e6,
            "tflops_algorithmic": flops / ms / 1e9}
    if T > 128:
        line["tflops_executed_256x256"] = 4.0 * 256 * 256 * 64 * n * H / ms / 1e9
    del qkv, out
    return line


def pipeline_lines(dev, steps, warmup, I=32, V=65):
    import types
    ctx = jb.get_context(dev)
    ctx.set_operand_type("f16")
    sd = jb.synth.make_vit_state_dict(seed=0, patch=16)
    model = jb.jclip.build_model(sd)
    largs = types.SimpleNamespace(encoder="vision", position="all", params=["q", "k", "v"], r=4, alpha=1,
                                  dropout_rate=0.25, backbone="ViT-B/16")
    layers = jb.apply_lora(largs, model)
    lora = jb.synth.make_lora(seed=7)
    for i, layer in enumerate(layers):
        for name, (A, B) in lora[i].items():
            getattr(layer, name).w_lora_A.data = A
            getattr(layer, name).w_lora_B.data = B
    Ts = [torch.from_numpy(jb.synth.make_text_features(seed=10 + i)) for i in range(3)]
    lp = jb.Channel_LP()
    lp.scale1.data, lp.bias1.data, lp.fc.weight.data, lp.fc.bias.data = jb.synth.make_head(2, Ts[2].numpy())
    hp = jb.HotPath(model, jb.TextBank(Ts[0], Ts[1], Ts[2], dev), lp, rank_by="cs5", k=5)
    imgs = (jb.synth.make_views_torch(1000, I, V, dev) * 255.0).round_().to(torch.uint8)
    step = lambda: hp.evaluate_base(imgs, topk_to_host=False)
    ms = time_ms(step, steps, warm=warmup)
    torch.cuda.synchronize()
    ctx.profile_start()
    t0 = time.perf_counter()
    step()
    torch.cuda.synchronize()
    prof_wall = (time.perf_counter() - t0) * 1e3
    prof = ctx.profile_stop()
    total = sum(v["ms"] for v in prof.values())
    views = I * V
    return {"what": "pipeline", "backbone": "ViT-B/16", "tokens": 197, "images": I, "views_per_image": V,
            "token_rows_per_pass": views * 197, "input": "uint8 device", "operands": "f16", "steps": steps,
            "ms_per_step": ms, "images_per_s": I / ms * 1e3, "views_per_s": views / ms * 1e3,
            "achieved_tflops": views * GFLOP_PER_VIEW / ms,        # GFLOP / ms = TFLOP/s
            "profiled_step": {"wall_ms": prof_wall, "sum_of_kernel_class_ms": total,
                              "ms_by_class": {k: v["ms"] for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"])},
                              "attention_share_of_kernel_time": prof.get("attention", {"ms": 0.0})["ms"] / total}}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True, help="output directory (created)")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--launches", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    dev = torch.device("cuda", 0)
    info = card()
    os.makedirs(args.out, exist_ok=True)
    lines = [attention_line(dev, 2048, 197, 12, args.launches), attention_line(dev, 8192, 50, 12, args.launches)]
    torch.cuda.empty_cache()
    lines.append(pipeline_lines(dev, args.steps, args.warmup))
    with open(os.path.join(args.out, "bench_vit_b16.jsonl"), "w") as f:
        for line in lines:
            line = {**line, **info}
            print(json.dumps(line))
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
