#!/usr/bin/env python
"""Micro-benchmarks of single kernels through the C-ABI (CUDA events, inputs larger than L2).
    python tools/bench_kernel.py attention|layernorm|mta|gemm [n_views]"""
import os
import sys
from ctypes import c_void_p

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import jclip_b200 as jb  # noqa: E402

what = sys.argv[1]
n = int(sys.argv[2]) if len(sys.argv) > 2 else 8192
OP = torch.float16 if os.environ.get("JCB_OPERANDS", "f16").lower().startswith("f") else torch.bfloat16
dev = torch.device("cuda", 0)
ctx = jb.get_context(dev)
ctx.bind_current_stream()
lib, h = ctx.lib, ctx.handle
P = lambda t: c_void_p(t.data_ptr())


def timeit(fn, iters=10, warm=3):
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


if what == "attention":
    T, H = 50, 12
    qkv = torch.randn(n * T, 3 * 768, device=dev).to(OP)
    out = torch.empty(n * T, 768, dtype=OP, device=dev)
    ms = timeit(lambda: jb.blocks.attention(qkv, n, T, H, out, sync=False))
    gb = n * T * 768 * 8 / 1e9
    print(f"attention n={n}: {ms:.3f} ms  {gb / ms * 1e3:.0f} GB/s")
elif what == "layernorm":
    x = torch.randn(n * 50, 768, device=dev)
    g, b = torch.ones(768, device=dev), torch.zeros(768, device=dev)
    y = torch.empty(n * 50, 768, dtype=OP, device=dev)
    ms = timeit(lambda: jb.blocks.layernorm(x, g, b, y))
    print(f"layernorm n={n}: {ms:.3f} ms  {n * 50 * 768 * 6 / 1e9 / ms * 1e3:.0f} GB/s")
elif what == "mta":
    I, V = n, 65
    feats = torch.from_numpy(jb.synth.make_unit_views(0, I, V)).to(dev)
    T = torch.from_numpy(jb.synth.make_text_features(seed=1)).t().contiguous().to(dev)
    ms = timeit(lambda: jb.solve_mta_batched(feats, T), iters=5, warm=2)
    print(f"mta I={I} V={V}: {ms:.3f} ms  ({ms / I * 1e3:.2f} us/image)")
elif what == "gemm":
    shapes = {"qkv": (2304, 768, 0), "out": (768, 768, 2), "fc1": (3072, 768, 1), "fc2": (768, 3072, 2)}
    M = n * 50
    for name, (N, K, epi) in shapes.items():
        A = torch.randn(M, K, device=dev).to(OP)
        B = (torch.randn(N, K, device=dev) * K ** -0.5).to(OP)
        bias = torch.randn(N, device=dev)
        out = torch.zeros(M, N, device=dev, dtype=torch.float32 if epi == 2 else OP)
        ms = timeit(lambda: jb.blocks.gemm(A, B, out, epi, bias=bias, sync=False))
        print(f"gemm {name} M={M} N={N} K={K}: {ms:.3f} ms  {2 * M * N * K / ms / 1e9:.0f} TFLOP/s")
elif what == "gemm_ln":
    # the two LayerNorm-preparing residual epilogues at the bench shape (out_proj: HBM-bound, c_proj: tensor-bound)
    C = jb._capi
    M = n * 50
    for name, (N, K, epi) in {"out_proj": (768, 768, C.EPI_RESID_LNPREP_SHORT), "c_proj": (768, 3072, C.EPI_RESID_LNPREP_LONG)}.items():
        A = torch.randn(M, K, device=dev).to(OP)
        B = (torch.randn(N, K, device=dev) * K ** -0.5).to(OP)
        bias = torch.randn(N, device=dev)
        resid = torch.zeros(M, N, device=dev)
        copy = torch.empty(M, N, device=dev, dtype=OP)
        st = [torch.zeros(M, 3, 2, device=dev) for _ in range(2)]
        sh = [torch.zeros(M, device=dev) for _ in range(2)]
        ms = timeit(lambda: jb.blocks.gemm(A, B, resid, epi, bias=bias, stats=st[1], out2=copy, stats_in=st[0], shift_in=sh[0],
                                           shift_out=sh[1], sync=False))
        gb = (2.0 * M * K + 10.0 * M * N) / 1e9
        print(f"gemm_ln {name} M={M} N={N} K={K}: {ms:.3f} ms  {2 * M * N * K / ms / 1e9:.0f} TFLOP/s  {gb / ms * 1e3:.0f} GB/s")
elif what == "tta":
    import numpy as np
    I = n
    rng = np.random.default_rng(0)
    imgs = [rng.integers(0, 256, (375, 500, 3), dtype=np.uint8) for _ in range(I)]
    gen = jb.TTAViews(n_crops=64, seed=0, emit=os.environ.get("EMIT", "views"))   # EMIT=patches: fused with the tower's front end
    jobs = gen.draw_jobs([im.shape[:2] for im in imgs])
    import time
    out = gen(imgs, jobs=jobs)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(3):
        out = gen(imgs, jobs=jobs)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / 3
    ctx.profile_start()
    out = gen(imgs, jobs=jobs)
    prof = ctx.profile_stop()
    print(f"tta I={I} x 65 views of 500x375: {dt * 1e3:.2f} ms per call incl. host packing + H2D ({I / dt:.0f} images/s); "
          f"kernels {prof['tta_views']['ms']:.2f} ms")
