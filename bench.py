#!/usr/bin/env python
"""Benchmark of the hot path: images/s for ViT-B/32 LoRA encode_image over the MTA crop batch
(N=64 crops + 1 centre view per image) -> MTA x3 -> LP++ head -> top-5, image-sharded over N GPUs.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

One "step" = one pass of the whole hot path over `--images-per-gpu` images x 65 views on every rank
(weak scaling: per-GPU work is fixed).  Rank 0 prints ONE JSON line:

  value      images/s, whole job, inputs resident in HBM (device pointers into jcb_pipeline)
  e2e        the same through HotPath.evaluate_stream with PINNED HOST images (two batches in flight): the
             host->device copies of every step's view chunks and the device->host read of its top-5 are inside
             the timed region; `blocking_call` is one HotPath.evaluate_base call per step
  roofline   the tcgen05 GEMM family (99 % of the FLOPs): algorithmic FLOPs / CUDA-event time of its
             launches, recorded on the launch stream inside the timed region, vs the measured bf16 peak
  cpu_baseline  the fp32 CPU oracle (a port: the reference needs Jittor, which is not installable) on a
             bounded sample of the same workload, on this box's host cores

`--impl reference` times that CPU oracle alone (rank 0 only), one image x 65 views per step.
"""
import argparse
import json
import os
import sys
import threading
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "images/sec (ViT-B/32 LoRA + MTA N=64 + LP++)"
UNIT = "images/s"
GFLOP_PER_VIEW = 8.8176          # SURVEY.md section 8(d): 8.7255 dense GEMM + 0.0922 attention
GEMM_GFLOP_PER_VIEW = 8.7255


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--images-per-gpu", type=int, default=128, help="images per step on every rank")
    ap.add_argument("--crops", type=int, default=64, help="N random crops per image (views = N + 1)")
    ap.add_argument("--chunk-views", type=int, default=0, help="views per pass through the tower (0 = library default)")
    ap.add_argument("--img-dtype", default="u8", choices=["u8", "f32"],
                    help="pixel format of the views: u8 (0..255, what an image decoder / the reference's PIL pipeline "
                         "produces before ToTensor; scaled by 1/255 on the device, bit-identical to ToTensor) or f32 in [0,1]")
    ap.add_argument("--host-chunk-views", type=int, default=0, help="views per pass when the input is in host memory")
    ap.add_argument("--no-balance", action="store_true",
                    help="N > 1: keep equal shards instead of sizing them by each rank's measured speed")
    ap.add_argument("--rebalance-every", type=int, default=5,
                    help="N > 1: every R timed steps the ranks exchange their step times and re-split the NEXT steps' global "
                         "batch by measured speed (no image moves); 0 = keep the calibrated split")
    ap.add_argument("--gather-every", type=int, default=0,
                    help="N > 1: all-gather the top-5 every G steps (1 = every step); 0 = once, at the end of the timed steps")
    ap.add_argument("--operands", default="f16", choices=["f16", "bf16"],
                    help="16-bit type of the tensor-core operands (fp32 accumulation either way, same tcgen05 rate): f16 meets "
                         "the north star's 1e-2 logit tolerance end to end, bf16 is its literal wording (0.02-0.07 off)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the top-5 class ids the last timed step returned for the whole global "
                         "batch (--impl reference: its one image) as DIR/topk.npy (float64 [images, 5]); the inputs are seeded, "
                         "so runs with the same arguments can be compared output for output (N > 1: needs --no-balance, the "
                         "balanced split depends on timings)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def workload_config(args, world, views_mib=None):
    """The `config` of both arms: the workload BASELINE.json's metric is quoted on (configs[2]/[3] at N = 64 crops)."""
    I, V = args.images_per_gpu, args.crops + 1
    if views_mib is None:
        views_mib = I * V * 3 * 224 * 224 * (1 if args.img_dtype == "u8" else 4) / 2**20
    return {
        "workload": f"ViT-B/32 LoRA(r=4 on q,k,v, merged) encode_image over {I} images x {V} views (N={args.crops} crops + "
                    f"centre) per GPU per step, {'uint8' if args.img_dtype == 'u8' else 'fp32'} 224x224 pixels (ToTensor scaling + CLIP "
                    f"normalisation fused on the device), MTA x3, LP++ head, "
                    f"top-5 of 403 classes",
        "images_per_gpu_per_step": I, "views_per_image": V, "parallelism": f"image-sharded dp{world}",
        "l2_policy": f"inputs larger than L2 ({views_mib:.0f} MiB of views per step)",
        "chunk_views_bound": args.chunk_views or 16384, "img_dtype": args.img_dtype, "gflop_per_view": GFLOP_PER_VIEW,
        "operands": f"{'fp16' if args.operands == 'f16' else 'bf16'} GEMM / attention operands, fp32 accumulation (TMEM), fp32 "
                    "residual stream / LayerNorm statistics / softmax / MTA / head",
    }


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"tflops": float(p["bf16_tflops_sustained"]), "hbm": float(p["hbm_gbs"]), "source": "measured"}
    except Exception:
        return {"tflops": 1590.0, "hbm": 6650.0, "source": "fallback"}


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons every 200 ms during the timed region (NVML; nvidia-smi as fallback)."""

    BAD = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, threading.Event(), [], set(), None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {"sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
                     "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                     "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                     "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                     "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80)}
            get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            while not self.stop_flag.is_set():
                self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                mask = get(h)
                for n, bit in names.items():
                    if mask & bit:
                        self.reasons.add(n)
                self.stop_flag.wait(0.2)
        except Exception as e:  # noqa: BLE001
            self.reasons.add(f"sampler_error:{type(e).__name__}")

    def summary(self):
        s = sorted(self.sm)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "samples": len(s),
                "reasons": sorted(self.reasons)}


def build_problem(jb, torch, dev, args, seed=0):
    """Random-init ViT-B/32 + LoRA (r=4 on q,k,v; merged in fp32), three text banks, LP++ head."""
    sd = jb.synth.make_vit_state_dict(seed=0)
    model = jb.jclip.build_model(sd)
    largs = types.SimpleNamespace(encoder="vision", position="all", params=["q", "k", "v"], r=4, alpha=1,
                                  dropout_rate=0.25, backbone="ViT-B/32")
    layers = jb.apply_lora(largs, model)
    lora = jb.synth.make_lora(seed=7)
    for i, layer in enumerate(layers):
        for name, (A, B) in lora[i].items():
            getattr(layer, name).w_lora_A.data = A
            getattr(layer, name).w_lora_B.data = B
    texts = [torch.from_numpy(jb.synth.make_text_features(seed=10 + i)) for i in range(3)]
    lp_np = jb.synth.make_head(2, texts[2].numpy())
    return sd, model, lora, texts, lp_np


def cpu_oracle_image(torch, sd, lora, texts, lp_t, imgs_np):
    """One image (V views) through the fp32 CPU oracle: tower -> MTA x3 -> head -> top-5."""
    from oracle import pipeline_image, vit_encode_image
    f = vit_encode_image(sd, imgs_np, lora=lora, scaling=0.5, apply_clip_norm=True, normalize=True)
    return pipeline_image(f, f, texts[0], texts[1], texts[2], lp_t, score="cs5")[0]


def run_reference(args):
    """The reference arm: its algorithm on the host cores.  Jittor 1.3.8.5 cannot be installed offline,
    so this is the oracle port (PyTorch CPU fp32, all host threads), one image x (N+1) views per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import torch
    import jclip_b200                  # synthetic inputs only: no native code is loaded on this arm
    jb_synth = jclip_b200.synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    V = args.crops + 1
    sd = jb_synth.make_vit_state_dict(seed=0)
    lora = jb_synth.make_lora(seed=7)
    texts = [torch.from_numpy(jb_synth.make_text_features(seed=10 + i)) for i in range(3)]
    lp_t = tuple(torch.from_numpy(a) for a in jb_synth.make_head(2, texts[2].numpy()))
    sd_t = {k: torch.from_numpy(v) for k, v in sd.items()}
    imgs = jb_synth.make_views(100, 1, V)[0]
    for _ in range(args.warmup):
        cpu_oracle_image(torch, sd_t, lora, texts, lp_t, imgs)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        top5 = cpu_oracle_image(torch, sd_t, lora, texts, lp_t, imgs)
    dt = time.perf_counter() - t0
    val = args.steps / dt
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "topk.npy"), top5.reshape(1, -1).numpy().astype(np.float64))
    sample = f"{args.steps} steps x 1 image x {V} views (224x224 fp32), full pipeline, oracle port on host cores"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        # the b200 arm's config; every step of THIS arm is a bounded sample of it (cpu_baseline.sample): one of the
        # step's images with all its views, so value = images/s of the same pipeline on the host cores
        "config": dict(workload_config(args, int(os.environ.get("WORLD_SIZE", "1"))), reference_sample_images_per_step=1),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import jclip_b200 as jb

    rank, world, local = jb.dist.init_from_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200 GPU: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = jb.dist.bind_to_gpu_numa(local)     # before any pinned allocation
    t_start = time.perf_counter()

    def stage(name):
        """Progress marker on stderr (stdout carries the one JSON line): which leg a run that hangs or is killed was in."""
        print(f"[bench rank {rank} +{time.perf_counter() - t_start:6.1f}s] {name}", file=sys.stderr, flush=True)
    if world != args.gpus and rank == 0:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)
    if args.dump_outputs and world > 1 and not args.no_balance:
        raise SystemExit("--dump-outputs on more than one GPU needs --no-balance: the balanced shards, and with them the "
                         "images of a step, depend on measured speeds")
    peaks = measured_peaks()
    V = args.crops + 1
    I = args.images_per_gpu
    K, W = args.steps, max(args.warmup, 0)

    sd, model, lora, texts, lp_np = build_problem(jb, torch, dev, args)
    # the path's only collectives: rank 0's text embeddings / head weights to everyone (once) ...
    bank_t = [t.to(dev) for t in texts]
    lp_dev = [torch.from_numpy(a).to(dev) for a in lp_np]
    jb.dist.broadcast_tensors(bank_t + lp_dev, src=0)
    lp = jb.Channel_LP()
    lp.scale1.data, lp.bias1.data, lp.fc.weight.data, lp.fc.bias.data = [t.cpu() for t in lp_dev]
    bank = jb.TextBank(bank_t[0], bank_t[1], bank_t[2], dev)
    hp = jb.HotPath(model, bank, lp, rank_by="cs5", k=5)
    ctx = jb.get_context(dev)
    ctx.set_operand_type(args.operands)      # before the first forward: the towers are packed lazily with this type
    if args.chunk_views:
        ctx.set_chunk_views(args.chunk_views)
    if args.host_chunk_views:
        ctx.set_host_chunk_views(args.host_chunk_views)

    # this rank's shard of the step's images: I_r images x V views, generated on the device
    def make_images(n):
        im = jb.synth.make_views_torch(1000 + rank, n, V, dev)
        return (im * 255.0).round_().to(torch.uint8) if args.img_dtype == "u8" else im

    n_total = I * world                      # the step's global batch: fixed, I images per GPU on average
    sizes = [I] * world
    # N > 1: every rank keeps a pool of I_max images and works on a prefix of it, so that the split of the global batch
    # can follow the ranks' speeds without generating or moving an image
    I_max = I if world == 1 else int(I * 1.15) + 2
    pool = make_images(I_max)
    images = pool[:I]
    stage("problem built")
    balance = None
    if world > 1 and not args.no_balance:
        # The GPUs of one box differ by a few per cent under the power cap, and every step ends in an all-gather: with
        # equal shards all ranks run at the pace of the slowest.  Images are independent, so the shard boundaries are
        # free: time this rank alone on the equal shard (no collective inside), exchange the timings, and size the shards
        # of the SAME global batch in proportion to speed (dist.balanced_shard_sizes).
        # Two rounds: the second one measures the re-sized shards themselves (and a warmer GPU) and corrects the first.
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        rounds = []
        for _round in range(2):
            for _ in range(3):
                hp.evaluate_base(images, topk_to_host=False)
            torch.cuda.synchronize()
            stage(f"calibration round {_round}: 3 untimed passes done")
            jb.dist.barrier()
            c0.record()
            for _ in range(5):
                hp.evaluate_base(images, topk_to_host=False)
            c1.record()
            torch.cuda.synchronize()
            ms_all = jb.dist.all_gather_floats(c0.elapsed_time(c1) / 5, dev)
            stage(f"calibration round {_round}: timed, exchanged")
            rounds.append({"shard_images": list(sizes), "ms_per_step_by_rank": [round(m, 2) for m in ms_all]})
            new_sizes = jb.dist.balanced_shard_sizes(n_total, [m / max(n, 1) for m, n in zip(ms_all, sizes)])
            if max(new_sizes) <= I_max:
                sizes = new_sizes
                images = pool[:sizes[rank]]
        balance = {"calibration": rounds, "shard_images": sizes}
    I_r = sizes[rank]
    lo_r = sum(sizes[:rank])

    # ... and the per-image top-5 to everyone (the path's other collective).  Default: the predictions of the K timed
    # steps are kept on the device and all-gathered ONCE, inside the timed region, the way the reference writes one result
    # file at the end of its loop; --gather-every 1 gathers after every step instead (asynchronously, so that the stream
    # computing step k+1 does not wait for the slowest rank's step k: dist.AsyncTopkGather).  Either way the ranks are not
    # in lockstep, and the timed region ends only when every gather has completed.
    G = max(args.gather_every, 0)
    gather = jb.dist.AsyncTopkGather(n_total, 5, dev, sizes=sizes, depth=4)
    # every rank's [K, I_max, 5] block (rows beyond a step's shard size are padding), gathered as one tensor
    gather_all = jb.dist.AsyncTopkGather(world * K * I_max, 5, dev, sizes=[K * I_max] * world, depth=1) if G != 1 else None
    kept = torch.zeros((K, I_max, 5), dtype=torch.int32, device=dev)
    step_no = [0]
    last_topk = [None]                       # this rank's predictions of the latest step (--dump-outputs)

    def step_device():
        topk = hp.evaluate_base(images, topk_to_host=False)
        last_topk[0] = topk
        if G == 1:
            return gather.submit(topk)
        kept[step_no[0] % K, :topk.shape[0]].copy_(topk, non_blocking=True)
        step_no[0] += 1
        return topk

    def finish_steps():
        """Inside the timed region, after the K steps: every rank's predictions of all K steps on every rank."""
        if G == 1:
            gather.drain()
            return None
        return gather_all.result(gather_all.submit(kept.view(K * I_max, 5)))

    # The main timed region with shards that FOLLOW the ranks' speeds (N > 1, --rebalance-every R > 0): the calibrated split
    # is static, but a GPU under the power cap drifts by a few per cent within seconds.  Every R steps each rank measures its
    # last R steps with CUDA events, the per-image times are exchanged (one all-gather of a float) and the NEXT steps' global
    # batch is re-split in proportion to speed (exponentially smoothed).  No image moves: a rank just evaluates a longer
    # or shorter prefix of its pool.  The step's global batch (n_total images) never changes.
    R = max(args.rebalance_every, 0) if (world > 1 and G != 1 and not args.no_balance) else 0
    split_history = []

    def timed_steps():
        cur = list(sizes)
        t_img = None
        w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0.record()
        done_in_window = 0
        for k in range(K):
            if R and k > 0 and k % R == 0:
                w1.record()
                w1.synchronize()
                mine = w0.elapsed_time(w1) / max(done_in_window, 1)
                per = jb.dist.all_gather_floats(mine, dev)
                t_img = per if t_img is None else [0.5 * a + 0.5 * b for a, b in zip(t_img, per)]
                new = jb.dist.balanced_shard_sizes(n_total, t_img)
                if max(new) <= I_max:
                    cur = new
                w0.record()
                done_in_window = 0
            n = cur[rank]
            topk = hp.evaluate_base(pool[:n], topk_to_host=False)
            kept[k, :n].copy_(topk, non_blocking=True)
            done_in_window += n
            split_history.append(list(cur))
        return finish_steps()

    for _ in range(max(W, 1)):
        r = step_device()
        out = gather.result(r if G == 1 else gather.submit(r))
    torch.cuda.synchronize()
    assert out.shape == (n_total, 5)
    # N > 1: the gathered rows of ANOTHER rank's shard, recomputed here from that rank's seeded images, must be bit-identical
    # (rows [lo, hi) of the gather = that rank's shard, in order; SURVEY.md section 4 "N ranks == 1 rank")
    shard_check = None
    if world > 1:
        other = (rank + 1) % world
        lo_o = sum(sizes[:other])
        im_o = jb.synth.make_views_torch(1000 + other, I_max, V, dev)[:sizes[other]]       # that rank's pool prefix
        im_o = (im_o * 255.0).round_().to(torch.uint8) if args.img_dtype == "u8" else im_o
        mine = hp.evaluate_base(im_o.contiguous(), topk_to_host=False)
        same = bool(torch.equal(mine, out[lo_o:lo_o + sizes[other]]))
        del im_o
        oks = jb.dist.all_gather_floats(1.0 if same else 0.0, dev)
        shard_check = {"what": "every rank recomputed the next rank's shard from its seeded images and compared it with the "
                               "rows it received in the all-gather", "bit_identical_by_rank": [bool(x) for x in oks]}
        assert all(oks), shard_check

    sampler = ClockSampler(local)
    stage("warm-up done, timed region")
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    jb.dist.barrier()
    torch.cuda.synchronize()
    n0 = ctx.launch_count
    ctx.profile_start()
    ev0.record()
    step_no[0] = 0
    if R:
        all_kept = timed_steps()
    else:
        for _ in range(K):
            step_device()
        all_kept = finish_steps()
    ev1.record()
    torch.cuda.synchronize()
    jb.dist.barrier()
    prof = ctx.profile_stop()
    if args.dump_outputs:
        # the global batch's predictions of the last timed step, shards in rank order (40 bytes per image: far below
        # 64 MB for any batch whose views fit in device memory)
        topk_last = jb.dist.all_gather_topk(last_topk[0], n_total, sizes)
        if rank == 0:
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "topk.npy"), topk_last.cpu().numpy().astype(np.float64))
    if R and all_kept is not None:
        # the gathered block of rank r, step k holds that step's shard of rank r in rows [0, split[k][r]): every step's
        # predictions cover the whole global batch exactly once
        blk = all_kept.view(world, K, I_max, 5)
        for k in (0, K - 1):
            rows = torch.cat([blk[r, k, :split_history[k][r]] for r in range(world)])
            assert rows.shape == (n_total, 5) and sum(split_history[k]) == n_total
        # step 0 used the calibrated split: its rows equal the warm-up step's gathered predictions
        assert torch.equal(torch.cat([blk[r, 0, :split_history[0][r]] for r in range(world)]), out)
        balance["rebalance"] = {"every_steps": R, "splits": [split_history[k] for k in range(0, K, R)],
                                "note": "per-image times exchanged every R steps (CUDA events), next steps' split by smoothed speed"}
    launches = ctx.launch_count - n0
    ms_total = jb.dist.max_over_ranks(ev0.elapsed_time(ev1), dev)
    ms_step = ms_total / K
    if balance is not None:
        balance["timed_ms_per_step_by_rank"] = [round(m / K, 2) for m in jb.dist.all_gather_floats(ev0.elapsed_time(ev1), dev)]
    value = n_total * K / (ms_total / 1e3)

    stage("timed region done; leg: cls_only_last_block")
    # ---- informational: the opt-in schedule that runs the last block on the class-token rows only (results agree to
    #      rounding; 0.53 of the 8.82 GFLOP per view are work whose output encode_image never returns)
    cls_only = None
    if not args.no_e2e:
        ctx.set_cls_only_last_block(True)
        try:
            for _ in range(2):
                r = step_device()
                out_c = gather.result(r if G == 1 else gather.submit(r))
            jb.dist.barrier()
            torch.cuda.synchronize()
            step_no[0] = 0
            ev0.record()
            for _ in range(K):
                step_device()
            finish_steps()
            ev1.record()
            torch.cuda.synchronize()
        finally:
            ctx.set_cls_only_last_block(False)
        ms_c = jb.dist.max_over_ranks(ev0.elapsed_time(ev1), dev) / K
        cls_only = {"value": n_total / (ms_c / 1e3), "unit": UNIT, "ms_per_step": ms_c, "executed_gflop_per_view": GFLOP_PER_VIEW - 0.5278,
                    "top5_agreement_with_full_schedule": float((out_c.sort(dim=1).values == out.sort(dim=1).values).all(dim=1).float().mean()),
                    "note": "jcb_ctx_set_cls_only_last_block(1): attention / out_proj / MLP of block 12 on 1 of 50 token rows; "
                            "NOT used for value / e2e / roofline"}

    stage("leg: e2e (host views)")
    # ---- end to end: pinned host images in, host top-5 out, copies inside the timed region
    e2e = None
    if not args.no_e2e:
        host_images = torch.empty(images.shape, dtype=images.dtype, pin_memory=True)
        host_images.copy_(images)
        torch.cuda.synchronize()
        for _ in range(max(W, 1)):
            tk = hp.evaluate_base(host_images)
        assert not tk.is_cuda and torch.equal(tk, out[lo_r:lo_r + I_r].cpu())
        # (a) one blocking call per step: nothing hides the first upload of a step or the final read
        jb.dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(K):
            tk = hp.evaluate_base(host_images)
            if G == 1:
                gather.submit(tk.to(dev))
            else:
                kept[k, :I_r].copy_(tk, non_blocking=True)
        finish_steps()
        torch.cuda.synchronize()
        dt_block = jb.dist.max_over_ranks(time.perf_counter() - t0, dev)
        # (b) the streaming form of the same call (HotPath.evaluate_stream, the reference's `for images in loader`
        #     loop): batch k+1 is submitted before batch k is collected, so its uploads overlap k's compute.  Every
        #     step still copies its own views from pinned host memory and reads its own top-5 back to the host.
        for tk2 in hp.evaluate_stream(host_images for _ in range(2)):
            assert torch.equal(tk2, tk)
        jb.dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k, tk2 in enumerate(hp.evaluate_stream(host_images for _ in range(K))):
            # stream-ordered (a blocking .to() would make the host wait for the batch submitted after this one)
            if G == 1:
                gather.submit(tk2.to(dev, non_blocking=True))
            else:
                kept[k, :I_r].copy_(tk2, non_blocking=True)
        finish_steps()
        torch.cuda.synchronize()
        dt = jb.dist.max_over_ranks(time.perf_counter() - t0, dev)
        assert torch.equal(tk2, tk)
        e2e = {"value": n_total * K / dt, "unit": UNIT, "ms_per_step": 1e3 * dt / K,
               "h2d_bytes_per_step": int(images.numel() * images.element_size()), "d2h_bytes_per_step": int(I_r * 5 * 4),
               "api": "HotPath.evaluate_stream(batches, depth=2): pinned host views in, host top-5 out, two batches in flight",
               "blocking_call": {"value": n_total * K / dt_block, "ms_per_step": 1e3 * dt_block / K,
                                 "api": "HotPath.evaluate_base(host_views), one blocking call per step"}}
        del host_images
    stage("leg: e2e_from_images")
    # ---- informational: the same step fed from DECODED IMAGES: crop boxes drawn on the host, one upload of the
    #      source image per image, views generated on the GPU (TTAViews, Pillow-exact), then the hot path
    e2e_img = None
    if not args.no_e2e:
        rng = np.random.default_rng(2000 + rank)
        src = [rng.integers(0, 256, (375, 500, 3), dtype=np.uint8) for _ in range(I_r)]
        gen = jb.TTAViews(n_crops=args.crops, scale=(0.5, 1.0), seed=rank, emit="patches")

        def run_images(steps, overlap=True):
            # HotPath.evaluate_image_stream: while the towers work on batch k, the host draws the boxes of batch k+1, packs
            # its images into the other pinned buffer, and upload + view generation are enqueued (overlap: on a second,
            # low-priority stream); the generator writes the conv1 patch matrix directly (no uint8 views, no im2col)
            topk = None
            for topk in hp.evaluate_image_stream((src for _ in range(steps)), gen, overlap=overlap):
                pass
            return topk

        run_images(4, overlap=False)     # first use: pinned staging, generator scratch (grows with the random crop sizes)
        jb.dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        run_images(K, overlap=False)
        torch.cuda.synchronize()
        dt_serial = jb.dist.max_over_ranks(time.perf_counter() - t0, dev)
        run_images(2)
        jb.dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        run_images(K)
        torch.cuda.synchronize()
        dt = jb.dist.max_over_ranks(time.perf_counter() - t0, dev)
        e2e_img = {"value": n_total * K / dt, "unit": UNIT, "ms_per_step": 1e3 * dt / K,
                   "h2d_bytes_per_step": int(sum(a.size for a in src)), "d2h_bytes_per_step": int(I_r * 5 * 4),
                   "api": "HotPath.evaluate_image_stream(batches of decoded images, TTAViews(emit='patches')): two batches in flight",
                   "in_stream_order": {"value": n_total * K / dt_serial, "ms_per_step": 1e3 * dt_serial / K,
                                       "api": "the same with overlap=False: view generation in stream order in front of the towers"},
                   "note": "host: 500x375 uint8 decoded images + crop-box draw; device: Pillow-exact centre view + "
                           f"{args.crops} RandomResizedCrop(0.5-1)+flip views per image written straight into the conv1 patch "
                           "matrix on a second stream while the previous batch's towers run, then the hot path"}
    stage("leg: single_image_call")
    # ---- informational: the reference's own call pattern, one image x (N+1) views per call (test.py:1692-1742), blocking,
    #      host top-5 out: launch-latency-bound (~200 launches per call; encoded TMA descriptors are cached per shape)
    single = None
    if not args.no_e2e:
        one = images[:1].contiguous()
        for _ in range(5):
            hp.evaluate_base(one, topk_to_host=True)
        torch.cuda.synchronize()
        n_calls = 50
        t0 = time.perf_counter()
        for _ in range(n_calls):
            hp.evaluate_base(one, topk_to_host=True)
        dt1 = (time.perf_counter() - t0) / n_calls
        single = {"ms_per_call": 1e3 * dt1, "images_per_s": 1.0 / dt1, "views_per_call": V, "cuda_graphs": ctx.graph_stats(),
                  "api": "HotPath.evaluate_base(1 image x views, device-resident), host top-5 back, one blocking call per image "
                         "(served from a CUDA graph from the third call on: jcb_ctx_set_graphs)"}
    stage("leg: other_operand_type")
    # ---- informational: the same device-resident step with the OTHER 16-bit operand type (the towers are re-packed)
    other_operands = None
    if not args.no_e2e:
        alt = "bf16" if args.operands == "f16" else "f16"
        ctx.set_operand_type(alt)
        try:
            for _ in range(2):
                r = step_device()
                out_a = gather.result(r if G == 1 else gather.submit(r))
            jb.dist.barrier()
            torch.cuda.synchronize()
            step_no[0] = 0
            ev0.record()
            for _ in range(K):
                step_device()
            finish_steps()
            ev1.record()
            torch.cuda.synchronize()
        finally:
            ctx.set_operand_type(args.operands)
        ms_a = jb.dist.max_over_ranks(ev0.elapsed_time(ev1), dev) / K
        other_operands = {"operands": alt, "value": n_total / (ms_a / 1e3), "unit": UNIT, "ms_per_step": ms_a,
                          "identical_top5_sets_vs_headline_operands": float((out_a.sort(dim=1).values == out.sort(dim=1).values).all(dim=1).float().mean()),
                          "note": "same kernels, tcgen05 kind::f16 runs fp16 and bf16 operands at the same rate; NOT used for value / e2e / roofline"}
    stage("leg: lora_applied")
    # ---- informational: the same device-resident step with the adapters APPLIED as low-rank GEMMs instead of merged
    #      (jcb_ctx_set_lora_mode; the towers are re-packed): what a caller that swaps adapters per request pays
    lora_applied = None
    if not args.no_e2e:
        ctx.set_lora_mode("applied")
        try:
            for _ in range(2):
                r = step_device()
                out_l = gather.result(r if G == 1 else gather.submit(r))
            jb.dist.barrier()
            torch.cuda.synchronize()
            step_no[0] = 0
            ev0.record()
            for _ in range(K):
                step_device()
            finish_steps()
            ev1.record()
            torch.cuda.synchronize()
        finally:
            ctx.set_lora_mode("merged")
        ms_l = jb.dist.max_over_ranks(ev0.elapsed_time(ev1), dev) / K
        lora_applied = {"value": n_total / (ms_l / 1e3), "unit": UNIT, "ms_per_step": ms_l,
                        "identical_top5_sets_vs_merged": float((out_l.sort(dim=1).values == out.sort(dim=1).values).all(dim=1).float().mean()),
                        "note": "jcb_ctx_set_lora_mode(JCB_LORA_APPLIED): y = W x + b + s B (A x) (test.py:388-398) as a narrow tcgen05 GEMM "
                                "+ a second TMA operand pair accumulated into the QKV tile, stand-alone LayerNorm schedule; "
                                "NOT used for value / e2e / roofline (those run the default merged mode)"}
    stage("legs done")
    sampler.stop_flag.set()
    sampler.join(timeout=2)
    clocks = sampler.summary()

    if rank != 0:
        return 0

    # ---- roofline: the dominant kernel = the tcgen05 GEMM instantiation with the largest share of the step
    #      (fc1: bias + QuickGELU epilogue); the whole GEMM family (patch / qkv / out / fc1 / fc2) is reported beside it
    gemm = {k: v for k, v in prof.items() if k.startswith("gemm_")}
    g_ms = sum(v["ms"] for v in gemm.values())
    g_fl = sum(v["flops"] * (v["timed_launches"] / max(v["launches"], 1)) for v in gemm.values())
    family = g_fl / (g_ms / 1e3) / 1e12 if g_ms > 0 else None
    per_kernel = {}
    for k, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"]):
        frac_timed = v["timed_launches"] / max(v["launches"], 1)
        ent = {"ms_per_step": v["ms"] / K / max(frac_timed, 1e-9), "launches_per_step": v["launches"] / K}
        if v["flops"] and v["ms"]:
            ent["tflops"] = v["flops"] * frac_timed / (v["ms"] / 1e3) / 1e12
        if v["bytes"] and v["ms"]:
            ent["gbs"] = v["bytes"] * frac_timed / (v["ms"] / 1e3) / 1e9
        per_kernel[k] = ent
    kernel_ms_step = sum(e["ms_per_step"] for e in per_kernel.values())
    top = max(gemm, key=lambda k: gemm[k]["ms"]) if gemm else None
    fold = int(os.environ.get("JCB_LN_FOLD", "2"))
    k2 = "gemm_tcgen05_2cta_kernel<256, %s, " + ("true" if args.operands == "f16" else "false") + ">"
    names = {"gemm_fc1": k2 % ("EPI_LNFOLD_GELU_BF16" if fold >= 2 else "EPI_BIAS_GELU_BF16") + " (MLP c_fc, M x 3072 x 768)",
             "gemm_fc2": k2 % ("EPI_RESID_LNPREP_LONG" if fold >= 1 else "EPI_BIAS_RESID_F32") + " (MLP c_proj, M x 768 x 3072)",
             "gemm_qkv": k2 % ("EPI_LNFOLD_BF16" if fold >= 1 else "EPI_BIAS_BF16") + " (packed QKV, M x 2304 x 768)",
             "gemm_out": k2 % ("EPI_RESID_LNPREP_SHORT" if fold >= 2 else "EPI_BIAS_RESID_F32") + " (attention out_proj, M x 768 x 768)",
             "gemm_patch": k2 % "EPI_F32" + " (conv1 as im2col GEMM)"}
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            tj = json.load(f)
        launches_per_step_top = per_kernel[top]["launches_per_step"]
        views_per_launch = I_r * V * model.visual.layers / launches_per_step_top
        if abs(views_per_launch - tj["views_per_launch"]) < 0.5 and tj.get("ln_fold", 1) == fold:
            traffic = tj["per_kernel_bytes"].get(top)
    except Exception:  # noqa: BLE001
        pass
    achieved = per_kernel[top].get("tflops") if top else None
    roofline = {
        "bound": "tensor", "kernel": names.get(top, top), "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s",
        "frac": (achieved / peaks["tflops"]) if achieved else None, "traffic": traffic,
        "traffic_unit": "bytes per launch (dram read + write, one ncu --set full capture at this launch shape; "
                        "profiles/ncu_traffic.json)" if traffic else None,
        "avg_launch_ms": (per_kernel[top]["ms_per_step"] / per_kernel[top]["launches_per_step"]) if top else None,
        "flops_per_launch": (gemm[top]["flops"] / gemm[top]["launches"]) if top else None,
        "peak_source": f"{peaks['source']} bf16_tflops_sustained (kernel timed inside a long step; tcgen05 kind::f16 runs fp16 and "
                       "bf16 operands at the same rate, so the measured bf16 figure is the denominator for both operand types)",
        "gemm_family_tflops": family, "gemm_family_frac": (family / peaks["tflops"]) if family else None,
        "gemm_ms_per_step": g_ms / K,
        "gemm_share_of_kernel_time": (g_ms / K) / kernel_ms_step if kernel_ms_step else None,
        # per GPU on average: the step's global batch / world (shards may be sized by rank speed)
        "whole_step_tflops": I * V * GFLOP_PER_VIEW / 1e3 / (ms_step / 1e3),
        "whole_step_frac": I * V * GFLOP_PER_VIEW / 1e3 / (ms_step / 1e3) / peaks["tflops"],
        "per_kernel": per_kernel,
    }

    # context for roofline.frac: the plain library GEMM (cuBLAS through torch.matmul: no bias / activation / LayerNorm work)
    # on the dominant kernel's own shape, back to back for ~0.5 s under the same power cap, after the timed region
    if world == 1 and top == "gemm_fc1" and not args.no_e2e:
        try:
            Mrows = I_r * V * 50
            op_dt = ctx.operand_torch_dtype
            ga = torch.randn(Mrows, 768, device=dev).to(op_dt)
            gw = torch.randn(3072, 768, device=dev).to(op_dt)
            go = torch.empty(Mrows, 3072, device=dev, dtype=op_dt)
            for _ in range(3):
                torch.matmul(ga, gw.t(), out=go)
            torch.cuda.synchronize()
            n_it = 300
            ev0.record()
            for _ in range(n_it):
                torch.matmul(ga, gw.t(), out=go)
            ev1.record()
            torch.cuda.synchronize()
            lib_ms = ev0.elapsed_time(ev1) / n_it
            roofline["library_same_shape"] = {
                "tflops": 2.0 * Mrows * 3072 * 768 / lib_ms / 1e9, "ms": lib_ms,
                "what": f"torch.matmul (cuBLAS) {args.operands} {Mrows} x 3072 x 768, plain GEMM without epilogue work, {n_it} launches "
                        "back to back after the timed region; informational, not the roofline denominator"}
            del ga, gw, go
        except Exception as e:  # noqa: BLE001
            roofline["library_same_shape"] = {"error": f"{type(e).__name__}: {e}"}

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        sd_t = {k: torch.from_numpy(v) for k, v in sd.items()}
        lp_t = tuple(torch.from_numpy(a) for a in lp_np)
        imgs_np = images[:4].cpu().float().numpy()
        if args.img_dtype == "u8":
            imgs_np = imgs_np / np.float32(255.0)          # == T.ToTensor on uint8 pixels
        t0 = time.perf_counter()
        cpu_oracle_image(torch, sd_t, lora, texts, lp_t, imgs_np[0])       # warm-up (thread pools, allocator)
        t_first = time.perf_counter() - t0
        n_img = max(1, min(3, int(15.0 / max(t_first, 1e-3))))
        t0 = time.perf_counter()
        cpu_top = [cpu_oracle_image(torch, sd_t, lora, texts, lp_t, imgs_np[1 + j]) for j in range(n_img)]
        dt = time.perf_counter() - t0
        agree = sum(len(set(cpu_top[j].tolist()) & set(out[1 + j].cpu().tolist())) for j in range(n_img)) / (5 * n_img)
        cpu_baseline = {"value": n_img / dt, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": f"{n_img} of the step's images x {V} views through the fp32 oracle (PyTorch CPU; the "
                                  f"reference's Jittor cannot be installed offline), after 1 warm-up image",
                        "top5_agreement_with_gpu": agree}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp16" if args.operands == "f16" else "bf16", "data": "synthetic",
        "config": dict(workload_config(args, world, I * V * 3 * 224 * 224 * (1 if args.img_dtype == "u8" else 4) / 2**20),
                       **({"shard_balance": dict(balance, note="same global batch (images_per_gpu_per_step x n_gpus); shards "
                                                               "sized by each rank's measured speed, dist.balanced_shard_sizes")}
                          if balance else {}),
                       **({"shard_check": shard_check} if shard_check else {}),
                       **({"topk_all_gather": "every step, asynchronous (dist.AsyncTopkGather)" if G == 1 else
                           f"once per {K} timed steps, inside the timed region"} if world > 1 else {})),
        "e2e": e2e, "e2e_from_images": e2e_img, "cls_only_last_block": cls_only, "other_operand_type": other_operands, "lora_applied": lora_applied, "single_image_call": single, "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline,
    }
    print(json.dumps(line))
    return 0


if __name__ == "__main__":
    rc = main()
    try:
        import torch.distributed as _d
        if _d.is_initialized():
            _d.destroy_process_group()
    except Exception:  # noqa: BLE001
        pass
    sys.exit(rc)
