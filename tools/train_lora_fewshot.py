#!/usr/bin/env python
"""Worked example: train image-tower LoRA adapters on a synthetic few-shot set with the reference's recipe
(lora_train_vlp.py:921-1024): logits 100 f T^T against fixed text features, cross-entropy, AdamW, cosine schedule;
then save the reference pickle and read it back with load_lora.
    python tools/train_lora_fewshot.py [--classes 10] [--shots 4] [--steps 30] [--layers 12] [--out DIR]
The images are seeded synthetic views (jclip_b200.synth), the text features random unit rows: the loss falls as the
adapters learn to separate the classes.  Prints the loss per step and the path of the saved pickle.
"""
import argparse
import os
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import jclip_b200 as jb  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--classes", type=int, default=10)
    ap.add_argument("--shots", type=int, default=4)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--layers", type=int, default=12)
    ap.add_argument("--lr", type=float, default=2e-3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    model = jb.jclip.build_model(jb.synth.make_vit_state_dict(seed=0, layers=a.layers))
    args = argparse.Namespace(encoder="vision", position="all", params=["q", "k", "v"], r=2, alpha=1, dropout_rate=0.25,
                              backbone="ViT-B/32", filename="lora_weights")
    layers = jb.apply_lora(args, model)
    trainer = jb.LoraTrainer(model, layers, seed=1)
    n = a.classes * a.shots
    images = torch.from_numpy(jb.synth.clip_normalize(jb.synth.make_views(7, 1, n).reshape(n, 3, 224, 224))).to(dev)
    labels = torch.arange(a.classes, device=dev).repeat_interleave(a.shots)
    g = torch.Generator().manual_seed(3)
    text = torch.nn.functional.normalize(torch.randn(a.classes, 512, generator=g), dim=-1).to(dev)
    opt = torch.optim.AdamW(trainer.parameters(), lr=a.lr, weight_decay=1e-2)
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, a.steps)
    for s in range(a.steps):
        f = trainer(images)
        loss = torch.nn.functional.cross_entropy(100 * f @ text.T, labels)
        opt.zero_grad()
        loss.backward()
        opt.step()
        sched.step()
        print(f"step {s:3d}  loss {loss.item():.4f}  lr {sched.get_last_lr()[0]:.2e}")
    out = a.out or tempfile.mkdtemp(prefix="lora_fewshot_")
    path = trainer.save(args, a.steps, layers, save_dir=out)
    trained = trainer.eval()(images)
    model2 = jb.jclip.build_model(jb.synth.make_vit_state_dict(seed=0, layers=a.layers))
    layers2 = jb.apply_lora(args, model2)
    jb.load_lora(args, layers2, path)
    same = torch.equal(trained, model2.visual(images, normalize=True))
    acc = float(((trained @ text.T).argmax(-1) == labels).float().mean())
    print(f"saved {path}; reloaded eval features identical: {same}; train accuracy {acc:.3f}")


if __name__ == "__main__":
    main()
