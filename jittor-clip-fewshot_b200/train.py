"""Training of image-tower LoRA adapters on the GPU: d(loss)/dA and d(loss)/dB through torch autograd.

The reference trains its adapters with `lora_train_vlp.py:921-1024` (cross-entropy of 100 f T^T logits, AdamW, cosine
schedule) and evaluates them with `test.py` after `save_lora` / `load_lora`.  `LoraTrainer` is the image-tower half of
that step: its forward runs the applied-LoRA tower (`W x + b + s B (A dropout(x))`) with a tape, and its backward runs
the tower's backward pass on the device (include/jclip_b200.h "LoRA training") and returns the gradients of A and B.
Everything else -- loss, optimiser, schedule -- stays in torch; it acts on a few hundred KB of parameters.

    layers = jb.apply_lora(args, model)                  # args.encoder == 'vision'
    trainer = jb.LoraTrainer(model, layers, seed=1)
    opt = torch.optim.AdamW(trainer.parameters(), lr=2e-4)
    f = trainer(views)                                   # [n, 512] unit rows, differentiable
    loss = F.cross_entropy(100 * f @ text.T, labels); loss.backward(); opt.step()
    trainer.save(args, epoch)                            # the reference pickle, readable by load_lora

Scope: towers of at most 256 tokens (ViT-B/32 and ViT-B/16, plain or IVLP), one adapter set, q / k / v / o on any blocks with the
ranks of q, k, v of a block summing to at most 64.  Base weights, biases, LayerNorms, embeddings and `visual.VPT` are
frozen.  The trainer switches the context to the applied LoRA mode (`Context.set_lora_mode("applied")`).
"""
import ctypes
from ctypes import byref, c_void_p

import numpy as np
import torch

from . import _capi
from ._capi import check
from .jclip.model import _LORA_PROJ
from .runtime import get_context, img_dtype_code, ptr


class _Tape:
    """Owns a jcb_tape*; released when the autograd graph that holds it goes away."""

    def __init__(self, lib, handle):
        self.lib, self.handle = lib, handle

    def release(self):
        if self.handle:
            self.lib.jcb_tape_release(self.handle)
            self.handle = None

    def __del__(self):
        self.release()


def _ptr_array(tensors):
    arr = (c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr() if t is not None else None
    return arr


class _TowerFn(torch.autograd.Function):
    @staticmethod
    def forward(fctx, trainer, views, *params):
        ctx, vit = trainer._ctx, trainer._vit
        n = views.shape[0]
        out = torch.empty((n, trainer.visual.output_dim), dtype=torch.float32, device=views.device)
        h = c_void_p()
        check(ctx.lib.jcb_vit_train_forward(vit, ptr(views), img_dtype_code(views), n, int(trainer.apply_clip_norm),
                                            int(trainer.normalize), float(trainer.dropout_rate), trainer.seed,
                                            trainer.step, ptr(out), byref(h)), ctx.handle)
        fctx.tape = _Tape(ctx.lib, h)
        fctx.trainer = trainer
        return out

    @staticmethod
    def backward(fctx, dout):
        trainer = fctx.trainer
        ctx = trainer._ctx
        grads = [torch.empty_like(p) for p in trainer._params]
        dA = [None] * (trainer.visual.layers * 4)
        dB = [None] * (trainer.visual.layers * 4)
        for (block, code), k in trainer._slots.items():
            dA[block * 4 + code], dB[block * 4 + code] = grads[2 * k], grads[2 * k + 1]
        ctx.bind_current_stream()
        check(ctx.lib.jcb_vit_train_backward(fctx.tape.handle, ptr(dout.contiguous()), _ptr_array(dA), _ptr_array(dB)),
              ctx.handle)
        fctx.tape.release()
        return (None, None) + tuple(grads)


class LoraTrainer:
    """Differentiable image tower over the LoRA adapters of `layers` (what `apply_lora` returned for `model`).

    parameters(): the adapters as CUDA fp32 leaf tensors, A [r, width] then B [width, r] per projection, in block order
    and q, k, v, o order.  `trainer(views)` -> features [n, embed_dim] fp32; in training mode (the default, `train()`)
    through the device backward pass with dropout `dropout_rate` (the layers' own rate unless given), in eval mode
    (`eval()`) exactly `model.encode_image` in the applied LoRA mode."""

    def __init__(self, model, layers, seed=0, dropout_rate=None, normalize=True, apply_clip_norm=False, device=None):
        self.visual = model.visual if hasattr(model, "visual") else model
        self.seed, self.step, self.training = int(seed), 0, True
        self.normalize, self.apply_clip_norm = bool(normalize), bool(apply_clip_norm)
        blocks = self.visual.transformer.resblocks
        dev = torch.device("cuda", get_context(device).device)
        self._params, self._slots, self._lins = [], {}, []
        rates = []
        for attn in layers:
            block = next((i for i, b in enumerate(blocks) if b.attn is attn), None)
            if block is None:
                raise ValueError("LoraTrainer trains image-tower adapters: a layer is not an attention of model.visual")
            for attr, code in _LORA_PROJ:
                lin = getattr(attn, attr)
                if not getattr(lin, "lora_enabled", False):
                    continue
                self._slots[(block, code)] = len(self._lins)
                self._lins.append(lin)
                rates.append(lin.dropout_rate)
                for arr in (lin.w_lora_A.data, lin.w_lora_B.data):
                    self._params.append(torch.tensor(np.asarray(arr, np.float32), device=dev, requires_grad=True))
        if not self._lins:
            raise ValueError("LoraTrainer: the layers carry no adapter")
        self.dropout_rate = float(rates[0] if dropout_rate is None else dropout_rate)
        self._ctx = get_context(dev)
        if self._ctx.lora_mode != "applied":
            self._ctx.set_lora_mode("applied")
            self.visual.mark_dirty()
        self._vit = None

    def parameters(self):
        return list(self._params)

    def train(self, mode=True):
        self.training = bool(mode)
        return self

    def eval(self):
        return self.train(False)

    def _sync_device(self, device):
        """Pack the current adapter values into the tower (no base-weight re-pack)."""
        with torch.cuda.device(device):
            ctx, vit = self.visual._engine(device)
            ctx.bind_current_stream()
            A = [None] * (self.visual.layers * 4)
            B = [None] * (self.visual.layers * 4)
            for (block, code), k in self._slots.items():
                A[block * 4 + code] = self._params[2 * k].detach()
                B[block * 4 + code] = self._params[2 * k + 1].detach()
            check(ctx.lib.jcb_vit_train_set_lora(vit, _ptr_array(A), _ptr_array(B)), ctx.handle)
        self._ctx, self._vit = ctx, vit

    def __call__(self, views):
        views = views.contiguous()
        if not views.is_cuda:
            raise ValueError("LoraTrainer takes device-resident views")
        self._sync_device(views.device)
        if not self.training:
            with torch.cuda.device(views.device):
                out = torch.empty((views.shape[0], self.visual.output_dim), dtype=torch.float32, device=views.device)
                check(self._ctx.lib.jcb_encode_image(self._vit, ptr(views), img_dtype_code(views), views.shape[0],
                                                     int(self.apply_clip_norm), int(self.normalize), ptr(out)),
                      self._ctx.handle)
            return out
        with torch.cuda.device(views.device):
            out = _TowerFn.apply(self, views, *self._params)
        self.step += 1
        return out

    def sync_to_model(self):
        """Copy the trained adapters back into the model's LoRA layers (numpy), e.g. before `save_lora`."""
        for k, lin in enumerate(self._lins):
            lin.w_lora_A.data = self._params[2 * k].detach().cpu().numpy().copy()
            lin.w_lora_B.data = self._params[2 * k + 1].detach().cpu().numpy().copy()

    def save(self, args, epoch, list_lora_layers, save_dir="lora_weights"):
        """`save_lora` (reference test.py:642-684) of the trained adapters; `load_lora` reads the pickle back."""
        from .lora import save_lora
        self.sync_to_model()
        return save_lora(args, epoch, list_lora_layers, save_dir)


def dropout_mask(seed, step, layer, proj, rows, cols, rate, device=None):
    """The keep mask [rows, cols] (uint8, on the device) of the training dropout of projection `proj` (JCB_PROJ_*) of
    block `layer` at `step`; row = view index * tokens + token within a call."""
    ctx = get_context(device)
    out = torch.empty((rows, cols), dtype=torch.uint8, device=torch.device("cuda", ctx.device))
    with torch.cuda.device(out.device):
        ctx.bind_current_stream()
        check(ctx.lib.jcb_lora_dropout_mask(ctx.handle, seed, step, layer, proj, rows, cols, float(rate), ptr(out)), ctx.handle)
    return out


# ---- host reproduction of the dropout mask (tests; the same Philox4x32-10 words as csrc/train.cu dropout_keep) ----
_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (curand_philox4x32_x.h) on uint64 numpy arrays holding 32-bit values; returns the 4 output words."""
    m32 = np.uint64(0xFFFFFFFF)
    c0, c1, c2, c3 = (np.asarray(x, np.uint64) & m32 for x in (c0, c1, c2, c3))
    k0, k1 = np.uint64(k0) & m32, np.uint64(k1) & m32
    for i in range(10):
        p0 = np.uint64(_M0) * c0
        p1 = np.uint64(_M1) * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & m32
        hi1, lo1 = p1 >> np.uint64(32), p1 & m32
        c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
        if i < 9:
            k0, k1 = (k0 + np.uint64(_W0)) & m32, (k1 + np.uint64(_W1)) & m32
    return c0, c1, c2, c3


def dropout_mask_host(seed, step, layer, proj, rows, cols, rate):
    """numpy reproduction of `dropout_mask`: element kept iff the top 24 bits of its Philox word >= floor(rate 2^24)."""
    r, c = np.meshgrid(np.arange(rows, dtype=np.uint64), np.arange(cols, dtype=np.uint64), indexing="ij")
    words = philox4x32_10(c >> np.uint64(2), r, np.uint64(step), np.uint64(layer * 4 + proj), seed & 0xFFFFFFFF, seed >> 32)
    sel = (c & np.uint64(3)).astype(np.int64)
    w = np.choose(sel, words)
    thr = np.uint64(int(np.float64(np.float32(rate)) * 16777216.0))
    return ((w >> np.uint64(8)) >= thr).astype(np.uint8)


__all__ = ["LoraTrainer", "dropout_mask", "dropout_mask_host", "philox4x32_10"]
