"""Host-side mirror of the reference's `jclip/model.py` module tree for the image-tower hot path.

Same names and attribute paths as the reference (`CLIP.visual.transformer.resblocks[i].attn`,
`CLIP.transformer.resblocks`, `CLIP.encode_image / encode_text`, `build_model(state_dict)`,
jclip/model.py:129-285) so that `apply_lora`, `load_lora` and the `ood.py` / `test.py` call sites work
unchanged -- but the objects are thin parameter containers: `encode_image` hands the whole forward
to the sm_100a library through the C-ABI (include/jclip_b200.h), with no per-op Python.

`encode_text` (SURVEY.md section 8 row f3: it runs once per run to produce the cached text embeddings,
`clip_classifier`, reference test.py:920-940) runs on the same library with a causal attention mask.
"""
import pickle
from typing import Dict

import numpy as np
import torch

from .. import _capi
from .._capi import byref, c_void_p, check
from ..runtime import as_torch, dlpack_capsule_pointer, get_context, img_dtype_code, ptr


def _np32(x):
    if isinstance(x, torch.Tensor):
        return x.detach().to("cpu", torch.float32).numpy()
    if hasattr(x, "numpy") and not isinstance(x, np.ndarray):   # jittor.Var
        x = x.numpy()
    return np.require(np.asarray(x), dtype=np.float32, requirements="C")


class Param:
    """A named fp32 parameter held on the host.  `.data` mirrors `jt.Var.data` (numpy view); assigning
    to it (reference test.py:723-733 `layer.q_proj.w_lora_A.data = ...`) marks the owning tower's
    packed device weights stale."""

    def __init__(self, value, owner=None):
        self._v = _np32(value)
        self._owner = owner
        self._version = 0

    @property
    def data(self):
        return self._v

    @data.setter
    def data(self, value):
        v = _np32(value)
        if v.shape != self._v.shape:
            raise ValueError(f"shape mismatch: parameter is {self._v.shape}, got {v.shape}")
        self._v = v
        self._version += 1
        if self._owner is not None:
            self._owner.mark_dirty()

    @property
    def shape(self):
        return self._v.shape

    @property
    def dtype(self):
        return torch.float32

    def numpy(self):
        return self._v

    def torch(self, device="cpu"):
        return torch.from_numpy(self._v).to(device)


class Module:
    """The sliver of `jittor.nn.Module` the reference call sites use."""

    def __init__(self):
        self.is_train = False

    def children(self):
        for k, v in self.__dict__.items():
            if k.startswith("_"):
                continue
            if isinstance(v, Module):
                yield v
            elif isinstance(v, (list, tuple)):
                for m in v:
                    if isinstance(m, Module):
                        yield m

    def named_parameters(self, prefix=""):
        out = []
        for k, v in self.__dict__.items():
            if k.startswith("_"):
                continue
            name = f"{prefix}{k}"
            if isinstance(v, Param):
                out.append((name, v))
            elif isinstance(v, Module):
                out.extend(v.named_parameters(name + "."))
            elif isinstance(v, (list, tuple)):
                for i, m in enumerate(v):
                    if isinstance(m, Module):
                        out.extend(m.named_parameters(f"{name}.{i}."))
        return out

    def parameters(self):
        return [p for _, p in self.named_parameters()]

    def state_dict(self):
        return {k: p.data for k, p in self.named_parameters()}

    def train(self, mode=True):
        # Jittor's Module.train()/eval() only flip `is_train` flags by DFS (SURVEY.md Appendix B)
        self.is_train = bool(mode)
        for c in self.children():
            c.train(mode)
        return self

    def eval(self):
        return self.train(False)

    def cuda(self):
        return self

    def __call__(self, *a, **kw):
        return self.execute(*a, **kw)


class LayerNorm(Module):
    def __init__(self, weight, bias, owner=None):
        super().__init__()
        self.weight = Param(weight, owner)
        self.bias = Param(bias, owner)


class Linear(Module):
    def __init__(self, weight, bias, owner=None):
        super().__init__()
        self.weight = Param(weight, owner)
        self.bias = Param(bias, owner) if bias is not None else None
        self.out_features, self.in_features = self.weight.shape


class MultiheadAttention(Module):
    """Packed-QKV attention container (reference jclip/mha.py:469-650: in_proj_weight [3E,E],
    in_proj_bias [3E], out_proj Linear)."""

    def __init__(self, embed_dim, num_heads, in_w, in_b, out_w, out_b, owner=None):
        super().__init__()
        self.embed_dim, self.num_heads = embed_dim, num_heads
        self.head_dim = embed_dim // num_heads
        self.in_proj_weight = Param(in_w, owner)
        self.in_proj_bias = Param(in_b, owner)
        self.out_proj = Linear(out_w, out_b, owner)
        self._owner = owner


class MLP(Module):
    def __init__(self, fc_w, fc_b, proj_w, proj_b, owner=None):
        super().__init__()
        self.c_fc = Linear(fc_w, fc_b, owner)
        self.c_proj = Linear(proj_w, proj_b, owner)


class ResidualAttentionBlock(Module):
    def __init__(self, sd, prefix, width, heads, owner=None, attn_mask=None):
        super().__init__()
        g = lambda k: sd[prefix + k]
        self.attn = MultiheadAttention(width, heads, g("attn.in_proj_weight"), g("attn.in_proj_bias"),
                                       g("attn.out_proj.weight"), g("attn.out_proj.bias"), owner)
        self.ln_1 = LayerNorm(g("ln_1.weight"), g("ln_1.bias"), owner)
        self.mlp = MLP(g("mlp.c_fc.weight"), g("mlp.c_fc.bias"), g("mlp.c_proj.weight"), g("mlp.c_proj.bias"), owner)
        self.ln_2 = LayerNorm(g("ln_2.weight"), g("ln_2.bias"), owner)
        self.attn_mask = attn_mask


class Transformer(Module):
    def __init__(self, sd, prefix, width, layers, heads, owner=None, attn_mask=None):
        super().__init__()
        self.width, self.layers = width, layers
        self.resblocks = [ResidualAttentionBlock(sd, f"{prefix}resblocks.{i}.", width, heads, owner, attn_mask)
                          for i in range(layers)]


class Conv2d(Module):
    def __init__(self, weight, owner=None):
        super().__init__()
        self.weight = Param(weight, owner)


_LORA_PROJ = (("q_proj", _capi.PROJ_Q), ("k_proj", _capi.PROJ_K), ("v_proj", _capi.PROJ_V), ("proj", _capi.PROJ_O))


class VisionTransformer(Module):
    """Parameter container + native engine of the image tower (reference jclip/model.py:80-126)."""

    def __init__(self, sd, input_resolution, patch_size, width, layers, heads, output_dim, design_details=None):
        super().__init__()
        self.input_resolution, self.output_dim = input_resolution, output_dim
        self.patch_size, self.width, self.layers, self.heads = patch_size, width, layers, heads
        # IVLP / VPT tower (reference jclip/model1.py:161-164, :192-196): n_ctx learnable tokens appended after
        # the positional embedding.  The vision transformer is built with prompts_needed=0 (model1.py:175),
        # so there are no per-layer prompts: `visual.VPT` is the only extra parameter.
        n_ctx = int((design_details or {}).get("vision_ctx", 0)) if "visual.VPT" not in sd else int(sd["visual.VPT"].shape[0])
        self.n_ctx = n_ctx
        if n_ctx > 0:
            vpt = sd.get("visual.VPT")
            if vpt is None:   # normal_(ctx_vectors, std=0.02), model1.py:163
                vpt = (np.random.default_rng(0).standard_normal((n_ctx, width)) * 0.02).astype(np.float32)
            self.VPT = Param(vpt, self)
        self.conv1 = Conv2d(sd["visual.conv1.weight"], self)
        self.class_embedding = Param(sd["visual.class_embedding"], self)
        self.positional_embedding = Param(sd["visual.positional_embedding"], self)
        self.ln_pre = LayerNorm(sd["visual.ln_pre.weight"], sd["visual.ln_pre.bias"], self)
        self.transformer = Transformer(sd, "visual.transformer.", width, layers, heads, self)
        self.ln_post = LayerNorm(sd["visual.ln_post.weight"], sd["visual.ln_post.bias"], self)
        self.proj = Param(sd["visual.proj"], self)
        self._dirty = True
        self._vit = None        # jcb_vit*
        self._ctx = None
        self._lora_slots = []   # LoRA slots 1 .. G-1: {layer: {proj code: (A, B, r, scaling)}} (set_lora_slots)

    def mark_dirty(self):
        self._dirty = True

    def set_lora_slots(self, slots, alpha=1.0):
        """Register LoRA slots 1 .. len(slots) of the image tower; slot 0 stays what `apply_lora` / `load_lora` put on the
        model.  Each entry is the path of a reference-layout LoRA pickle (`save_lora`) or a dict {layer: {proj: (A, B)}}
        (proj in "q", "k", "v", "o"; A [r, width], B [width, r]; scaling alpha / sqrt(r), or pass (A, B, scaling)).
        A call then picks a slot per view (`visual(x, slot_of_view=...)`) or per image (HotPath `slot_of_image`), and
        each view comes out bit-identical to a tower that carries only its slot.  Slots need the applied LoRA mode
        (`Context.set_lora_mode("applied")`).  `set_lora_slots([])` drops them."""
        from ..lora import slot_adapters
        slots = list(slots)
        if len(slots) + 1 > _capi.MAX_LORA_SLOTS:
            raise ValueError(f"{len(slots) + 1} LoRA slots (slot 0 + {len(slots)}); at most {_capi.MAX_LORA_SLOTS}")
        self._lora_slots = [slot_adapters(s, self.layers, self.width, alpha) for s in slots]
        self._dirty = True

    @property
    def lora_slots(self):
        """G: slot 0 plus the slots registered with set_lora_slots."""
        return 1 + len(self._lora_slots)

    # ---- native engine ------------------------------------------------------------------------
    def _engine(self, device=None):
        """Create / refresh the device-side packed weights (fp32 LoRA merge, then bf16)."""
        ctx = get_context(device)
        if self._vit is not None and self._ctx is not ctx:
            self.release()
        if self._vit is None:
            cfg = _capi.VitConfig(self.layers, self.width, self.patch_size, self.input_resolution, self.output_dim,
                                  self.n_ctx)
            h = c_void_p()
            check(ctx.lib.jcb_vit_create(ctx.handle, byref(cfg), byref(h)), ctx.handle)
            self._vit, self._ctx, self._dirty = h, ctx, True
        if not self._dirty and (ctx.lib.jcb_vit_operand_type(self._vit) != ctx.lib.jcb_ctx_get_operand_type(ctx.handle) or
                                ctx.lib.jcb_vit_lora_mode(self._vit) != ctx.lib.jcb_ctx_get_lora_mode(ctx.handle)):
            self._dirty = True      # the context's operand type / LoRA mode changed since the weights were packed
        if self._dirty:
            lib = ctx.lib
            for name, p in self.named_parameters("visual."):
                if "lora_" in name:
                    continue
                a = np.ascontiguousarray(p.data, dtype=np.float32)
                check(lib.jcb_vit_set_param(self._vit, name.encode(), a.ctypes.data_as(c_void_p), a.size), ctx.handle)
            check(lib.jcb_vit_clear_lora(self._vit), ctx.handle)
            for i, block in enumerate(self.transformer.resblocks):
                attn = block.attn
                if not getattr(attn, "is_lora", False):
                    continue
                for attr, code in _LORA_PROJ:
                    lin = getattr(attn, attr)
                    if not getattr(lin, "lora_enabled", False):
                        continue
                    A = np.ascontiguousarray(lin.w_lora_A.data, dtype=np.float32)
                    B = np.ascontiguousarray(lin.w_lora_B.data, dtype=np.float32)
                    check(lib.jcb_vit_set_lora(self._vit, i, code, A.ctypes.data_as(c_void_p),
                                               B.ctypes.data_as(c_void_p), lin.r, float(lin.scaling)), ctx.handle)
            if self._lora_slots:   # every registered slot counts, also one that carries no adapter
                check(lib.jcb_vit_set_lora_slot_count(self._vit, 1 + len(self._lora_slots)), ctx.handle)
            for g, slot in enumerate(self._lora_slots, 1):
                for i, projs in sorted(slot.items()):
                    for code, (A, B, r, scaling) in sorted(projs.items()):
                        check(lib.jcb_vit_set_lora_slot(self._vit, g, i, code, A.ctypes.data_as(c_void_p),
                                                        B.ctypes.data_as(c_void_p), r, scaling), ctx.handle)
            check(lib.jcb_vit_finalize(self._vit), ctx.handle)
            self._dirty = False
        return ctx, self._vit

    def named_parameters(self, prefix=""):
        # reference key names: LoRA wrappers expose the wrapped attention's packed parameters under
        # `attn.in_proj_weight` etc., so the state-dict contract (SURVEY.md Appendix D) is unchanged
        return super().named_parameters(prefix)

    def release(self):
        if self._vit is not None and self._ctx is not None and self._ctx.handle:
            self._ctx.lib.jcb_vit_destroy(self._vit)
        self._vit, self._ctx = None, None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass

    def execute(self, x, apply_clip_norm=False, normalize=False, slot_of_view=None):
        """[B,3,R,R] -> [B,output_dim] float32.  Device tensors (torch, or anything exporting DLPack
        such as a jittor.Var) are used in place; host arrays go through the *_host entry point.
        slot_of_view: None, or B LoRA slot indices (set_lora_slots): view b is encoded with slot slot_of_view[b] only."""
        was_numpy = isinstance(x, np.ndarray)
        t = as_torch(x)
        R = self.input_resolution
        if t.dim() != 4 or t.shape[1] != 3 or t.shape[2] != R or t.shape[3] != R:
            raise ValueError(f"expected images of shape [n, 3, {R}, {R}], got {tuple(t.shape)}")
        if t.dtype == torch.float64 or t.dtype == torch.float16:
            t = t.float()
        code = img_dtype_code(t)
        t = t.contiguous()
        n = t.shape[0]
        if slot_of_view is not None:
            # host images are copied to the device first (the slot entry point takes device input)
            slots = slot_array(slot_of_view, n, "slot_of_view")
            on_device = t.is_cuda
            dev = t.device if on_device else torch.device("cuda", get_context(None).device)
            with torch.cuda.device(dev):
                t = t.to(dev)
                ctx, vit = self._engine(dev)
                ctx.bind_current_stream()
                out = torch.empty((n, self.output_dim), dtype=torch.float32, device=dev)
                check(ctx.lib.jcb_encode_image_slots(vit, ptr(t), code, n, slots.ctypes.data_as(c_void_p),
                                                     int(apply_clip_norm), int(normalize), ptr(out)), ctx.handle)
            if on_device:
                return out
            return out.cpu().numpy() if was_numpy else out.cpu()
        if t.is_cuda:
            with torch.cuda.device(t.device):
                ctx, vit = self._engine(t.device)
                ctx.bind_current_stream()
                out = torch.empty((n, self.output_dim), dtype=torch.float32, device=t.device)
                check(ctx.lib.jcb_encode_image(vit, ptr(t), code, n, int(apply_clip_norm), int(normalize), ptr(out)),
                      ctx.handle)
            return out
        ctx, vit = self._engine(None)
        with torch.cuda.device(ctx.device):
            ctx.bind_current_stream()
            out = torch.empty((n, self.output_dim), dtype=torch.float32)
            check(ctx.lib.jcb_encode_image_host(vit, ptr(t), code, n, int(apply_clip_norm), int(normalize), ptr(out)),
                  ctx.handle)
        return out.numpy() if was_numpy else out

    def execute_dlpack(self, images, out, apply_clip_norm=False, normalize=False):
        """Zero-copy DLPack entry (jcb_encode_image_dlpack): `images` and `out` are objects with
        `__dlpack__` (e.g. jittor Vars); `out` is written in place."""
        ctx, vit = self._engine(None)
        cin, cout = images.__dlpack__(), out.__dlpack__()
        with torch.cuda.device(ctx.device):
            ctx.bind_current_stream()
            check(ctx.lib.jcb_encode_image_dlpack(vit, dlpack_capsule_pointer(cin), dlpack_capsule_pointer(cout),
                                                  int(apply_clip_norm), int(normalize)), ctx.handle)
        return out

    def debug_tokens(self, x, apply_clip_norm=False):
        t = as_torch(x).contiguous()
        with torch.cuda.device(t.device):
            ctx, vit = self._engine(t.device)
            ctx.bind_current_stream()
            T = (self.input_resolution // self.patch_size) ** 2 + 1 + self.n_ctx
            out = torch.empty((t.shape[0], T, self.width), dtype=torch.float32, device=t.device)
            check(ctx.lib.jcb_vit_debug_tokens(vit, ptr(t), img_dtype_code(t), t.shape[0], int(apply_clip_norm), ptr(out)),
                  ctx.handle)
        return out


def slot_array(slots, n, name):
    """A host int32 array of n LoRA slot indices (the library validates their range)."""
    a = np.ascontiguousarray(as_torch(slots).cpu().numpy() if isinstance(slots, torch.Tensor) else np.asarray(slots),
                             dtype=np.int32)
    if a.shape != (n,):
        raise ValueError(f"{name} must hold {n} slot indices, got shape {a.shape}")
    return a


class Embedding(Module):
    def __init__(self, weight, owner=None):
        super().__init__()
        self.weight = Param(weight, owner)


class CLIP(Module):
    """reference jclip/model.py:129-232."""

    def __init__(self, sd, embed_dim, image_resolution, vision_layers, vision_width, vision_patch_size,
                 context_length, vocab_size, transformer_width, transformer_heads, transformer_layers,
                 design_details=None):
        super().__init__()
        self.context_length = context_length
        vision_heads = vision_width // 64                         # jclip/model.py:152
        self.visual = VisionTransformer(sd, image_resolution, vision_patch_size, vision_width, vision_layers,
                                        vision_heads, embed_dim, design_details)
        # the text tower's parameters are owned by this object: assigning to any of them (e.g. LoRA weights on
        # the text blocks) marks the packed device copy of the text tower stale
        self.transformer = Transformer(sd, "transformer.", transformer_width, transformer_layers, transformer_heads,
                                       self, attn_mask=self.build_attention_mask())
        self.vocab_size = vocab_size
        self.token_embedding = Embedding(sd["token_embedding.weight"], self)
        self.positional_embedding = Param(sd["positional_embedding"], self)
        self.ln_final = LayerNorm(sd["ln_final.weight"], sd["ln_final.bias"], self)
        self.text_projection = Param(sd["text_projection"], self)
        self.logit_scale = Param(sd.get("logit_scale", np.log(1 / 0.07)))
        self._text_dirty, self._text, self._text_ctx = True, None, None

    def mark_dirty(self):
        self._text_dirty = True

    def _text_engine(self, device=None):
        """Create / refresh the device-side packed text tower (jcb_text_*; LoRA merged in fp32, then bf16)."""
        ctx = get_context(device)
        if self._text is not None and self._text_ctx is not ctx:
            self.release_text()
        lib = ctx.lib
        if self._text is None:
            W = self.transformer.width
            cfg = _capi.TextConfig(self.transformer.layers, W, self.context_length, self.vocab_size,
                                   self.text_projection.shape[1])
            h = c_void_p()
            check(lib.jcb_text_create(ctx.handle, byref(cfg), byref(h)), ctx.handle)
            self._text, self._text_ctx, self._text_dirty = h, ctx, True
        if not self._text_dirty and (lib.jcb_text_operand_type(self._text) != lib.jcb_ctx_get_operand_type(ctx.handle) or
                                     lib.jcb_text_lora_mode(self._text) != lib.jcb_ctx_get_lora_mode(ctx.handle)):
            self._text_dirty = True
        if self._text_dirty:
            named = [("token_embedding.weight", self.token_embedding.weight), ("positional_embedding", self.positional_embedding),
                     ("ln_final.weight", self.ln_final.weight), ("ln_final.bias", self.ln_final.bias),
                     ("text_projection", self.text_projection)]
            named += [(n, p) for n, p in self.transformer.named_parameters("transformer.") if "lora_" not in n]
            for name, p in named:
                a = np.ascontiguousarray(p.data, dtype=np.float32)
                check(lib.jcb_text_set_param(self._text, name.encode(), a.ctypes.data_as(c_void_p), a.size), ctx.handle)
            check(lib.jcb_text_clear_lora(self._text), ctx.handle)
            for i, block in enumerate(self.transformer.resblocks):
                attn = block.attn
                if not getattr(attn, "is_lora", False):
                    continue
                for attr, code in _LORA_PROJ:
                    lin = getattr(attn, attr)
                    if getattr(lin, "lora_enabled", False):
                        A = np.ascontiguousarray(lin.w_lora_A.data, dtype=np.float32)
                        B = np.ascontiguousarray(lin.w_lora_B.data, dtype=np.float32)
                        check(lib.jcb_text_set_lora(self._text, i, code, A.ctypes.data_as(c_void_p),
                                                    B.ctypes.data_as(c_void_p), lin.r, float(lin.scaling)), ctx.handle)
            check(lib.jcb_text_finalize(self._text), ctx.handle)
            self._text_dirty = False
        return ctx, self._text

    def release_text(self):
        if self._text is not None and self._text_ctx is not None and self._text_ctx.handle:
            self._text_ctx.lib.jcb_text_destroy(self._text)
        self._text, self._text_ctx = None, None

    def __del__(self):
        try:
            self.release_text()
        except Exception:
            pass

    def build_attention_mask(self):
        mask = torch.full((self.context_length, self.context_length), float("-inf"))
        return torch.triu(mask, 1)

    @property
    def dtype(self):
        return self.visual.conv1.weight.dtype

    def encode_image(self, image):
        # jclip/model.py:199-200
        return self.visual(image)

    def encode_text(self, text, normalize=False):
        """jclip/model.py:202-215 on the sm_100a library (jcb_encode_text): [n, context_length] token ids ->
        [n, embed_dim] float32 on the GPU."""
        tok = as_torch(text)
        if tok.dim() != 2 or tok.shape[1] != self.context_length:
            raise ValueError(f"expected tokens of shape [n, {self.context_length}], got {tuple(tok.shape)}")
        if not tok.is_cuda:
            if not torch.cuda.is_available():
                raise RuntimeError("encode_text runs on a B200 GPU only; there is no CPU fallback")
            tok = tok.cuda()
        tok = tok.to(torch.int64).contiguous()
        with torch.cuda.device(tok.device):
            ctx, handle = self._text_engine(tok.device)
            ctx.bind_current_stream()
            out = torch.empty((tok.shape[0], self.text_projection.shape[1]), dtype=torch.float32, device=tok.device)
            check(ctx.lib.jcb_encode_text(handle, ptr(tok), tok.shape[0], int(normalize), ptr(out)), ctx.handle)
        return out

    def execute(self, image, text):
        # jclip/model.py:217-232
        fi = as_torch(self.encode_image(image))
        ft = as_torch(self.encode_text(text)).to(fi.device)
        fi = fi / fi.norm(dim=1, keepdim=True)
        ft = ft / ft.norm(dim=1, keepdim=True)
        scale = float(np.exp(self.logit_scale.data))
        li = scale * fi @ ft.t()
        return li, li.t()

    # ---- (de)serialisation: pickled {key: numpy} like `jt.save` / `jt.load` of a state dict ------
    def state_dict(self):
        return {k: p.data for k, p in self.named_parameters()}

    def save(self, path):
        with open(path, "wb") as f:
            pickle.dump(self.state_dict(), f, protocol=4)

    def load_parameters(self, sd):
        mine = dict(self.named_parameters())
        for k, v in sd.items():
            if k in mine:
                mine[k].data = v

    def load(self, path):
        with open(path, "rb") as f:
            self.load_parameters(pickle.load(f))


def build_model(state_dict: Dict[str, np.ndarray], design_details=None):
    """Shape inference from state-dict keys, exactly as the reference does (jclip/model.py:235-285).
    With `design_details` (or a `visual.VPT` key) this is jclip/model1.py:322-374, the IVLP variant."""
    if "visual.proj" not in state_dict:
        raise NotImplementedError("only ViT checkpoints are supported on this path (mode='vit'); the ResNet "
                                  "variant jclip/model_res.py is outside the hot path")
    sd = {k: _np32(v) for k, v in state_dict.items() if k not in ("input_resolution", "context_length", "vocab_size")}
    vision_width = sd["visual.conv1.weight"].shape[0]
    vision_layers = len([k for k in sd if k.startswith("visual.") and k.endswith(".attn.in_proj_weight")])
    vision_patch_size = sd["visual.conv1.weight"].shape[-1]
    grid_size = round((sd["visual.positional_embedding"].shape[0] - 1) ** 0.5)
    image_resolution = vision_patch_size * grid_size
    embed_dim = sd["text_projection"].shape[1]
    context_length = sd["positional_embedding"].shape[0]
    vocab_size = sd["token_embedding.weight"].shape[0]
    transformer_width = sd["ln_final.weight"].shape[0]
    transformer_heads = transformer_width // 64
    transformer_layers = len(set(k.split(".")[2] for k in sd if k.startswith("transformer.resblocks")))
    model = CLIP(sd, embed_dim, image_resolution, vision_layers, vision_width, vision_patch_size, context_length,
                 vocab_size, transformer_width, transformer_heads, transformer_layers, design_details)
    return model.eval()
