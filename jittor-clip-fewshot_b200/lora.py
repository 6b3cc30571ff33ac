"""LoRA adapters on the attention projections: containers, `apply_lora`, and the pickle I/O.

Mirrors reference test.py:277-816 (identical copies in ood.py / slow_pace.py / lora_train_vlp.py):
`LoRALayer` (scaling = alpha / sqrt(r), test.py:288-289), `LinearLoRA`, `PlainMultiheadAttentionLoRA`
(splits the packed in_proj into q/k/v, test.py:487-505), `apply_lora` (test.py:608-640), `save_lora`
(:642-684), `load_lora` (:695-735), `load_lora_swa` (:736-816).  The on-disk layout is the reference's
(SURVEY.md Appendix D) and the shipped `lora_weights1/lora_weights.pkl` loads unchanged.

These objects only *hold* the adapters.  The arithmetic -- W' = W + scaling * B A in fp32, then bf16 --
happens once, on the device, when the image tower re-packs its weights (jcb_vit_set_lora /
jcb_vit_finalize); mathematically identical to the reference's eval path, which applies
W x + b + scaling * x (B A)^T un-merged (test.py:388-398).
"""
import math
import os
import pickle

import numpy as np

from .jclip.model import Module, MultiheadAttention, Param

INDEX_POSITIONS_TEXT = {                                           # test.py:52-61
    'top1': [11], 'top2': [10, 11], 'top3': [9, 10, 11], 'bottom': [0, 1, 2, 3], 'mid': [4, 5, 6, 7],
    'up': [8, 9, 10, 11], 'half-up': [6, 7, 8, 9, 10, 11], 'half-bottom': [0, 1, 2, 3, 4, 5],
    'all': list(range(12))}
_B = {'bottom': [0, 1, 2, 3], 'mid': [4, 5, 6, 7], 'up': [8, 9, 10, 11], 'half-up': [6, 7, 8, 9, 10, 11],
      'half-bottom': [0, 1, 2, 3, 4, 5], 'all': list(range(12))}
INDEX_POSITIONS_VISION = {                                         # test.py:63-88
    'ViT-B/16': dict(_B, top=[11], top3=[9, 10, 11]),
    'ViT-B/32': dict(_B),
    'ViT-L/14': dict(_B, all=list(range(21))),
}


class LoRALayer:
    """test.py:277-337 (only what inference needs)."""

    def __init__(self, r, lora_alpha, fan_in_fan_out=False, dropout_rate=0.0):
        self.r = r
        self.lora_alpha = lora_alpha
        self.dropout_rate = dropout_rate
        if self.r > 0:
            self.scaling = self.lora_alpha / math.sqrt(self.r)    # test.py:288-289: NOT alpha / r
        self.merged = False
        self.fan_in_fan_out = fan_in_fan_out


class LinearLoRA(Module, LoRALayer):
    """One projection (a row block of the packed in_proj, or out_proj) plus its adapter.

    `weight` / `bias` are views of the wrapped attention's parameters; `w_lora_A` [r, in] starts
    kaiming-uniform(a=sqrt 5) and `w_lora_B` [out, r] zero as in the reference (test.py:301-305)."""

    def __init__(self, weight, bias, r, lora_alpha, dropout_rate, owner, rng):
        Module.__init__(self)
        LoRALayer.__init__(self, r, lora_alpha, dropout_rate=dropout_rate)
        self.out_features, self.in_features = weight.shape
        self._weight, self._bias = weight, bias
        self.lora_enabled = r > 0
        if self.lora_enabled:
            bound = 1.0 / math.sqrt(self.in_features)             # kaiming_uniform_(a=sqrt(5)) on [r, in]
            self.w_lora_A = Param(rng.uniform(-bound, bound, (r, self.in_features)).astype(np.float32), owner)
            self.w_lora_B = Param(np.zeros((self.out_features, r), np.float32), owner)

    @property
    def weight(self):
        return self._weight

    @property
    def bias(self):
        return self._bias

    def merge_BA(self):
        return self.w_lora_B.data @ self.w_lora_A.data             # test.py:310-313


class PlainMultiheadAttentionLoRA(MultiheadAttention):
    """test.py:469-605.  Keeps the packed parameters of the attention it wraps (so the state-dict keys
    of jclip/model.py:235-285 still resolve) and adds `q_proj`, `k_proj`, `v_proj`, `proj`."""

    is_lora = True

    def __init__(self, existing_mha, enable_lora=('q', 'k', 'v', 'o'), r=0, lora_alpha=1, dropout_rate=0.0,
                 seed=None):
        E = existing_mha.embed_dim
        Module.__init__(self)
        self.embed_dim, self.num_heads, self.head_dim = E, existing_mha.num_heads, existing_mha.head_dim
        self.in_proj_weight = existing_mha.in_proj_weight
        self.in_proj_bias = existing_mha.in_proj_bias
        self.out_proj = existing_mha.out_proj
        self._owner = existing_mha._owner
        self.dropout = 0.0
        rng = np.random.default_rng(seed)
        W, b = self.in_proj_weight, self.in_proj_bias

        def make(lo, hi, key, src_w=None, src_b=None):
            on = key in enable_lora
            w = (lambda: W.data[lo:hi]) if src_w is None else (lambda: src_w.data)
            bb = (lambda: b.data[lo:hi]) if src_b is None else (lambda: src_b.data)
            return LinearLoRA(_View(w, (hi - lo, E)), _View(bb, (hi - lo,)), r if on else 0, lora_alpha,
                              dropout_rate, self._owner, rng)

        self.q_proj = make(0, E, 'q')                              # rows 0:E      test.py:491-494
        self.k_proj = make(E, 2 * E, 'k')                          # rows E:2E     test.py:495-498
        self.v_proj = make(2 * E, 3 * E, 'v')                      # rows 2E:3E    test.py:499-501
        self.proj = make(0, E, 'o', self.out_proj.weight, self.out_proj.bias)
        if self._owner is not None:
            self._owner.mark_dirty()


class _View:
    """Read-only window on a slice of another parameter (no copy; follows later `.data` updates)."""

    def __init__(self, getter, shape):
        self._get, self.shape = getter, shape

    @property
    def data(self):
        return self._get()


def apply_lora(args, clip_model):
    """test.py:608-640.  `args` needs .encoder, .position, .params, .r, .alpha, .dropout_rate, .backbone."""
    list_lora_layers = []
    if args.encoder in ('text', 'both'):
        indices = INDEX_POSITIONS_TEXT[args.position]
        for i, block in enumerate(clip_model.transformer.resblocks):
            if i in indices and block.attn.__class__.__name__ == 'MultiheadAttention':
                block.attn = PlainMultiheadAttentionLoRA(block.attn, enable_lora=args.params, r=args.r,
                                                         lora_alpha=args.alpha, dropout_rate=args.dropout_rate)
                list_lora_layers.append(block.attn)
    if args.encoder in ('vision', 'both'):
        indices = INDEX_POSITIONS_VISION[args.backbone][args.position]
        for i, block in enumerate(clip_model.visual.transformer.resblocks):
            if i in indices and block.attn.__class__.__name__ == 'MultiheadAttention':
                block.attn = PlainMultiheadAttentionLoRA(block.attn, enable_lora=args.params, r=args.r,
                                                         lora_alpha=args.alpha, dropout_rate=args.dropout_rate)
                list_lora_layers.append(block.attn)
    return list_lora_layers


_KEYS = (('q', 'q_proj'), ('k', 'k_proj'), ('v', 'v_proj'), ('o', 'proj'))


def lora_state(args, list_lora_layers):
    weights = {}
    for i, layer in enumerate(list_lora_layers):
        lw = {}
        for p, name in _KEYS:
            if p in args.params:
                lin = getattr(layer, name)
                lw[name] = {'w_lora_A': np.array(lin.w_lora_A.data), 'w_lora_B': np.array(lin.w_lora_B.data)}
        weights[f'layer_{i}'] = lw
    metadata = {'r': args.r, 'alpha': args.alpha, 'encoder': args.encoder, 'params': args.params,
                'position': args.position}
    return {'weights': weights, 'metadata': metadata}


def save_lora(args, epoch, list_lora_layers, save_dir='lora_weights'):
    """test.py:642-684: pickle {'weights': {'layer_i': {...}}, 'metadata': {...}} (protocol 4, numpy)."""
    os.makedirs(save_dir, exist_ok=True)
    save_path = f'{save_dir}/{epoch}_{args.filename}.pkl'
    with open(save_path, 'wb') as f:
        pickle.dump(lora_state(args, list_lora_layers), f, protocol=4)
    print(f'LoRA weights saved to {save_path}')
    return save_path


def _check_metadata(args, metadata, alpha):
    if metadata['r'] != args.r:
        raise ValueError(f"r mismatch: expected {args.r}, found {metadata['r']}")
    if metadata['alpha'] != alpha:
        raise ValueError(f"alpha mismatch: expected {alpha}, found {metadata['alpha']}")
    if metadata['encoder'] != args.encoder:
        raise ValueError(f"Encoder mismatch: expected {args.encoder}, found {metadata['encoder']}")
    if list(metadata['params']) != list(args.params):
        raise ValueError(f"Params mismatch: expected {args.params}, found {metadata['params']}")
    if metadata['position'] != args.position:
        raise ValueError(f"Position mismatch: expected {args.position}, found {metadata['position']}")


def _assign(args, list_lora_layers, weights):
    for i, layer in enumerate(list_lora_layers):
        lw = weights[f'layer_{i}']
        for p, name in _KEYS:
            if p in args.params and name in lw:
                lin = getattr(layer, name)
                lin.w_lora_A.data = lw[name]['w_lora_A']
                lin.w_lora_B.data = lw[name]['w_lora_B']


def load_lora(args, list_lora_layers, load_path):
    """test.py:695-735 (same exceptions: FileNotFoundError, ValueError on metadata mismatch)."""
    if not os.path.exists(load_path):
        raise FileNotFoundError(f'File {load_path} does not exist.')
    with open(load_path, 'rb') as f:
        loaded = pickle.load(f)
    _check_metadata(args, loaded['metadata'], args.alpha)
    _assign(args, list_lora_layers, loaded['weights'])
    print(f'LoRA weights loaded from {load_path}')


def load_lora_swa(args, list_lora_layers, swa_weights_folder):
    """test.py:736-816: average every pickle in a folder (the reference checks `args.alpha_lora` here)."""
    if not os.path.exists(swa_weights_folder):
        raise FileNotFoundError(f'folder {swa_weights_folder} does not exist.')
    acc, count = None, 0
    for filename in os.listdir(swa_weights_folder):
        path = os.path.join(swa_weights_folder, filename)
        if os.path.isdir(path):
            continue
        with open(path, 'rb') as f:
            loaded = pickle.load(f)
        _check_metadata(args, loaded['metadata'], getattr(args, 'alpha_lora', args.alpha))
        w = loaded['weights']
        if acc is None:
            acc = {ln: {pn: {k: np.zeros_like(np.asarray(v, np.float32)) for k, v in pw.items()}
                        for pn, pw in lw.items()} for ln, lw in w.items()}
        for ln, lw in w.items():
            for pn, pw in lw.items():
                for k, v in pw.items():
                    acc[ln][pn][k] += np.asarray(v, np.float32)
        count += 1
    if count == 0:
        raise FileNotFoundError(f'no LoRA pickles in {swa_weights_folder}')
    for lw in acc.values():
        for pw in lw.values():
            for k in pw:
                pw[k] /= count
    _assign(args, list_lora_layers, acc)


_PROJ_CODE = {'q': 0, 'k': 1, 'v': 2, 'o': 3}
_NAME_PROJ = {name: p for p, name in _KEYS}


def _vision_blocks(metadata, layers):
    """Image-tower block index of each `layer_i` entry of a pickle written by save_lora: apply_lora's order, text blocks
    first for encoder 'both' (test.py:608-640)."""
    enc, pos = metadata['encoder'], metadata['position']
    if enc not in ('vision', 'both'):
        raise ValueError(f"the pickle holds {enc!r} adapters; LoRA slots are image-tower adapters")
    table = INDEX_POSITIONS_VISION['ViT-L/14' if layers > 12 else 'ViT-B/16']
    blocks = [i for i in table[pos] if i < layers]
    skip = len(INDEX_POSITIONS_TEXT[pos]) if enc == 'both' else 0
    return skip, blocks


def slot_adapters(entry, layers, width, alpha=1.0):
    """One LoRA slot as {block: {proj code: (A [r, width], B [width, r], r, scaling)}} float32, from a reference-layout
    pickle path (scaling = metadata alpha / sqrt(r), test.py:288-289) or from a dict {block: {proj: (A, B)}} with proj in
    'q', 'k', 'v', 'o' (scaling alpha / sqrt(r), or given as a third element)."""
    out = {}

    def put(block, proj, A, B, scaling):
        A = np.ascontiguousarray(A, dtype=np.float32)
        B = np.ascontiguousarray(B, dtype=np.float32)
        r = A.shape[0]
        if not 0 <= block < layers:
            raise ValueError(f"LoRA slot: block {block} outside the tower's {layers} blocks")
        if A.shape != (r, width) or B.shape != (width, r):
            raise ValueError(f"LoRA slot, block {block} proj {proj}: A {A.shape} / B {B.shape}, expected [r, {width}] / [{width}, r]")
        out.setdefault(block, {})[_PROJ_CODE[proj]] = (A, B, r, float(alpha / math.sqrt(r) if scaling is None else scaling))

    if isinstance(entry, (str, os.PathLike)):
        if not os.path.exists(entry):
            raise FileNotFoundError(f'File {entry} does not exist.')
        with open(entry, 'rb') as f:
            loaded = pickle.load(f)
        md = loaded['metadata']
        skip, blocks = _vision_blocks(md, layers)
        for i, block in enumerate(blocks):
            for name, w in loaded['weights'].get(f'layer_{skip + i}', {}).items():
                put(block, _NAME_PROJ[name], w['w_lora_A'], w['w_lora_B'], md['alpha'] / math.sqrt(md['r']))
        return out
    for block, projs in entry.items():
        for proj, ab in projs.items():
            if proj not in _PROJ_CODE:
                raise ValueError(f"LoRA slot: unknown projection {proj!r} (q, k, v, o)")
            put(int(block), proj, ab[0], ab[1], ab[2] if len(ab) > 2 else None)
    return out
