"""Per-GPU context of the native library plus the tensor hand-off helpers of the Python host side.

PyTorch is plumbing here: device memory, streams and (dist.py) torch.distributed.  Every device
tensor crosses the C-ABI as a raw pointer; Jittor Vars and other frameworks' arrays come in through
DLPack (zero copy).  Nothing in this module computes.
"""
import ctypes
import threading

import numpy as np
import torch

from . import _capi
from ._capi import byref, c_void_p, check

_contexts = {}
_lock = threading.Lock()


class Context:
    """One jcb_ctx per process and GPU (replaces `jt.flags.use_cuda = 1`, reference test.py:25)."""

    def __init__(self, device):
        self.lib = _capi.load_library()
        self.device = int(device)
        h = c_void_p()
        check(self.lib.jcb_ctx_create(self.device, byref(h)))
        self.handle = h
        self._stream = None
        # the pass bounds last set through this object (the library's defaults until then, include/jclip_b200.h)
        self.chunk_views, self.host_chunk_views = 16384, 2048

    def bind_current_stream(self):
        """Run the library's kernels on torch's current stream so they order with the caller's work."""
        s = torch.cuda.current_stream(self.device).cuda_stream
        if s != self._stream:
            check(self.lib.jcb_ctx_set_stream(self.handle, c_void_p(s)), self.handle)
            self._stream = s

    def set_chunk_views(self, n):
        check(self.lib.jcb_ctx_set_chunk_views(self.handle, int(n)), self.handle)
        self.chunk_views = int(n)

    def set_host_chunk_views(self, n):
        check(self.lib.jcb_ctx_set_host_chunk_views(self.handle, int(n)), self.handle)
        self.host_chunk_views = int(n)

    def set_cls_only_last_block(self, on):
        """Opt-in: last block of the image tower on the class-token rows only (include/jclip_b200.h)."""
        check(self.lib.jcb_ctx_set_cls_only_last_block(self.handle, int(bool(on))), self.handle)

    def set_operand_type(self, name):
        """16-bit operand type of the towers packed from now on: "f16" (default; logits within 1e-2 of the fp32
        reference end to end) or "bf16" (include/jclip_b200.h jcb_ctx_set_operand_type).  Models re-pack lazily."""
        try:
            code = _capi.OPERAND_NAMES[str(name).lower()]
        except KeyError:
            raise ValueError(f"operand type must be 'f16' or 'bf16', got {name!r}") from None
        check(self.lib.jcb_ctx_set_operand_type(self.handle, code), self.handle)

    @property
    def operand_type(self):
        return "f16" if self.lib.jcb_ctx_get_operand_type(self.handle) == _capi.OPERAND_F16 else "bf16"

    def set_lora_mode(self, name):
        """How the towers packed from now on carry their LoRA adapters: "merged" (default: W + s B A in fp32, rounded once)
        or "applied" (y = W x + b + s B (A x) as low-rank tcgen05 GEMMs accumulated into the projection's TMEM tile, the
        branch the reference evaluates, test.py:388-398; include/jclip_b200.h jcb_ctx_set_lora_mode).  Models re-pack lazily."""
        try:
            code = _capi.LORA_MODES[str(name).lower()]
        except KeyError:
            raise ValueError(f"lora mode must be 'merged' or 'applied', got {name!r}") from None
        check(self.lib.jcb_ctx_set_lora_mode(self.handle, code), self.handle)

    @property
    def lora_mode(self):
        return "applied" if self.lib.jcb_ctx_get_lora_mode(self.handle) == _capi.LORA_APPLIED else "merged"

    @property
    def operand_torch_dtype(self):
        return torch.float16 if self.operand_type == "f16" else torch.bfloat16

    def sync(self):
        check(self.lib.jcb_sync(self.handle), self.handle)

    def set_graphs(self, on=True, max_views=0):
        """CUDA graphs for small jcb_pipeline calls (include/jclip_b200.h jcb_ctx_set_graphs)."""
        check(self.lib.jcb_ctx_set_graphs(self.handle, int(bool(on)), int(max_views)), self.handle)

    def graph_stats(self):
        c, n, f = ctypes.c_int64(), ctypes.c_int64(), ctypes.c_int64()
        check(self.lib.jcb_ctx_graph_stats(self.handle, byref(c), byref(n), byref(f)), self.handle)
        return {"captured": c.value, "launched": n.value, "failed": f.value}

    def trim(self):
        """Release the context's grow-only scratch (re-reserved on demand)."""
        check(self.lib.jcb_ctx_trim(self.handle), self.handle)

    @property
    def launch_count(self):
        return int(self.lib.jcb_ctx_launch_count(self.handle))

    def info(self):
        sms, maj, mnr, ws = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(), ctypes.c_size_t()
        check(self.lib.jcb_ctx_info(self.handle, byref(sms), byref(maj), byref(mnr), byref(ws)), self.handle)
        return {"num_sms": sms.value, "cc": (maj.value, mnr.value), "workspace_bytes": ws.value}

    def profile_start(self):
        check(self.lib.jcb_ctx_profile(self.handle, 1), self.handle)

    def profile_stop(self):
        """Stop and return {kernel class: {ms, launches, timed_launches, flops, bytes}} (CUDA events on
        the launch stream around every launch since profile_start)."""
        check(self.lib.jcb_ctx_profile(self.handle, 0), self.handle)
        out = {}
        for kc in range(_capi.KC_COUNT):
            ms, fl, by = ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
            n, nt = ctypes.c_int64(), ctypes.c_int64()
            check(self.lib.jcb_ctx_profile_read(self.handle, kc, byref(ms), byref(n), byref(nt), byref(fl), byref(by)),
                  self.handle)
            if n.value:
                out[self.lib.jcb_kernel_class_name(kc).decode()] = {
                    "ms": ms.value, "launches": n.value, "timed_launches": nt.value, "flops": fl.value,
                    "bytes": by.value}
        return out

    def close(self):
        if self.handle:
            self.lib.jcb_ctx_destroy(self.handle)
            self.handle = None


def get_context(device=None):
    if device is None:
        if not torch.cuda.is_available():
            raise RuntimeError("jclip_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        device = torch.cuda.current_device()
    if isinstance(device, torch.device):
        device = device.index if device.index is not None else torch.cuda.current_device()
    with _lock:
        ctx = _contexts.get(device)
        if ctx is None:
            ctx = _contexts[device] = Context(device)
    return ctx


# ------------------------------------------------------------------------------------------------
_IMG_DTYPES = {torch.float32: _capi.IMG_F32, torch.bfloat16: _capi.IMG_BF16, torch.uint8: _capi.IMG_U8}


def img_dtype_code(t):
    """JCB_IMG_* of an image tensor [..., 3, R, R] -- or, for a 16-bit tensor whose last two dims are NOT a square image
    ([..., patches, 3 * P * P]: the patch matrix TTAViews(emit="patches") writes), JCB_IMG_PATCHES_*."""
    if t.dim() >= 3 and t.shape[-1] != t.shape[-2] and t.dtype in (torch.float16, torch.bfloat16):
        return _capi.IMG_PATCHES_F16 if t.dtype == torch.float16 else _capi.IMG_PATCHES_BF16
    try:
        return _IMG_DTYPES[t.dtype]
    except KeyError:
        raise TypeError(f"images must be float32, bfloat16 or uint8, got {t.dtype}") from None


def as_torch(x, device=None):
    """Borrow `x` as a torch tensor without copying when it already lives on a device.

    torch.Tensor -> itself; objects exporting DLPack (jittor.Var, cupy, ...) -> torch.from_dlpack;
    numpy / sequences -> a host tensor (the caller decides whether to use the *_host entry point)."""
    if isinstance(x, torch.Tensor):
        return x
    if hasattr(x, "__dlpack__"):
        return torch.from_dlpack(x)
    if hasattr(x, "dlpack"):          # jittor.Var.dlpack() returns a capsule
        return torch.utils.dlpack.from_dlpack(x.dlpack())
    return torch.from_numpy(np.ascontiguousarray(x))


def dev_f32(x, device):
    """fp32 contiguous tensor on `device` (copies only if needed)."""
    t = as_torch(x)
    return t.to(device=device, dtype=torch.float32).contiguous()


def ptr(t):
    return c_void_p(t.data_ptr()) if t is not None else c_void_p(0)


def dlpack_capsule_pointer(capsule):
    """DLManagedTensor* inside a 'dltensor' PyCapsule (for jcb_encode_image_dlpack)."""
    api = ctypes.pythonapi
    api.PyCapsule_GetPointer.restype = ctypes.c_void_p
    api.PyCapsule_GetPointer.argtypes = [ctypes.py_object, ctypes.c_char_p]
    return ctypes.c_void_p(api.PyCapsule_GetPointer(capsule, b"dltensor"))
