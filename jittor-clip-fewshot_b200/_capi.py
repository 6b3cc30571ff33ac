"""ctypes binding of libjclip_b200.so: one prototype per declaration in include/jclip_b200.h.

This is the only place the Python host side touches native code.  There is no CPU fallback: if the
library is missing the import of any product module fails with instructions to build it, and a
context cannot be created without an sm_100 GPU.
"""
import ctypes
import os
from ctypes import (POINTER, Structure, byref, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t,
                    c_void_p)
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = PKG_DIR / "libjclip_b200.so"

JCB_OK = 0
JCB_E_INVALID, JCB_E_CUDA, JCB_E_STATE, JCB_E_NO_DEVICE, JCB_E_KERNEL, JCB_E_NOMEM = -1, -2, -3, -4, -5, -6
JCB_ABI_VERSION = 4
MAX_INFLIGHT = 4   # JCB_MAX_INFLIGHT
MAX_LORA_SLOTS = 8   # JCB_MAX_LORA_SLOTS
IMG_F32, IMG_BF16, IMG_U8, IMG_PATCHES_BF16, IMG_PATCHES_F16 = 0, 1, 2, 3, 4
PROJ_Q, PROJ_K, PROJ_V, PROJ_O = 0, 1, 2, 3
SCORE_NAMES = ("logits", "cs", "cs1", "cs2", "cs3", "cs4", "cs5")
SCORE_INDEX = {n: i for i, n in enumerate(SCORE_NAMES)}
KC_COUNT = 19
FILTER_BILINEAR, FILTER_BICUBIC = 0, 1
# JCB_EPI_* (epilogue 3, the conv1 scatter, no longer exists)
EPI_BIAS_16, EPI_BIAS_GELU_16, EPI_BIAS_RESID_F32, EPI_F32 = 0, 1, 2, 4
EPI_LNFOLD_16, EPI_LNFOLD_GELU_16, EPI_RESID_LNPREP_SHORT, EPI_RESID_LNPREP_LONG = 5, 6, 7, 8
OPERAND_BF16, OPERAND_F16 = 0, 1
LORA_MERGED, LORA_APPLIED = 0, 1
LORA_MODES = {"merged": LORA_MERGED, "applied": LORA_APPLIED}
OPERAND_NAMES = {"bf16": OPERAND_BF16, "f16": OPERAND_F16, "fp16": OPERAND_F16, "float16": OPERAND_F16,
                 "bfloat16": OPERAND_BF16}

_ERR_NAMES = {-1: "JCB_E_INVALID", -2: "JCB_E_CUDA", -3: "JCB_E_STATE", -4: "JCB_E_NO_DEVICE", -5: "JCB_E_KERNEL",
              -6: "JCB_E_NOMEM"}


class VitConfig(Structure):
    _fields_ = [("layers", c_int32), ("width", c_int32), ("patch", c_int32), ("resolution", c_int32),
                ("embed_dim", c_int32), ("vpt_tokens", c_int32)]


class TextConfig(Structure):
    _fields_ = [("layers", c_int32), ("width", c_int32), ("context_length", c_int32), ("vocab_size", c_int32),
                ("embed_dim", c_int32)]


class MtaParams(Structure):
    _fields_ = [("lambda_y", c_float), ("lambda_q", c_float), ("th", c_float), ("temperature", c_float),
                ("k_frac", c_double), ("max_iter", c_int32), ("reserved", c_int32)]


class HeadWeights(Structure):
    _fields_ = [("scale1", c_void_p), ("bias1", c_void_p), ("fc_w", c_void_p), ("fc_b", c_void_p)]


class SrcImage(Structure):
    _fields_ = [("offset", c_int64), ("height", c_int32), ("width", c_int32)]


class ViewJob(Structure):
    _fields_ = [("image", c_int32), ("top", c_int32), ("left", c_int32), ("crop_h", c_int32), ("crop_w", c_int32),
                ("out_h", c_int32), ("out_w", c_int32), ("off_y", c_int32), ("off_x", c_int32), ("filter", c_int32),
                ("flip", c_int32), ("reserved", c_int32)]


class GemmArgs(Structure):
    _fields_ = [("A_dev", c_void_p), ("B_dev", c_void_p), ("M", c_int32), ("N", c_int32), ("K", c_int32),
                ("operand_type", c_int32), ("bias_dev", c_void_p), ("epilogue", c_int32), ("stats_slots", c_int32),
                ("out_dev", c_void_p), ("ldo", c_int64), ("stats_dev", c_void_p), ("colsum_dev", c_void_p),
                ("out2_dev", c_void_p), ("stats_in_dev", c_void_p), ("shift_in_dev", c_void_p),
                ("shift_out_dev", c_void_p), ("stats_in_row_stride", c_int64),
                ("A2_dev", c_void_p), ("B2_dev", c_void_p), ("K2", c_int32), ("lda2", c_int64), ("ldb2", c_int64)]


class PipelineArgs(Structure):
    _fields_ = [
        ("images", c_void_p), ("img_dtype", c_int32), ("images_on_host", c_int32), ("n_images", c_int64),
        ("n_views", c_int32), ("apply_clip_norm", c_int32),
        ("text_pt_dev", c_void_p), ("text_hand_dev", c_void_p), ("text_zs_dev", c_void_p),
        ("text_pt_t_dev", c_void_p), ("text_hand_t_dev", c_void_p), ("text_zs_t_dev", c_void_p),
        ("lp", HeadWeights), ("n_classes", c_int32), ("rank_by", c_int32), ("k", c_int32),
        ("topk_on_host", c_int32),
        ("out_topk", c_void_p), ("out_feats_dev", c_void_p), ("out_scores_dev", c_void_p),
    ]


# name -> (restype, argtypes); mirrors include/jclip_b200.h line by line
PROTOTYPES = {
    "jcb_abi_version": (c_int, []),
    "jcb_ctx_create": (c_int, [c_int, POINTER(c_void_p)]),
    "jcb_ctx_destroy": (c_int, [c_void_p]),
    "jcb_ctx_set_stream": (c_int, [c_void_p, c_void_p]),
    "jcb_ctx_set_chunk_views": (c_int, [c_void_p, c_int64]),
    "jcb_ctx_set_host_chunk_views": (c_int, [c_void_p, c_int64]),
    "jcb_ctx_set_cls_only_last_block": (c_int, [c_void_p, c_int]),
    "jcb_ctx_set_operand_type": (c_int, [c_void_p, c_int]),
    "jcb_ctx_get_operand_type": (c_int, [c_void_p]),
    "jcb_vit_operand_type": (c_int, [c_void_p]),
    "jcb_text_operand_type": (c_int, [c_void_p]),
    "jcb_ctx_set_lora_mode": (c_int, [c_void_p, c_int]),
    "jcb_ctx_get_lora_mode": (c_int, [c_void_p]),
    "jcb_vit_lora_mode": (c_int, [c_void_p]),
    "jcb_text_lora_mode": (c_int, [c_void_p]),
    "jcb_ctx_trim": (c_int, [c_void_p]),
    "jcb_sync": (c_int, [c_void_p]),
    "jcb_last_error": (c_char_p, [c_void_p]),
    "jcb_ctx_info": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_size_t)]),
    "jcb_ctx_launch_count": (c_int64, [c_void_p]),
    "jcb_ctx_profile": (c_int, [c_void_p, c_int]),
    "jcb_ctx_profile_read": (c_int, [c_void_p, c_int, POINTER(c_double), POINTER(c_int64), POINTER(c_int64),
                                     POINTER(c_double), POINTER(c_double)]),
    "jcb_kernel_class_name": (c_char_p, [c_int]),
    "jcb_vit_create": (c_int, [c_void_p, POINTER(VitConfig), POINTER(c_void_p)]),
    "jcb_vit_destroy": (c_int, [c_void_p]),
    "jcb_vit_set_param": (c_int, [c_void_p, c_char_p, c_void_p, c_int64]),
    "jcb_vit_set_lora": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_float]),
    "jcb_vit_set_lora_slot": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_float]),
    "jcb_vit_set_lora_slot_count": (c_int, [c_void_p, c_int]),
    "jcb_vit_lora_slots": (c_int, [c_void_p]),
    "jcb_vit_clear_lora": (c_int, [c_void_p]),
    "jcb_vit_finalize": (c_int, [c_void_p]),
    "jcb_encode_image": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int, c_int, c_void_p]),
    "jcb_encode_image_slots": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_void_p, c_int, c_int, c_void_p]),
    "jcb_encode_image_host": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int, c_int, c_void_p]),
    "jcb_vit_debug_tokens": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int, c_void_p]),
    "jcb_text_create": (c_int, [c_void_p, POINTER(TextConfig), POINTER(c_void_p)]),
    "jcb_text_destroy": (c_int, [c_void_p]),
    "jcb_text_set_param": (c_int, [c_void_p, c_char_p, c_void_p, c_int64]),
    "jcb_text_set_lora": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_float]),
    "jcb_text_clear_lora": (c_int, [c_void_p]),
    "jcb_text_finalize": (c_int, [c_void_p]),
    "jcb_encode_text": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    "jcb_class_mean": (c_int, [c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_void_p]),
    "jcb_tta_views": (c_int, [c_void_p, c_void_p, c_void_p, POINTER(SrcImage), c_int32, POINTER(ViewJob), c_int64, c_int32,
                              c_void_p]),
    "jcb_tta_patches": (c_int, [c_void_p, c_void_p, c_void_p, POINTER(SrcImage), c_int32, POINTER(ViewJob), c_int64,
                                c_int32, c_int32, c_int32, c_int32, c_void_p]),
    "jcb_mta_default_params": (None, [POINTER(MtaParams)]),
    "jcb_mta": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, POINTER(MtaParams),
                        c_void_p, c_void_p]),
    "jcb_mta_debug": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, POINTER(MtaParams),
                              c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "jcb_head": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                         POINTER(HeadWeights), c_int64, c_int32, c_int32, c_int32, c_int32, c_void_p, c_void_p,
                         c_void_p]),
    "jcb_cosine_topk": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_float, c_int32,
                                c_void_p, c_void_p]),
    "jcb_channel_lp": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_int32, POINTER(HeadWeights), c_void_p]),
    "jcb_logit_normalize": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_void_p]),
    "jcb_pipeline": (c_int, [c_void_p, c_void_p, POINTER(PipelineArgs)]),
    "jcb_pipeline_slots": (c_int, [c_void_p, c_void_p, POINTER(PipelineArgs), c_void_p]),
    "jcb_ctx_set_graphs": (c_int, [c_void_p, c_int, c_int64]),
    "jcb_ctx_graph_stats": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int64), POINTER(c_int64)]),
    "jcb_pipeline_submit": (c_int, [c_void_p, c_void_p, POINTER(PipelineArgs), POINTER(c_int64)]),
    "jcb_pipeline_submit_slots": (c_int, [c_void_p, c_void_p, POINTER(PipelineArgs), c_void_p, POINTER(c_int64)]),
    "jcb_pipeline_wait": (c_int, [c_void_p, c_int64]),
    "jcb_gemm": (c_int, [c_void_p, POINTER(GemmArgs)]),
    "jcb_fold_ln": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p,
                            c_void_p, c_void_p]),
    "jcb_layernorm": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_int32, c_void_p]),
    "jcb_attention": (c_int, [c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_int32, c_void_p]),
    "jcb_attention_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_int32, c_int32, c_void_p]),
    "jcb_im2col": (c_int, [c_void_p, c_void_p, c_int32, c_int64, c_int32, c_int32, c_int32, c_int32, c_void_p]),
    "jcb_tensor_map_cache_stats": (None, [POINTER(ctypes.c_uint64), POINTER(ctypes.c_uint64)]),
    "jcb_encode_image_dlpack": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int]),
    "jcb_vit_train_set_lora": (c_int, [c_void_p, c_void_p, c_void_p]),
    "jcb_vit_train_forward": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int, c_int, c_float, ctypes.c_uint64, c_int64,
                                      c_void_p, POINTER(c_void_p)]),
    "jcb_vit_train_forward_dlpack": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, ctypes.c_uint64, c_int64,
                                             POINTER(c_void_p)]),
    "jcb_vit_train_backward": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "jcb_tape_release": (c_int, [c_void_p]),
    "jcb_lora_dropout_mask": (c_int, [c_void_p, ctypes.c_uint64, c_int64, c_int, c_int, c_int64, c_int32, c_float, c_void_p]),
}


class JcbError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"{_ERR_NAMES.get(code, code)}: {message}")
        self.code = code


_lib = None


def load_library(path=None):
    """dlopen libjclip_b200.so and attach the prototypes.  Raises if it has not been built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = Path(path) if path else Path(os.environ.get("JCB_LIB_PATH") or LIB_PATH)   # JCB_LIB_PATH: A/B builds only
    if not p.exists():
        raise RuntimeError(
            f"{p} is missing: the hot path is CUDA-only and has no CPU fallback.  Build it with "
            f"`python {PKG_DIR / 'build.py'}` (needs nvcc with sm_100a support).")
    lib = ctypes.CDLL(str(p))
    for name, (restype, argtypes) in PROTOTYPES.items():
        fn = getattr(lib, name)   # AttributeError here = header / library mismatch
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.jcb_abi_version() != JCB_ABI_VERSION:
        raise RuntimeError(f"ABI version mismatch: library {lib.jcb_abi_version()}, binding {JCB_ABI_VERSION}")
    if path is None:
        _lib = lib
    return lib


def check(rc, ctx_handle=None):
    if rc == JCB_OK:
        return
    msg = ""
    if ctx_handle:
        raw = load_library().jcb_last_error(ctx_handle)
        msg = raw.decode("utf-8", "replace") if raw else ""
    if rc == JCB_E_NO_DEVICE and not msg:
        msg = "no CUDA device of compute capability 10.x (B200); this library has no CPU fallback"
    raise JcbError(rc, msg)


__all__ = ["load_library", "check", "JcbError", "VitConfig", "MtaParams", "HeadWeights", "PipelineArgs", "PROTOTYPES",
           "byref", "c_void_p", "SCORE_NAMES", "SCORE_INDEX"]
