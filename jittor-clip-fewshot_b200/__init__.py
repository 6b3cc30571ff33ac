"""jittor-clip-fewshot_b200: the B200-native (sm_100a) hot path of Dokumushikun/jittor-clip-fewshot.

    encode_image (CLIP ViT-B/32, LoRA merged on q/k/v/o) over the MTA crop batch
      -> solve_mta (MeanShift mode seeking)  ->  cosine / LP++ logits  ->  top-5

behind the reference's own Python API: `jclip.load`, `model.encode_image`, `apply_lora`, `load_lora`,
`solve_mta`, `Channel_LP`, `logit_normalize`.  All arithmetic lives in `libjclip_b200.so`
(csrc/*.cu; C-ABI in include/jclip_b200.h), called through ctypes.  There is no CPU fallback.

The directory name has hyphens, so import it through the repo-root shim:  `import jclip_b200`.
"""
from . import _capi, blocks, dist, jclip, lora, methods, pipeline, runtime, synth, train, tta  # noqa: F401
from ._capi import JcbError, load_library  # noqa: F401
from .jclip import clip  # noqa: F401
from .lora import apply_lora, load_lora, load_lora_swa, save_lora  # noqa: F401
from .methods import Channel_LP, clip_classifier, cls_acc, cosine_topk, logit_normalize, solve_mta, solve_mta_batched, solve_mta_logits  # noqa: F401
from .pipeline import HotPath, TextBank, clean_results, evaluate_new_batch, merge_results, split_ood_batch  # noqa: F401
from .runtime import get_context  # noqa: F401
from .train import LoraTrainer  # noqa: F401
from .tta import TTAViews  # noqa: F401

__version__ = "0.1.0"
