"""The whole hot path for a shard of images in one native call, and the batched forms of the
reference's per-image evaluation loops.

The reference iterates `for image in loader:` with batch size 1 and, per image, runs encode_image on
the 1+N views, three `solve_mta`, two `channel_lp`, three `logit_normalize`, three cosine-logit
matmuls, the fusion and `topk(5)` -- each a handful of Jittor kernels plus a host sync
(test.py:1692-1742, :1759-1779, ood.py:867-883).  `HotPath.evaluate_base` does the same arithmetic
for I images at once with ONE C-ABI call (jcb_pipeline): the image tower over I*(N+1) views in
L2-sized chunks, one MTA launch (3 problems per image), one head launch.
"""
import re

import numpy as np
import torch

from . import _capi
from ._capi import check
from .jclip.model import slot_array
from .methods import Channel_LP, cosine_topk, solve_mta_batched
from .runtime import as_torch, dev_f32, get_context, img_dtype_code, ptr

OOD_BASE_MAX = 372   # reference ood.py:880 routes `pred <= 372` to the base list (bug-compatible, SURVEY C-2)


class TextBank:
    """The cached text embeddings of the hot path, resident on the device in both orientations:
    T [C, D] for the cosine logits (test.py:1729-1731) and T^T [D, C] for solve_mta (test.py:1708)."""

    def __init__(self, text_pt, text_hand, text_zs, device):
        self.device = torch.device(device)
        self.pt, self.hand, self.zs = (dev_f32(t, self.device) for t in (text_pt, text_hand, text_zs))
        self.pt_t, self.hand_t, self.zs_t = (t.t().contiguous() for t in (self.pt, self.hand, self.zs))
        self.num_classes, self.dim = self.pt.shape


class _Ticket:
    """One un-collected submission: keeps the input / output buffers and the argument struct alive."""

    def __init__(self, ctx, ticket_id, topk, keep):
        self.ctx, self.id, self.topk, self.keep = ctx, ticket_id, topk, keep


class HotPath:
    """encode_image -> L2 normalise -> solve_mta x3 -> Channel_LP / logit_normalize / fusion -> top-k."""

    def __init__(self, clip_model, text_bank, channel_lp, clip_model_zs=None, rank_by="cs1", k=5,
                 apply_clip_norm=True):
        """rank_by: the score whose top-k is returned.  Default "cs1" = cosine_similarity1, what the reference's
        evaluate_base writes to its result file (test.py:1738); "cs5" is the LP++ fusion the reference computes beside it
        (test.py:1735) and BASELINE.json's headline config names -- bench.py and the parity tests pass it explicitly."""
        if rank_by not in _capi.SCORE_INDEX:
            raise ValueError(f"rank_by must be one of {sorted(_capi.SCORE_INDEX)}, got {rank_by!r}")
        self.model, self.model_zs = clip_model, clip_model_zs
        self.text, self.lp = text_bank, channel_lp
        self.rank_by, self.k, self.apply_clip_norm = rank_by, k, apply_clip_norm

    @staticmethod
    def _check_input(images):
        """[I, V, 3, R, R] pixels (float32 / bfloat16 / uint8, device or pinned host) or the device-resident patch matrix
        [I, V, patches, 3 * P * P] of TTAViews(emit="patches")."""
        t = as_torch(images)
        is_patches = t.dim() == 4 and t.dtype in (torch.float16, torch.bfloat16) and t.is_cuda
        if t.dim() != 5 and not is_patches:
            raise ValueError(f"expected images [I, V, 3, R, R] (or a device patch matrix [I, V, patches, 3 P P]), got {tuple(t.shape)}")
        return t.contiguous()

    def _args(self, images, I, V, on_host, out_topk, out_feats, out_scores, device):
        a = _capi.PipelineArgs()
        a.images = images.data_ptr()
        a.img_dtype = img_dtype_code(images)
        a.images_on_host = int(on_host)
        a.n_images, a.n_views = I, V
        a.apply_clip_norm = int(self.apply_clip_norm)
        tb = self.text
        a.text_pt_dev, a.text_hand_dev, a.text_zs_dev = tb.pt.data_ptr(), tb.hand.data_ptr(), tb.zs.data_ptr()
        a.text_pt_t_dev, a.text_hand_t_dev, a.text_zs_t_dev = tb.pt_t.data_ptr(), tb.hand_t.data_ptr(), tb.zs_t.data_ptr()
        a.lp = self.lp.head_struct(device)
        a.n_classes = tb.num_classes
        a.rank_by = _capi.SCORE_INDEX[self.rank_by]
        a.k = self.k
        a.topk_on_host = int(not out_topk.is_cuda)
        a.out_topk = out_topk.data_ptr()
        a.out_feats_dev = out_feats.data_ptr() if out_feats is not None else None
        a.out_scores_dev = out_scores.data_ptr() if out_scores is not None else None
        return a

    def evaluate_base(self, images, return_feats=False, return_scores=False, topk_to_host=None, slot_of_image=None):
        """images [I, V, 3, R, R] (V = N+1 views, view 0 un-augmented; reference test.py:1700), float32 /
        bfloat16 / uint8, on the device or in (pinned) host memory.  Returns int32 top-k [I, k] -- on the
        host when the images were on the host (the end-to-end call), else on the device.
        slot_of_image: None, or I LoRA slot indices of the image tower (VisionTransformer.set_lora_slots): every view of
        image i runs slot slot_of_image[i]; the zero-shot tower runs its own slot 0."""
        t = self._check_input(images)
        I, V = t.shape[0], t.shape[1]
        slots = slot_array(slot_of_image, I, "slot_of_image") if slot_of_image is not None else None
        on_host = not t.is_cuda
        device = self.text.device
        if topk_to_host is None:
            topk_to_host = on_host
        with torch.cuda.device(device):
            ctx, vit = self.model.visual._engine(device)
            vit_zs = self.model_zs.visual._engine(device)[1] if self.model_zs is not None else None
            ctx.bind_current_stream()
            topk = torch.empty((I, self.k), dtype=torch.int32, device="cpu" if topk_to_host else device,
                               pin_memory=topk_to_host)
            feats = torch.empty((I * V, self.text.dim), dtype=torch.float32, device=device) if return_feats else None
            scores = torch.empty((I, self.text.num_classes), dtype=torch.float32, device=device) if return_scores else None
            a = self._args(t, I, V, on_host, topk, feats, scores, device)
            if slots is None:
                check(ctx.lib.jcb_pipeline(vit, vit_zs, _capi.byref(a)), ctx.handle)
            else:
                check(ctx.lib.jcb_pipeline_slots(vit, vit_zs, _capi.byref(a), slots.ctypes.data_as(_capi.c_void_p)),
                      ctx.handle)
        out = [topk]
        if return_feats:
            out.append(feats.view(I, V, -1))
        if return_scores:
            out.append(scores)
        return out[0] if len(out) == 1 else tuple(out)

    # ---- streams of batches: the reference's `for images in loader:` loop with the next batch's uploads
    #      overlapping this batch's compute (jcb_pipeline_submit / jcb_pipeline_wait)
    def submit(self, images, slot_of_image=None):
        """Enqueue evaluate_base(images, slot_of_image=...) without waiting and return a ticket for `collect`.  `images`
        as in evaluate_base; host images must be page-locked (pin_memory) for the copies to overlap compute and
        must not be modified until `collect` returns."""
        t = self._check_input(images)
        I, V = t.shape[0], t.shape[1]
        slots = slot_array(slot_of_image, I, "slot_of_image") if slot_of_image is not None else None
        device = self.text.device
        with torch.cuda.device(device):
            ctx, vit = self.model.visual._engine(device)
            vit_zs = self.model_zs.visual._engine(device)[1] if self.model_zs is not None else None
            ctx.bind_current_stream()
            topk = torch.empty((I, self.k), dtype=torch.int32, device="cpu", pin_memory=True)
            a = self._args(t, I, V, not t.is_cuda, topk, None, None, device)
            ticket = _capi.c_int64()
            if slots is None:
                check(ctx.lib.jcb_pipeline_submit(vit, vit_zs, _capi.byref(a), _capi.byref(ticket)), ctx.handle)
            else:
                check(ctx.lib.jcb_pipeline_submit_slots(vit, vit_zs, _capi.byref(a), slots.ctypes.data_as(_capi.c_void_p),
                                                        _capi.byref(ticket)), ctx.handle)
        return _Ticket(ctx, ticket.value, topk, (t, a))

    def collect(self, ticket):
        """Block until the submission has completed; returns its int32 top-k [I, k] on the host."""
        check(ticket.ctx.lib.jcb_pipeline_wait(ticket.ctx.handle, ticket.id), ticket.ctx.handle)
        ticket.keep = None
        return ticket.topk

    def evaluate_stream(self, batches, depth=2):
        """Generator over an iterable of image batches: yields the host top-k of each batch in order while up to
        `depth` batches are in flight (depth 2 = the uploads of batch k+1 overlap the compute of batch k).  An item of
        `batches` is an image batch, or an (images, slot_of_image) pair to run LoRA slots per image (see submit)."""
        if not 1 <= depth <= _capi.MAX_INFLIGHT:
            raise ValueError(f"depth must be in 1..{_capi.MAX_INFLIGHT}")
        pending = []
        for item in batches:
            images, slots = item if isinstance(item, tuple) else (item, None)
            pending.append(self.submit(images, slot_of_image=slots))
            if len(pending) >= depth:
                yield self.collect(pending.pop(0))
        while pending:
            yield self.collect(pending.pop(0))

    def evaluate_image_stream(self, image_batches, tta, overlap=True):
        """The reference's test loop from DECODED images (`for images in loader`, test.py:1692, with JtDataset building the
        1 + N views per image, :1547-1560): `image_batches` yields lists of [H, W, 3] uint8 arrays, `tta` is a TTAViews.
        Yields the host top-k of each batch in order.  Software pipeline, two batches in flight: while the towers work on
        batch k, the host packs batch k + 1 and enqueues its upload and view generation.

        overlap=True: the generator runs on a second, LOW-priority stream and the towers on a high-priority one, so its
        integer work fills the issue slots the tensor-core kernels leave free (the generator has its own scratch in the
        library) without delaying the persistent GEMM grids at kernel boundaries.  overlap=False: everything in stream
        order on the current stream."""
        device = self.text.device
        with torch.cuda.device(device):
            ctx, _ = self.model.visual._engine(device)
            if overlap:
                if getattr(self, "_streams", None) is None:
                    lo, hi = torch.cuda.Stream.priority_range() if hasattr(torch.cuda.Stream, "priority_range") else (0, -1)
                    self._streams = (torch.cuda.Stream(device, priority=hi), torch.cuda.Stream(device, priority=lo))
                main, side = self._streams
                main.wait_stream(torch.cuda.current_stream(device))   # weights / text banks prepared by the caller's stream
            else:
                main = side = torch.cuda.current_stream(device)
            bufs, produced, consumed = [None, None], [torch.cuda.Event(), torch.cuda.Event()], [None, None]
            pending = None
            for k, imgs in enumerate(image_batches):
                b = k & 1
                shape, dtype = tta.out_shape_dtype(len(imgs), ctx)
                n = 1
                for d in shape:
                    n *= d
                if bufs[b] is None or bufs[b].numel() < n or bufs[b].dtype != dtype:
                    bufs[b] = torch.empty(n, dtype=dtype, device=device)
                    main.wait_stream(torch.cuda.current_stream(device))
                    if overlap:      # written on `side`, read on `main`, allocated on the caller's stream: the caching
                        bufs[b].record_stream(side)      # allocator must not hand the block out again (after a later
                        bufs[b].record_stream(main)      # re-size) before both streams are done with it
                if overlap and consumed[b] is not None:
                    side.wait_event(consumed[b])            # the towers have read what this buffer held two batches ago
                views = tta(imgs, out=bufs[b][:n], stream=side if overlap else None)
                with torch.cuda.stream(main):
                    if overlap:
                        produced[b].record(side)
                        main.wait_event(produced[b])
                    ticket = self.submit(views.view(shape))     # queued BEHIND batch k - 1: the tower stream never drains
                    if overlap:
                        consumed[b] = torch.cuda.Event()
                        consumed[b].record(main)
                if pending is not None:
                    yield self.collect(pending)             # returns when batch k - 1 is done, i.e. as batch k starts: the
                pending = ticket                            # host then packs batch k + 1 while the GPU runs batch k
            if pending is not None:
                yield self.collect(pending)

    def evaluate_new(self, images, text_zs=None):
        """evaluate_new (test.py:1759-1779): zero-shot tower -> solve_mta -> 100 f T^T -> top-5."""
        model = self.model_zs if self.model_zs is not None else self.model
        return evaluate_new_batch(model, images, self.text.zs if text_zs is None else text_zs, k=self.k,
                                  apply_clip_norm=self.apply_clip_norm)


def _encode_views(model, images, apply_clip_norm):
    t = as_torch(images)
    I, V = t.shape[0], t.shape[1]
    f = model.visual(t.reshape(I * V, *t.shape[2:]), apply_clip_norm=apply_clip_norm, normalize=True)
    return as_torch(f).view(I, V, -1)


def evaluate_new_batch(model, images, text_zs, k=5, apply_clip_norm=True):
    feats = _encode_views(model, images, apply_clip_norm)
    if not feats.is_cuda:
        feats = feats.cuda()
    tz = dev_f32(text_zs, feats.device)
    mode = solve_mta_batched(feats, tz.t().contiguous())
    return cosine_topk(mode, tz, k=k)


def split_ood_batch(model, images, text_features, apply_clip_norm=False):
    """split_ood (ood.py:857-883): zero-shot MTA logits -> argmax -> base/new routing.
    Returns (pred [I] int32, is_base [I] bool) with `is_base = pred <= 372` exactly as ood.py:880.
    ood.py normalises in the PIL transform, hence apply_clip_norm defaults to False here."""
    feats = _encode_views(model, images, apply_clip_norm)
    if not feats.is_cuda:
        feats = feats.cuda()
    tz = dev_f32(text_features, feats.device)
    mode = solve_mta_batched(feats, tz.t().contiguous())
    pred = cosine_topk(mode, tz, k=1)[:, 0]
    return pred, pred <= OOD_BASE_MAX


# ---- result files (reference test.py:1738-1747, :1788-1796, :1837-1849; ood.py:866-883) ----------
def format_result_line(impath, labels):
    """`f"{impath} {top5_str}"` where impath is the batch-1 loader's list repr, e.g. "['a/b.jpg'] 1 2 3 4 5"."""
    return f"{impath} {' '.join(map(str, [int(x) for x in labels]))}"


def process_line(line):
    """test.py:1788-1796: replace "['dir/file.jpg']" by "file.jpg"."""
    m = re.search(r"\['(.*?)'\]", line)
    if m:
        line = line.replace(m.group(0), m.group(1).split('/')[-1])
    return line


def write_results(path, impaths, topk, clean=False):
    topk = as_torch(topk).cpu().numpy()
    with open(path, "w") as f:
        for p, row in zip(impaths, topk):
            line = format_result_line([p] if not isinstance(p, list) else p, row)
            f.write((process_line(line) if clean else line) + "\n")


def write_ood_split(base_path, new_path, impaths, is_base):
    """ood.py:879-883: one path per line into TestSetB_1.txt (base) / TestSetB_2.txt (new)."""
    is_base = as_torch(is_base).cpu().numpy().astype(bool)
    with open(base_path, "w") as fb, open(new_path, "w") as fn:
        for p, b in zip(impaths, is_base):
            (fb if b else fn).write(f"{p}\n")


def read_results(path):
    """A result file as {first field: [remaining fields]} in file order; a repeated key keeps its first position and
    its last values (reference load_txt_to_dict, test.py:1650-1658: whitespace-split lines into a dict).  A blank line
    raises, as it does in the reference (`parts[0]` of an empty split)."""
    out = {}
    with open(path, "r") as f:
        for line in f:
            fields = line.split()
            if not fields:
                raise IndexError(f"{path}: blank line in a result file")
            out[fields[0]] = fields[1:]
    return out


def save_results(entries, path):
    """reference save_dict_to_txt (test.py:1660-1664): "<key> <v1> <v2> ...\n" per entry, single spaces."""
    with open(path, "w") as f:
        for key, values in entries.items():
            f.write(f"{key} {' '.join(values)}\n")


def merge_results(base_txt, update_txt):
    """The merger that ends run_test1 (reference update_txt_file, test.py:1666-1674, called at :1837-1840): the base
    list written by evaluate_base is overwritten, entry by entry, by the list evaluate_new wrote for the images the
    OOD router sent to the zero-shot tower; files only in the update list are appended.  Rewrites `base_txt` in place."""
    merged = read_results(base_txt)
    merged.update(read_results(update_txt))
    save_results(merged, base_txt)
    return merged


def clean_results(input_txt, output_txt):
    """test.py:1843-1849: every line through process_line ("['dir/file.jpg']" -> "file.jpg") into result.txt."""
    with open(input_txt, "r") as fi, open(output_txt, "w") as fo:
        for line in fi:
            fo.write(process_line(line))
