"""Engine: packed weights + per-shape plans behind ``VQAModel.forward``.

One Engine belongs to one VQAModel on one CUDA device.  Weights are packed once
(``program.build_weights``); a plan (workspace + op list + tensor maps) is built per
(batch, length, input format, mask dtype, aux, top-k) and cached.
"""
from __future__ import annotations

from collections import OrderedDict
from typing import Dict, Optional, Tuple

import torch

from . import program as P
from .runtime import Plan, VqaError, lib


class ImageCache:
    """Question-independent half of the forward for ``n_images`` images: K/V of every cross-attention layer
    (``kv[l]`` fp32 ``[n_images, 49, 2 * embed_dim]``, K in the first embed_dim columns).  The reference recomputes these
    per (image, question) pair (models/fusion.py:284, models/cross_attention.py:160-161,286-287); ``Engine.encode_images``
    computes them once and ``Engine.answer`` runs only the question side against them.  A model without cross-attention
    layers caches nothing but the number of images."""

    def __init__(self, kv, n_images: Optional[int] = None):
        self.kv = list(kv)
        if n_images is None:
            if not self.kv:
                raise ValueError("an ImageCache without K/V tensors needs n_images")
            n_images = int(self.kv[0].shape[0])
        self.n_images = int(n_images)

    @property
    def nbytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in self.kv)

    def select(self, index) -> "ImageCache":
        """Cache rows ``index`` (LongTensor / list, repeats allowed): one entry per question for ``Engine.answer``."""
        idx = torch.as_tensor(index, dtype=torch.long, device=self.kv[0].device if self.kv else "cpu").reshape(-1)
        return ImageCache([t.index_select(0, idx) for t in self.kv], int(idx.numel()))

    @staticmethod
    def cat(caches) -> "ImageCache":
        caches = list(caches)
        return ImageCache([torch.cat([c.kv[l] for c in caches], 0) for l in range(len(caches[0].kv))],
                          sum(c.n_images for c in caches))


MAX_TOP_K = 128      # softmax_topk_kernel selects one winner per block-wide pass
MAX_TOP_K_ANSWERS = 50000   # softmax_topk_kernel keeps a row of logits in shared memory (206 KB at 50 000)


def check_cacheable(cfg: dict):
    """The question-side program reads each cached layer's K/V from its own external slot: one per layer, up to
    ``program.MAX_CACHED_LAYERS``."""
    if cfg["num_cross_layers"] > P.MAX_CACHED_LAYERS:
        raise NotImplementedError(f"the image cache holds up to {P.MAX_CACHED_LAYERS} cross-attention layers, the model "
                                  f"has {cfg['num_cross_layers']}: use forward / predict")


class Engine:
    def __init__(self, model, weights: Optional[P.Weights] = None, max_plans: int = 16):
        p = next(model.parameters())
        if p.device.type != "cuda":
            raise VqaError("vqa_b200.VQAModel runs on CUDA (sm_100a) only: move the model with .cuda() "
                           "(there is no CPU path)")
        lib()  # fail early if the library is missing
        self.device = p.device
        self.cfg = dict(model.config)
        with torch.no_grad():
            self.weights = weights if weights is not None else P.build_weights(
                model.state_dict(), self.cfg, self.device, precision=getattr(model, "precision", "bf16"))
        # LRU of plans: a plan owns a workspace (7.4 MB per pair: 1.9 GB at batch 256), so a server fed arbitrary batch
        # sizes must not keep one per shape for ever.  An evicted plan stays alive while somebody (a captured CUDA graph,
        # see ``last_plan``) still holds a reference; its workspace is released with the last reference.
        self.max_plans = max(1, int(max_plans))
        self._plans: "OrderedDict[tuple, Tuple[P.Program, Plan]]" = OrderedDict()
        self.last_plan: Optional[Tuple[P.Program, Plan]] = None   # plan of the latest run (graph captures pin it)
        self.window = True

    # ------------------------------------------------------------------ plans
    def plan_for(self, B: int, L: int, in_fmt: str, mask_dtype: int, want_aux: bool, top_k: int, n_images: int = 0,
                 side: str = "both", slot: int = 0):
        """``slot``: plans with different slot numbers have their own workspace, so forwards issued on different
        streams may overlap on the GPU (the pipelined predict path runs two)."""
        n_images = n_images or B
        if top_k < 0 or top_k > min(MAX_TOP_K, self.cfg["num_answers"]):
            raise ValueError(f"top_k must be between 1 and min({MAX_TOP_K}, num_answers={self.cfg['num_answers']}), got {top_k}")
        if top_k and self.cfg["num_answers"] > MAX_TOP_K_ANSWERS:
            raise ValueError(f"top-k selection runs for at most {MAX_TOP_K_ANSWERS} answers, the model has "
                             f"{self.cfg['num_answers']}: call forward and select from the logits")
        key = (B, L, in_fmt, mask_dtype, want_aux, top_k, self.window, n_images, side, slot)
        hit = self._plans.get(key)
        if hit is not None:
            self._plans.move_to_end(key)
        if hit is None:
            if L > self.cfg["max_question_length"]:
                raise RuntimeError(f"sequence length {L} exceeds max_question_length "
                                   f"{self.cfg['max_question_length']} (size of the positional-encoding buffer)")
            prog = P.Program(self.weights, self.cfg, B, L, in_fmt, mask_dtype, want_aux, top_k, self.device,
                             window=self.window, n_images=n_images, side=side)
            idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
            hit = (prog, Plan(prog.ops, idx))
            self._plans[key] = hit
            while len(self._plans) > self.max_plans:
                self._plans.popitem(last=False)
        self.last_plan = hit
        return hit

    @staticmethod
    def _mask_code(mask: Optional[torch.Tensor]) -> int:
        if mask is None:
            return P.MASK_NONE
        return {torch.int64: P.MASK_I64, torch.float32: P.MASK_F32, torch.int32: P.MASK_I32,
                torch.bool: P.MASK_U8, torch.uint8: P.MASK_U8}.get(mask.dtype, -1)

    # ------------------------------------------------------------------ execution
    def _check_images(self, images: torch.Tensor):
        if images.device != self.device:
            raise VqaError(f"inputs must live on {self.device} (got images on {images.device})")
        if images.dim() != 4:
            raise ValueError("images must be [B,3,224,224] float32 (NCHW) or [B,224,224,3] uint8 (HWC)")
        if images.dtype == torch.uint8:
            if tuple(images.shape[1:]) != (224, 224, 3):
                raise ValueError("uint8 images must be [B,224,224,3]")
            return "hwc_u8", images.contiguous()
        if tuple(images.shape[1:]) != (3, 224, 224):
            raise ValueError("float images must be [B,3,224,224]")
        return "nchw_f32", images.float().contiguous()

    def _check_question(self, token_ids, attention_mask):
        if token_ids.device != self.device:
            raise VqaError(f"inputs must live on {self.device} (got ids on {token_ids.device})")
        B, L = token_ids.shape
        ids = token_ids.contiguous()
        if ids.dtype != torch.int64:
            ids = ids.long()
        mask = attention_mask
        code = self._mask_code(mask)
        if mask is not None:
            if mask.device != self.device:
                raise VqaError("attention_mask must live on the model's device")
            if code < 0:
                mask, code = mask.float(), P.MASK_F32
            if tuple(mask.shape) != (B, L):
                raise ValueError("attention_mask must be [B, L]")
            mask = mask.contiguous()
        return ids, mask, code

    def encode_images(self, images: torch.Tensor) -> ImageCache:
        """Image side only (SURVEY 8f row f2): backbone, projector and the K/V projections of every cross-attention
        layer for ``images``; the result can be kept across calls and answered against with ``answer``."""
        in_fmt, images = self._check_images(images)
        Bi = int(images.shape[0])
        if Bi < 1:
            raise ValueError("encode_images needs at least one image")
        prog, plan = self.plan_for(Bi, 1, in_fmt, P.MASK_NONE, False, 0, Bi, side="image")
        ext = [0] * len(P.EXT)
        ext[P.EXT["images"]] = images.data_ptr()
        stream = torch.cuda.current_stream(self.device)
        plan.run(ext, stream.cuda_stream)     # the library selects the plan's device itself
        if not torch.cuda.is_current_stream_capturing():
            images.record_stream(stream)
        D2 = 2 * self.cfg["embed_dim"]
        return ImageCache([prog.tensor(f"x.{l}.kv").view(Bi, 49, D2).clone() for l in range(prog.n_cross_layers)], Bi)

    def answer(self, cache: ImageCache, token_ids: torch.Tensor, attention_mask: Optional[torch.Tensor] = None,
               top_k: int = 0):
        """Question side only against cached images: text encoder, cross-attention over ``cache``, gate, head.
        ``cache.n_images`` must divide the number of questions (image i answers the next B / n_images questions; use
        ``cache.select(index)`` for an arbitrary question -> image assignment).  Returns (logits, top_idx, top_probs);
        logits are bit-identical to ``run`` on the same images."""
        ids, mask, code = self._check_question(token_ids, attention_mask)
        B, L = ids.shape
        Bi = cache.n_images
        if Bi < 1 or B % Bi != 0:
            raise ValueError("the number of questions must be a multiple of the number of cached images")
        prog, plan = self.plan_for(B, L, "nchw_f32", code, False, top_k, Bi, side="question")
        if len(cache.kv) != prog.n_cross_layers:
            raise ValueError(f"cache has {len(cache.kv)} layers, the model has {prog.n_cross_layers}")
        D2 = 2 * self.cfg["embed_dim"]
        kv = []
        for t in cache.kv:
            if t.device != self.device or t.dtype != torch.float32 or tuple(t.shape) != (Bi, 49, D2):
                raise ValueError(f"cache entries must be fp32 [{Bi}, 49, {D2}] on {self.device}")
            kv.append(t.contiguous())
        NA = self.cfg["num_answers"]
        logits = torch.empty(B, NA, dtype=torch.float32, device=self.device)
        top_idx = torch.empty(B, max(top_k, 1), dtype=torch.int64, device=self.device)
        top_p = torch.empty(B, max(top_k, 1), dtype=torch.float32, device=self.device)
        ext = [0] * len(P.EXT)
        ext[P.EXT["ids"]] = ids.data_ptr()
        ext[P.EXT["mask"]] = mask.data_ptr() if mask is not None else 0
        ext[P.EXT["logits"]] = logits.data_ptr()
        ext[P.EXT["top_idx"]] = top_idx.data_ptr()
        ext[P.EXT["top_probs"]] = top_p.data_ptr()
        for l, t in enumerate(kv):
            ext[P.EXT[f"kv{l}"]] = t.data_ptr()
        stream = torch.cuda.current_stream(self.device)
        plan.run(ext, stream.cuda_stream)
        if not torch.cuda.is_current_stream_capturing():
            for t in (ids, mask, *kv):
                if t is not None:
                    t.record_stream(stream)
        return logits, top_idx, top_p

    def run(self, images: torch.Tensor, token_ids: torch.Tensor, attention_mask: Optional[torch.Tensor],
            want_aux: bool = False, top_k: int = 0, slot: int = 0):
        """Launch the forward on the current stream.  Returns (logits, top_idx, top_probs, program)."""
        if images.device != self.device or token_ids.device != self.device:
            raise VqaError(f"inputs must live on {self.device} (got images on {images.device}, "
                           f"ids on {token_ids.device})")
        if images.dim() != 4:
            raise ValueError("images must be [B,3,224,224] float32 (NCHW) or [B,224,224,3] uint8 (HWC)")
        if images.dtype == torch.uint8:
            in_fmt = "hwc_u8"
            if tuple(images.shape[1:]) != (224, 224, 3):
                raise ValueError("uint8 images must be [B,224,224,3]")
        else:
            in_fmt = "nchw_f32"
            if tuple(images.shape[1:]) != (3, 224, 224):
                raise ValueError("float images must be [B,3,224,224]")
            if images.dtype != torch.float32:
                images = images.float()
        B, L = token_ids.shape
        Bi = int(images.shape[0])
        if Bi < 1 or B % Bi != 0:
            # Bi == B is the reference contract; Bi < B (one image, many questions) is this engine's extension:
            # image i answers the B / Bi consecutive questions i * B/Bi .. (i + 1) * B/Bi - 1
            raise ValueError("the number of questions must be a multiple of the number of images")
        images = images.contiguous()
        ids = token_ids.contiguous()
        if ids.dtype != torch.int64:
            ids = ids.long()
        mask = attention_mask
        code = self._mask_code(mask)
        if mask is not None:
            if mask.device != self.device:
                raise VqaError("attention_mask must live on the model's device")
            if code < 0:
                mask, code = mask.float(), P.MASK_F32
            if tuple(mask.shape) != (B, L):
                raise ValueError("attention_mask must be [B, L]")
            mask = mask.contiguous()
        prog, plan = self.plan_for(B, L, in_fmt, code, want_aux, top_k, Bi, slot=slot)
        NA = self.cfg["num_answers"]
        logits = torch.empty(B, NA, dtype=torch.float32, device=self.device)
        top_idx = torch.empty(B, max(top_k, 1), dtype=torch.int64, device=self.device)
        top_p = torch.empty(B, max(top_k, 1), dtype=torch.float32, device=self.device)
        ext = [0] * len(P.EXT)
        ext[P.EXT["images"]] = images.data_ptr()
        ext[P.EXT["ids"]] = ids.data_ptr()
        ext[P.EXT["mask"]] = mask.data_ptr() if mask is not None else 0
        ext[P.EXT["logits"]] = logits.data_ptr()
        ext[P.EXT["top_idx"]] = top_idx.data_ptr()
        ext[P.EXT["top_probs"]] = top_p.data_ptr()
        stream = torch.cuda.current_stream(self.device)
        plan.run(ext, stream.cuda_stream)
        if not torch.cuda.is_current_stream_capturing():
            for t in (images, ids, mask):  # keep inputs alive until the stream has consumed them
                if t is not None:
                    t.record_stream(stream)
        return logits, top_idx, top_p, prog

    def forward(self, images, token_ids, attention_mask=None, return_aux=False):
        logits, _, _, prog = self.run(images, token_ids, attention_mask, want_aux=return_aux)
        if not return_aux:
            return logits, None
        B, L = token_ids.shape
        D = self.cfg["embed_dim"]
        aux = {
            "image_features": prog.tensor("aux.image_features").clone(),
            "text_features": prog.tensor("text_features").view(B, L, D).clone(),
            "text_pooled": prog.tensor("text_pooled").clone(),
            "fused": prog.tensor("fused").clone(),
            "cross_attention_weights": [prog.tensor(n).clone() for n in prog.xattn_weights],
            "image_projected": prog.tensor("image_projected").view(-1, 49, D).clone(),
            "attended_pooled": prog.tensor("attended_pooled").clone(),
        }
        return logits, aux

    def predict(self, images, token_ids, attention_mask=None, top_k=5, slot: int = 0):
        if top_k < 1:
            raise ValueError("top_k must be at least 1")
        _, idx, probs, _ = self.run(images, token_ids, attention_mask, top_k=top_k, slot=slot)
        return idx, probs
