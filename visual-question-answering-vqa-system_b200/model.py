"""Drop-in ``VQAModel`` whose eval-mode forward runs on hand-written sm_100a kernels.

Boundary #1 of SURVEY.md section 8b: same constructor, ``config`` dict, 225-key
``state_dict`` and ``forward(images, token_ids, attention_mask=None, return_aux=False)``
signature as the reference (models/vqa_model.py:132-311), same ``predict`` /
``get_attention_maps`` / ``get_num_parameters`` helpers (:313-380) and the same
``create_vqa_model`` / ``load_vqa_model`` factories (:383-432).

There is no PyTorch fallback: ``forward`` needs CUDA tensors, eval mode and the in-tree
``libvqa_b200.so``; anything else raises.
"""
from __future__ import annotations

from typing import Any, Dict, Optional, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F

from .modules import AnswerHead, CustomResNet, MultimodalFusion, TransformerTextEncoder

_SUPPORTED = ("The sm_100a engine runs embed_dim 128..512 in steps of 64 with head_dim = embed_dim / num_attention_heads "
              "in {16, 32, 64} and ffn_hidden_dim 64..4096 in steps of 64 (the reference defaults are 256 / 8 heads / 1024); "
              "max_question_length is at most 512.  Layer counts (0 included), vocab sizes, answer counts, se_reduction and "
              "the SE/spatial/gating ablation switches are free, with two limits: top-k selection (predict, VQAInference) "
              "runs for at most 50000 answers (forward has no limit), and the image cache (encode_images / answer, "
              "VQAInference(image_cache_size>0)) holds at most 8 cross-attention layers.")


def supported_config(embed_dim: int, num_attention_heads: int, ffn_hidden_dim: int, max_question_length: int) -> bool:
    """Whether the engine has kernels for these widths (``_SUPPORTED``).  embed_dim is the K of the text and fusion
    Linears (32-element chunks of the tf32 GEMM, 64-element chunks of the fp16 ones) and the width of the LayerNorm and
    fusion-tail kernels; head_dim selects the attention kernels' instantiation; the cross-attention FFN is 4 * embed_dim."""
    D, H, F = embed_dim, num_attention_heads, ffn_hidden_dim
    return (D % 64 == 0 and 128 <= D <= 512 and H >= 1 and D % H == 0 and D // H in (16, 32, 64)
            and F % 64 == 0 and 64 <= F <= 4096 and max_question_length <= 512)


class VQAModel(nn.Module):
    def __init__(self, vocab_size: int = 10000, embed_dim: int = 256, num_answers: int = 1000,
                 use_se_attention: bool = True, use_spatial_attention: bool = True, se_reduction: int = 16,
                 num_transformer_layers: int = 4, num_attention_heads: int = 8, ffn_hidden_dim: int = 1024,
                 max_question_length: int = 20, num_cross_layers: int = 2, use_gating: bool = True,
                 dropout: float = 0.1, answer_dropout: float = 0.3, precision: str = "bf16"):
        super().__init__()
        self.embed_dim = embed_dim
        self.num_answers = num_answers
        self.image_encoder = CustomResNet(use_se=use_se_attention, use_spatial=use_spatial_attention,
                                          se_reduction=se_reduction)
        self.text_encoder = TransformerTextEncoder(
            vocab_size=vocab_size, embed_dim=embed_dim, num_layers=num_transformer_layers,
            num_heads=num_attention_heads, ffn_hidden_dim=ffn_hidden_dim, max_length=max_question_length,
            dropout=dropout, pad_idx=0)
        self.fusion = MultimodalFusion(
            image_channels=self.image_encoder.output_channels,
            image_spatial_size=self.image_encoder.output_spatial_size, embed_dim=embed_dim,
            num_heads=num_attention_heads, num_cross_layers=num_cross_layers, dropout=dropout,
            use_gating=use_gating)
        self.answer_head = AnswerHead(input_dim=embed_dim, hidden_dim=embed_dim * 2,
                                      num_answers=num_answers, dropout=answer_dropout)
        self.config = {
            "vocab_size": vocab_size, "embed_dim": embed_dim, "num_answers": num_answers,
            "use_se_attention": use_se_attention, "use_spatial_attention": use_spatial_attention,
            "se_reduction": se_reduction, "num_transformer_layers": num_transformer_layers,
            "num_attention_heads": num_attention_heads, "ffn_hidden_dim": ffn_hidden_dim,
            "max_question_length": max_question_length, "num_cross_layers": num_cross_layers,
            "use_gating": use_gating, "dropout": dropout, "answer_dropout": answer_dropout,
        }
        # not part of the reference config: arithmetic mode of the engine ("bf16" | "tf32")
        self.precision = precision
        self._engine = None

    # ------------------------------------------------------------------ engine plumbing
    def _check_supported(self):
        c = self.config
        if not supported_config(c["embed_dim"], c["num_attention_heads"], c["ffn_hidden_dim"], c["max_question_length"]):
            raise NotImplementedError(_SUPPORTED)

    def engine(self):
        """The CUDA engine bound to this module's current parameters (built lazily)."""
        from .engine import Engine  # imports ctypes binding; fails loudly if the .so is missing
        self._check_supported()
        if self._engine is None:
            self._engine = Engine(self)
        return self._engine

    def invalidate_engine(self):
        """Drop packed weights / plans (call after mutating parameters in place)."""
        self._engine = None

    def load_state_dict(self, *a, **k):
        out = super().load_state_dict(*a, **k)
        self._engine = None
        return out

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self._engine = None
        return out

    # ------------------------------------------------------------------ reference API
    def forward(self, images: torch.Tensor, token_ids: torch.Tensor,
                attention_mask: Optional[torch.Tensor] = None, return_aux: bool = False
                ) -> Tuple[torch.Tensor, Optional[Dict]]:
        if self.training:
            raise NotImplementedError(
                "vqa_b200.VQAModel implements the eval-mode inference path only; call .eval() "
                "(training / autograd through the fused kernels is out of scope)")
        return self.engine().forward(images, token_ids, attention_mask, return_aux)

    def predict(self, images: torch.Tensor, token_ids: torch.Tensor,
                attention_mask: Optional[torch.Tensor] = None, top_k: int = 5
                ) -> Tuple[torch.Tensor, torch.Tensor]:
        self.eval()
        with torch.no_grad():
            return self.engine().predict(images, token_ids, attention_mask, top_k)

    # ------------------------------------------------------------------ extension: image cache (SURVEY 8f row f2)
    def encode_images(self, images: torch.Tensor):
        """Question-independent half of ``forward`` (backbone, projector, cross-attention K/V) for ``images``: an
        ``ImageCache`` that can be kept across calls.  ``answer(cache, ids, mask)`` then equals ``forward`` bit for bit."""
        if self.training:
            raise NotImplementedError("eval-mode inference path only; call .eval()")
        from .engine import check_cacheable
        check_cacheable(self.config)
        with torch.no_grad():
            return self.engine().encode_images(images)

    def answer(self, cache, token_ids: torch.Tensor, attention_mask: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Logits ``[B, num_answers]`` of ``token_ids`` asked about the cached images (``cache.n_images`` divides B)."""
        if self.training:
            raise NotImplementedError("eval-mode inference path only; call .eval()")
        with torch.no_grad():
            return self.engine().answer(cache, token_ids, attention_mask)[0]

    def get_attention_maps(self, images, token_ids, attention_mask=None) -> Dict[str, torch.Tensor]:
        _, aux = self.forward(images, token_ids, attention_mask, return_aux=True)
        vis = self.fusion.get_attention_visualization(
            aux["cross_attention_weights"], spatial_size=self.image_encoder.output_spatial_size)
        return {"cross_attention": aux["cross_attention_weights"], "cross_attention_spatial": vis}

    def get_num_parameters(self) -> Dict[str, int]:
        counts = {name: sum(p.numel() for p in getattr(self, name).parameters())
                  for name in ("image_encoder", "text_encoder", "fusion", "answer_head")}
        counts["total"] = sum(counts.values())
        return counts


def create_vqa_model(vocab_size: int = 10000, num_answers: int = 1000, use_attention: bool = True,
                     **kwargs: Any) -> VQAModel:
    return VQAModel(vocab_size=vocab_size, num_answers=num_answers, use_se_attention=use_attention,
                    use_spatial_attention=use_attention, **kwargs)


def load_vqa_model(checkpoint_path: str, device: str = "cpu") -> VQAModel:
    """Load a reference checkpoint ``{'config': ..., 'model_state_dict': ...}`` (training/train.py:280-288)."""
    ckpt = torch.load(checkpoint_path, map_location=device)
    model = VQAModel(**ckpt.get("config", {}))
    model.load_state_dict(ckpt["model_state_dict"])
    return model.to(device)
