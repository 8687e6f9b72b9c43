"""Shared by the model-width tests (tests/test_model_widths_cpu.py, tests/test_gpu_model_widths.py): the widths they run
and fp64 references whose head width and embedding width are parameters.  tests/question_ref.py fixes head_dim 32 for
the default model; these restate its attention and LayerNorm rows for any width.
"""
from __future__ import annotations

import math

import torch

# (embed_dim, num_attention_heads, ffn_hidden_dim) -> what each covers
CONFIGS = {
    "a": (256, 4, 1024),    # head_dim 64, fused post-attention chains (D = 256)
    "b": (256, 16, 512),    # head_dim 16, chains at FFN width 512
    "c": (512, 8, 2048),    # head_dim 64, LayerNorm / fusion tail at 512, unfused FFN, cross FFN 2048
    "d": (128, 4, 256),     # LayerNorm / fusion tail at 128
    "e": (192, 6, 768),     # embed_dim not a multiple of 128 (float2 LayerNorm rows, 64-column GEMM tiles)
}


def ctor(name, **kw):
    D, H, F = CONFIGS[name]
    return dict(embed_dim=D, num_attention_heads=H, ffn_hidden_dim=F, **kw)


def attention(q, k, v, heads, key_mask=None, q_per_kv=1):
    """softmax(Q K^T / sqrt(head_dim) + mask) V with head_dim = D / heads.  q [B, L, D]; k, v [B / q_per_kv, T, D];
    key_mask [B, T], 0 = masked.  Returns (context [B, L, D], weights [B, heads, L, T]) in fp64."""
    q, k, v = (t.to(torch.float64) for t in (q, k, v))
    B, L, D = q.shape
    T, hd = k.shape[1], D // heads
    k, v = k.repeat_interleave(q_per_kv, dim=0), v.repeat_interleave(q_per_kv, dim=0)
    qh = q.view(B, L, heads, hd).transpose(1, 2)
    kh = k.view(B, T, heads, hd).transpose(1, 2)
    vh = v.view(B, T, heads, hd).transpose(1, 2)
    s = qh @ kh.transpose(-2, -1) / math.sqrt(hd)
    if key_mask is not None:
        s = s.masked_fill(key_mask.view(B, 1, 1, T) == 0, float("-inf"))
    w = torch.softmax(s, dim=-1)
    return (w @ vh).transpose(1, 2).reshape(B, L, D), w


def ln_params(g, D, n=3):
    out = {}
    for k in range(1, n + 1):
        out[f"g{k}"] = torch.rand(D, generator=g) + 0.5
        out[f"b{k}"] = torch.randn(D, generator=g) * 0.1
    return out


def ln_rows(g, D, n_random):
    """Rows of each kind: random, constant (zero variance: the output is beta), large common offset."""
    rows = [torch.randn(n_random, D, generator=g) * 2]
    rows.append(torch.tensor([0.0, 3.0, -1.5, 1024.0]).view(4, 1).expand(4, D))
    rows.append(torch.randn(4, D, generator=g) + torch.tensor([100.0, -300.0, 1e3, 1e4]).view(4, 1))
    kinds = ["random"] * n_random + ["constant"] * 4 + ["offset"] * 4
    return torch.cat(rows).contiguous(), kinds
