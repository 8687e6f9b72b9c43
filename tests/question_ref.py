"""fp64 references for the question-side kernels (attention core, LayerNorm-256, embedding, masked pools + gate + output
norm) and the error measure for their three output forms.

Every function takes the kernel's own fp32 inputs and computes in fp64.  The references restate the reference modules
(oracle/vqa_oracle.py) op by op -- masked keys get -inf, so a fully masked row is NaN (SURVEY T5); pools divide by the
weight sum clamped to at least 1 -- and share no code with the kernels or the CPU emulator.
"""
from __future__ import annotations

import math

import torch

HD = 32          # head_dim of every attention in the engine


def attention(q, k, v, heads, key_mask=None, q_per_kv=1):
    """softmax(Q K^T / sqrt(32) + mask) V.  q [B, L, D]; k, v [B / q_per_kv, T, D] (query b reads K / V of row
    b // q_per_kv); key_mask [B, T], 0 = masked.  Returns (context [B, L, D], weights [B, heads, L, T]) in fp64."""
    q, k, v = (t.to(torch.float64) for t in (q, k, v))
    B, L, D = q.shape
    T = k.shape[1]
    k, v = k.repeat_interleave(q_per_kv, dim=0), v.repeat_interleave(q_per_kv, dim=0)
    qh = q.view(B, L, heads, HD).transpose(1, 2)
    kh = k.view(B, T, heads, HD).transpose(1, 2)
    vh = v.view(B, T, heads, HD).transpose(1, 2)
    s = qh @ kh.transpose(-2, -1) / math.sqrt(HD)
    if key_mask is not None:
        s = s.masked_fill(key_mask.view(B, 1, 1, T) == 0, float("-inf"))
    w = torch.softmax(s, dim=-1)
    return (w @ vh).transpose(1, 2).reshape(B, L, D), w


def layernorm(x, gamma, beta, eps=1e-5):
    """LayerNorm over the last dimension: biased variance, eps inside the square root."""
    x = x.to(torch.float64)
    mean = x.mean(dim=-1, keepdim=True)
    var = (x - mean).pow(2).mean(dim=-1, keepdim=True)
    return (x - mean) / torch.sqrt(var + eps) * gamma.to(torch.float64) + beta.to(torch.float64)


def embed(table, pe, ids):
    """table[id] + pe[position] (the table is stored pre-scaled by sqrt(D)); ids [B, L]."""
    L = ids.shape[1]
    return table.to(torch.float64)[ids] + pe.to(torch.float64)[:L].unsqueeze(0)


def masked_pool(x, weights):
    """sum_l x[:, l] * w[:, l] / clamp(sum_l w[:, l], min=1) (models/fusion.py:303-313); x [B, L, D], weights [B, L]."""
    w = weights.to(torch.float64).unsqueeze(-1)
    return (x.to(torch.float64) * w).sum(dim=1) / w.sum(dim=1).clamp(min=1)


def gate_mix(ap, tp, pre):
    """sigmoid(pre) * att + (1 - sigmoid(pre)) * txt (models/fusion.py:159-166)."""
    g = torch.sigmoid(pre.to(torch.float64))
    return g * ap.to(torch.float64) + (1 - g) * tp.to(torch.float64)


# ----------------------------------------------------------------------------- output forms
def half_ulp(x, form):
    """Half a unit in the last place at |x| of the output format: 0 for fp32 (compared at the fp32 gate),
    2^(e - 12) for tf32 and fp16 (11 significant bits), fp16 with its subnormal floor 2^-24."""
    if form == "f32":
        return torch.zeros_like(x)
    _, e = torch.frexp(x.abs())                  # |x| = m * 2^e, m in [0.5, 1)
    e = e.to(torch.float64) - 12
    if form == "f16":
        e = e.clamp(min=-25)
    return torch.where(x == 0, torch.zeros_like(x) if form == "tf32" else torch.full_like(x, 2.0 ** -25), torch.exp2(e))


def is_tf32(t):
    """True where the fp32 value has no bits below the 10-bit tf32 mantissa."""
    return (t.contiguous().view(torch.int32) & 0x1FFF) == 0


def form_error(got, want, form):
    """Worst error of a kernel output against its fp64 reference, beyond the rounding its format allows:
    max(|got - want| - half_ulp(want)) / max|want| over the elements where the reference is finite.  NaN positions are
    checked separately (``nan_mismatch``)."""
    got, want = got.to(torch.float64), want.to(torch.float64)
    ok = ~torch.isnan(want)
    if not bool(ok.any()):
        return 0.0
    g, w = got[ok], want[ok]
    excess = (g - w).abs() - half_ulp(w, form)
    amax = float(w.abs().max())
    return float(torch.nan_to_num(excess, nan=math.inf).max().clamp(min=0)) / (amax if amax > 0 else 1.0)


def nan_mismatch(got, want) -> int:
    """Elements where exactly one of kernel and reference is NaN."""
    return int((torch.isnan(got.to(torch.float64)) != torch.isnan(want.to(torch.float64))).sum())
