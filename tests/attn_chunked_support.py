"""Test infrastructure for VQA_OP_ATTN_CHUNKED (questions longer than 64 tokens): the CPU emulator's restatement of the
op and its row of the schedule's access table.

Importing this module registers both: ``emulator.Emulator.op_attn_chunked`` (the emulator dispatches on ``"op_" +
kind``) and ``schedule.ACCESS["attn_chunked"]``.  The tests of long questions import it; so does any test that builds a
program with more than 64 tokens.
"""
import torch

import emulator as E
import schedule as S


def op_attn_chunked(self, op, ext):
    """Self-attention (q and kv both the packed qkv rows, key mask) or cross-attention (q_per_kv questions per image, no
    mask) of questions longer than 64 tokens, with the emulator's own attention (``Emulator._attend``)."""
    i = op.i
    B, L, H, hd, T = i["B"], i["L"], i["H"], i["hd"], i["T"]
    D = H * hd
    q = torch.as_strided(E._t(op.p["q"], torch.float32, ext), (B * L, D), (i["ld_q"], 1)).view(B, L, H, hd).transpose(1, 2)
    kvf = E._t(op.p["kv"], torch.float32, ext)
    qk = max(i.get("q_per_kv", 1), 1)           # consecutive queries that share one image's K / V
    Bi = B // qk
    k = torch.as_strided(kvf[i["k_off"]:], (Bi * T, D), (i["ld_kv"], 1)).view(Bi, T, H, hd).transpose(1, 2)
    v = torch.as_strided(kvf[i["v_off"]:], (Bi * T, D), (i["ld_kv"], 1)).view(Bi, T, H, hd).transpose(1, 2)
    k, v = k.repeat_interleave(qk, dim=0), v.repeat_interleave(qk, dim=0)
    mask = None
    if op.p.get("mask") is not None:
        mask = E._t(op.p["mask"], torch.int32, ext)[: B * T].view(B, T)
    ctx, w = self._attend(q, k, v, hd, mask)
    self._attn_store(op.p["out"], i.get("no_round", 0), ctx.transpose(1, 2).reshape(B, L, D), ext)
    if op.p.get("weights") is not None:
        E._t(op.p["weights"], torch.float32, ext)[: B * H * L * T].view(B, H, L, T).copy_(w)


E.Emulator.op_attn_chunked = op_attn_chunked
S.ACCESS.setdefault("attn_chunked", dict(q=S.R, kv=S.R, mask=S.R, out=S.W, weights=S.W))
