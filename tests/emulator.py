"""CPU interpreter for vqa_b200.program op lists (TEST INFRASTRUCTURE).

Executes the exact op list the CUDA library receives, on CPU tensors, with the same storage
dtypes (bf16 activations, tf32-truncated GEMM operands).  It validates the layout and tap
algebra of ``program.py`` against the oracle without a GPU, and on the GPU box it serves as
the per-op expected value for the kernels in ``csrc/``.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

import topk_ref as TR
from vqa_b200 import program as P

MEAN = torch.tensor([0.485, 0.456, 0.406])
STD = torch.tensor([0.229, 0.224, 0.225])


def trunc_tf32(t):
    return (t.contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


def _t(ref, dtype, ext):
    """Flat typed view of a Buf / external tensor."""
    if ref is None:
        return None
    if isinstance(ref, P.ExtRef):
        return ext[ref.slot]
    return ref.arena.tensor[ref.offset:].view(dtype)


def _grid_index(B, H, W, Pp, rpi):
    n = torch.arange(B).view(B, 1, 1)
    h = torch.arange(H).view(1, H, 1)
    w = torch.arange(W).view(1, 1, W)
    return (n * rpi + h * Pp + w).reshape(-1)  # [B*H*W] flat rows, NHW order


class Emulator:
    def __init__(self, prog: P.Program, tf32_truncate: bool = True):
        self.prog = prog
        self.tf32_truncate = tf32_truncate

    def run(self, ext, first=0, last=None):
        ops = self.prog.ops[first:last]
        for op in ops:
            getattr(self, "op_" + op.kind)(op, ext)

    # ------------------------------------------------------------------ ops
    def op_ingest(self, op, ext):
        i = op.i
        B, Pp, rows = i["B"], i["P"], i["rows"]
        src = ext[op.p["src"].slot]
        if i["mode"] == 0:
            x = src.float().view(B, 3, 224, 224)
        else:
            x = src.view(B, 224, 224, 3).float().div(255.0)
            x = ((x - MEAN) / STD).permute(0, 3, 1, 2)
        adt = torch.float32 if i.get("f32") else torch.bfloat16
        dst = _t(op.p["dst"], adt, ext)[: rows * 16].view(rows, 16)
        dst.zero_()
        # [B,3,112,2,112,2] -> [B,112,112,ph,pw,c]
        xp = x.reshape(B, 3, 112, 2, 112, 2).permute(0, 2, 4, 3, 5, 1)
        packed = torch.zeros(B, 112, 112, 2, 2, 4)
        packed[..., :3] = xp
        if i.get("ones"):
            packed[..., 0, :, 3] = 1.0   # bias columns of the fused stem (phases (0,0) and (0,1))
        idx = _grid_index(B, 112, 112, Pp, Pp * Pp)
        dst[idx] = P.round_tf32(packed.reshape(-1, 16)) if i.get("f32") else packed.reshape(-1, 16).to(torch.bfloat16)

    def op_gemm(self, op, ext):
        i = op.i
        dt = {P.DT_BF16: torch.bfloat16, P.DT_TF32: torch.float32, P.DT_F16: torch.float16}[i["dtype"]]
        chunk = i.get("row_bytes", 128) // (4 if i["dtype"] == P.DT_TF32 else 2)
        M, N, Npad, Ktot = i["M"], i["N"], i["Npad"], i["Ktot"]
        amaps = []
        for k in ("a0", "a1"):
            ref = op.p.get(k)
            if ref is None:
                amaps.append(None)
                continue
            rows, cols, ld = i[k + "_rows"], i[k + "_cols"], i[k + "_ld"]
            flat = _t(ref, dt, ext)
            amaps.append(torch.as_strided(flat, (rows, cols), (ld, 1)))
        Wt = _t(op.p["b"], dt, ext)[: Npad * Ktot].view(Npad, Ktot).float()
        sf, sf_step = i.get("sf", 1) or 1, i.get("sf_step", 1) or 1
        Mx = M + (sf - 1) * sf_step          # shift-fused form: accumulator rows past M feed the last outputs
        acc = torch.zeros(Mx, Npad)
        m = torch.arange(Mx)
        halo = i["halo"]
        covered = 0
        for g in range(i["ngroups"]):
            A = amaps[i[f"g_map{g}"]]
            delta, acol, nch = i[f"g_delta{g}"], i[f"g_acol{g}"], i[f"g_chunks{g}"]
            ntaps, kbase, tap0 = i[f"g_ntaps{g}"], i[f"g_kbase{g}"], i[f"g_tap0{g}"]
            kw = nch * chunk
            for t in range(ntaps):
                idx = m + delta - halo + i[f"tap_rel{tap0 + t}"]
                ok = (idx >= 0) & (idx < A.shape[0])
                a = torch.zeros(Mx, kw)
                a[ok] = A[idx[ok], acol: acol + kw].float()
                if i["dtype"] == P.DT_TF32 and self.tf32_truncate:
                    a = trunc_tf32(a)
                kcol = kbase + t * kw
                acc += a @ Wt[:, kcol: kcol + kw].t()
                covered += kw
        assert covered == Ktot
        if sf > 1:   # out[m] = sum_j acc[m + j*step, j*BN + n]
            bn = i["BN"]
            acc = sum(acc[j * sf_step: j * sf_step + M, j * bn: j * bn + N] for j in range(sf))
        else:
            acc = acc[:, :N]
        m = torch.arange(M)
        if op.p.get("bias") is not None:
            acc = acc + _t(op.p["bias"], torch.float32, ext)[:N]
        if op.p.get("res") is not None:
            rdt = torch.bfloat16 if i["res_dtype"] == P.OUT_BF16 else torch.float32
            r = torch.as_strided(_t(op.p["res"], rdt, ext), (M, N), (i["ldr"], 1)).float()
            acc = acc + r
        if i["relu"]:
            acc = acc.clamp_min(0)
        if i["mask_en"]:
            rem = m % i["mRPI"]
            valid = ((rem // i["mP"]) < i["mH"]) & ((rem % i["mP"]) < i["mW"])
            acc = torch.where(valid.view(-1, 1), acc, torch.zeros(()))
        if i["round_tf32"]:
            acc = P.round_tf32(acc)
        odt = {P.OUT_BF16: torch.bfloat16, P.OUT_F32: torch.float32, P.OUT_F16: torch.float16}[i["out_dtype"]]
        if i.get("pool"):
            # fused 3x3/2 max-pool of the (bf16-rounded) conv map, written to the pooled padded grid
            B, H, W_ = i["n_imgs"], i["mH"], i["mW"]
            conv = acc.to(odt)[_grid_index(B, H, W_, i["mP"], i["mRPI"])].float().view(B, H, W_, N)
            y = F.max_pool2d(conv.permute(0, 3, 1, 2), 3, 2, 1).permute(0, 2, 3, 1).reshape(-1, N)
            rows_o = B * i["pool_rpio"]
            dst = _t(op.p["out"], odt, ext)[: rows_o * N].view(rows_o, N)
            dst.zero_()
            dst[_grid_index(B, i["pool_Ho"], i["pool_Wo"], i["pool_Po"], i["pool_rpio"])] = y.to(odt)
            return
        out = torch.as_strided(_t(op.p["out"], odt, ext), (M, N), (i["ldo"], 1))
        out.copy_(acc.to(odt))
        if op.p.get("sums") is not None:   # column sums of every 32-row slab (fp32, before the 16-bit rounding)
            ns = (M + 31) // 32
            padded = torch.zeros(ns * 32, N)
            padded[:M] = acc
            _t(op.p["sums"], torch.float32, ext)[: ns * N].view(ns, N).copy_(padded.view(ns, 32, N).sum(dim=1))
        if i.get("topk"):                  # fused softmax + top-k of the stored rows (the answer head's last Linear)
            k = i["topk"]
            probs, idx = F.softmax(acc, dim=-1).topk(k, dim=-1)
            ext[op.p["topk_idx"].slot].view(M, k).copy_(idx)
            ext[op.p["topk_probs"].slot].view(M, k).copy_(probs)

    def op_stem_pool(self, op, ext):
        """Two-row fused stem: acc[m, :64] = conv at flat position m, acc[m, 64:] = conv at m + P (same A window)."""
        i = op.i
        B, H, W_, Pp, rpi = i["B"], i["H"], i["W"], i["P"], i["RPI"]
        rows = i["a_rows"]
        A = _t(op.p["a"], torch.bfloat16, ext)[: rows * 16].view(rows, 16).float()
        Wt = _t(op.p["w"], torch.bfloat16, ext)[: 128 * 320].view(128, 320).float()
        m = torch.arange(B * rpi)
        acc = torch.zeros(B * rpi, 128)
        for ia in range(5):
            for ib in range(4):
                idx = m + (ia - 2) * Pp + (ib - 2)
                ok = (idx >= 0) & (idx < rows)
                a = torch.zeros(B * rpi, 16)
                a[ok] = A[idx[ok]]
                t = ia * 4 + ib
                acc += a @ Wt[:, t * 16:(t + 1) * 16].t()
        gi = _grid_index(B, H, W_, Pp, rpi)
        conv = acc[:, :64].clamp_min(0).to(torch.bfloat16)
        nxt = acc[:, 64:].clamp_min(0).to(torch.bfloat16)
        inner = _grid_index(B, H - 1, W_, Pp, rpi)          # block 1 of row h is block 0 of row h + 1
        assert torch.equal(nxt[inner], conv[inner + Pp]), "two-row stem weight blocks disagree"
        y = F.max_pool2d(conv[gi].float().view(B, H, W_, 64).permute(0, 3, 1, 2), 3, 2, 1).permute(0, 2, 3, 1).reshape(-1, 64)
        rows_o = B * i["RPIo"]
        dst = _t(op.p["out"], torch.bfloat16, ext)[: rows_o * 64].view(rows_o, 64)
        dst.zero_()
        dst[_grid_index(B, i["Ho"], i["Wo"], i["Po"], i["RPIo"])] = y.to(torch.bfloat16)

    def op_mlp_chain(self, op, ext):
        """x1 = xres + ctx Wo^T; x2 = x1 + relu(LN(x1) W1^T + b1) W2^T + b2; y = LN'(x2) Wn^T (fp16 operands, fp32 accumulate)."""
        i = op.i
        T, D, Fh, Nn = i["T"], i["D"], i["F"], i["Nn"]
        f16, f32 = torch.float16, torch.float32
        ctx = _t(op.p["ctx"], f16, ext)[: T * D].view(T, D).float()
        xres = _t(op.p["xres"], f32, ext)[: T * D].view(T, D).clone()
        wo = _t(op.p["wo"], f16, ext)[: D * D].view(D, D).float()
        w1 = _t(op.p["w1"], f16, ext)[: Fh * D].view(Fh, D).float()
        w2 = _t(op.p["w2"], f16, ext)[: D * Fh].view(D, Fh).float()
        b1 = _t(op.p["b1"], f32, ext)[:Fh]
        b2 = _t(op.p["b2"], f32, ext)[:D]
        x1 = xres + ctx @ wo.t()
        xn = F.layer_norm(x1, (D,), _t(op.p["ln_g"], f32, ext)[:D], _t(op.p["ln_b"], f32, ext)[:D], op.f["eps"]).half().float()
        h = F.relu(xn @ w1.t() + b1).half().float()
        x2 = x1 + h @ w2.t() + b2
        if Nn:
            wn = _t(op.p["wn"], f16, ext)[: Nn * D].view(Nn, D).float()
            xn2 = F.layer_norm(x2, (D,), _t(op.p["n_g"], f32, ext)[:D], _t(op.p["n_b"], f32, ext)[:D], op.f["eps_n"]).half().float()
            _t(op.p["y"], f32, ext)[: T * Nn].view(T, Nn).copy_(xn2 @ wn.t())
        _t(op.p["xout"], f32, ext)[: T * D].view(T, D).copy_(x2)

    def op_maxpool(self, op, ext):
        i = op.i
        B, C = i["B"], i["C"]
        adt = torch.float32 if i.get("f32") else torch.bfloat16
        src = _t(op.p["src"], adt, ext)[: B * i["RPIin"] * C].view(B * i["RPIin"], C)
        idx = _grid_index(B, i["Hin"], i["Win"], i["Pin"], i["RPIin"])
        x = src[idx].float().view(B, i["Hin"], i["Win"], C).permute(0, 3, 1, 2)
        y = F.max_pool2d(x, 3, 2, 1).permute(0, 2, 3, 1).reshape(-1, C)
        dst = _t(op.p["dst"], adt, ext)[: B * i["RPIout"] * C].view(B * i["RPIout"], C)
        dst.zero_()
        dst[_grid_index(B, i["Hout"], i["Wout"], i["Pout"], i["RPIout"])] = y.to(adt)

    def _grid_nhwc(self, ref, ext, B, C, H, W, Pp, rpi, dtype=torch.bfloat16):
        src = _t(ref, dtype, ext)[: B * rpi * C].view(B * rpi, C)
        return src[_grid_index(B, H, W, Pp, rpi)].float().view(B, H, W, C)

    def op_se_squeeze(self, op, ext):
        i = op.i
        B, C, H, W, S = i["B"], i["C"], i["H"], i["W"], i["S"]
        x = self._grid_nhwc(op.p["src"], ext, B, C, H, W, i["P"], i["RPI"]).reshape(B, H * W, C)
        per = (H * W + S - 1) // S
        part = torch.zeros(B, S, C)
        for k in range(S):   # slice partial sums, added in slice order by se_excite
            part[:, k] = x[:, k * per: (k + 1) * per].sum(dim=1)
        _t(op.p["sums"], torch.float32, ext)[: B * S * C].view(B, S, C).copy_(part)

    def op_se_excite(self, op, ext):
        i = op.i
        B, C, R, S = i["B"], i["C"], i["R"], i["S"]
        mean = _t(op.p["sums"], torch.float32, ext)[: B * S * C].view(B, S, C).sum(dim=1) / i["HW"]
        w1 = _t(op.p["w1"], torch.float32, ext)[: R * C].view(R, C)
        w2t = _t(op.p["w2"], torch.float32, ext)[: R * C].view(R, C)   # stored transposed
        sc = torch.sigmoid(F.relu(mean @ w1.t()) @ w2t)
        _t(op.p["scale"], torch.float32, ext)[: B * C].view(B, C).copy_(sc)

    def op_spatial_map(self, op, ext):
        i = op.i
        B, C, H, W, ks = i["B"], i["C"], i["H"], i["W"], i["ksize"]
        x = self._grid_nhwc(op.p["src"], ext, B, C, H, W, i["P"], i["RPI"])
        if op.p.get("scale") is not None:
            x = x * _t(op.p["scale"], torch.float32, ext)[: B * C].view(B, 1, 1, C)
        pooled = torch.stack([x.max(dim=3)[0], x.mean(dim=3)], dim=1)  # [B,2,H,W], max first
        w = _t(op.p["wconv"], torch.float32, ext)[: 2 * ks * ks].view(1, 2, ks, ks)
        att = torch.sigmoid(F.conv2d(pooled, w, None, padding=ks // 2))
        _t(op.p["att"], torch.float32, ext)[: B * H * W].view(B, H * W).copy_(att.view(B, H * W))

    def op_scale_relayout(self, op, ext):
        i = op.i
        B, C, H, W = i["B"], i["C"], i["H"], i["W"]
        x = self._grid_nhwc(op.p["src"], ext, B, C, H, W, i["P"], i["RPI"])
        if op.p.get("scale") is not None:
            x = x * _t(op.p["scale"], torch.float32, ext)[: B * C].view(B, 1, 1, C)
        if op.p.get("att") is not None:
            x = x * _t(op.p["att"], torch.float32, ext)[: B * H * W].view(B, H, W, 1)
        x = x.to(torch.bfloat16)
        if i["mode"] == 0:
            dst = _t(op.p["dst"], torch.bfloat16, ext)[: B * i["RPIo"] * C].view(B * i["RPIo"], C)
            dst.zero_()
            dst[_grid_index(B, H, W, i["Po"], i["RPIo"])] = x.reshape(-1, C)
        else:
            pr = i["phase_rows"]
            dst = _t(op.p["dst"], torch.bfloat16, ext)[: 4 * pr * C].view(4, pr, C)
            dst.zero_()
            idx = _grid_index(B, H // 2, W // 2, i["Po"], i["RPIo"])
            for ph in range(2):
                for pw in range(2):
                    dst[ph * 2 + pw][idx] = x[:, ph::2, pw::2, :].reshape(-1, C)

    def op_grid_to_nchw(self, op, ext):
        i = op.i
        x = self._grid_nhwc(op.p["src"], ext, i["B"], i["C"], i["H"], i["W"], i["P"], i["RPI"],
                            torch.float32 if i.get("f32") else torch.bfloat16)
        n = i["B"] * i["C"] * i["H"] * i["W"]
        _t(op.p["dst"], torch.float32, ext)[:n].view(i["B"], i["C"], i["H"], i["W"]).copy_(x.permute(0, 3, 1, 2))

    def op_stage_tail(self, op, ext):
        i = op.i
        B, C, H, W = i["B"], i["C"], i["H"], i["W"]
        adt = torch.float32 if i.get("f32") else torch.bfloat16
        x = self._grid_nhwc(op.p["src"], ext, B, C, H, W, i["P"], i["RPI"], adt)     # [B,H,W,C] fp32 values
        sc = torch.ones(B, C)
        if op.p.get("w1") is not None:
            R = i["R"]
            mean = x.reshape(B, H * W, C).sum(dim=1) / (H * W)
            w1 = _t(op.p["w1"], torch.float32, ext)[: R * C].view(R, C)
            w2t = _t(op.p["w2"], torch.float32, ext)[: R * C].view(R, C)
            sc = torch.sigmoid(F.relu(mean @ w1.t()) @ w2t)
            if op.p.get("scale") is not None:
                _t(op.p["scale"], torch.float32, ext)[: B * C].view(B, C).copy_(sc)
        xs = x * sc.view(B, 1, 1, C)
        att = torch.ones(B, H, W)
        if op.p.get("wconv") is not None:
            ks = i["ks"]
            pooled = torch.stack([xs.max(dim=3)[0], xs.mean(dim=3)], dim=1)
            w = _t(op.p["wconv"], torch.float32, ext)[: 2 * ks * ks].view(1, 2, ks, ks)
            att = torch.sigmoid(F.conv2d(pooled, w, None, padding=ks // 2)).view(B, H, W)
            if op.p.get("att") is not None:
                _t(op.p["att"], torch.float32, ext)[: B * H * W].view(B, H * W).copy_(att.view(B, H * W))
        y = x * sc.view(B, 1, 1, C) * att.view(B, H, W, 1)
        y = P.round_tf32(y) if i.get("f32") else y.to(torch.bfloat16)
        Po, RPIo = i["Po"], i["RPIo"]
        if i["mode"]:
            pr = i["phase_rows"]
            dst = _t(op.p["dst"], adt, ext)[: 4 * pr * C].view(4, pr, C)
            dst.zero_()
            idx = _grid_index(B, H // 2, W // 2, Po, RPIo)
            for ph in range(2):
                for pw in range(2):
                    dst[ph * 2 + pw][idx] = y[:, ph::2, pw::2, :].reshape(-1, C)
        else:
            dst = _t(op.p["dst"], adt, ext)[: B * RPIo * C].view(B * RPIo, C)
            dst.zero_()
            dst[_grid_index(B, H, W, Po, RPIo)] = y.reshape(-1, C)

    def op_split_tf32(self, op, ext):
        i = op.i
        M, K = i["M"], i["K"]
        src = torch.as_strided(_t(op.p["src"], torch.float32, ext), (M, K), (i["ld_src"], 1))
        hi = P.round_tf32(src)
        dst = _t(op.p["dst"], torch.float32, ext)[: M * 2 * K].view(M, 2 * K)
        dst[:, :K] = hi
        dst[:, K:] = P.round_tf32(src - hi)

    def op_copy_rows(self, op, ext):
        i = op.i
        src = torch.as_strided(_t(op.p["src"], torch.float32, ext), (i["rows"], i["cols"]), (i["ld_src"], 1))
        torch.as_strided(_t(op.p["dst"], torch.float32, ext), (i["rows"], i["cols"]), (i["ld_dst"], 1)).copy_(src)

    def op_mask_prep(self, op, ext):
        i = op.i
        src = ext[op.p["src"].slot]
        _t(op.p["dst"], torch.int32, ext)[: i["B"] * i["L"]].view(i["B"], i["L"]).copy_((src != 0).to(torch.int32))
        if op.p.get("dstf") is not None:   # pooling weights: attention_mask.float()
            _t(op.p["dstf"], torch.float32, ext)[: i["B"] * i["L"]].view(i["B"], i["L"]).copy_(src.float())

    def op_embed(self, op, ext):
        i = op.i
        B, L, D, V = i["B"], i["L"], i["D"], i["V"]
        ids = ext[op.p["ids"].slot].view(B, L)
        table = _t(op.p["table"], torch.float32, ext)[: V * D].view(V, D)
        pe = _t(op.p["pe"], torch.float32, ext)
        x = table[ids] + pe[: L * D].view(1, L, D)
        _t(op.p["dst"], torch.float32, ext)[: B * L * D].view(B, L, D).copy_(x)
        if op.p.get("gamma") is not None:     # + the first encoder layer's LayerNorm (+ mask normalisation), same launch
            y = F.layer_norm(x.view(B * L, D), (D,), _t(op.p["gamma"], torch.float32, ext)[:D],
                             _t(op.p["beta"], torch.float32, ext)[:D], op.f["eps"])
            self._ln_store(op.p["ln_dst"], i.get("round_tf32", 0), y, ext)
            if op.p.get("mask_dst") is not None:
                src = ext[op.p["mask_src"].slot]
                _t(op.p["mask_dst"], torch.int32, ext)[: B * L].view(B, L).copy_((src != 0).to(torch.int32))
                if op.p.get("mask_dstf") is not None:
                    _t(op.p["mask_dstf"], torch.float32, ext)[: B * L].view(B, L).copy_(src.to(torch.float32))

    @staticmethod
    def _ln_store(ref, rnd, y, ext):
        rows, D = y.shape
        if rnd == 2:                          # fp16 operand of the next Linear
            _t(ref, torch.float16, ext)[: rows * D].view(rows, D).copy_(y.half())
        else:
            _t(ref, torch.float32, ext)[: rows * D].view(rows, D).copy_(P.round_tf32(y) if rnd else y)

    def op_layernorm(self, op, ext):
        i = op.i
        rows, D = i["rows"], i["D"]
        g = _t(op.p["gamma"], torch.float32, ext)[:D]
        b = _t(op.p["beta"], torch.float32, ext)[:D]
        flat = _t(op.p["src"], torch.float32, ext)
        if i["mode"] == 0:
            x = torch.as_strided(flat, (rows, D), (i["ld_src"], 1))
        else:
            S = i["S"]
            Bn = rows // (S * S)
            idx = _grid_index(Bn, S, S, i["Pg"], i["RPIg"])
            x = torch.as_strided(flat, (Bn * i["RPIg"], D), (i["ld_src"], 1))[idx]
        y = F.layer_norm(x, (D,), g, b, op.f["eps"])
        if i["mode"] == 1:
            S = i["S"]
            pos = _t(op.p["pos"], torch.float32, ext)[: S * S * D].view(1, S * S, D)
            y = (y.view(-1, S * S, D) + pos).view(rows, D)
        for k in (2, 3):                      # chained LayerNorms of the unrounded first output
            if op.p.get(f"gamma{k}") is not None:
                z = F.layer_norm(y, (D,), _t(op.p[f"gamma{k}"], torch.float32, ext)[:D],
                                 _t(op.p[f"beta{k}"], torch.float32, ext)[:D], op.f["eps"])
                self._ln_store(op.p[f"dst{k}"], i.get(f"rnd{k}", 0), z, ext)
        self._ln_store(op.p["dst"], i["round_tf32"], y, ext)

    @staticmethod
    def _attend(q, k, v, hd, key_mask=None):
        s = torch.matmul(q, k.transpose(-2, -1)) / math.sqrt(hd)
        if key_mask is not None:
            s = s.masked_fill(key_mask.view(key_mask.shape[0], 1, 1, -1) == 0, float("-inf"))
        w = F.softmax(s, dim=-1)
        return torch.matmul(w, v), w

    def op_self_attn(self, op, ext):
        i = op.i
        B, L, H, hd, ld = i["B"], i["L"], i["H"], i["hd"], i["ld_qkv"]
        D = H * hd
        qkv = _t(op.p["qkv"], torch.float32, ext)[: B * L * ld].view(B, L, ld)
        q, k, v = (qkv[..., j * D:(j + 1) * D].reshape(B, L, H, hd).transpose(1, 2) for j in range(3))
        mask = None
        if op.p.get("mask") is not None:
            mask = _t(op.p["mask"], torch.int32, ext)[: B * L].view(B, L)
        ctx, _ = self._attend(q, k, v, hd, mask)
        self._attn_store(op.p["out"], i.get("no_round", 0), ctx.transpose(1, 2).reshape(B, L, D), ext)

    @staticmethod
    def _attn_store(ref, no_round, ctx, ext):
        """Attention output forms: 2 = fp16, 1 = fp32, 0 = tf32-rounded fp32."""
        odt = torch.float16 if no_round == 2 else torch.float32
        _t(ref, odt, ext)[: ctx.numel()].view(ctx.shape).copy_(ctx.to(odt) if no_round else P.round_tf32(ctx))

    def op_cross_attn(self, op, ext):
        i = op.i
        B, L, H, hd, T = i["B"], i["L"], i["H"], i["hd"], i["T"]
        D = H * hd
        q = torch.as_strided(_t(op.p["q"], torch.float32, ext), (B * L, D), (i["ld_q"], 1)).view(B, L, H, hd).transpose(1, 2)
        kvf = _t(op.p["kv"], torch.float32, ext)
        qk = max(i.get("q_per_kv", 1), 1)           # consecutive queries that share one image's K / V
        Bi = B // qk
        k = torch.as_strided(kvf[i["k_off"]:], (Bi * T, D), (i["ld_kv"], 1)).view(Bi, T, H, hd).transpose(1, 2)
        v = torch.as_strided(kvf[i["v_off"]:], (Bi * T, D), (i["ld_kv"], 1)).view(Bi, T, H, hd).transpose(1, 2)
        k, v = k.repeat_interleave(qk, dim=0), v.repeat_interleave(qk, dim=0)
        ctx, w = self._attend(q, k, v, hd)
        self._attn_store(op.p["out"], i.get("no_round", 0), ctx.transpose(1, 2).reshape(B, L, D), ext)
        if op.p.get("weights") is not None:
            _t(op.p["weights"], torch.float32, ext)[: B * H * L * T].view(B, H, L, T).copy_(w)

    def op_pool_gate_ln(self, op, ext):
        i = op.i
        B, L, D = i["B"], i["L"], i["D"]
        phase = i.get("phase", 0)
        buf = lambda key, n: _t(op.p[key], torch.float32, ext)[:n]
        if phase != 2:
            xa = buf("xatt", B * L * D).view(B, L, D)
            tx = buf("text", B * L * D).view(B, L, D)
            if op.p.get("mask") is not None:
                m = _t(op.p["mask"], torch.float32, ext)[: B * L].view(B, L, 1)
            else:
                m = torch.ones(B, L, 1)
            den = m.sum(dim=1).clamp(min=1)
            ap = (xa * m).sum(dim=1) / den
            tp = (tx * m).sum(dim=1) / den
            buf("att_pooled", B * D).view(B, D).copy_(ap)
            buf("txt_pooled", B * D).view(B, D).copy_(tp)
            if phase == 1:      # pools only; [att;txt] as the tf32 A operand of the gate GEMM
                cat = torch.cat([ap, tp], dim=-1)
                if i.get("no_round") == 2:
                    _t(op.p["cat"], torch.float16, ext)[: B * 2 * D].view(B, 2 * D).copy_(cat.half())
                else:
                    buf("cat", B * 2 * D).view(B, 2 * D).copy_(cat if i.get("no_round") else P.round_tf32(cat))
                return
            assert not i["use_gate"]
            fz = ap + tp
        else:                   # gate pre-activation comes from the GEMM
            ap, tp = buf("att_pooled", B * D).view(B, D), buf("txt_pooled", B * D).view(B, D)
            g = torch.sigmoid(buf("pre", B * D).view(B, D))
            fz = g * ap + (1 - g) * tp
        fz = F.layer_norm(fz, (D,), buf("gamma", D), buf("beta", D), op.f["eps"])
        buf("fused", B * D).view(B, D).copy_(fz)
        if i.get("no_round") == 2 and op.p.get("cat") is not None:
            _t(op.p["cat"], torch.float16, ext)[: B * D].view(B, D).copy_(fz.half())

    def op_softmax_topk(self, op, ext):
        i = op.i
        B, N, k = i["B"], i["N"], i["k"]
        logits = torch.as_strided(ext[op.p["logits"].slot].view(-1), (B, N), (i["ld"], 1))
        probs, idx = F.softmax(logits, dim=-1).topk(k, dim=-1)
        nan_rows = torch.isnan(logits).any(dim=1)
        if bool(nan_rows.any()):                 # the kernel's order: NaN ties go to the lower index
            idx[nan_rows] = TR.ref_order(logits[nan_rows], k)
        ext[op.p["idx"].slot].view(B, k).copy_(idx)
        ext[op.p["probs"].slot].view(B, k).copy_(probs)


def run_program(prog: P.Program, images, ids, mask, top_k=0, tf32_truncate=True, extra=None):
    """Run a CPU-resident program; returns (logits, ext list).  ``extra``: {slot name: flat tensor} for further
    external slots (the cached K/V of a question-side program)."""
    B = prog.B
    NA = prog.cfg["num_answers"]
    ext = [None] * len(P.EXT)
    for name, t in (extra or {}).items():
        ext[P.EXT[name]] = t
    ext[P.EXT["images"]] = images
    ext[P.EXT["ids"]] = ids
    ext[P.EXT["mask"]] = mask
    ext[P.EXT["logits"]] = torch.zeros(B, NA)
    ext[P.EXT["top_idx"]] = torch.zeros(B, max(top_k, 1), dtype=torch.int64)
    ext[P.EXT["top_probs"]] = torch.zeros(B, max(top_k, 1))
    Emulator(prog, tf32_truncate).run(ext)
    return ext[P.EXT["logits"]], ext
