"""Host-side compiler: state_dict -> packed weights + a flat list of kernel ops.

This is where the network is *defined*; the CUDA library (csrc/) only knows how to run
individual op kinds.  ``build_weights`` does the load-time weight algebra of SURVEY.md
Appendix B (BN fold, OHWI repack, shortcut-as-extra-K, QKV concatenation) and
``build_program`` lays activations out in HBM and emits the op list for one (batch, length,
input format) shape.  The same op list is (a) serialised to ``VqaOp`` structs for
``vqa_plan_create`` and (b) interpreted on the CPU by ``tests/emulator.py`` to validate the
layout / tap algebra against the oracle without a GPU.

HBM layout ("padded-flat NHWC"): a feature map [B,H,W,C] is stored as rows of C channels on a
grid with ``pad`` zero columns at the END of every image row and ``pad`` zero rows at the END
of every image:  row(n,h,w) = n*Hp*P + h*P + w,  P = W+pad, Hp = H+pad.  Because the pads are
shared between neighbouring rows / images, a 3x3 tap (dh,dw) is the pure 1-D row shift
dh*P+dw, so a convolution is a GEMM whose A operand is the same 2-D tensor loaded at shifted
row coordinates (TMA zero-fills out-of-range rows).  Stride-2 convolutions read a 4-phase
split of their input (phase (ph,pw) holds x[2a+ph, 2b+pw]) whose grid geometry equals the
output's.  The 7x7/2 stem reads a phase-packed input (16 bf16 per phase-pixel) through an
overlapping-row tensor map so that 4 horizontal taps form one 64-wide K chunk.
"""
from __future__ import annotations

import math
import os
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import torch

EXT_TAG = 1 << 63
MAX_TAPS = 16     # total taps over all groups of one GEMM op
MAX_GROUPS = 12

# ----------------------------------------------------------------------------- op field tables
KINDS = {
    "ingest": 1, "gemm": 2, "maxpool": 3, "se_squeeze": 4, "se_excite": 5, "spatial_map": 6,
    "scale_relayout": 7, "embed": 8, "layernorm": 9, "self_attn": 10, "cross_attn": 11,
    "pool_gate_ln": 12, "softmax_topk": 13, "mask_prep": 14, "grid_to_nchw": 15,
    "copy_rows": 16, "stage_tail": 17, "split_tf32": 18, "stem_pool": 19, "mlp_chain": 20, "attn_chunked": 21,
}

_GROUPS = [f"g_{k}{g}" for k in ("map", "delta", "acol", "chunks", "ntaps", "kbase", "tap0")
           for g in range(MAX_GROUPS)]
_TAPS = [f"tap_rel{t}" for t in range(MAX_TAPS)]

FIELDS: Dict[str, Dict[str, List[str]]] = {
    "ingest": {"i": ["B", "mode", "HW", "P", "rows", "ones", "f32"], "p": ["src", "dst"], "f": []},
    "gemm": {"i": ["dtype", "M", "N", "Npad", "Ktot", "BN", "MT", "halo", "a0_rows", "a0_cols", "a0_ld",
                   "a1_rows", "a1_cols", "a1_ld", "ngroups", "ntaps", "out_dtype", "ldo", "res_dtype", "ldr",
                   "relu", "round_tf32", "mask_en", "mP", "mRPI", "mH", "mW", "smem_budget", "max_ctas", "row_bytes",
                   "halo_hi", "tiles_per_img", "tile_stride", "tile_row0", "img_rows", "n_imgs", "pool", "pool_P",
                   "pool_W", "pool_Wo", "pool_Ho", "pool_Po", "pool_rpio", "pair", "sf", "sf_step", "topk"]
                  + _GROUPS + _TAPS,
             "p": ["a0", "a1", "b", "out", "bias", "res", "dbg", "sums", "topk_idx", "topk_probs", "topk_part", "topk_cnt"], "f": []},
    "maxpool": {"i": ["B", "C", "Hin", "Win", "Pin", "RPIin", "Hout", "Wout", "Pout", "RPIout", "f32"],
                "p": ["src", "dst"], "f": []},
    "se_squeeze": {"i": ["B", "C", "H", "W", "P", "RPI", "S"], "p": ["src", "sums"], "f": []},
    "se_excite": {"i": ["B", "C", "R", "HW", "S"], "p": ["sums", "w1", "w2", "scale"], "f": []},
    "spatial_map": {"i": ["B", "C", "H", "W", "P", "RPI", "ksize"],
                    "p": ["src", "scale", "wconv", "att"], "f": []},
    "scale_relayout": {"i": ["B", "C", "H", "W", "P", "RPI", "mode", "Po", "RPIo", "phase_rows"],
                       "p": ["src", "scale", "att", "dst"], "f": []},
    "embed": {"i": ["B", "L", "D", "V", "round_tf32", "mask_dtype"],
              "p": ["ids", "table", "pe", "dst", "gamma", "beta", "ln_dst", "mask_src", "mask_dst", "mask_dstf"], "f": ["eps"]},
    "layernorm": {"i": ["rows", "D", "ld_src", "mode", "round_tf32", "S", "Pg", "RPIg", "rnd2", "rnd3"],
                  "p": ["src", "gamma", "beta", "dst", "pos", "gamma2", "beta2", "dst2", "gamma3", "beta3", "dst3"], "f": ["eps"]},
    "self_attn": {"i": ["B", "L", "H", "hd", "ld_qkv", "no_round"], "p": ["qkv", "mask", "out"], "f": []},
    "cross_attn": {"i": ["B", "L", "H", "hd", "T", "ld_q", "ld_kv", "k_off", "v_off", "no_round", "q_per_kv"],
                   "p": ["q", "kv", "out", "weights"], "f": []},
    "pool_gate_ln": {"i": ["B", "L", "D", "use_gate", "phase", "no_round"],
                     "p": ["xatt", "text", "mask", "wg", "bg", "gamma", "beta", "fused",
                           "att_pooled", "txt_pooled", "cat", "pre"], "f": ["eps"]},
    "softmax_topk": {"i": ["B", "N", "k", "ld"], "p": ["logits", "idx", "probs"], "f": []},
    "mask_prep": {"i": ["B", "L", "dtype"], "p": ["src", "dst", "dstf"], "f": []},
    "grid_to_nchw": {"i": ["B", "C", "H", "W", "P", "RPI", "f32"], "p": ["src", "dst"], "f": []},
    "copy_rows": {"i": ["rows", "cols", "ld_src", "ld_dst"], "p": ["src", "dst"], "f": []},
    "split_tf32": {"i": ["M", "K", "ld_src"], "p": ["src", "dst"], "f": []},
    "stage_tail": {"i": ["B", "C", "H", "W", "P", "RPI", "R", "ks", "mode", "Po", "RPIo", "phase_rows", "CS", "f32", "split"],
                   "p": ["src", "w1", "w2", "wconv", "dst", "scale", "att", "sums"], "f": []},
    "stem_pool": {"i": ["B", "H", "W", "P", "RPI", "Ho", "Wo", "Po", "RPIo", "run_len", "a_rows", "max_ctas"],
                  "p": ["a", "w", "out", "dbg"], "f": []},
    "mlp_chain": {"i": ["T", "D", "F", "Nn", "Nn_pad", "max_ctas", "CS"],
                  "p": ["ctx", "xres", "xout", "wo", "w1", "b1", "w2", "b2", "ln_g", "ln_b", "n_g", "n_b", "wn", "y"],
                  "f": ["eps", "eps_n"]},
    "attn_chunked": {"i": ["B", "L", "H", "hd", "T", "ld_q", "ld_kv", "k_off", "v_off", "no_round", "q_per_kv"],
                     "p": ["q", "kv", "mask", "out", "weights"], "f": []},
}

DT_BF16, DT_TF32, DT_F16 = 0, 1, 2      # gemm operand dtype
OUT_BF16, OUT_F32, OUT_F16 = 0, 1, 2    # gemm output / residual dtype
MASK_NONE, MASK_I64, MASK_F32, MASK_I32, MASK_U8 = 0, 1, 2, 3, 4

# external slots (order of the ext[] array given to vqa_plan_run)
EXT = {"images": 0, "ids": 1, "mask": 2, "logits": 3, "top_idx": 4, "top_probs": 5}
MAX_CACHED_LAYERS = 8
# attn_mma_kernel (self_attn / cross_attn) holds every key of a (pair, head) in one warp: up to 64.  Longer questions run
# attn_chunked_kernel, which streams the keys in chunks of 64 (up to 512).  Programs of at most 64 tokens keep the
# single-warp kernel, so their results stay bit for bit what they were (DESIGN.md, "Long questions").
ATTN_MMA_MAX_L = 64
MAX_QUESTION_LENGTH = 512
TOPK_FUSED_MAX = 8   # kTopKMax in csrc/gemm_tcgen05.cu: winners an epilogue thread keeps; larger k uses softmax_topk_kernel
# K/V of a cached image side (question-side programs): one slot per cross-attention layer
EXT.update({f"kv{l}": 6 + l for l in range(MAX_CACHED_LAYERS)})


def generate_fields_header() -> str:
    """csrc/op_fields.h is generated from FIELDS so both sides of the ABI cannot drift."""
    out = ["// GENERATED by vqa_b200/program.py::generate_fields_header -- do not edit.",
           "#pragma once", ""]
    for kind, spec in FIELDS.items():
        up = kind.upper()
        for cls in ("i", "p", "f"):
            names = spec[cls]
            out.append(f"enum {{ " + " ".join(f"{up}_{cls.upper()}_{n} = {k}," for k, n in enumerate(names))
                       + f" {up}_N{cls.upper()} = {len(names)} }};")
        out.append("")
    return "\n".join(out)


# ----------------------------------------------------------------------------- memory
class Arena:
    """Bump allocator over one torch.uint8 tensor (device or CPU)."""

    def __init__(self, device):
        self.device = torch.device(device)
        self.size = 0
        self.tensor: Optional[torch.Tensor] = None
        self._bufs: List["Buf"] = []

    def alloc(self, nbytes: int, name: str = "", align: int = 1024) -> "Buf":
        off = (self.size + align - 1) // align * align
        self.size = off + int(nbytes)
        b = Buf(self, off, int(nbytes), name)
        self._bufs.append(b)
        return b

    def commit(self, zero: bool = False):
        n = (self.size + 4096 + 15) // 16 * 16  # slack: the stem's overlapping tensor map reads 96 B past its last row
        self.tensor = (torch.zeros if zero else torch.empty)(n, dtype=torch.uint8, device=self.device)
        return self


@dataclass
class Buf:
    arena: Arena
    offset: int
    nbytes: int
    name: str = ""

    def view(self, dtype: torch.dtype, *shape) -> torch.Tensor:
        t = self.arena.tensor[self.offset: self.offset + self.nbytes].view(dtype)
        return t.view(*shape) if shape else t

    def addr(self) -> int:
        return self.arena.tensor.data_ptr() + self.offset


@dataclass
class ExtRef:
    slot: int

    def addr(self) -> int:
        return EXT_TAG | self.slot


@dataclass
class Op:
    kind: str
    name: str
    i: Dict[str, int] = field(default_factory=dict)
    p: Dict[str, object] = field(default_factory=dict)   # Buf | ExtRef | None
    f: Dict[str, float] = field(default_factory=dict)
    lane: int = 0   # bit 0: 0 = caller's stream, 1 = side stream; LANE_JOIN: wait for the other lane's work so far


LANE_JOIN = 4      # VQA_LANE_JOIN: this op needs everything issued so far on the other lane


@dataclass
class Grid:
    B: int
    H: int
    W: int
    pad: int = 1

    @property
    def P(self):
        return self.W + self.pad

    @property
    def Hp(self):
        return self.H + self.pad

    @property
    def rpi(self):
        return self.Hp * self.P

    @property
    def rows(self):
        return self.B * self.rpi


# ----------------------------------------------------------------------------- weights
def _fold_bn(sd, conv_key, bn_prefix):
    """W' = W*s[cout], b' = beta - mu*s with s = gamma/sqrt(var+eps) (SURVEY Appendix B)."""
    w = sd[conv_key].float()
    s = sd[bn_prefix + ".weight"].float() / torch.sqrt(sd[bn_prefix + ".running_var"].float() + 1e-5)
    b = sd[bn_prefix + ".bias"].float() - sd[bn_prefix + ".running_mean"].float() * s
    return w * s.view(-1, 1, 1, 1), b


# Stride-2 3x3 convolution over the 4-phase split, taps grouped by the phase they read (one A window per phase):
# phase (1,1) serves (kh,kw) = (0,0),(0,2),(2,0),(2,2); phase (1,0) serves (0,1),(2,1); phase (0,1) serves (1,0),(1,2);
# phase (0,0) serves the centre tap.  The weight matrix of the windowed form is stored in this tap order.
PHASE_TAP_ORDER = [(0, 0), (0, 2), (2, 0), (2, 2), (0, 1), (2, 1), (1, 0), (1, 2), (1, 1)]


def _ohwi_phase_order(w):
    """[Cout,Cin,3,3] -> [Cout, 9*Cin] with the taps in PHASE_TAP_ORDER (K index = tap*Cin + c)."""
    return torch.cat([w[:, :, kh, kw] for kh, kw in PHASE_TAP_ORDER], dim=1).contiguous()


def _stem_two_row_matrix(m):
    """[64, 256] stem matrix (4 vertical x 4 horizontal phase-pixel taps x 16) -> [128, 320] for the two-row form of the
    fused stem (csrc/stem_tcgen05.cu): 5 vertical tap positions ia' = 0..4 against ONE A window; rows 0..63 produce conv
    row r with W[ia'] (nothing at ia' = 4), rows 64..127 produce conv row r+1 with W[ia' - 1] (nothing at ia' = 0)."""
    m = m.reshape(64, 4, 4, 16)
    out = torch.zeros(128, 5, 4, 16, dtype=m.dtype, device=m.device)
    out[:64, 0:4] = m
    out[64:, 1:5] = m
    return out.reshape(128, 320)


def _ohwi_shift_fused(w):
    """[Cout,Cin,3,3] -> [3*Cout, 3*Cin] for the shift-fused form of a 3x3 convolution: row kw*Cout + co holds the
    weights of horizontal tap kw, K index = kh*Cin + c.  One N = 3*Cout MMA per vertical tap then produces the three
    horizontal taps' partial sums side by side; the epilogue adds them with row shifts 0 / 1 / 2."""
    cout, cin = w.shape[:2]
    return w.permute(3, 0, 2, 1).reshape(3 * cout, 3 * cin).contiguous()


def _ohwi(w):
    """[Cout,Cin,kh,kw] -> [Cout, kh*kw*Cin] with K index = (kh*KW+kw)*Cin + c."""
    return w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).contiguous()


def _stem_matrix(w):
    """7x7/2 stem as a 4x4/1 conv over the 2x2 phase-packed input: [64,3,7,7] -> [64, 256].

    K index = ((ia*4 + ib)*2 + ph)*2*4 + pw*4 + c with vertical tap da = ia-2, horizontal db = ib-2,
    source pixel (2*(i+da)+ph, 2*(j+db)+pw) = (2i + kh - 3, 2j + kw - 3).
    """
    cout = w.shape[0]
    m = torch.zeros(cout, 4, 4, 2, 2, 4, dtype=torch.float32, device=w.device)
    for kh in range(7):
        u = kh - 3
        da, ph = u // 2, u % 2
        for kw in range(7):
            v = kw - 3
            db, pw = v // 2, v % 2
            m[:, da + 2, db + 2, ph, pw, :3] = w[:, :, kh, kw]
    return m.reshape(cout, 256)


class Weights:
    """Packed device-resident parameters (one arena; this is what gets NCCL-broadcast)."""

    def __init__(self, device):
        self.precision = "bf16"     # "bf16": bf16 backbone operands | "tf32": fp32 activations, tf32 operands everywhere
        self.arena = Arena(device)
        self.items: Dict[str, Tuple[Buf, torch.dtype, Tuple[int, ...]]] = {}
        self._pending: List[Tuple[str, torch.Tensor]] = []

    def add(self, name: str, t: torch.Tensor, dtype: torch.dtype):
        t = t.detach().to(dtype).contiguous()
        buf = self.arena.alloc(t.numel() * t.element_size(), name)
        self.items[name] = (buf, dtype, tuple(t.shape))
        self._pending.append((name, t))
        return buf

    def finalize(self):
        self.arena.commit(zero=True)
        for name, t in self._pending:
            buf, dtype, shape = self.items[name]
            buf.view(dtype, *shape).copy_(t)
        self._pending = []
        return self

    def buf(self, name) -> Buf:
        return self.items[name][0]

    def tensor(self, name) -> torch.Tensor:
        buf, dtype, shape = self.items[name]
        return buf.view(dtype, *shape)

    def __contains__(self, name):
        return name in self.items


def _pad_rows(w: torch.Tensor, mult: int) -> torch.Tensor:
    n = w.shape[0]
    npad = (n + mult - 1) // mult * mult
    if npad == n:
        return w
    out = torch.zeros((npad,) + tuple(w.shape[1:]), dtype=w.dtype, device=w.device)
    out[:n] = w
    return out


def round_tf32(t: torch.Tensor) -> torch.Tensor:
    """Round-to-nearest-even to 10 mantissa bits (what cvt.rna.tf32 does, ties aside)."""
    i = t.contiguous().view(torch.int32)
    r = (i + 0x0FFF + ((i >> 13) & 1)) & ~0x1FFF
    return r.view(torch.float32)


def build_weights(sd: Dict[str, torch.Tensor], cfg: dict, device, precision: str = "bf16") -> Weights:
    """All load-time algebra; every product is formed in fp32 before the bf16 / tf32 cast.

    precision="tf32" (the tolerance mode of BASELINE.json: logits within 1e-3 of the fp32 reference) stores the
    backbone weights as tf32-rounded fp32 instead of bf16; everything else is identical."""
    assert precision in ("bf16", "tf32")
    W = Weights(device)
    W.precision = precision
    sd = {k: v.detach().to("cpu") for k, v in sd.items()}
    bf, f32 = torch.bfloat16, torch.float32
    tf = precision == "tf32"
    cw = f32 if tf else bf                                    # storage type of the backbone GEMM operands
    cast = (lambda m: round_tf32(m.float())) if tf else (lambda m: m)

    def lin(name, w):
        """A tf32 Linear weight; in tf32 precision mode also its 3xTF32 form [hi | hi | lo] along K, consumed with
        A = [a_hi | a_lo]: a_hi*hi + a_lo*hi + a_hi*lo recovers fp32-level products on the tf32 tensor pipe."""
        w = w.float()
        hi = round_tf32(w)
        W.add(name, hi, f32)
        if tf:
            W.add(name + ".x3", torch.cat([hi, hi, round_tf32(w - hi)], dim=1), f32)
        else:
            # throughput mode: fp16 operands -- the 11-bit significand of tf32 in half the bytes and at twice
            # the MMA rate (the Linears of this path are bound by their operand fill, 40-48 B/clk per SM)
            W.add(name + ".h", w, torch.float16)

    # ---- backbone (BN folded, OHWI, bf16 operands, fp32 bias)
    w, b = _fold_bn(sd, "image_encoder.stem.0.weight", "image_encoder.stem.1")
    W.add("stem.w", cast(_stem_matrix(w)), cw)
    W.add("stem.b", b, f32)
    # bias folded into K: ingest(ones=1) stores 1.0 in the spare channel of phases (0,0) and (0,1) of every
    # in-image block; the centre tap's weights there carry the bias as a bf16 hi + lo pair (error ~2^-17)
    mb = _stem_matrix(w).view(-1, 4, 4, 2, 2, 4).clone()
    hi = b.to(bf).float()
    mb[:, 2, 2, 0, 0, 3] = hi
    mb[:, 2, 2, 0, 1, 3] = (b - hi).to(bf).float()
    if not tf:
        W.add("stem.wb", mb.reshape(-1, 256), bf)
        W.add("stem.w2", _stem_two_row_matrix(mb.reshape(-1, 256)), bf)
    for s in (1, 2, 3, 4):
        p = f"image_encoder.stage{s}"
        blk = 0
        while f"{p}.blocks.{blk}.conv1.weight" in sd:
            q = f"{p}.blocks.{blk}"
            w1, b1 = _fold_bn(sd, q + ".conv1.weight", q + ".bn1")
            w2, b2 = _fold_bn(sd, q + ".conv2.weight", q + ".bn2")
            m2 = _ohwi(w2)
            if q + ".downsample.0.weight" in sd:  # shortcut 1x1 becomes extra K columns of conv2
                wd, bd = _fold_bn(sd, q + ".downsample.0.weight", q + ".downsample.1")
                m2 = torch.cat([m2, _ohwi(wd)], dim=1)
                b2 = b2 + bd
            W.add(f"s{s}.b{blk}.conv1.w", cast(_ohwi(w1)), cw)
            if not tf and q + ".downsample.0.weight" in sd and tuple(w1.shape[2:]) == (3, 3) and w1.shape[0] != w1.shape[1]:
                W.add(f"s{s}.b{blk}.conv1.wp", _ohwi_phase_order(w1), cw)     # stride-2 block entry, windowed form
            W.add(f"s{s}.b{blk}.conv1.b", b1, f32)
            if not tf and w1.shape[0] == 64 and w1.shape[1] == 64 and q + ".downsample.0.weight" not in sd:
                # 64-channel layers: shift-fused form (N = 192 MMAs; a 128x64 MMA is bound by its shared-memory reads)
                W.add(f"s{s}.b{blk}.conv1.wsf", _ohwi_shift_fused(w1), cw)
                W.add(f"s{s}.b{blk}.conv2.wsf", _ohwi_shift_fused(w2), cw)
            W.add(f"s{s}.b{blk}.conv2.w", cast(m2), cw)
            W.add(f"s{s}.b{blk}.conv2.b", b2, f32)
            blk += 1
        if f"{p}.attention.se.fc1.weight" in sd:
            W.add(f"s{s}.se.w1", sd[f"{p}.attention.se.fc1.weight"], f32)
            W.add(f"s{s}.se.w2", sd[f"{p}.attention.se.fc2.weight"].t(), f32)   # stored [R, C] (coalesced reads)
        if f"{p}.attention.spatial.conv.weight" in sd:
            W.add(f"s{s}.spatial.w", sd[f"{p}.attention.spatial.conv.weight"].reshape(2, -1), f32)

    # ---- text encoder (fp32 storage, tf32-rounded GEMM operands)
    t = "text_encoder"
    D = cfg["embed_dim"]
    # the reference scales after the lookup (F.embedding(ids, emb) * math.sqrt(D)); both are the same fp32 product of each
    # table element and fp32(sqrt(D)), so scaling the table once gives the same bits for every D, a perfect square or not
    W.add("text.emb", sd[t + ".token_embedding.weight"].float() * math.sqrt(D), f32)
    W.add("text.pe", sd[t + ".positional_encoding.pe"][0], f32)
    layer = 0
    while f"{t}.layers.{layer}.norm1.weight" in sd:
        q = f"{t}.layers.{layer}"
        W.add(f"text.{layer}.ln1.g", sd[q + ".norm1.weight"], f32)
        W.add(f"text.{layer}.ln1.b", sd[q + ".norm1.bias"], f32)
        qkv = torch.cat([sd[q + f".self_attention.W_{n}.weight"] for n in "qkv"], dim=0)
        lin(f"text.{layer}.qkv.w", qkv)
        lin(f"text.{layer}.o.w", sd[q + ".self_attention.W_o.weight"])
        W.add(f"text.{layer}.ln2.g", sd[q + ".norm2.weight"], f32)
        W.add(f"text.{layer}.ln2.b", sd[q + ".norm2.bias"], f32)
        lin(f"text.{layer}.fc1.w", sd[q + ".ffn.fc1.weight"])
        W.add(f"text.{layer}.fc1.b", sd[q + ".ffn.fc1.bias"], f32)
        lin(f"text.{layer}.fc2.w", sd[q + ".ffn.fc2.weight"])
        W.add(f"text.{layer}.fc2.b", sd[q + ".ffn.fc2.bias"], f32)
        layer += 1
    W.add("text.lnf.g", sd[t + ".final_norm.weight"], f32)
    W.add("text.lnf.b", sd[t + ".final_norm.bias"], f32)

    # ---- fusion
    fz = "fusion"
    W.add("proj.w", cast(sd[fz + ".image_projector.projection.0.weight"]), cw)   # A operand is the backbone output
    W.add("proj.b", sd[fz + ".image_projector.projection.0.bias"], f32)
    W.add("proj.ln.g", sd[fz + ".image_projector.projection.1.weight"], f32)
    W.add("proj.ln.b", sd[fz + ".image_projector.projection.1.bias"], f32)
    W.add("proj.pos", sd[fz + ".image_projector.position_embedding"][0], f32)
    layer = 0
    while f"{fz}.cross_attention.layers.{layer}.norm_query.weight" in sd:
        q = f"{fz}.cross_attention.layers.{layer}"
        for nm, key in (("lnq", "norm_query"), ("lnkv", "norm_kv"), ("lnf", "norm_ffn")):
            W.add(f"x.{layer}.{nm}.g", sd[f"{q}.{key}.weight"], f32)
            W.add(f"x.{layer}.{nm}.b", sd[f"{q}.{key}.bias"], f32)
        lin(f"x.{layer}.q.w", sd[q + ".cross_attention.W_q.weight"])
        kv = torch.cat([sd[q + ".cross_attention.W_k.weight"], sd[q + ".cross_attention.W_v.weight"]], dim=0)
        lin(f"x.{layer}.kv.w", kv)
        lin(f"x.{layer}.o.w", sd[q + ".cross_attention.W_o.weight"])
        lin(f"x.{layer}.fc1.w", sd[q + ".ffn.0.weight"])
        W.add(f"x.{layer}.fc1.b", sd[q + ".ffn.0.bias"], f32)
        lin(f"x.{layer}.fc2.w", sd[q + ".ffn.3.weight"])
        W.add(f"x.{layer}.fc2.b", sd[q + ".ffn.3.bias"], f32)
        layer += 1
    if fz + ".gate.gate.0.weight" in sd:
        lin("gate.w", sd[fz + ".gate.gate.0.weight"])
        W.add("gate.b", sd[fz + ".gate.gate.0.bias"], f32)
    W.add("out.ln.g", sd[fz + ".output_norm.weight"], f32)
    W.add("out.ln.b", sd[fz + ".output_norm.bias"], f32)

    # ---- answer head (N padded to the GEMM tile so TMA boxes never leave the tensor)
    h = "answer_head.classifier"
    for idx, nm in ((0, "head0"), (3, "head1"), (6, "head2")):
        b = sd[f"{h}.{idx}.bias"].float()
        lin(nm + ".w", _pad_rows(sd[f"{h}.{idx}.weight"].float(), 256))
        W.add(nm + ".b", _pad_rows(b, 256), f32)
    return W.finalize()


# ----------------------------------------------------------------------------- program
def _bn_tile(n: int) -> int:
    for t in (64, 128, 256):
        if n <= t:
            return t
    return 256


class OpList:
    """A workspace arena plus a list of ops over it (the unit ``vqa_plan_create`` consumes)."""

    def __init__(self, weights: Weights, device=None, window: bool = True):
        self.W = weights
        self.tf32 = getattr(weights, "precision", "bf16") == "tf32"
        self.window = window
        self.stem_window = window
        self.half_tail = not self.tf32              # fp16 operands for the text / fusion / head Linears
        self.out_mode = 1 if self.tf32 else 2       # producers of Linear operands: 1 = unrounded fp32 (3xTF32), 2 = fp16
        self.tdt = torch.float16 if self.half_tail else torch.float32   # storage of their A operands
        self.fuse_pool = window and not self.tf32
        # SE squeeze partial sums in the epilogue of each stage's last convolution + streaming stage tail.  Correct and
        # tested, but measured slower on B200 (the 31-shuffle column-sum butterfly costs the stage-1 convolution 14 us and
        # the per-CTA scale chain of the streaming tail does not beat the staged one), so it is opt-in.  It also makes the
        # SE mean depend on where an image's rows fall in the 32-row slab grid, i.e. on its position in the batch.
        self.se_epilogue = window and os.environ.get("VQA_SE_EPILOGUE", "0") != "0"
        # fused post-attention chains (W_o + residual + LayerNorm + FFN + residual + next block's LayerNorm + projection
        # in one kernel, csrc/chain_tcgen05.cu) for the fp16-operand text / fusion path; "0" = one launch per Linear / LayerNorm
        self.chain = self.half_tail and os.environ.get("VQA_CHAIN", "1") != "0"
        # fused stem: two conv rows per N = 128 MMA, vertical max in registers (stem_pool op); "0" = the 3-row gemm form
        self.stem_two_row = os.environ.get("VQA_STEM_TWO_ROW", "1") != "0"
        # LayerNorms that follow each other (or the embedding) share a launch: embedding + first encoder norm + mask
        # normalisation, final text norm + first query norm, projector norm + key/value norms; "0" = one launch each
        self.fuse_ln = os.environ.get("VQA_FUSE_LN", "1") != "0"
        self.fused_tail = window or self.tf32
        self.pair = window and not self.tf32
        self.phase_windows = os.environ.get("VQA_PHASE_WINDOWS", "1") != "0"   # A/B switch for the stride-2 block entries
        # shift-fused form of the 64-channel 3x3 convolutions (N = 192 MMAs + shuffle epilogue): correct and tested, but
        # measured slower than the 9-tap form on B200 (70-82 us against 66-78 us per stage-1 convolution: the MMAs reach
        # their 96-cycle floor, the epilogue's two shuffles per output do not keep up), so it is opt-in
        self.shift_fused = window and not self.tf32 and os.environ.get("VQA_SHIFT_FUSED", "0") != "0"
        self.ws = Arena(device if device is not None else weights.arena.device)
        self.ops: List[Op] = []
        self.named: Dict[str, Tuple[Buf, torch.dtype, Tuple[int, ...]]] = {}
        self.lane = 0

    def commit(self):
        self.ws.commit(zero=True)
        return self

    # -- helpers
    def _buf(self, name, dtype, *shape) -> Buf:
        n = 1
        for s in shape:
            n *= s
        b = self.ws.alloc(n * torch.empty((), dtype=dtype).element_size(), name)
        self.named[name] = (b, dtype, tuple(shape))
        return b

    def tensor(self, name) -> torch.Tensor:
        b, dtype, shape = self.named[name]
        return b.view(dtype, *shape)

    def _op(self, kind, name, i=None, p=None, f=None):
        spec = FIELDS[kind]
        i, p, f = i or {}, p or {}, f or {}
        assert set(i) <= set(spec["i"]) and set(p) <= set(spec["p"]) and set(f) <= set(spec["f"]), (kind, i, p, f)
        self.ops.append(Op(kind, name, i, p, f, self.lane))

    def gemm(self, name, *, dtype, M, N, a0, a0_shape, groups, w, bias, out, ldo, out_dtype,
             a1=None, a1_shape=None, res=None, res_dtype=-1, ldr=0, relu=False, rnd=False,
             grid: Optional[Grid] = None, halo: int = 0, MT: int = 1, row_bytes: int = 128,
             halo_hi: Optional[int] = None, pool_to: Optional[Grid] = None, pair: Optional[bool] = None,
             sf: int = 1, sf_step: int = 1, sums=None, topk=None):
        """Tap-shifted GEMM.  ``groups``: list of (map, row_delta, a_col, n_chunks, [tap_rel...]).

        For K-chunk c of group g the kernel loads ONE window of A rows
        [m0 + delta - halo, m0 + delta - halo + 128*MT + 2*halo) x 64 channels (a_col + 64c) and
        issues one MMA set per tap t whose A rows start ``tap_rel[t]`` rows into the window,
        against weight columns kbase_g + (t*n_chunks + c)*chunk.  a*_shape = (rows, cols, ld).
        ``row_bytes`` is the K-chunk width in bytes: 128 (SWIZZLE_128B, 4 MMAs per chunk) or 32
        (SWIZZLE_32B, one K=16 MMA per chunk: the stem, whose "channels" are 16 packed values).
        The window may be asymmetric: ``halo`` rows before the tile, ``halo_hi`` (default = halo) after.

        ``sf`` > 1 (shift-fused form, N <= 64): the weight matrix has ``sf`` row blocks of BN rows and every MMA is
        sf*BN columns wide; the epilogue forms out[m] = sum_j acc[m + j*sf_step, j*BN + n].  A 128-row tile then
        yields 128 - (sf-1)*sf_step output rows (the M tiling is strided accordingly).

        ``topk`` = (k, idx, probs): fused softmax + top-k of the fp32 output rows in the epilogue (k <= TOPK_FUSED_MAX,
        16-bit operands, 128-column tiles): winners and their probabilities go to ``idx`` [M, k] int64 / ``probs`` [M, k].
        """
        wbuf, _, wshape = self.W.items[w]
        npad, ktot = wshape
        chunk = row_bytes // (4 if dtype == DT_TF32 else 2)
        halo_hi = halo if halo_hi is None else halo_hi
        bn = _bn_tile(N)
        # small-M layers (text / fusion / head): halve the N tile when that still leaves fewer tiles than SMs,
        # so more SMs work and each CTA's epilogue is shorter
        if bn == 256 and ((M + 127) // 128) * ((N + 255) // 256) < 100 and npad % 128 == 0 and MT == 1:
            bn = 128
        # 256-row window convolutions with >= 256 output channels: 128-column tiles on a CTA pair (512 rows x 128
        # columns per pair) keep two accumulator stages in TMEM, so the epilogue overlaps the next tile's MMAs
        # (measured: stage 3 conv 66 -> 57 us; the 256-column tile fills TMEM with one stage)
        if bn == 256 and dtype == DT_BF16 and out_dtype == OUT_BF16 and MT == 2 and self.pair and halo > 0:
            bn = 128
        # experiment switch: "MT,BN,pair" for the window convolutions with >= 256 output channels (stages 3 and 4)
        wide = os.environ.get("VQA_WIDE_CONV", "")
        if wide and N >= 256 and dtype == DT_BF16 and out_dtype == OUT_BF16 and halo > 0 and sf == 1 and grid is not None:
            MT, bn, pair = (int(v) for v in wide.split(","))
            pair = bool(pair) and self.pair
        if topk is not None:
            assert dtype != DT_TF32 and out_dtype == OUT_F32 and res is None and not relu and MT == 1 and npad % 128 == 0
            assert 0 < topk[0] <= min(TOPK_FUSED_MAX, N)
            bn = 128
        # CTA pairs (cta_group::2): bf16 convolutions with a bf16 output; each CTA loads half of every weight tile
        if pair is None:
            pair_bns = [int(v) for v in os.environ.get("VQA_PAIR_BN", "128").split(",") if v]
            pair = (self.pair and dtype == DT_BF16 and out_dtype == OUT_BF16 and bn in pair_bns
                    and not (row_bytes == 32 and MT == 1))
            if sf > 1:
                pair = self.pair and os.environ.get("VQA_SF_PAIR", "0") != "0"
        # Small batches (batch-1 `predict`, BASELINE configs[3]): the big tiles leave most SMs without a tile -- one image at
        # 7x7 is ONE 512-row pair tile per 128 output channels, 8 CTAs each walking K = 4608 alone.  While fewer than a third of
        # the SMs would get a tile, shrink it: 128-row sub-tiles, single CTAs instead of pairs, then 64-column tiles, so that more
        # CTAs share the weight stream and the serial MMA chain of each gets shorter.  Large batches never take this path.
        if (dtype == DT_BF16 and out_dtype == OUT_BF16 and grid is not None and sf == 1 and pool_to is None and topk is None
                and sums is None and row_bytes == 128 and os.environ.get("VQA_SMALL_M", "1") != "0"):
            def n_tiles_of(mt_, bn_, pair_):
                return -(-M // (128 * mt_ * (2 if pair_ else 1))) * -(-N // bn_)
            for step in ("mt", "pair", "bn"):
                if n_tiles_of(MT, bn, pair) >= 48:      # measured: 64 big tiles (batch 128 at 7x7) beat 128 small ones
                    break
                if step == "mt" and MT == 2:
                    MT = 1
                elif step == "pair" and pair:
                    pair = False
                elif step == "bn" and bn > 64 and npad % 64 == 0:
                    bn = 64
        # widths that are multiples of 64 but not of the chosen tile (embed_dim 192, 320, 448 and their multiples, FFN
        # widths such as 320): the largest tile that divides the weight rows
        while npad % bn and bn > 64 and sf == 1 and topk is None:
            bn //= 2
        assert npad % bn == 0 and npad >= N, (name, npad, bn)
        assert len(groups) <= MAX_GROUPS and MT * bn * sf <= 512
        assert sf == 1 or (1 < sf <= 3 and npad == sf * bn and MT == 1 and pool_to is None and (sf - 1) * sf_step <= 4)
        i = dict(dtype=dtype, M=M, N=N, Npad=npad, Ktot=ktot, BN=bn, MT=MT, halo=halo,
                 a0_rows=a0_shape[0], a0_cols=a0_shape[1], a0_ld=a0_shape[2],
                 a1_rows=a1_shape[0] if a1_shape else 0, a1_cols=a1_shape[1] if a1_shape else 0,
                 a1_ld=a1_shape[2] if a1_shape else 0, ngroups=len(groups), out_dtype=out_dtype, ldo=ldo,
                 res_dtype=res_dtype, ldr=ldr, relu=int(relu), round_tf32=int(rnd),
                 mask_en=int(grid is not None), mP=grid.P if grid else 1, mRPI=grid.rpi if grid else 1,
                 mH=grid.H if grid else 1, mW=grid.W if grid else 1, smem_budget=0, max_ctas=0,
                 row_bytes=row_bytes, halo_hi=halo_hi, sf=sf, sf_step=sf_step, topk=topk[0] if topk else 0)
        if sf > 1:   # strided M tiling: tile t covers accumulator rows [t*stride, t*stride + 128), outputs the first `stride`
            stride = 128 * MT - (sf - 1) * sf_step
            i.update(tiles_per_img=(M + stride - 1) // stride, tile_stride=stride, tile_row0=0, img_rows=M, n_imgs=1)
        i["pair"] = int(bool(pair))
        if pool_to is not None:
            # fused 3x3/2 max-pool epilogue: tile t = (image, pooled row i') covers conv rows 2i'-1 .. 2i'+1
            assert grid is not None and MT == 3 and 3 * grid.P <= 384 and pool_to.H * 2 == grid.H
            i.update(tiles_per_img=pool_to.H, tile_stride=2 * grid.P, tile_row0=-grid.P, img_rows=grid.rpi,
                     n_imgs=grid.B, pool=1, pool_P=grid.P, pool_W=grid.W, pool_Wo=pool_to.W, pool_Ho=pool_to.H,
                     pool_Po=pool_to.P, pool_rpio=pool_to.rpi)
        kbase = tap0 = 0
        for g, (mp, delta, acol, nch, rels) in enumerate(groups):
            assert all(0 <= r <= halo + halo_hi for r in rels), (name, rels, halo, halo_hi)
            i[f"g_map{g}"], i[f"g_delta{g}"], i[f"g_acol{g}"], i[f"g_chunks{g}"] = mp, delta, acol, nch
            i[f"g_ntaps{g}"], i[f"g_kbase{g}"], i[f"g_tap0{g}"] = len(rels), kbase, tap0
            for r in rels:
                i[f"tap_rel{tap0}"] = r
                tap0 += 1
            kbase += len(rels) * nch * chunk
        assert kbase == ktot, (name, kbase, ktot)
        assert tap0 <= MAX_TAPS
        i["ntaps"] = tap0
        # ``sums``: fp32 [ceil(M/32), N] -- the epilogue also writes the column sums of every 32-row slab of the output
        p = dict(a0=a0, a1=a1, b=wbuf, out=out, bias=self.W.buf(bias) if bias else None, res=res, sums=sums)
        if topk is not None:
            n_tiles = npad // bn
            p.update(topk_idx=topk[1], topk_probs=topk[2],
                     topk_part=self._buf(name + ".topk_part", torch.float32, M, 2 * n_tiles, 4 + 2 * TOPK_FUSED_MAX),
                     topk_cnt=self._buf(name + ".topk_cnt", torch.int32, (M + 127) // 128))
        self._op("gemm", name, i, p)

    def linear(self, name, a, M, K, w, bias, out, N, ldo=None, res=None, relu=False, rnd=False, lda=None, topk=None):
        """fp32/TF32 dense layer: out[M,N] = a[M,K] @ W^T (+bias)(+res)(relu).

        tf32 precision mode: 3xTF32.  ``a`` (unrounded fp32) is split into [a_hi | a_lo] by a small kernel and the
        GEMM runs three K groups against [W_hi | W_hi | W_lo]; the tf32 rounding of the plain path (5e-4 per
        operand, the dominant term of the tail's error) drops to ~1e-6."""
        if self.tf32 and (w + ".x3") in self.W:
            sp = self._buf(name + ".split", torch.float32, M, 2 * K)
            self._op("split_tf32", name + ".split", dict(M=M, K=K, ld_src=lda or K), dict(src=a, dst=sp))
            kc = K // 32
            self.gemm(name, dtype=DT_TF32, M=M, N=N, a0=sp, a0_shape=(M, 2 * K, 2 * K),
                      groups=[(0, 0, 0, kc, [0]), (0, 0, K, kc, [0]), (0, 0, 0, kc, [0])],
                      w=w + ".x3", bias=bias, out=out, ldo=ldo or N, out_dtype=OUT_F32, res=res,
                      res_dtype=OUT_F32 if res is not None else -1, ldr=(ldo or N), relu=relu, rnd=False)
            return
        if self.half_tail and (w + ".h") in self.W:
            # fp16 operands; an output that feeds another Linear (rnd=True) is stored as fp16 too
            assert not (rnd and res is not None)
            self.gemm(name, dtype=DT_F16, M=M, N=N, a0=a, a0_shape=(M, K, lda or K), groups=[(0, 0, 0, K // 64, [0])],
                      w=w + ".h", bias=bias, out=out, ldo=ldo or N, out_dtype=OUT_F16 if rnd else OUT_F32, res=res,
                      res_dtype=OUT_F32 if res is not None else -1, ldr=(ldo or N), relu=relu, rnd=False, topk=topk)
            return
        assert topk is None, "the fused top-k epilogue exists for the fp16-operand Linears only"
        self.gemm(name, dtype=DT_TF32, M=M, N=N, a0=a, a0_shape=(M, K, lda or K), groups=[(0, 0, 0, K // 32, [0])],
                  w=w, bias=bias, out=out, ldo=ldo or N, out_dtype=OUT_F32, res=res,
                  res_dtype=OUT_F32 if res is not None else -1, ldr=(ldo or N), relu=relu, rnd=rnd)

    def stem_pool(self, name, a, g0: Grid, w, out, g: Grid, run_len: Optional[int] = None, max_ctas: int = 0):
        """Fused conv7x7/2 + ReLU + max-pool 3x3/2 over the phase-packed input ``a`` on grid ``g0`` (pad = 2) into the
        pooled grid ``g`` (csrc/stem_tcgen05.cu).  A CTA walks runs of ``run_len`` consecutive pooled rows of one image
        (the previous conv row is carried in registers); the default keeps every SM busy for small batches and costs one
        primer tile per 14 rows for large ones."""
        assert g0.pad == 2 and g0.P <= 128 and g.H * 2 == g0.H and g.W * 2 == g0.W and g.B == g0.B
        if run_len is None:
            run_len = next((r for r in (14, 8, 7, 4, 2, 1) if g.H % r == 0 and g0.B * (g.H // r) >= 148), 1)
        assert g.H % run_len == 0
        self._op("stem_pool", name, dict(B=g0.B, H=g0.H, W=g0.W, P=g0.P, RPI=g0.rpi, Ho=g.H, Wo=g.W, Po=g.P, RPIo=g.rpi,
                                         run_len=run_len, a_rows=g0.rows, max_ctas=max_ctas),
                 dict(a=a, w=self.W.buf(w), out=out))

    def mlp_chain(self, name, *, ctx, xres, xout, T, prefix, ln, nxt=None, max_ctas: int = 0, cs: int = 0):
        """One kernel for xout = x1 + FFN(LN(x1)), x1 = xres + ctx W_o^T, and optionally y = LN'(xout) W_n^T.

        ``prefix``: weight name prefix with ``.o.w.h / .fc1.w.h / .fc1.b / .fc2.w.h / .fc2.b``; ``ln``: name prefix of the
        LayerNorm between W_o and the FFN (``.g / .b``); ``nxt`` = (LayerNorm prefix, weight name, y buffer, Nn)."""
        W = self.W
        F = W.items[prefix + ".fc1.w.h"][2][0]
        p = dict(ctx=ctx, xres=xres, xout=xout, wo=W.buf(prefix + ".o.w.h"), w1=W.buf(prefix + ".fc1.w.h"),
                 b1=W.buf(prefix + ".fc1.b"), w2=W.buf(prefix + ".fc2.w.h"), b2=W.buf(prefix + ".fc2.b"),
                 ln_g=W.buf(ln + ".g"), ln_b=W.buf(ln + ".b"), n_g=None, n_b=None, wn=None, y=None)
        Nn = npad = 0
        if nxt is not None:
            nln, wn, y, Nn = nxt
            npad = W.items[wn][2][0]
            p.update(n_g=W.buf(nln + ".g"), n_b=W.buf(nln + ".b"), wn=W.buf(wn), y=y)
        # cs: CTAs per cluster that share the multicast weight stream (0 = by the number of 128-row tiles)
        cs = cs or int(os.environ.get("VQA_CHAIN_CS", "0"))
        self._op("mlp_chain", name, dict(T=T, D=256, F=F, Nn=Nn, Nn_pad=npad, max_ctas=max_ctas, CS=cs), p, dict(eps=1e-5, eps_n=1e-5))

    def _conv3x3_groups(self, g: Grid, nchunks: int, cout: int, residual: bool = False):
        """Stride-1 3x3 conv on a padded-flat grid -> (groups, halo, MT).

        window=True: ONE A window (tile rows + P+1 rows of halo on both sides) is loaded per K chunk
        and the 9 taps read row-shifted views of it in shared memory (9x less A traffic);
        window=False: every tap loads its own A tile at the shifted row coordinate.
        """
        if self.window:
            halo = g.P + 1
            rels = [halo + (kh - 1) * g.P + (kw - 1) for kh in range(3) for kw in range(3)]
            # 256-row tiles (less halo per output row); measured at 64 channels: 76 -> 65 us without residual, 76 -> 78 us
            # with one, so the residual convs of stage 1 keep 128-row tiles.  The tf32 kernels are instantiated for MT = 1.
            mt = 2 if (cout >= 128 or not residual) and not self.tf32 else 1
            return [(0, 0, 0, nchunks, rels)], halo, mt
        return [(0, (kh - 1) * g.P + (kw - 1), 0, nchunks, [0]) for kh in range(3) for kw in range(3)], 0, 1

    def _conv3x3_sf(self, g: Grid, nchunks: int):
        """Shift-fused stride-1 3x3 conv (64 output channels): 3 vertical taps per K chunk, each one MMA that is
        3 x 64 columns wide (horizontal taps kw = 0, 1, 2 side by side).  acc_kw[r] = sum_kh A[r + (kh-1)P - 1] W[kh,kw]
        and out[m] = acc_0[m] + acc_1[m+1] + acc_2[m+2]  ->  (groups, halo, halo_hi)."""
        halo = g.P + 1
        rels = [halo + (kh - 1) * g.P - 1 for kh in range(3)]
        return [(0, 0, 0, nchunks, rels)], halo, g.P - 1

    def _ln_mode(self, rnd):
        # output mode: 0 = fp32, 1 = tf32-rounded fp32, 2 = fp16 (operand of an fp16 Linear); tf32 precision mode:
        # consumers split the unrounded value into hi + lo
        return 0 if (not rnd or self.tf32) else (2 if self.half_tail else 1)

    def _ln_extra(self, extra):
        """``extra``: up to two (gamma, beta, dst, rnd) -- further LayerNorms of the first one's unrounded output, same launch."""
        i, p = {}, {}
        assert len(extra) <= 2
        for k, (g2, b2, dst2, rnd2) in enumerate(extra, start=2):
            i[f"rnd{k}"] = self._ln_mode(rnd2)
            p.update({f"gamma{k}": self.W.buf(g2), f"beta{k}": self.W.buf(b2), f"dst{k}": dst2})
        return i, p

    def layernorm(self, name, src, g, b, dst, rows, rnd=False, ld=None, extra=()):
        D = self.W.items[g][2][0]        # the width of the norm is that of its gamma
        xi, xp = self._ln_extra(extra)
        self._op("layernorm", name, dict(rows=rows, D=D, ld_src=ld or D, mode=0, round_tf32=self._ln_mode(rnd), S=0, Pg=0, RPIg=0, **xi),
                 dict(src=src, gamma=self.W.buf(g), beta=self.W.buf(b), dst=dst, pos=None, **xp), dict(eps=1e-5))


class Program(OpList):
    """Op list + workspace of the whole VQA forward for one (B, L, input format, aux) shape."""

    def __init__(self, weights: Weights, cfg: dict, B: int, L: int, in_fmt: str = "nchw_f32",
                 mask_dtype: int = MASK_I64, want_aux: bool = False, top_k: int = 0, device=None,
                 window: bool = True, n_images: Optional[int] = None, side: str = "both"):
        """``n_images`` (default B): the image side runs on n_images images and every image answers B / n_images
        consecutive questions (BASELINE config "one image, many questions": backbone, projector and the K/V
        projections of both cross-attention layers run once per image, SURVEY 8f row f2).

        ``side`` splits the forward at the only place the two modalities meet, the cross-attention K/V
        (models/cross_attention.py:160-161,286-287 recompute them per pair although they do not depend on the question):
        "image" = ingest .. backbone .. projector .. K/V projections of every layer (the per-image cache entry, buffers
        ``x.{l}.kv``); "question" = text encoder, cross-attention against K/V given as external slots ``kv{l}``, gate,
        head; "both" = the whole forward in one op list."""
        super().__init__(weights, device, window)
        assert side in ("both", "image", "question"), side
        self.side = side
        assert not (want_aux and side != "both"), "aux outputs need the whole forward"
        self.cfg = cfg
        self.B, self.L = B, L
        self.Bi = B if n_images is None else int(n_images)
        assert self.Bi >= 1 and B % self.Bi == 0, "the number of questions must be a multiple of the number of images"
        self.in_fmt = in_fmt
        self.mask_dtype = mask_dtype
        self.want_aux = want_aux
        self.top_k = top_k
        self._build()
        self.commit()

    # -- network definition
    def _build(self):
        B, L, W, cfg = self.Bi, self.L, self.W, self.cfg   # B = images on this side of the program
        bf, f32, i32 = torch.bfloat16, torch.float32, torch.int32
        if self.side == "question":
            self._build_text_fusion(None, None)
            return

        # ================= image side =================
        tf = self.tf32
        act = f32 if tf else bf                      # backbone activation storage
        esz = 4 if tf else 2
        self.act, self.cdt, self.codt = act, (DT_TF32 if tf else DT_BF16), (OUT_F32 if tf else OUT_BF16)
        self.cchunk = 32 if tf else 64               # channels per 128-byte K chunk
        g0 = Grid(B, 112, 112, pad=2)
        GUARD = 32   # zero phase-pixels in front of the data (only the overlapping-row variants need them)
        s0g = self._buf("stem_in", act, g0.rows + GUARD + 1, 16)
        s0 = Buf(s0g.arena, s0g.offset + GUARD * 16 * esz, g0.rows * 16 * esz, "stem_in.data")
        fused = self.stem_window and self.fuse_pool
        self._op("ingest", "ingest", dict(B=B, mode=0 if self.in_fmt == "nchw_f32" else 1, HW=224, P=g0.P, rows=g0.rows,
                                          ones=int(fused), f32=int(tf)),
                 dict(src=ExtRef(EXT["images"]), dst=s0))
        g = Grid(B, 56, 56)
        x = self._buf("s1.in", act, g.rows, 64)
        if tf:
            # tf32 mode: a phase-pixel is 16 fp32 = 64 bytes; every A row is TWO horizontally adjacent phase-pixels
            # (32 fp32 = one 128-byte chunk) through an overlapping-row tensor map (rows start every 16 elements),
            # 4 vertical x 2 horizontal taps; tap (ia, jb) covers weight columns (ia*4 + 2*jb)*16 .. +32
            s1 = self._buf("stem_out", act, g0.rows, 64)
            taps = [(0, (ia - 2) * g0.P + (2 * jb - 2) + GUARD, 0, 1, [0]) for ia in range(4) for jb in range(2)]
            self.gemm("stem.conv", dtype=DT_TF32, M=g0.rows, N=64, a0=s0g, a0_shape=(g0.rows + GUARD, 32, 16), groups=taps,
                      w="stem.w", bias="stem.b", out=s1, ldo=64, out_dtype=OUT_F32, relu=True, rnd=True, grid=g0)
            self._op("maxpool", "stem.pool", dict(B=B, C=64, Hin=112, Win=112, Pin=g0.P, RPIin=g0.rpi,
                                                  Hout=56, Wout=56, Pout=g.P, RPIout=g.rpi, f32=1), dict(src=s1, dst=x))
        elif fused and self.stem_two_row:
            self.stem_pool("stem.conv+pool", s0, g0, "stem.w2", x, g)
        elif fused:
            lo, hi = 2 * g0.P + 2, g0.P + 1
            rels = [lo + (ia - 2) * g0.P + (ib - 2) for ia in range(4) for ib in range(4)]
            self.gemm("stem.conv+pool", dtype=DT_BF16, M=g0.rows, N=64, a0=s0, a0_shape=(g0.rows, 16, 16),
                      groups=[(0, 0, 0, 1, rels)], w="stem.wb", bias=None, out=x, ldo=64, out_dtype=OUT_BF16,
                      relu=True, grid=g0, halo=lo, halo_hi=hi, MT=3, row_bytes=32, pool_to=g)
        else:
            self._stem_unfused(g0, s0, s0g, GUARD, g, x)
        self._build_rest(g, x)

    def _stem_unfused(self, g0, s0, s0g, GUARD, g, x):
        B = self.Bi
        bf = torch.bfloat16
        s1 = self._buf("stem_out", bf, g0.rows, 64)
        if self.stem_window:
            # 32-byte rows (one phase-pixel = 16 packed bf16), SWIZZLE_32B: ONE window of phase-pixels per
            # 256-row tile; the 16 taps (4 vertical x 4 horizontal phase-pixel offsets) are row-shifted
            # K=16 MMAs into it.  Window = tile + 2P+2 rows before (da=-2, db=-2) and P+1 after (da=+1, db=+1).
            lo, hi = 2 * g0.P + 2, g0.P + 1
            rels = [lo + (ia - 2) * g0.P + (ib - 2) for ia in range(4) for ib in range(4)]
            self.gemm("stem.conv", dtype=DT_BF16, M=g0.rows, N=64, a0=s0, a0_shape=(g0.rows, 16, 16),
                      groups=[(0, 0, 0, 1, rels)], w="stem.w", bias="stem.b", out=s1, ldo=64, out_dtype=OUT_BF16,
                      relu=True, grid=g0, halo=lo, halo_hi=hi, MT=2, row_bytes=32)
        else:
            # 4 vertical taps; each A row = 4 consecutive phase-pixels (64 bf16) through an overlapping-row
            # tensor map (rows start every 16 elements); 4x the shared-memory fill traffic of the window form
            # (a row is addressed by its FIRST pixel, so rows starting at pixel -1/-2 must be in-range
            # coordinates, hence the GUARD offset instead of relying on TMA out-of-bounds zero fill)
            taps = [(0, (ia - 2) * g0.P - 2 + GUARD, 0, 1, [0]) for ia in range(4)]
            self.gemm("stem.conv", dtype=DT_BF16, M=g0.rows, N=64, a0=s0g, a0_shape=(g0.rows + GUARD, 64, 16), groups=taps,
                      w="stem.w", bias="stem.b", out=s1, ldo=64, out_dtype=OUT_BF16, relu=True, grid=g0)
        self._op("maxpool", "stem.pool", dict(B=B, C=64, Hin=112, Win=112, Pin=g0.P, RPIin=g0.rpi,
                                              Hout=56, Wout=56, Pout=g.P, RPIout=g.rpi), dict(src=s1, dst=x))

    def _stage_tail(self, s, x, g, cout, has_se, has_sp, sums=None):
        """One fused kernel per stage: SE squeeze/excite, spatial attention, scaling and the relayout.  ``sums``: per-slab
        channel sums written by the epilogue of the stage's last convolution (SE squeeze for free); without spatial
        attention the tail is then a pure streaming pass (``split`` CTAs per image), with it the staged kernel skips
        its own reduction."""
        B, W = self.Bi, self.W
        bf, f32 = torch.bfloat16, torch.float32
        scale = self._buf(f"s{s}.se.scale", f32, B, cout) if has_se else None
        att = self._buf(f"s{s}.spatial.att", f32, B, g.H * g.W) if has_sp else None
        ks = int(round(math.sqrt(W.items[f"s{s}.spatial.w"][2][1]))) if has_sp else 0
        r = W.items[f"s{s}.se.w1"][2][0] if has_se else 0
        if s < 4:
            gn = Grid(B, g.H // 2, g.W // 2)
            nxt = self._buf(f"s{s + 1}.in", self.act, 4 * gn.rows, cout)
            mode, Po, RPIo, prow, out = 1, gn.P, gn.rpi, gn.rows, (nxt, True, gn.rows)
        else:
            nxt = self._buf("features", self.act, g.rows, cout)
            mode, Po, RPIo, prow, out = 0, g.P, g.rpi, g.rows, (nxt, False, 0)
        # cluster size: rows per CTA small enough for two CTAs per SM (<= ~100 KB of pixels), whole image with spatial
        cs = 1
        if not has_sp:
            lim = (200 if self.tf32 else 104) * 1024     # fp32 rows: one CTA per SM
            esz = 4 if self.tf32 else 2
            while (g.H // cs) * g.W * cout * esz > lim and cs < 8 and (g.H // (2 * cs)) % 2 == 0 and g.H % (2 * cs) == 0:
                cs *= 2
        split = 0
        if sums is not None and not has_sp:
            # streaming form: ~6k 16-byte vectors per CTA, rows per CTA even for the phase split
            split = 1
            while ((g.H // split) * g.W * cout // 8 > 8192 and g.H % (2 * split) == 0
                   and (mode == 0 or (g.H // (2 * split)) % 2 == 0)):
                split *= 2
            cs = 1
        self._op("stage_tail", f"s{s}.tail",
                 dict(B=B, C=cout, H=g.H, W=g.W, P=g.P, RPI=g.rpi, R=r, ks=ks, mode=mode, Po=Po, RPIo=RPIo,
                      phase_rows=prow, CS=cs, f32=int(self.tf32), split=split),
                 dict(src=x, w1=W.buf(f"s{s}.se.w1") if has_se else None, w2=W.buf(f"s{s}.se.w2") if has_se else None,
                      wconv=W.buf(f"s{s}.spatial.w") if has_sp else None, dst=nxt, scale=scale, att=att, sums=sums))
        return out

    def _build_rest(self, g, x):
        B, L, W, cfg = self.Bi, self.L, self.W, self.cfg   # B = images on this side of the program
        bf, f32, i32 = torch.bfloat16, torch.float32, torch.int32
        cin = 64
        x_is_phase = False
        phase_rows = 0
        for s, cout in ((1, 64), (2, 128), (3, 256), (4, 512)):
            if s > 1:
                g = Grid(B, g.H // 2, g.W // 2)
            nblk = 0
            while f"s{s}.b{nblk}.conv1.w" in W:
                nblk += 1
            for blk in range(nblk):
                y = self._buf(f"s{s}.b{blk}.mid", self.act, g.rows, cout)
                o = self._buf(f"s{s}.b{blk}.out", self.act, g.rows, cout)
                nch_in = cin // self.cchunk
                cdt, codt, rnd = self.cdt, self.codt, self.tf32   # tf32 mode: outputs are the next GEMM's tf32 operands
                w1name, halo1_hi = f"s{s}.b{blk}.conv1.w", None
                if blk == 0 and x_is_phase:   # stride-2 3x3 over the 4-phase split
                    taps = []
                    for kh in range(3):
                        ph, di = (1, -1) if kh == 0 else ((0, 0) if kh == 1 else (1, 0))
                        for kw in range(3):
                            pw, dj = (1, -1) if kw == 0 else ((0, 0) if kw == 1 else (1, 0))
                            taps.append((0, (ph * 2 + pw) * phase_rows + di * g.P + dj, 0, nch_in, [0]))
                    a_rows, halo1, mt1 = 4 * phase_rows, 0, (2 if cout >= 128 and not self.tf32 else 1)   # 256-row tiles (s2: 55 -> 43 us, s3/s4: one wave instead of 1.7)
                    if self.window and self.phase_windows and not self.tf32 and f"s{s}.b{blk}.conv1.wp" in W:
                        # one A window per PHASE instead of one A tile per tap: the 9 taps read 4 phases, and the taps of
                        # one phase are row shifts (-P-1, -P, -1, 0) of each other, so 4 windows of tile + P+1 rows
                        # replace 9 tiles in shared memory (these layers are bound by the L2 -> shared-memory fill)
                        halo1, halo1_hi, w1name = g.P + 1, 0, f"s{s}.b{blk}.conv1.wp"
                        rel = lambda di, dj: halo1 + di * g.P + dj
                        taps = [(0, 3 * phase_rows, 0, nch_in, [rel(-1, -1), rel(-1, 0), rel(0, -1), rel(0, 0)]),
                                (0, 2 * phase_rows, 0, nch_in, [rel(-1, 0), rel(0, 0)]),
                                (0, 1 * phase_rows, 0, nch_in, [rel(0, -1), rel(0, 0)]),
                                (0, 0, 0, nch_in, [rel(0, 0)])]
                else:
                    taps, halo1, mt1 = self._conv3x3_groups(g, nch_in, cout)
                    a_rows = g.rows
                sf = 3 if (self.shift_fused and f"s{s}.b{blk}.conv1.wsf" in W) else 1
                if sf > 1:
                    (taps, halo1, halo1_hi), mt1, w1name = self._conv3x3_sf(g, nch_in), 1, f"s{s}.b{blk}.conv1.wsf"
                self.gemm(f"s{s}.b{blk}.conv1", dtype=cdt, M=g.rows, N=cout, a0=x, a0_shape=(a_rows, cin, cin),
                          groups=taps, w=w1name, bias=f"s{s}.b{blk}.conv1.b", out=y, ldo=cout,
                          out_dtype=codt, relu=True, rnd=rnd, grid=g, halo=halo1, halo_hi=halo1_hi, MT=mt1, sf=sf)
                has_ds = W.items[f"s{s}.b{blk}.conv2.w"][2][1] > 9 * cout
                # the stage's last convolution also writes the SE squeeze partial sums (one row per 32-row slab)
                se_sums = None
                if (blk == nblk - 1 and self.se_epilogue and self.fused_tail and not self.tf32 and sf == 1
                        and f"s{s}.se.w1" in W):
                    se_sums = self._buf(f"s{s}.se.slabs", f32, (g.rows + 31) // 32, cout)
                taps2, halo2, mt2 = self._conv3x3_groups(g, cout // self.cchunk, cout, residual=not has_ds)
                halo2_hi, w2name = None, f"s{s}.b{blk}.conv2.w"
                if sf > 1:
                    (taps2, halo2, halo2_hi), mt2, w2name = self._conv3x3_sf(g, cout // self.cchunk), 1, f"s{s}.b{blk}.conv2.wsf"
                if has_ds:
                    # shortcut conv1x1/stride as extra K columns: phase (0,0) of the block input, same flat row index
                    # (the identity residual as K columns too was measured: 77 -> 85 us at 64 channels, not used)
                    assert x_is_phase or cin != cout
                    taps2.append((1, 0, 0, nch_in, [halo2]))
                    self.gemm(f"s{s}.b{blk}.conv2", dtype=cdt, M=g.rows, N=cout, a0=y,
                              a0_shape=(g.rows, cout, cout), a1=x,
                              a1_shape=(phase_rows if x_is_phase else g.rows, cin, cin), groups=taps2,
                              w=f"s{s}.b{blk}.conv2.w", bias=f"s{s}.b{blk}.conv2.b", out=o, ldo=cout,
                              out_dtype=codt, relu=True, rnd=rnd, grid=g, halo=halo2, MT=mt2, sums=se_sums)
                else:
                    assert not x_is_phase
                    self.gemm(f"s{s}.b{blk}.conv2", dtype=cdt, M=g.rows, N=cout, a0=y,
                              a0_shape=(g.rows, cout, cout), groups=taps2, w=w2name,
                              bias=f"s{s}.b{blk}.conv2.b", out=o, ldo=cout, out_dtype=codt, relu=True, rnd=rnd,
                              res=x, res_dtype=codt, ldr=cin, grid=g, halo=halo2, halo_hi=halo2_hi, MT=mt2, sf=sf,
                              sums=se_sums)
                x, cin, x_is_phase = o, cout, False
            # ---- stage attention + relayout for the next stage
            has_se, has_sp = f"s{s}.se.w1" in W, f"s{s}.spatial.w" in W
            if self.fused_tail and (s < 4 or has_se or has_sp):
                x, x_is_phase, phase_rows = self._stage_tail(s, x, g, cout, has_se, has_sp, sums=se_sums if nblk else None)
                continue
            scale = att = None
            if has_se:
                hw = g.H * g.W
                S = 8 if hw >= 2048 else (4 if hw >= 512 else (2 if hw >= 128 else 1))   # pixel slices per image
                sums = self._buf(f"s{s}.se.sums", f32, B, S, cout)
                scale = self._buf(f"s{s}.se.scale", f32, B, cout)
                self._op("se_squeeze", f"s{s}.se.squeeze", dict(B=B, C=cout, H=g.H, W=g.W, P=g.P, RPI=g.rpi, S=S),
                         dict(src=x, sums=sums))
                r = W.items[f"s{s}.se.w1"][2][0]
                self._op("se_excite", f"s{s}.se.excite", dict(B=B, C=cout, R=r, HW=g.H * g.W, S=S),
                         dict(sums=sums, w1=W.buf(f"s{s}.se.w1"), w2=W.buf(f"s{s}.se.w2"), scale=scale))
            if has_sp:
                att = self._buf(f"s{s}.spatial.att", f32, B, g.H * g.W)
                ks = int(round(math.sqrt(W.items[f"s{s}.spatial.w"][2][1])))
                self._op("spatial_map", f"s{s}.spatial.map", dict(B=B, C=cout, H=g.H, W=g.W, P=g.P, RPI=g.rpi, ksize=ks),
                         dict(src=x, scale=scale, wconv=W.buf(f"s{s}.spatial.w"), att=att))
            if s < 4:
                gn = Grid(B, g.H // 2, g.W // 2)
                nxt = self._buf(f"s{s + 1}.in", bf, 4 * gn.rows, cout)
                self._op("scale_relayout", f"s{s}.relayout",
                         dict(B=B, C=cout, H=g.H, W=g.W, P=g.P, RPI=g.rpi, mode=1, Po=gn.P, RPIo=gn.rpi, phase_rows=gn.rows),
                         dict(src=x, scale=scale, att=att, dst=nxt))
                x, x_is_phase, phase_rows = nxt, True, gn.rows
            elif scale is not None or att is not None:
                nxt = self._buf("features", bf, g.rows, cout)
                self._op("scale_relayout", f"s{s}.relayout",
                         dict(B=B, C=cout, H=g.H, W=g.W, P=g.P, RPI=g.rpi, mode=0, Po=g.P, RPIo=g.rpi, phase_rows=g.rows),
                         dict(src=x, scale=scale, att=att, dst=nxt))
                x = nxt
        feat, gf = x, g          # [B*64, 512] bf16 on the 7x7 (+1 pad) grid
        self.feat_name = next(k for k, v in self.named.items() if v[0] is feat)
        if self.want_aux:
            nchw = self._buf("aux.image_features", f32, B, 512, 7, 7)
            self._op("grid_to_nchw", "aux.image_features", dict(B=B, C=512, H=7, W=7, P=gf.P, RPI=gf.rpi, f32=int(self.tf32)),
                     dict(src=feat, dst=nchw))
        self._build_text_fusion(feat, gf)

    def _build_text_fusion(self, feat, gf):
        L, W, cfg = self.L, self.W, self.cfg
        bf, f32, i32 = torch.bfloat16, torch.float32, torch.int32
        Bi, B = self.Bi, self.B                    # from here on B = (image, question) pairs
        D, H, F = cfg["embed_dim"], cfg["num_attention_heads"], cfg["ffn_hidden_dim"]
        T = B * L
        S = 7
        TI = Bi * S * S
        n_layers = 0
        while f"x.{n_layers}.q.w" in W:
            n_layers += 1
        self.n_cross_layers = n_layers
        if self.side == "image":
            # the cache entry of these images: projector + LayerNorm + position, then K/V of every cross-attention layer
            praw = self._buf("proj.raw", f32, gf.rows, D)
            self.gemm("proj", dtype=self.cdt, M=gf.rows, N=D, a0=feat, a0_shape=(gf.rows, 512, 512),
                      groups=[(0, 0, 0, 512 // self.cchunk, [0])], w="proj.w", bias="proj.b", out=praw, ldo=D, out_dtype=OUT_F32)
            img = self._buf("image_projected", f32, TI, D)
            imns = [self._buf(f"x.{l}.imgn", self.tdt, TI, D) for l in range(n_layers)]
            n_fused = min(n_layers, 2) if self.fuse_ln else 0   # key/value norms that ride in the projector norm's launch
            xi, xp = self._ln_extra([(f"x.{l}.lnkv.g", f"x.{l}.lnkv.b", imns[l], True) for l in range(n_fused)])
            self._op("layernorm", "proj.ln", dict(rows=TI, D=D, ld_src=D, mode=1, round_tf32=0, S=S, Pg=gf.P, RPIg=gf.rpi, **xi),
                     dict(src=praw, gamma=W.buf("proj.ln.g"), beta=W.buf("proj.ln.b"), dst=img, pos=W.buf("proj.pos"), **xp),
                     dict(eps=1e-5))
            for l in range(n_layers):
                kv = self._buf(f"x.{l}.kv", f32, TI, 2 * D)
                if l >= n_fused:
                    self.layernorm(f"x.{l}.lnkv", img, f"x.{l}.lnkv.g", f"x.{l}.lnkv.b", imns[l], TI, rnd=True)
                self.linear(f"x.{l}.kv", imns[l], TI, D, f"x.{l}.kv.w", None, kv, 2 * D)
            return
        cached = self.side == "question"
        if cached and n_layers > MAX_CACHED_LAYERS:
            raise NotImplementedError(f"cached image side supports up to {MAX_CACHED_LAYERS} cross-attention layers")

        # ================= text side (independent of the image side: runs on the side stream) =================
        self.lane = 0 if cached else 1             # question-side programs are a single chain: one lane
        # the key mask of the self-attention is binary (mask == 0 -> -inf, models/text_encoder.py:244); the masked mean
        # pools weigh every token with attention_mask.float() (models/fusion.py:299-312): both forms are kept
        mask = maskw = None
        fuse_embed = self.fuse_ln and D == 256 and "text.0.ln1.g" in W
        if self.mask_dtype != MASK_NONE:
            mask = self._buf("mask_i32", i32, B, L)
            maskw = self._buf("mask_f32", f32, B, L)
            if not fuse_embed:
                self._op("mask_prep", "mask", dict(B=B, L=L, dtype=self.mask_dtype),
                         dict(src=ExtRef(EXT["mask"]), dst=mask, dstf=maskw))
        n_text = 0
        while f"text.{n_text}.qkv.w" in W:
            n_text += 1
        xt = self._buf("text.x", f32, T, D)
        xn = self._buf("text.xn", self.tdt, T, D) if n_text else None
        qkv = self._buf("text.qkv", f32, T, 3 * D) if n_text else None
        ctx = self._buf("text.ctx", self.tdt, T, D) if n_text else None
        chain = self.chain and D == 256 and F % 128 == 0 and F <= 1024
        # FFN hidden state of the text layers (F) and of the cross-attention layers (4 * D, modules.py:203), one buffer for
        # both; the chain kernels keep it on chip
        Fx = W.items["x.0.fc1.w"][2][0] if n_layers else F
        hid = None if chain or not (n_text or n_layers) else self._buf("text.hid", self.tdt, T, max(F, Fx))
        V = W.items["text.emb"][2][0]
        if fuse_embed:   # embedding + position, the first layer's LayerNorm and the mask normalisation in one launch
            self._op("embed", "text.embed", dict(B=B, L=L, D=D, V=V, round_tf32=self._ln_mode(True), mask_dtype=self.mask_dtype),
                     dict(ids=ExtRef(EXT["ids"]), table=W.buf("text.emb"), pe=W.buf("text.pe"), dst=xt,
                          gamma=W.buf("text.0.ln1.g"), beta=W.buf("text.0.ln1.b"), ln_dst=xn,
                          mask_src=ExtRef(EXT["mask"]) if mask is not None else None, mask_dst=mask, mask_dstf=maskw),
                     dict(eps=1e-5))
        else:
            self._op("embed", "text.embed", dict(B=B, L=L, D=D, V=V),
                     dict(ids=ExtRef(EXT["ids"]), table=W.buf("text.emb"), pe=W.buf("text.pe"), dst=xt))
        layer = 0
        while f"text.{layer}.qkv.w" in W:
            p = f"text.{layer}"
            if not (chain and layer > 0):         # chains: the previous layer's kernel already produced this layer's q, k, v
                if not (fuse_embed and layer == 0):
                    self.layernorm(p + ".ln1", xt, p + ".ln1.g", p + ".ln1.b", xn, T, rnd=True)
                self.linear(p + ".qkv", xn, T, D, p + ".qkv.w", None, qkv, 3 * D)
            if L <= ATTN_MMA_MAX_L:
                self._op("self_attn", p + ".attn", dict(B=B, L=L, H=H, hd=D // H, ld_qkv=3 * D, no_round=self.out_mode),
                         dict(qkv=qkv, mask=mask, out=ctx))
            else:
                self._op("attn_chunked", p + ".attn", dict(B=B, L=L, H=H, hd=D // H, T=L, ld_q=3 * D, ld_kv=3 * D, k_off=D,
                                                           v_off=2 * D, no_round=self.out_mode, q_per_kv=1),
                         dict(q=qkv, kv=qkv, mask=mask, out=ctx))
            if chain:
                q1 = f"text.{layer + 1}"
                nxt = (q1 + ".ln1", q1 + ".qkv.w.h", qkv, 3 * D) if (q1 + ".qkv.w") in W else None
                self.mlp_chain(p + ".chain", ctx=ctx, xres=xt, xout=xt, T=T, prefix=p, ln=p + ".ln2", nxt=nxt)
                layer += 1
                continue
            self.linear(p + ".o", ctx, T, D, p + ".o.w", None, xt, D, res=xt)
            self.layernorm(p + ".ln2", xt, p + ".ln2.g", p + ".ln2.b", xn, T, rnd=True)
            self.linear(p + ".fc1", xn, T, D, p + ".fc1.w", p + ".fc1.b", hid, F, relu=True, rnd=True)
            self.linear(p + ".fc2", hid, T, F, p + ".fc2.w", p + ".fc2.b", xt, D, res=xt)
            layer += 1
        text = self._buf("text_features", f32, T, D)
        qn0 = self._buf("x.0.qn", self.tdt, T, D) if n_layers else None
        fuse_lnq = self.fuse_ln and n_layers > 0
        self.layernorm("text.lnf", xt, "text.lnf.g", "text.lnf.b", text, T,
                       extra=[("x.0.lnq.g", "x.0.lnq.b", qn0, True)] if fuse_lnq else ())

        # ================= fusion =================
        # Two lanes stay busy: the side lane (which just finished the text encoder) goes on with the first layer's
        # query projection (needs only the text) and later with the K/V projections of layers >= 1 (need only the
        # projected image); the main lane runs projector -> K/V of layer 0 -> attention / FFN chain and joins the
        # side lane right before each attention.  Ops are issued in list order, so a JOIN waits only for what
        # precedes it in the list.
        q = qn = qp = cx = None
        if n_layers:
            q = self._buf("x.q", f32, T, D)          # running query (residual stream)
            qn = None if chain else self._buf("x.qn", self.tdt, T, D)   # chains: each layer's kernel normalises the next query
            qp = self._buf("x.qp", f32, T, D)
            cx = self._buf("x.ctx", self.tdt, T, D)
        if cached:
            imns, kvs = [], [ExtRef(EXT[f"kv{l}"]) for l in range(n_layers)]
        else:
            imns = [self._buf(f"x.{l}.imgn", self.tdt, TI, D) for l in range(n_layers)]
            kvs = [self._buf(f"x.{l}.kv", f32, TI, 2 * D) for l in range(n_layers)]
        if n_layers:                              # side lane: LN_q + W_q of layer 0
            if not fuse_lnq:
                self.layernorm("x.0.lnq", text, "x.0.lnq.g", "x.0.lnq.b", qn0, T, rnd=True)
            self.linear("x.0.q", qn0, T, D, "x.0.q.w", None, qp, D)
        self.lane = 0
        if not cached:
            praw = self._buf("proj.raw", f32, gf.rows, D)
            self.gemm("proj", dtype=self.cdt, M=gf.rows, N=D, a0=feat, a0_shape=(gf.rows, 512, 512),
                      groups=[(0, 0, 0, 512 // self.cchunk, [0])], w="proj.w", bias="proj.b", out=praw, ldo=D, out_dtype=OUT_F32)
            img = self._buf("image_projected", f32, Bi * S * S, D)
            n_fused = min(n_layers, 2) if self.fuse_ln else 0   # key/value norms that ride in the projector norm's launch
            xi, xp = self._ln_extra([(f"x.{l}.lnkv.g", f"x.{l}.lnkv.b", imns[l], True) for l in range(n_fused)])
            self._op("layernorm", "proj.ln", dict(rows=Bi * S * S, D=D, ld_src=D, mode=1, round_tf32=0, S=S, Pg=gf.P, RPIg=gf.rpi, **xi),
                     dict(src=praw, gamma=W.buf("proj.ln.g"), beta=W.buf("proj.ln.b"), dst=img, pos=W.buf("proj.pos"), **xp),
                     dict(eps=1e-5))

        def kv_proj(l):
            if l >= n_fused:
                self.layernorm(f"x.{l}.lnkv", img, f"x.{l}.lnkv.g", f"x.{l}.lnkv.b", imns[l], TI, rnd=True)
            self.linear(f"x.{l}.kv", imns[l], TI, D, f"x.{l}.kv.w", None, kvs[l], 2 * D)

        if n_layers and not cached:
            kv_proj(0)
        src_q = text
        self.xattn_weights = []
        for layer in range(n_layers):
            p = f"x.{layer}"
            if layer > 0 and not chain:           # chains: the previous layer's kernel already produced this layer's query
                self.layernorm(p + ".lnq", src_q, p + ".lnq.g", p + ".lnq.b", qn, T, rnd=True)
                self.linear(p + ".q", qn, T, D, p + ".q.w", None, qp, D)
            wts = None
            if self.want_aux:
                wts = self._buf(f"aux.xattn.{layer}", f32, B, H, L, S * S)
                self.xattn_weights.append(f"aux.xattn.{layer}")
            xi = dict(B=B, L=L, H=H, hd=D // H, T=S * S, ld_q=D, ld_kv=2 * D, k_off=0, v_off=D, no_round=self.out_mode,
                      q_per_kv=B // Bi)
            if L <= ATTN_MMA_MAX_L:
                self._op("cross_attn", p + ".attn", xi, dict(q=qp, kv=kvs[layer], out=cx, weights=wts))
            else:
                self._op("attn_chunked", p + ".attn", xi, dict(q=qp, kv=kvs[layer], mask=None, out=cx, weights=wts))
            if not cached:
                self.ops[-1].lane |= LANE_JOIN    # needs the side lane's q (layer 0) / K,V (layers >= 1)
            if layer == 0 and n_layers > 1 and not cached:   # side lane: K/V of every later layer, concurrent with this layer's chain
                self.lane = 1
                first = len(self.ops)
                for l in range(1, n_layers):
                    kv_proj(l)
                self.ops[first].lane |= LANE_JOIN  # needs image_projected from the main lane
                self.lane = 0
            if chain:
                q1 = f"x.{layer + 1}"
                nxt = (q1 + ".lnq", q1 + ".q.w.h", qp, D) if layer + 1 < n_layers else None
                self.mlp_chain(p + ".chain", ctx=cx, xres=src_q, xout=q, T=T, prefix=p, ln=p + ".lnf", nxt=nxt)
                src_q = q
                continue
            # q = src_q + W_o ctx   (first layer reads the text features as residual, writes the stream buffer)
            self.linear(p + ".o", cx, T, D, p + ".o.w", None, q, D, res=src_q)
            self.layernorm(p + ".lnf", q, p + ".lnf.g", p + ".lnf.b", qn, T, rnd=True)
            self.linear(p + ".fc1", qn, T, D, p + ".fc1.w", p + ".fc1.b", hid, Fx, relu=True, rnd=True)
            self.linear(p + ".fc2", hid, T, Fx, p + ".fc2.w", p + ".fc2.b", q, D, res=q)
            src_q = q
        # without a cross layer no attention op has joined the lanes: the fusion tail reads the side lane's text features
        # and float mask, so its first op joins them
        tail_join = len(self.ops) if n_layers == 0 and not cached else None
        fused = self._buf("fused", f32, B, D)
        attp = self._buf("attended_pooled", f32, B, D)
        txtp = self._buf("text_pooled", f32, B, D)
        use_gate = "gate.w" in W
        fused_h = self._buf("fused.h", torch.float16, B, D) if self.half_tail else None   # fp16 operand of head0
        tail_p = dict(xatt=src_q, text=text, mask=maskw, wg=None, bg=None, gamma=W.buf("out.ln.g"), beta=W.buf("out.ln.b"),
                      fused=fused, att_pooled=attp, txt_pooled=txtp, cat=None, pre=None)
        if use_gate:
            # masked pools -> [att;txt] (tf32) -> gate pre-activation on the tensor cores (the 512 KB gate matrix is
            # read once instead of once per pair) -> sigmoid gate, mix, LayerNorm
            cat = self._buf("fusion.cat", self.tdt, B, 2 * D)
            pre = self._buf("fusion.gate_pre", f32, B, D)
            self._op("pool_gate_ln", "fusion.pool", dict(B=B, L=L, D=D, use_gate=1, phase=1, no_round=self.out_mode),
                     dict(tail_p, cat=cat), dict(eps=1e-5))
            self.linear("fusion.gate", cat, B, 2 * D, "gate.w", "gate.b", pre, D)
            self._op("pool_gate_ln", "fusion.mix", dict(B=B, L=L, D=D, use_gate=1, phase=2, no_round=self.out_mode),
                     dict(tail_p, pre=pre, cat=fused_h), dict(eps=1e-5))
        else:
            self._op("pool_gate_ln", "fusion.tail", dict(B=B, L=L, D=D, use_gate=0, phase=0, no_round=self.out_mode),
                     dict(tail_p, cat=fused_h), dict(eps=1e-5))
        if tail_join is not None:
            self.ops[tail_join].lane |= LANE_JOIN

        # ================= answer head =================
        NA = cfg["num_answers"]
        h0 = self._buf("head.h0", self.tdt, B, 2 * D)
        h1 = self._buf("head.h1", self.tdt, B, D)
        self.linear("head0", fused_h if self.half_tail else fused, B, D, "head0.w", "head0.b", h0, 2 * D, relu=True, rnd=True)
        self.linear("head1", h0, B, 2 * D, "head1.w", "head1.b", h1, D, relu=True, rnd=True)
        # softmax + top-k fused into the last Linear's epilogue (models/vqa_model.py:336-337, api/inference.py:231-234):
        # per-thread running max / exp-sum / k best while the logits are drained from TMEM, merged by the CTA that finishes
        # an M tile's last N tile.  Correct and tested (tests/test_gpu_gemm.py), but OPT-IN (VQA_FUSED_TOPK=1): one thread
        # per row and partial selects among its 64 columns, against 256 threads per row in softmax_topk_kernel, and this
        # GEMM (K = 256) has no MMA time to hide that behind -- measured 55.6 us against 14.2 + 14.2 us at 256 rows.
        fuse_topk = (0 < self.top_k <= TOPK_FUSED_MAX and NA % 4 == 0 and self.half_tail and "head2.w.h" in W
                     and W.items["head2.w.h"][2][0] % 128 == 0 and os.environ.get("VQA_FUSED_TOPK", "0") != "0")
        if NA % 4 == 0:
            self.linear("head2", h1, B, D, "head2.w", "head2.b", ExtRef(EXT["logits"]), NA, ldo=NA,
                        topk=(self.top_k, ExtRef(EXT["top_idx"]), ExtRef(EXT["top_probs"])) if fuse_topk else None)
        else:
            # the GEMM epilogue stores through TMA (16-byte row pitch and N granules): an odd num_answers goes
            # through a padded scratch matrix (the padded weight rows / bias entries are zero)
            nap = (NA + 3) // 4 * 4
            lg = self._buf("head.logits_padded", f32, B, nap)
            self.linear("head2", h1, B, D, "head2.w", "head2.b", lg, nap, ldo=nap)
            self._op("copy_rows", "head2.unpad", dict(rows=B, cols=NA, ld_src=nap, ld_dst=NA),
                     dict(src=lg, dst=ExtRef(EXT["logits"])))
        if self.top_k and not fuse_topk:
            self._op("softmax_topk", "topk", dict(B=B, N=NA, k=self.top_k, ld=NA),
                     dict(logits=ExtRef(EXT["logits"]), idx=ExtRef(EXT["top_idx"]), probs=ExtRef(EXT["top_probs"])))
