"""Layer-by-layer parity of a program run against an fp64 restatement of each reference module (TEST INFRASTRUCTURE).

The op list runs in ranges on one stream.  After the last op of a module its outputs are decoded from the workspace and
compared with the oracle function of that module (oracle/vqa_oracle.py, on the reference state dict cast to fp64)
applied to the module's inputs, decoded from the same workspace.  Each module therefore sees the upstream state the
kernels produced, and an error is charged to the layer that made it, at the image / pair and element where it sits.
The references use the reference's own unfolded weights, so the load-time algebra of program.py (BN folding, tap
orders, phase splits, packed and fused forms) is checked together with the kernels.

The same walker drives the CPU emulator (tests/test_layer_parity_cpu.py) and libvqa_b200 (tests/test_gpu_layer_parity.py).
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Callable, List, Optional

import torch

import emulator as E
from oracle import vqa_oracle as O
from vqa_b200 import program as P
from vqa_b200.model import VQAModel
from vqa_b200.synth import randomise_state, synth_batch

# Gates on max|err| / max|ref| per module output, by arithmetic class and precision mode, at 2-3x the worst value measured
# on B200 (1000 W power limit) over every module and case of tests/test_gpu_layer_parity.py (B = 1 .. 1024), shown beside.
GATES = {
    "bf16": {
        "ingest": 4e-3,   # 2.95e-3: one bf16 rounding of the normalised image, <= 2^-8 of max|x|
        "conv": 1e-2,     # 4.76e-3: bf16 operands and output, fp32 accumulation (stem, convolutions, stage tails, projector)
        "linear": 2e-3,   # 8.35e-4: fp16 operands, fp32 accumulation (text / cross layers, K/V, gate, head)
        "fp32": 1e-6,     # 4.40e-7: fp32 arithmetic on the module's inputs (embedding, LayerNorm, pools, SE scale, spatial map)
    },
    "tf32": {
        "ingest": 1e-3,   # 3.69e-4: one tf32 rounding, <= 2^-11
        "conv": 1.5e-3,   # 6.49e-4: tf32 operands, fp32 activations
        "linear": 3e-5,   # 1.10e-5: 3xTF32 (the CPU emulator, accumulating in IEEE fp32, gets 1.4e-6)
        "fp32": 1e-6,     # 2.91e-7
    },
}
# max over channels of |mean error of the channel| / rms(ref), convolution class: a wrong bias, BN shift or scale moves a
# whole channel.  Its floor is the rounding of the folded weights, which is fixed per channel (B200: 9.17e-3 / 1.07e-3).
CHANNEL_GATES = {"bf16": 2e-2, "tf32": 3e-3}


def _absmax(t) -> float:
    return float(t.float().abs().max()) if t.numel() else 0.0


# ----------------------------------------------------------------------------- decoders
def grid_pads(prog, name, H, W, pad=1):
    """Max |value| over the pad rows and columns of every image of a padded-flat grid buffer."""
    t = prog.tensor(name)
    B = t.shape[0] // ((H + pad) * (W + pad))
    g = t[: B * (H + pad) * (W + pad)].view(B, H + pad, W + pad, t.shape[-1])
    return max(_absmax(g[:, H:]), _absmax(g[:, :H, W:]))


def grid_nchw(prog, name, H, W, imgs=None):
    """A padded-flat NHWC grid buffer (program.py, "HBM layout") -> (fp64 NCHW of the valid pixels of images ``imgs``
    (default: all), max |value| over the pad rows and columns of EVERY image)."""
    t = prog.tensor(name)
    C = t.shape[-1]
    B = t.shape[0] // ((H + 1) * (W + 1))
    g = t[: B * (H + 1) * (W + 1)].view(B, H + 1, W + 1, C)
    if imgs is not None:
        g = g[imgs]
    return g[:, :H, :W].permute(0, 3, 1, 2).to(torch.float64), grid_pads(prog, name, H, W)


def phases_nchw(prog, name, H, W, imgs=None):
    """The 4-phase split a stage tail writes for the next stage's stride-2 convolution (phase (ph,pw) holds x[2a+ph, 2b+pw]
    on the half-resolution padded grid) -> (fp64 NCHW [b, C, H, W], max |value| over the pads of every phase and image)."""
    t = prog.tensor(name)
    C = t.shape[-1]
    h2, w2 = H // 2, W // 2
    B = t.shape[0] // (4 * (h2 + 1) * (w2 + 1))
    ph = t[: 4 * B * (h2 + 1) * (w2 + 1)].view(4, B, h2 + 1, w2 + 1, C)
    pad = max(_absmax(ph[:, :, h2]), _absmax(ph[:, :, :h2, w2]))
    if imgs is not None:
        ph = ph[:, imgs]
    v = ph[:, :, :h2, :w2].reshape(2, 2, -1, h2, w2, C)                # [ph, pw, b, i, j, c]
    return v.permute(2, 5, 3, 0, 4, 1).reshape(-1, C, H, W).to(torch.float64), pad


def stem_in_nchw(prog, imgs=None):
    """The phase-packed ingest buffer (16 values per phase-pixel: [ph][pw][c of 4], 112 x 112 grid with 2 pad rows and
    columns, 32 guard rows in front) -> (fp64 NCHW image [b, 3, 224, 224], max deviation of every other cell -- pads,
    guards, the spare channel -- from what it must hold: 0, or 1.0 in the bias column of the fused stem)."""
    t = prog.tensor("stem_in")
    op = next(o for o in prog.ops if o.kind == "ingest")
    B, Pp = op.i["B"], op.i["P"]
    guard = t.shape[0] - 1 - B * Pp * Pp
    d = t[guard: guard + B * Pp * Pp].view(B, Pp, Pp, 2, 2, 4)
    spare = d[:, :112, :112, :, :, 3].float()
    if op.i["ones"]:
        spare = spare.clone()
        spare[:, :, :, 0] -= 1.0
    pad = max(_absmax(t[:guard]), _absmax(t[guard + B * Pp * Pp:]), _absmax(d[:, 112:]), _absmax(d[:, :112, 112:]),
              _absmax(spare))
    if imgs is not None:
        d = d[imgs]
    img = d[:, :112, :112, :, :, :3].permute(0, 5, 1, 3, 2, 4).reshape(-1, 3, 224, 224)
    return img.to(torch.float64), pad


def tokens(prog, name, B, L):
    """A row-major token buffer (fp32 or fp16) -> fp64 [B, L, D]."""
    t = prog.tensor(name)
    return t.reshape(-1, t.shape[-1])[: B * L].reshape(B, L, -1).to(torch.float64)


# ----------------------------------------------------------------------------- report
@dataclass
class Row:
    module: str
    output: str
    cls: str            # gate class ("pads": exactly 0; "topk": exact winners)
    err: float          # max|err| / max|ref| (pads: max |pad value|; topk: mismatching winners)
    rms: float          # rms(err) / rms(ref)
    where: str
    gate: float
    chan: Optional[float] = None       # convolution class: max |channel mean error| / rms(ref)
    chan_gate: Optional[float] = None
    kernel: str = ""

    @property
    def ok(self) -> bool:
        ok = self.err <= self.gate                      # NaN fails
        if self.chan is not None:
            ok = ok and self.chan <= self.chan_gate
        return ok


class Report:
    def __init__(self, title):
        self.title = title
        self.rows: List[Row] = []

    def failures(self) -> List[Row]:
        return [r for r in self.rows if not r.ok]

    def failing_modules(self) -> List[str]:
        out = []
        for r in self.failures():
            if r.module not in out:
                out.append(r.module)
        return out

    def worst(self, cls) -> float:
        return max((r.err for r in self.rows if r.cls == cls), default=0.0)

    def table(self) -> str:
        lines = [self.title,
                 f"{'module':<20} {'output':<22} {'class':<7} {'max/absmax':>10} {'gate':>8} {'rms/rms':>9} "
                 f"{'chan':>9} {'':4} where / kernel"]
        for r in self.rows:
            chan = "" if r.chan is None else f"{r.chan:9.2e}"
            lines.append(f"{r.module:<20} {r.output:<22} {r.cls:<7} {r.err:10.2e} {r.gate:8.1e} {r.rms:9.2e} "
                         f"{chan:>9} {'ok' if r.ok else 'FAIL':4} {r.where}  {r.kernel}")
        return "\n".join(lines)


def _where(idx, shape, labels, index_map=None):
    pos = []
    for d in reversed(shape):
        pos.append(idx % d)
        idx //= d
    pos = pos[::-1]
    if index_map is not None:
        pos[0] = int(index_map[pos[0]])
    return " ".join(f"{lab}{p}" for lab, p in zip(labels, pos))


# ----------------------------------------------------------------------------- the checker
class Checker:
    """Walks ``prog`` with ``runner(first, last)`` (runs ops [first, last) and returns when they are done) and compares
    every module with its fp64 reference.  ``imgs``: the images whose backbone layers are checked (default all); pads,
    projector, K/V and the whole text / fusion / head side are checked for every image and pair."""

    def __init__(self, prog: P.Program, sd, ext, runner: Callable[[int, int], None], imgs=None,
                 kernel_name: Optional[Callable[[int], str]] = None, title: str = ""):
        self.prog, self.ext, self.runner = prog, ext, runner
        self.dev = prog.ws.tensor.device
        self.sd = {k: v.detach().to(self.dev, torch.float64) for k, v in sd.items()}
        self.cfg = prog.cfg
        self.heads = self.cfg["num_attention_heads"]
        self.mode = "tf32" if prog.tf32 else "bf16"
        self.imgs = None if imgs is None else torch.as_tensor(imgs, dtype=torch.long, device=self.dev)
        self.kernel_name = kernel_name or (lambda k: "")
        self.idx = {op.name: k for k, op in enumerate(prog.ops)}
        self.report = Report(title or f"B={prog.B} images={prog.Bi} L={prog.L} {prog.in_fmt} {self.mode}")
        self.snaps = {}
        self.steps = []

    # -- bookkeeping
    def _last(self, pred) -> int:
        return max(k for k, op in enumerate(self.prog.ops) if pred(op.name))

    def _step(self, at, fn):
        self.steps.append((at, fn))

    def _snap(self, key, at, fn):
        """Decode a buffer that later ops rewrite in place, right after op ``at``."""
        self._step(at, lambda: self.snaps.__setitem__(key, fn()))

    def _cmp(self, module, output, cls, got, want, labels, at, index_map=None, chan=False):
        got, want = got.to(torch.float64), want.to(torch.float64)
        assert got.shape == want.shape, (module, output, tuple(got.shape), tuple(want.shape))
        d = got - want
        err = d.abs()
        amax = float(want.abs().max())
        k = int(torch.nan_to_num(err, nan=math.inf).argmax())
        rms_ref = float(want.pow(2).mean().sqrt())
        row = Row(module, output, cls, float(err.max()) / amax, float(err.pow(2).mean().sqrt()) / rms_ref,
                  _where(k, got.shape, labels, index_map), GATES[self.mode][cls], kernel=self.kernel_name(at))
        if chan:
            row.chan = float(d.mean(dim=(0, 2, 3)).abs().max()) / rms_ref
            row.chan_gate = CHANNEL_GATES[self.mode]
        self.report.rows.append(row)

    def _pads(self, module, output, value, at):
        self.report.rows.append(Row(module, output, "pads", value, 0.0, "", 0.0, kernel=self.kernel_name(at)))

    def _conv(self, module, output, got, want, at):
        self._cmp(module, output, "conv", got, want, ("img ", "c", "h", "w"), at, self.imgs, chan=True)

    # -- module list
    def _ref_image(self):
        x = self.ext[P.EXT["images"]]
        if self.imgs is not None:
            x = x[self.imgs.to(x.device)]
        if self.prog.in_fmt == "hwc_u8":
            return O.preprocess_u8(x.cpu()).to(self.dev, torch.float64)
        return x.to(self.dev, torch.float64)

    def _backbone(self):
        sd, prog, imgs, idx = self.sd, self.prog, self.imgs, self.idx
        k = idx["ingest"]

        def ingest():
            got, pad = stem_in_nchw(prog, imgs)
            self._cmp("ingest", "stem_in", "ingest", got, self._ref_image(), ("img ", "c", "y", "x"), k, imgs)
            self._pads("ingest", "stem_in pads", pad, k)
        self._step(k, ingest)

        k_stem = self._last(lambda n: n.startswith("stem."))

        def stem():
            x, _ = stem_in_nchw(prog, imgs)
            got, pad = grid_nchw(prog, "s1.in", 56, 56, imgs)
            self._conv("stem", "s1.in", got, O.stem(sd, x), k_stem)
            self._pads("stem", "s1.in pads", pad, k_stem)
            if "stem_out" in prog.named:
                self._pads("stem", "stem_out pads", grid_pads(prog, "stem_out", 112, 112, pad=2), k_stem)
        self._step(k_stem, stem)

        for s in (1, 2, 3, 4):
            hw = 56 >> (s - 1)
            nblk = sum(1 for b in range(8) if f"s{s}.b{b}.conv1" in idx)
            p = f"image_encoder.stage{s}"
            for b in range(nblk):
                self._block(s, b, hw, p + f".blocks.{b}")
            self._tail(s, hw, nblk, p)

    def _block_input(self, s, b, hw):
        if b > 0:
            return grid_nchw(self.prog, f"s{s}.b{b - 1}.out", hw, hw, self.imgs)[0]
        if s == 1:
            return grid_nchw(self.prog, "s1.in", hw, hw, self.imgs)[0]
        return phases_nchw(self.prog, f"s{s}.in", 2 * hw, 2 * hw, self.imgs)[0]

    def _block(self, s, b, hw, p):
        stride = 2 if (s > 1 and b == 0) else 1
        k1, k2 = self.idx[f"s{s}.b{b}.conv1"], self.idx[f"s{s}.b{b}.conv2"]

        def conv1():
            got, pad = grid_nchw(self.prog, f"s{s}.b{b}.mid", hw, hw, self.imgs)
            self._conv(f"s{s}.b{b}.conv1", f"s{s}.b{b}.mid", got, O.block_conv1(self.sd, p, self._block_input(s, b, hw), stride), k1)
            self._pads(f"s{s}.b{b}.conv1", f"s{s}.b{b}.mid pads", pad, k1)

        def conv2():
            mid = grid_nchw(self.prog, f"s{s}.b{b}.mid", hw, hw, self.imgs)[0]
            got, pad = grid_nchw(self.prog, f"s{s}.b{b}.out", hw, hw, self.imgs)
            want = O.block_tail(self.sd, p, self._block_input(s, b, hw), mid, stride)
            self._conv(f"s{s}.b{b}.conv2", f"s{s}.b{b}.out", got, want, k2)
            self._pads(f"s{s}.b{b}.conv2", f"s{s}.b{b}.out pads", pad, k2)
        self._step(k1, conv1)
        self._step(k2, conv2)

    def _tail(self, s, hw, nblk, p):
        prog, sd = self.prog, self.sd
        ops = [k for k, op in enumerate(prog.ops) if op.name.startswith(f"s{s}.") and not op.name.split(".")[1].startswith("b")]
        if not ops:
            return                                  # stage 4 without attention: its last block output is the feature map
        k = max(ops)
        has_se, has_sp = (p + ".attention.se.fc1.weight") in sd, (p + ".attention.spatial.conv.weight") in sd
        name = f"s{s}.tail"

        def tail():
            x = grid_nchw(prog, f"s{s}.b{nblk - 1}.out", hw, hw, self.imgs)[0]
            y = x
            if has_se:
                sc = O.se_scale(sd, p + ".attention.se", x)
                got = prog.tensor(f"s{s}.se.scale")
                got = got[self.imgs] if self.imgs is not None else got
                self._cmp(name, f"s{s}.se.scale", "fp32", got, sc, ("img ", "c"), k, self.imgs)
                y = x * sc.view(x.shape[0], -1, 1, 1)
            if has_sp:
                amap = O.spatial_map(sd, p + ".attention.spatial", y)
                got = prog.tensor(f"s{s}.spatial.att").view(-1, 1, hw, hw)
                got = got[self.imgs] if self.imgs is not None else got
                self._cmp(name, f"s{s}.spatial.att", "fp32", got, amap, ("img ", "c", "h", "w"), k, self.imgs)
                y = y * amap
            if s < 4:
                got, pad = phases_nchw(prog, f"s{s + 1}.in", hw, hw, self.imgs)
                out = f"s{s + 1}.in"
            else:
                got, pad = grid_nchw(prog, prog.feat_name, hw, hw, self.imgs)
                out = prog.feat_name
            self._conv(name, out, got, y, k)
            self._pads(name, out + " pads", pad, k)
        self._step(k, tail)

    def _image_side_linears(self):
        prog, sd, idx = self.prog, self.sd, self.idx
        Bi, D = prog.Bi, self.cfg["embed_dim"]
        k = idx["proj.ln"]

        def image_projected():
            return prog.tensor("image_projected").view(Bi, 49, D).to(torch.float64)

        def proj():
            feats = grid_nchw(prog, prog.feat_name, 7, 7)[0]
            self._cmp("proj", "image_projected", "conv", image_projected(), O.image_projector(sd, feats),
                      ("img ", "pos", "d"), k)
        self._step(k, proj)
        for l in range(prog.n_cross_layers):
            kk = idx[f"x.{l}.kv"]

            def kv(l=l, kk=kk):
                lp = f"fusion.cross_attention.layers.{l}"
                n = O._ln(sd, lp + ".norm_kv", image_projected())
                want = torch.cat([O._lin(sd, lp + ".cross_attention.W_k", n), O._lin(sd, lp + ".cross_attention.W_v", n)], -1)
                got = prog.tensor(f"x.{l}.kv").view(Bi, 49, 2 * D)
                self._cmp(f"x.{l}.kv", f"x.{l}.kv", "linear", got, want, ("img ", "pos", "d"), kk)
            self._step(kk, kv)

    def _text_fusion_head(self):
        prog, sd, idx, ext = self.prog, self.sd, self.idx, self.ext
        B, Bi, L = prog.B, prog.Bi, prog.L
        ids = ext[P.EXT["ids"]].to(self.dev)
        mask = ext[P.EXT["mask"]]
        mask = None if mask is None else mask.to(self.dev)
        tok = ("pair ", "tok ", "d")
        k = idx["text.embed"]
        self._snap("text.x", k, lambda: tokens(prog, "text.x", B, L))
        self._step(k, lambda: self._cmp("text.embed", "text.x", "fp32", self.snaps["text.x"], O.text_embed(sd, ids), tok, k))
        n_text = sum(1 for l in range(64) if f"text.{l}.attn" in idx)
        for l in range(n_text):
            kl = idx.get(f"text.{l}.chain", idx.get(f"text.{l}.fc2"))

            def layer(l=l, kl=kl):
                x_in = self.snaps.pop("text.x")
                want = O.text_layer(sd, f"text_encoder.layers.{l}", x_in, mask, self.heads)
                self.snaps["text.x"] = tokens(prog, "text.x", B, L)
                self._cmp(f"text.{l}", "text.x", "linear", self.snaps["text.x"], want, tok, kl)
            self._step(kl, layer)
        k = idx["text.lnf"]

        def final_norm():
            want = O._ln(sd, "text_encoder.final_norm", self.snaps.pop("text.x"))
            self._cmp("text.lnf", "text_features", "fp32", tokens(prog, "text_features", B, L), want, tok, k)
        self._step(k, final_norm)

        q_name = "text_features"
        for l in range(prog.n_cross_layers):
            kl = idx.get(f"x.{l}.chain", idx.get(f"x.{l}.fc2"))

            def cross(l=l, kl=kl, q_name=q_name):
                q_in = self.snaps.pop("x.q") if q_name == "x.q" else tokens(prog, "text_features", B, L)
                img = prog.tensor("image_projected").view(Bi, 49, -1).to(torch.float64).repeat_interleave(B // Bi, dim=0)
                want, w = O.cross_layer(sd, f"fusion.cross_attention.layers.{l}", q_in, img, self.heads)
                self.snaps["x.q"] = tokens(prog, "x.q", B, L)
                self._cmp(f"x.{l}", "x.q", "linear", self.snaps["x.q"], want, tok, kl)
                if prog.want_aux:
                    got = prog.tensor(f"aux.xattn.{l}").view(B, self.heads, L, 49)
                    self._cmp(f"x.{l}", f"aux.xattn.{l}", "linear", got, w, ("pair ", "head ", "tok ", "key "), kl)
            self._step(kl, cross)
            q_name = "x.q"
        kf = self._last(lambda n: n.startswith("fusion."))

        def fusion(q_name=q_name):
            q = self.snaps.pop("x.q") if q_name == "x.q" else tokens(prog, "text_features", B, L)
            fused, ap, tp = O.fusion_tail(sd, q, tokens(prog, "text_features", B, L), mask)
            for name, want, cls in (("attended_pooled", ap, "fp32"), ("text_pooled", tp, "fp32"), ("fused", fused, "linear")):
                self._cmp("fusion", name, cls, prog.tensor(name), want, ("pair ", "d"), kf)
        self._step(kf, fusion)

        kh = idx.get("head2.unpad", idx["head2"])
        logits = ext[P.EXT["logits"]]

        def head():
            want = O.answer_head(sd, prog.tensor("fused").to(torch.float64))
            self._cmp("head", "logits", "linear", logits, want, ("pair ", "answer "), kh)
        self._step(kh, head)
        if prog.top_k:
            kt = idx.get("topk", kh)

            def topk():
                wi, wp = O.predict_topk(logits.to(torch.float64), prog.top_k)
                gi, gp = ext[P.EXT["top_idx"]], ext[P.EXT["top_probs"]]
                bad = (gi != wi).any(dim=1)
                first = int(bad.nonzero()[0]) if bool(bad.any()) else -1
                self.report.rows.append(Row("topk", "top_idx", "topk", float(bad.sum()), 0.0,
                                            f"first pair {first}" if first >= 0 else "", 0.0, kernel=self.kernel_name(kt)))
                self._cmp("topk", "top_probs", "fp32", gp, wp, ("pair ", "rank "), kt)
            self._step(kt, topk)

    # -- run
    def run(self) -> Report:
        if self.prog.side == "both":
            self._backbone()
            self._image_side_linears()
        self._text_fusion_head()
        done = 0
        with torch.no_grad():
            for at, fn in sorted(self.steps, key=lambda s: s[0]):     # stable: snapshots before checks of the same op
                if at + 1 > done:
                    self.runner(done, at + 1)
                    done = at + 1
                fn()
            if done < len(self.prog.ops):
                self.runner(done, len(self.prog.ops))
        return self.report


# ----------------------------------------------------------------------------- cases
ABLATE = dict(use_se_attention=False, use_spatial_attention=False, use_gating=False, num_transformer_layers=1,
              num_cross_layers=1, max_question_length=12, vocab_size=500, num_answers=37)
NOSPATIAL = dict(use_spatial_attention=False)


def make_case(ctor, B, L=None, in_fmt="nchw_f32", mask_kind="i64", precision="bf16", window=True, n_images=None,
              device="cpu", seed=1234, top_k=5):
    """A seeded model (randomised BN / LayerNorm state), its program on ``device`` and the external slots.
    Returns (prog, sd, ext)."""
    torch.manual_seed(0)
    model = VQAModel(**ctor).eval()
    sd = randomise_state(model.state_dict(), 1)
    cfg = model.config
    L = L or cfg["max_question_length"]
    Bi = B if n_images is None else n_images
    u8, img, ids, mask = synth_batch(B, seed, max_len=L, vocab=cfg["vocab_size"])
    images = (u8 if in_fmt == "hwc_u8" else img)[:Bi]
    code = {"i64": P.MASK_I64, "f32": P.MASK_F32, "none": P.MASK_NONE}[mask_kind]
    m = {"i64": mask, "f32": mask.float(), "none": None}[mask_kind]
    W = P.build_weights(sd, cfg, device, precision=precision)
    prog = P.Program(W, cfg, B, L, in_fmt, code, want_aux=True, top_k=top_k, device=device, window=window, n_images=n_images)
    NA = cfg["num_answers"]
    ext = [images, ids, m, torch.zeros(B, NA), torch.zeros(B, max(top_k, 1), dtype=torch.int64), torch.zeros(B, max(top_k, 1))]
    ext = [None if t is None else t.to(device) for t in ext]
    return prog, sd, ext


def emulator_runner(prog, ext):
    emu = E.Emulator(prog)
    return lambda first, last: emu.run(ext, first, last)


def check_on_emulator(prog, sd, ext, imgs=None, title="") -> Report:
    return Checker(prog, sd, ext, emulator_runner(prog, ext), imgs=imgs, kernel_name=lambda k: "", title=title).run()
