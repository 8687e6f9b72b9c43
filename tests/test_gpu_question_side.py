"""The question side against fp64 at every question length, mask shape and image-to-question ratio the API accepts.

1. The attention core (attn_mma_kernel through VQA_OP_SELF_ATTN / VQA_OP_CROSS_ATTN) against softmax(QK^T/sqrt(32) +
   mask) V in fp64 on the same fp32 inputs: every key-tile template (3, 4, 7, 8 tiles of 8 keys) and both sides of each
   boundary, one and two query blocks, seven key-mask shapes (a fully masked row is NaN, at exactly the reference's
   elements), the three output forms, near one-hot softmaxes, cross-attention with several questions per image, and the
   launcher's refusals.
2. layernorm256_kernel (both modes, up to two chained norms, every output form), embed_kernel / embed_ln_kernel (every
   mask dtype, first and last id, lengths whose tok % L differ) and pool_gate_ln_kernel (phases 0, 1, 2 with weighted,
   negative, sub-unit and zero-sum masks) against fp64, on random, constant and large-offset rows.
3. The whole question side through tests/layer_parity.py at max_question_length 1, 9, 32, 33 and 64, at token counts
   T = B * L below, at, one past and several 128-row tiles, every mask shape and dtype, 2 and 3 images with 2 and 5
   questions each, bf16 and tf32 with a fully masked question, and the cached path (image side, then question side).

VQA_DRY=1 runs every case on the CPU emulator instead of the library (a rehearsal of the test's Python side).

Output forms are compared beyond the rounding their format allows: |got - ref| - half an ulp of the format at ref
(tf32 and fp16: 11 significant bits; fp32: 0), over max|ref|.  tf32 outputs must also be exact tf32 values.

Worst error measured on B200 (1000 W power limit), by check and output form (fp32 / tf32 / fp16):

    self-attention, randn inputs       1.35e-6 / 3.83e-7 / 4.23e-7
    self-attention, inputs x8          1.58e-5 / 1.32e-5 / 9.98e-6
    cross-attention output             2.08e-6 / 7.35e-7 / 6.33e-7   weights 1.83e-6
    layernorm256_kernel                1.68e-7 / 1.91e-8 / 2.35e-8   large-offset rows 2.35e-4 (within 3x torch fp32)
    embed_kernel / embed_ln_kernel     1.87e-7 / 1.38e-8 / 1.86e-8
    pool_gate_ln_kernel                3.85e-7 / 4.31e-9 / 3.67e-8

End to end (layer_parity.GATES classes), worst over the bf16 cases: linear 8.00e-4, fp32 1.91e-7, conv 4.86e-3.  The
whole file takes about 10 s on a B200.
"""
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

import emulator as E  # noqa: E402
import layer_parity as LP  # noqa: E402
import question_ref as R  # noqa: E402
from vqa_b200 import program as P  # noqa: E402

DRY = bool(os.environ.get("VQA_DRY"))     # CPU-only rehearsal of the test's Python side: the emulator stands in
DEV = "cpu" if DRY else "cuda"
H, D = 8, 256

# max over elements of (|err| - half ulp of the output format) / max|ref|, at 2-3x the worst measured on B200 (1000 W)
GATES = {
    "attn": 5e-6,        # 2.08e-6 (cross-attention output, fp32 form): 3xTF32 products, fp32 softmax
    "attn_x8": 4e-5,     # 1.58e-5: inputs x8 make scores 64x larger, so their fp32 rounding moves the near one-hot softmax 64x more
    "ln": 1e-6,          # 3.85e-7 (a pooled row): fp32 LayerNorm, embedding, pools
}
ROW_SUM_GATE = 1e-5      # |sum of a cross-attention weight row - 1|
FORMS = {0: "tf32", 1: "f32", 2: "f16"}      # attention no_round / pool no_round -> output format
LN_FORMS = {0: "f32", 1: "tf32", 2: "f16"}   # LayerNorm rnd -> output format


def _weights(device, **tensors):
    W = P.Weights(device)
    W.add("dummy", torch.zeros(8), torch.float32)
    for name, t in tensors.items():
        W.add(name, t, torch.float32)
    return W.finalize()


def _named(ol, name):
    b, dtype, shape = ol.named[name]
    return b.view(dtype, *shape)


def _run(build, ext=None):
    """``build(device) -> OpList`` with its inputs written; runs it on the library (or the emulator under VQA_DRY).
    Returns (oplist, ext on the device)."""
    ol = build(DEV)
    ext = [None if t is None else t.to(DEV) for t in (ext or [None] * 6)]
    if DRY:
        E.Emulator(ol).run(ext)
    else:
        from vqa_b200.runtime import Plan
        plan = Plan(ol.ops, 0)
        plan.run([0 if t is None else t.data_ptr() for t in ext], torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
    return ol, ext


def _check(tag, got, want, form, gate):
    got, want = got.cpu(), want.cpu()
    assert R.nan_mismatch(got, want) == 0, f"{tag}: NaN at different elements than the fp64 reference"
    if form == "tf32":
        fin = ~torch.isnan(got)
        assert bool(R.is_tf32(got.float())[fin].all()), f"{tag}: output is not tf32-rounded"
    err = R.form_error(got, want, form)
    print(f"WORST {tag} {form} {err:.3e}")
    assert err <= gate, f"{tag}: {err:.3e} > {gate:.1e}"
    return err


# ============================================================================ 1. attention core
SELF_LENGTHS = [1, 2, 7, 8, 9, 16, 17, 24, 25, 31, 32, 33, 40, 48, 56, 57, 63, 64]
MASK_KINDS = ("all", "prefix", "left", "first", "last", "holes", "none")


def key_mask(kind, L):
    """One [L] int32 key mask of the given shape."""
    m = torch.zeros(L, dtype=torch.int32)
    if kind == "all":
        m[:] = 1
    elif kind == "prefix":
        m[: max(1, (2 * L) // 3)] = 1
    elif kind == "left":                        # left-padded: the valid tokens at the end of the row
        m[L - max(1, L // 2):] = 1
    elif kind == "first":
        m[0] = 1
    elif kind == "last":
        m[L - 1] = 1
    elif kind == "holes":
        m[0::2] = 1
    else:
        assert kind == "none", kind             # a fully masked row: NaN in the reference
    return m


@pytest.mark.parametrize("L", SELF_LENGTHS)
def test_self_attention_matches_fp64(L):
    """One pair per mask shape (7 pairs), each output form at unit and x8 input scale (6 ops on one mask)."""
    B = len(MASK_KINDS)
    mask = torch.stack([key_mask(k, L) for k in MASK_KINDS])
    cases = [(nr, sc) for nr in (0, 1, 2) for sc in (1.0, 8.0)]
    g = torch.Generator().manual_seed(100 + L)
    inputs = [torch.randn(B * L, 3 * D, generator=g) * sc for _, sc in cases]

    def build(device):
        ol = P.OpList(_weights(device), device)
        m = ol._buf("mask", torch.int32, B, L)
        for c, (nr, _) in enumerate(cases):
            qkv = ol._buf(f"qkv{c}", torch.float32, B * L, 3 * D)
            out = ol._buf(f"out{c}", torch.float16 if nr == 2 else torch.float32, B * L, D)
            ol._op("self_attn", f"attn{c}", dict(B=B, L=L, H=H, hd=32, ld_qkv=3 * D, no_round=nr),
                   dict(qkv=qkv, mask=m, out=out))
        ol.commit()
        _named(ol, "mask").copy_(mask)
        for c, x in enumerate(inputs):
            _named(ol, f"qkv{c}").copy_(x)
        return ol
    ol, _ = _run(build)
    for c, (nr, sc) in enumerate(cases):
        x = inputs[c].view(B, L, 3 * D)
        want, _ = R.attention(x[..., :D], x[..., D:2 * D], x[..., 2 * D:], H, mask)
        got = _named(ol, f"out{c}").view(B, L, D)
        assert bool(torch.isnan(want[MASK_KINDS.index("none")]).all()) and not bool(torch.isnan(want[:-1]).any())
        _check(f"self L{L} x{sc:g}", got, want, FORMS[nr], GATES["attn" if sc == 1 else "attn_x8"])


CROSS_CASES = [(L, Bi, qpk) for L in (1, 17, 33, 64) for Bi in (1, 3) for qpk in (1, 2, 5)]


@pytest.mark.parametrize("T", [49, 1, 8, 9, 25, 33, 57, 64])
def test_cross_attention_matches_fp64(T):
    """T = 49 (the image tokens): L in {1, 17, 33, 64} x images {1, 3} x questions per image {1, 2, 5}.  The other key
    counts cover the launcher's envelope and every template at one configuration each."""
    cases = CROSS_CASES if T == 49 else [(33, 2, 2)]
    g = torch.Generator().manual_seed(200 + T)
    data = []
    for c, (L, Bi, qpk) in enumerate(cases):
        B = Bi * qpk
        data.append((torch.randn(B * L, D, generator=g), torch.randn(Bi * T, 2 * D, generator=g), c % 3))

    def build(device):
        ol = P.OpList(_weights(device), device)
        for c, (L, Bi, qpk) in enumerate(cases):
            B, nr = Bi * qpk, data[c][2]
            q = ol._buf(f"q{c}", torch.float32, B * L, D)
            kv = ol._buf(f"kv{c}", torch.float32, Bi * T, 2 * D)
            out = ol._buf(f"out{c}", torch.float16 if nr == 2 else torch.float32, B * L, D)
            w = ol._buf(f"w{c}", torch.float32, B, H, L, T)
            ol._op("cross_attn", f"x{c}", dict(B=B, L=L, H=H, hd=32, T=T, ld_q=D, ld_kv=2 * D, k_off=0, v_off=D,
                                               no_round=nr, q_per_kv=qpk), dict(q=q, kv=kv, out=out, weights=w))
        ol.commit()
        for c, (q, kv, _) in enumerate(data):
            _named(ol, f"q{c}").copy_(q)
            _named(ol, f"kv{c}").copy_(kv)
        return ol
    ol, _ = _run(build)
    for c, (L, Bi, qpk) in enumerate(cases):
        B = Bi * qpk
        q, kv, nr = data[c]
        kv = kv.view(Bi, T, 2 * D)
        want, wref = R.attention(q.view(B, L, D), kv[..., :D], kv[..., D:], H, None, qpk)
        tag = f"cross T{T} L{L} images{Bi} x{qpk}"
        _check(tag, _named(ol, f"out{c}").view(B, L, D), want, FORMS[nr], GATES["attn"])
        w = _named(ol, f"w{c}").cpu()
        _check(tag + " weights", w, wref, "f32", GATES["attn"])
        rows = (w.double().sum(dim=-1) - 1).abs().max().item()
        print(f"WORST {tag} row sums {rows:.3e}")
        assert rows <= ROW_SUM_GATE, f"{tag}: a weight row sums to 1 +- {rows:.2e}"


@pytest.mark.skipif(DRY, reason="the launcher's refusals are the library's; the emulator does not model them")
@pytest.mark.parametrize("kind", ["cross_T65", "self_L65", "cross_batch_not_multiple"])
def test_attention_launcher_refuses_out_of_envelope(kind):
    """65 keys, 65 tokens and a batch that is not a multiple of q_per_kv are errors, and nothing is launched."""
    from vqa_b200.runtime import Plan, VqaError, launch_count

    def build(device):
        ol = P.OpList(_weights(device), device)
        if kind == "self_L65":
            B, L = 2, 65
            qkv = ol._buf("qkv", torch.float32, B * L, 3 * D)
            mask = ol._buf("mask", torch.int32, B, L)
            out = ol._buf("out", torch.float32, B * L, D)
            ol._op("self_attn", "attn", dict(B=B, L=L, H=H, hd=32, ld_qkv=3 * D, no_round=1), dict(qkv=qkv, mask=mask, out=out))
        else:
            B, L, T, qpk = (2, 20, 65, 1) if kind == "cross_T65" else (5, 20, 49, 2)
            q = ol._buf("q", torch.float32, B * L, D)
            kv = ol._buf("kv", torch.float32, B * T, 2 * D)
            out = ol._buf("out", torch.float32, B * L, D)
            w = ol._buf("w", torch.float32, B, H, L, T)
            ol._op("cross_attn", "x", dict(B=B, L=L, H=H, hd=32, T=T, ld_q=D, ld_kv=2 * D, k_off=0, v_off=D, no_round=1,
                                           q_per_kv=qpk), dict(q=q, kv=kv, out=out, weights=w))
        ol.commit()
        _named(ol, "out").fill_(7.0)
        return ol
    ol = build("cuda")
    plan = Plan(ol.ops, 0)
    torch.cuda.synchronize()
    n0 = launch_count()
    with pytest.raises(VqaError):
        plan.run([0] * 6, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert launch_count() == n0, "a kernel was launched"
    assert bool((_named(ol, "out") == 7.0).all()), "the output was written"


# ============================================================================ 2. LayerNorm, embedding, pools
def _ln_params(g, n=3):
    out = {}
    for k in range(1, n + 1):
        out[f"g{k}"] = torch.rand(D, generator=g) + 0.5
        out[f"b{k}"] = torch.randn(D, generator=g) * 0.1
    return out


def ln_rows(g, n_random):
    """Rows of each kind: random, constant (zero variance: the output is beta), large common offset."""
    rows = [torch.randn(n_random, D, generator=g) * 2]
    rows.append(torch.tensor([0.0, 3.0, -1.5, 1024.0]).view(4, 1).expand(4, D))
    rows.append(torch.randn(4, D, generator=g) + torch.tensor([100.0, -300.0, 1e3, 1e4]).view(4, 1))
    kinds = ["random"] * n_random + ["constant"] * 4 + ["offset"] * 4
    return torch.cat(rows).contiguous(), kinds


def _offset_gate(x, gamma, beta, kinds):
    """Gate for the large-offset rows: 3x the error of torch's fp32 layer_norm on the same rows (and at least the fp32
    gate).  The kernel is not asked to beat fp32."""
    sel = torch.tensor([k == "offset" for k in kinds])
    ref = R.layernorm(x[sel], gamma, beta)
    err = float((F.layer_norm(x[sel], (D,), gamma, beta, 1e-5).double() - ref).abs().max() / ref.abs().max())
    return max(GATES["ln"], 3 * err), sel


@pytest.mark.parametrize("mode", [0, 1])
def test_layernorm_matches_fp64(mode):
    """mode 0 (token rows) and mode 1 (the projector's 7x7 grid rows + position embedding), with 0, 1 or 2 chained
    norms of the first output, every output form on each output."""
    g = torch.Generator().manual_seed(300 + mode)
    prm = _ln_params(g)
    pos = torch.randn(49, D, generator=g) * 0.5
    x, kinds = ln_rows(g, 41 if mode == 0 else 139)      # mode 1: 3 images of 49 pixels
    rows = x.shape[0]
    if mode == 1:
        assert rows == 3 * 49
        grid = torch.full((3, 8, 8, D), float("nan"))      # pad cells NaN: a read of one shows
        grid[:, :7, :7] = x.view(3, 7, 7, D)
        src = grid.reshape(3 * 64, D)
    else:
        src = x
    cases = [(ne, rnd) for ne in (0, 1, 2) for rnd in (0, 1, 2)]

    def build(device):
        W = _weights(device, pos=pos, **prm)
        ol = P.OpList(W, device)
        s = ol._buf("src", torch.float32, *src.shape)
        dt = lambda r: torch.float16 if r == 2 else torch.float32
        for c, (ne, rnd) in enumerate(cases):
            dst = ol._buf(f"y{c}", dt(rnd), rows, D)
            i = dict(rows=rows, D=D, ld_src=D, mode=mode, round_tf32=rnd, S=7 if mode else 0, Pg=8 if mode else 0,
                     RPIg=64 if mode else 0)
            p = dict(src=s, gamma=W.buf("g1"), beta=W.buf("b1"), dst=dst, pos=W.buf("pos") if mode else None)
            for k in range(2, 2 + ne):
                r = (rnd + k - 1) % 3
                i[f"rnd{k}"] = r
                p.update({f"gamma{k}": W.buf(f"g{k}"), f"beta{k}": W.buf(f"b{k}"), f"dst{k}": ol._buf(f"y{c}.{k}", dt(r), rows, D)})
            ol._op("layernorm", f"ln{c}", i, p, dict(eps=1e-5))
        ol.commit()
        _named(ol, "src").copy_(src)
        return ol
    ol, _ = _run(build)
    y = R.layernorm(x, prm["g1"], prm["b1"])
    if mode == 1:
        y = (y.view(3, 49, D) + pos.double()).view(rows, D)
    refs = {1: y, 2: R.layernorm(y, prm["g2"], prm["b2"]), 3: R.layernorm(y, prm["g3"], prm["b3"])}
    off_gate, off = _offset_gate(x, prm["g1"], prm["b1"], kinds)
    for c, (ne, rnd) in enumerate(cases):
        outs = [(1, f"y{c}", rnd)] + [(k, f"y{c}.{k}", (rnd + k - 1) % 3) for k in range(2, 2 + ne)]
        for k, name, r in outs:
            got = _named(ol, name).cpu()
            tag = f"layernorm mode{mode} extras{ne} out{k}"
            _check(tag, got[~off], refs[k][~off], LN_FORMS[r], GATES["ln"])
            if k == 1:
                _check(tag + " offset rows", got[off], refs[k][off], LN_FORMS[r], off_gate)
    const = torch.tensor([k == "constant" for k in kinds])
    if mode == 0:                                       # zero variance: beta, to the fp32 gate
        _check("layernorm constant rows = beta", _named(ol, "y0").cpu()[const], prm["b1"].double().expand(4, D), "f32",
               GATES["ln"])


V_EMB, MAXL = 50, 64
MASK_DTYPES = ["i64", "f32", "i32", "bool", "u8"]


def _mask_of(dtype, B, L, g):
    """A [B, L] mask of the given dtype: binary prefix / left-padded rows; f32 with fractional, negative and zero
    weights; u8 with weights 0..3."""
    base = torch.stack([key_mask(("prefix", "left", "holes", "all", "first")[b % 5], L) for b in range(B)])
    if dtype == "f32":
        w = torch.randn(B, L, generator=g)
        w[0] = torch.rand(L, generator=g)                   # fractional, positive
        return torch.where(base != 0, w, torch.zeros(()))
    if dtype == "u8":
        return (base * torch.randint(0, 4, (B, L), generator=g)).to(torch.uint8)
    return base.to({"i64": torch.int64, "i32": torch.int32, "bool": torch.bool}[dtype])


@pytest.mark.parametrize("mask_dtype", MASK_DTYPES)
@pytest.mark.parametrize("B,L", [(3, 9), (2, 20), (2, 64)])
def test_embedding_matches_fp64(B, L, mask_dtype):
    """embed_kernel and embed_ln_kernel (+ the first LayerNorm, + the mask's int32 key form and float pooling weights):
    ids 0 and V-1, lengths whose tok % L differ, every mask dtype."""
    g = torch.Generator().manual_seed(400 + 7 * L + MASK_DTYPES.index(mask_dtype))
    table = torch.randn(V_EMB, D, generator=g) * 16
    pe = torch.randn(MAXL, D, generator=g)
    prm = _ln_params(g, 1)
    ids = torch.randint(0, V_EMB, (B, L), generator=g)
    ids[0, 0], ids[-1, -1] = 0, V_EMB - 1
    ids[B // 2, L // 2] = V_EMB - 1
    mask = _mask_of(mask_dtype, B, L, g)
    code = LP.MASK_CODES[mask.dtype]
    rnd = MASK_DTYPES.index(mask_dtype) % 3

    def build(device):
        W = _weights(device, table=table, pe=pe, **prm)
        ol = P.OpList(W, device)
        xs = [ol._buf(f"x{c}", torch.float32, B * L, D) for c in range(2)]
        y = ol._buf("y", torch.float16 if rnd == 2 else torch.float32, B * L, D)
        mi, mf = ol._buf("mask_i32", torch.int32, B, L), ol._buf("mask_f32", torch.float32, B, L)
        ids_ref, tb, pb = P.ExtRef(P.EXT["ids"]), W.buf("table"), W.buf("pe")
        ol._op("embed", "fused", dict(B=B, L=L, D=D, V=V_EMB, round_tf32=rnd, mask_dtype=code),
               dict(ids=ids_ref, table=tb, pe=pb, dst=xs[0], gamma=W.buf("g1"), beta=W.buf("b1"), ln_dst=y,
                    mask_src=P.ExtRef(P.EXT["mask"]), mask_dst=mi, mask_dstf=mf), dict(eps=1e-5))
        ol._op("embed", "plain", dict(B=B, L=L, D=D, V=V_EMB), dict(ids=ids_ref, table=tb, pe=pb, dst=xs[1]))
        ol.commit()
        return ol
    ol, _ = _run(build, [None, ids, mask, None, None, None])
    want = R.embed(table, pe, ids).view(B * L, D)
    for c, kernel in enumerate(("embed_ln", "embed")):
        _check(f"{kernel} B{B} L{L}", _named(ol, f"x{c}").cpu(), want, "f32", GATES["ln"])
    _check(f"embed_ln LayerNorm B{B} L{L}", _named(ol, "y").cpu(), R.layernorm(want, prm["g1"], prm["b1"]), LN_FORMS[rnd],
           GATES["ln"])
    assert torch.equal(_named(ol, "mask_i32").cpu(), (mask != 0).to(torch.int32)), "key mask"
    assert torch.equal(_named(ol, "mask_f32").cpu(), mask.float()), "pooling weights"


POOL_ROWS = ("prefix", "fractional", "negative", "sum_0.3", "sum_0", "cancel", "heavy", "constant")


def pool_weights(L, g):
    """[len(POOL_ROWS), L] float pooling weights: a binary prefix, fractional weights, signed weights, two weights that
    sum to 0.3, all zero, +-0.5 that cancel, weights summing to more than one, and a binary row for constant features."""
    w = torch.zeros(len(POOL_ROWS), L)
    w[0, : max(1, L // 2)] = 1
    w[1] = torch.rand(L, generator=g)
    w[2] = torch.randn(L, generator=g)
    w[3, 0] = 0.1
    w[3, L - 1] += 0.2
    if L > 1:
        w[5, 0], w[5, 1] = 0.5, -0.5
    w[6] = torch.rand(L, generator=g) * 3
    w[7] = 1
    return w


@pytest.mark.parametrize("L", [1, 20, 64])
def test_pool_gate_ln_matches_fp64(L):
    """Phase 1 (masked mean pools + the gate GEMM's operand row in each form), phase 2 (sigmoid gate, mix, output
    norm) and phase 0 (pools, sum, output norm), denominators clamped to 1 as in the reference."""
    g = torch.Generator().manual_seed(500 + L)
    B = len(POOL_ROWS)
    w = pool_weights(L, g)
    xatt, text = torch.randn(B, L, D, generator=g), torch.randn(B, L, D, generator=g) * 0.5
    xatt[-1], text[-1] = 1.5, -0.25                        # constant features: zero-variance fused row in phase 0
    ap_in, tp_in, pre = torch.randn(B, D, generator=g), torch.randn(B, D, generator=g), torch.randn(B, D, generator=g) * 2
    prm = _ln_params(g, 1)
    cases = [(1, 0), (1, 1), (1, 2), (2, 1), (2, 2), (0, 1), (0, 2)]     # (phase, no_round)

    def build(device):
        W = _weights(device, **prm)
        ol = P.OpList(W, device)
        xa, tx, m = ol._buf("xatt", torch.float32, B * L, D), ol._buf("text", torch.float32, B * L, D), ol._buf("w", torch.float32, B, L)
        for c, (ph, nr) in enumerate(cases):
            ap, tp = ol._buf(f"ap{c}", torch.float32, B, D), ol._buf(f"tp{c}", torch.float32, B, D)
            fused = ol._buf(f"fused{c}", torch.float32, B, D)
            ncat = 2 * D if ph == 1 else D
            cat = ol._buf(f"cat{c}", torch.float16 if nr == 2 else torch.float32, B, ncat) if (ph == 1 or nr == 2) else None
            pr = ol._buf(f"pre{c}", torch.float32, B, D) if ph == 2 else None
            ol._op("pool_gate_ln", f"pool{c}", dict(B=B, L=L, D=D, use_gate=int(ph > 0), phase=ph, no_round=nr),
                   dict(xatt=xa, text=tx, mask=m, gamma=W.buf("g1"), beta=W.buf("b1"), fused=fused, att_pooled=ap,
                        txt_pooled=tp, cat=cat, pre=pr), dict(eps=1e-5))
        ol.commit()
        _named(ol, "xatt").copy_(xatt.view(B * L, D))
        _named(ol, "text").copy_(text.view(B * L, D))
        _named(ol, "w").copy_(w)
        for c, (ph, _) in enumerate(cases):
            if ph == 2:
                _named(ol, f"ap{c}").copy_(ap_in)
                _named(ol, f"tp{c}").copy_(tp_in)
                _named(ol, f"pre{c}").copy_(pre)
        return ol
    ol, _ = _run(build)
    ap, tp = R.masked_pool(xatt, w), R.masked_pool(text, w)
    for c, (ph, nr) in enumerate(cases):
        tag = f"pool_gate_ln L{L} phase{ph} no_round{nr}"
        if ph != 2:
            _check(tag + " att_pooled", _named(ol, f"ap{c}").cpu(), ap, "f32", GATES["ln"])
            _check(tag + " txt_pooled", _named(ol, f"tp{c}").cpu(), tp, "f32", GATES["ln"])
        if ph == 1:
            _check(tag + " cat", _named(ol, f"cat{c}").cpu(), torch.cat([ap, tp], -1), FORMS[nr], GATES["ln"])
            continue
        f = ap + tp if ph == 0 else R.gate_mix(ap_in, tp_in, pre)
        want = R.layernorm(f, prm["g1"], prm["b1"])
        _check(tag + " fused", _named(ol, f"fused{c}").cpu(), want, "f32", GATES["ln"])
        if nr == 2:
            _check(tag + " fused fp16", _named(ol, f"cat{c}").cpu(), want, "f16", GATES["ln"])
        if ph == 0:
            assert float((want[-1] - prm["b1"].double()).abs().max()) == 0.0    # the constant row's reference is beta


# ============================================================================ 3. whole question side, layer by layer
def question_mask(kinds, L, dtype, g):
    """[len(kinds), L] mask of ``dtype`` with one row per kind (MASK_KINDS); "f32" rows carry fractional and negative
    weights on their valid tokens, "u8" rows weights 1..3."""
    m = torch.stack([key_mask(k, L) for k in kinds])
    if dtype == "f32":
        w = torch.rand(m.shape, generator=g) * 1.5 + 0.05
        w[::3] *= -1                                        # some questions with negative weights
        return torch.where(m != 0, w, torch.zeros(()))
    if dtype == "u8":
        return (m * torch.randint(1, 4, m.shape, generator=g)).to(torch.uint8)
    return m.to({"i64": torch.int64, "i32": torch.int32, "bool": torch.bool}[dtype])


def _parity(prog, sd, ext, title, imgs=None, image_projected=None):
    if DRY:
        rep = LP.check_on_emulator(prog, sd, ext, imgs=imgs, title=title, image_projected=image_projected)
    else:
        from vqa_b200.runtime import Plan
        plan = Plan(prog.ops, 0)
        ptrs = [0 if t is None else t.data_ptr() for t in ext]
        stream = torch.cuda.current_stream().cuda_stream

        def runner(first, last):
            plan.run(ptrs, stream, first, last)
            torch.cuda.synchronize()
        rep = LP.Checker(prog, sd, ext, runner, imgs=imgs, kernel_name=plan.kernel_name, title=title,
                         image_projected=image_projected).run()
    print(rep.table())
    print("WORST", title, {c: f"{rep.worst(c):.2e}" for c in ("conv", "linear", "fp32")})
    assert not rep.failures(), rep.table()
    return rep


VALID = ("all", "prefix", "left", "first", "last", "holes")
# (max_question_length, L, questions, images, mask dtype, precision, fully masked question)
# T = questions * L: 5, 90, 42, 128, 120, 495 (3 tiles + 111), 250, 128, 129, 320, 68, 80
E2E = [
    (1, 1, 5, 1, "i64", "bf16", False),
    (9, 9, 10, 2, "f32", "bf16", False),
    (9, 7, 6, 3, "i32", "bf16", False),
    (32, 32, 4, 2, "bool", "bf16", False),
    (32, 20, 6, 3, "u8", "bf16", False),
    (33, 33, 15, 3, "i64", "bf16", False),
    (33, 25, 10, 2, "f32", "bf16", False),
    (64, 64, 2, 1, "u8", "bf16", False),
    (64, 43, 3, 3, "i32", "bf16", False),
    (64, 64, 5, 1, "bool", "bf16", False),
    (17, 17, 4, 2, "f32", "bf16", True),
    (20, 16, 5, 1, "u8", "tf32", True),
]


def _questions(maxL, L, B, dtype, empty, seed, vocab):
    g = torch.Generator().manual_seed(seed)
    kinds = [VALID[(b + seed) % len(VALID)] for b in range(B)]
    if empty:
        kinds[1] = "none"
    ids = torch.randint(0, vocab, (B, L), generator=g)
    ids[0, 0], ids[-1, -1] = 0, vocab - 1
    return ids, question_mask(kinds, L, dtype, g)


@pytest.mark.parametrize("case", E2E, ids=lambda c: f"maxlen{c[0]}-L{c[1]}-B{c[2]}-img{c[3]}-{c[4]}-{c[5]}"
                         + ("-empty" if c[6] else ""))
def test_question_side_layers_match_fp64(case):
    maxL, L, B, Bi, dtype, precision, empty = case
    ids, mask = _questions(maxL, L, B, dtype, empty, 31 * maxL + L, 10000)
    prog, sd, ext = LP.make_case(dict(max_question_length=maxL), B, L=L, n_images=Bi, precision=precision, device=DEV,
                                 seed=maxL + L, ids=ids, mask=mask)
    assert prog.Bi == Bi and prog.B * prog.L == B * L
    rep = _parity(prog, sd, ext, f"maxlen {maxL} L {L} B {B} images {Bi} {dtype} {precision}",
                  imgs=sorted({0, Bi - 1}))
    if empty:                                           # the fully masked question is NaN end to end, like the reference
        assert bool(torch.isnan(ext[P.EXT["logits"]][1]).all()) and not bool(torch.isnan(ext[P.EXT["logits"]][0]).any())
    assert any(r.module == "text.0" for r in rep.rows)


def test_cached_question_side_matches_fp64():
    """The cached path: the image side of 2 images (the cache entry: projector and K/V of every cross layer), then the
    question side of 5 questions per image against that K/V, each module of the question side against fp64."""
    maxL, L, B, Bi = 33, 30, 10, 2
    ids, mask = _questions(maxL, L, B, "f32", False, 7, 10000)
    prog, sd, ext = LP.make_case(dict(max_question_length=maxL), B, L=L, n_images=Bi, device=DEV, seed=3, ids=ids,
                                 mask=mask, side="question")
    img = P.Program(prog.W, prog.cfg, Bi, 1, "nchw_f32", P.MASK_NONE, n_images=Bi, device=DEV, side="image")
    img_ext = [ext[P.EXT["images"]]] + [None] * 5
    if DRY:
        E.Emulator(img).run(img_ext)
    else:
        from vqa_b200.runtime import Plan
        Plan(img.ops, 0).run([0 if t is None else t.data_ptr() for t in img_ext], torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
    for l in range(img.n_cross_layers):
        ext[P.EXT[f"kv{l}"]] = img.tensor(f"x.{l}.kv").reshape(-1)
    _parity(prog, sd, ext, "cached: 2 images x 5 questions",
            image_projected=img.tensor("image_projected").view(Bi, 49, D).clone())
