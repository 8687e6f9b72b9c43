"""Models whose embed_dim, head count or FFN width differ from the reference defaults, on the GPU.

1. Each new kernel instantiation against fp64 (tests/model_widths_support.py), with the gates test_gpu_question_side.py
   uses for the same output form: layernorm_kernel<D> in modes 0 and 1 with 0-2 chained norms and every output form;
   pool_gate_ln_kernel<D> in phases 0, 1 and 2; attn_mma_kernel (L <= 64) and attn_chunked_kernel (L = 1 .. 512) at
   head_dim 16 and 64: self-attention under the mask shapes of test_gpu_long_questions.py, cross-attention over 49
   image tokens with its weights; the launchers' refusals of other widths.
2. The question side layer by layer against fp64 (tests/layer_parity.py on a poisoned workspace) at each width of
   MW.CONFIGS, bf16 and tf32, at 20 and at 128 tokens.
3. The API at each width: logits against the fp32 oracle (bf16: the repo's logit gate; tf32: 1e-3) with return_aux,
   encode_images + answer, predict, load_vqa_model; VQAInference through a non-default checkpoint.
4. Whole plan and CUDA graph against the serial run at config c (embed_dim 512, head_dim 64, FFN 2048).

VQA_DRY=1 runs parts 1 and 2 on the CPU emulator instead of the library.
"""
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

from conftest import REPO  # noqa: E402
import attn_chunked_support  # noqa: E402,F401
import layer_parity as LP  # noqa: E402
import model_widths_support as MW  # noqa: E402
import question_ref as R  # noqa: E402
import test_gpu_long_questions as LQ  # noqa: E402
import test_gpu_question_side as QS  # noqa: E402
from vqa_b200 import program as P  # noqa: E402

sys.path.insert(0, REPO)
from oracle import vqa_oracle as O  # noqa: E402

DRY, DEV = QS.DRY, QS.DEV
GATES, FORMS, LN_FORMS, ROW_SUM_GATE = QS.GATES, QS.FORMS, QS.LN_FORMS, QS.ROW_SUM_GATE
LOGIT_REL_TOL = {"bf16": 2e-2, "tf32": 1e-3}     # test_gpu_model.py's bf16 logit gate; the tf32 mode's 1e-3
needs_gpu = pytest.mark.skipif(DRY, reason="runs the library itself (engine, graphs, streams)")
WIDTHS = [128, 192, 320, 512]                     # float4 rows (128, 512) and float2 rows (192, 320)


# ============================================================================ 1. kernels
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("D", WIDTHS)
def test_layernorm_matches_fp64(D, mode):
    g = torch.Generator().manual_seed(3000 + D + mode)
    prm = MW.ln_params(g, D)
    pos = torch.randn(49, D, generator=g) * 0.5
    x, kinds = MW.ln_rows(g, D, 41 if mode == 0 else 139)
    rows = x.shape[0]
    if mode == 1:
        grid = torch.full((3, 8, 8, D), float("nan"))      # pad cells NaN: a read of one shows
        grid[:, :7, :7] = x.view(3, 7, 7, D)
        src = grid.reshape(3 * 64, D)
    else:
        src = x
    cases = [(ne, rnd) for ne in (0, 1, 2) for rnd in (0, 1, 2)]

    def build(device):
        W = QS._weights(device, pos=pos, **prm)
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
        QS._named(ol, "src").copy_(src)
        return ol
    ol, _ = QS._run(build)
    y = R.layernorm(x, prm["g1"], prm["b1"])
    if mode == 1:
        y = (y.view(3, 49, D) + pos.double()).view(rows, D)
    refs = {1: y, 2: R.layernorm(y, prm["g2"], prm["b2"]), 3: R.layernorm(y, prm["g3"], prm["b3"])}
    off = torch.tensor([k == "offset" for k in kinds])
    ref_off = R.layernorm(x[off], prm["g1"], prm["b1"])
    torch_err = float((torch.nn.functional.layer_norm(x[off], (D,), prm["g1"], prm["b1"], 1e-5).double() - ref_off).abs().max()
                      / ref_off.abs().max())
    off_gate = max(GATES["ln"], 3 * torch_err)           # the large-offset rows: within 3x torch's fp32 layer_norm
    for c, (ne, rnd) in enumerate(cases):
        outs = [(1, f"y{c}", rnd)] + [(k, f"y{c}.{k}", (rnd + k - 1) % 3) for k in range(2, 2 + ne)]
        for k, name, r in outs:
            got = QS._named(ol, name).cpu()
            tag = f"layernorm D{D} mode{mode} extras{ne} out{k}"
            QS._check(tag, got[~off], refs[k][~off], LN_FORMS[r], GATES["ln"])
            if k == 1:
                QS._check(tag + " offset rows", got[off], refs[k][off], LN_FORMS[r], off_gate)
    if mode == 0:
        const = torch.tensor([k == "constant" for k in kinds])
        QS._check(f"layernorm D{D} constant rows = beta", QS._named(ol, "y0").cpu()[const],
                  prm["b1"].double().expand(4, D), "f32", GATES["ln"])


@pytest.mark.parametrize("L", [1, 20, 64])
@pytest.mark.parametrize("D", WIDTHS)
def test_pool_gate_ln_matches_fp64(D, L):
    g = torch.Generator().manual_seed(5000 + D + L)
    B = len(QS.POOL_ROWS)
    w = QS.pool_weights(L, g)
    xatt, text = torch.randn(B, L, D, generator=g), torch.randn(B, L, D, generator=g) * 0.5
    xatt[-1], text[-1] = 1.5, -0.25
    ap_in, tp_in, pre = torch.randn(B, D, generator=g), torch.randn(B, D, generator=g), torch.randn(B, D, generator=g) * 2
    prm = MW.ln_params(g, D, 1)
    cases = [(1, 0), (1, 1), (1, 2), (2, 1), (2, 2), (0, 1), (0, 2)]     # (phase, no_round)

    def build(device):
        W = QS._weights(device, **prm)
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
        QS._named(ol, "xatt").copy_(xatt.view(B * L, D))
        QS._named(ol, "text").copy_(text.view(B * L, D))
        QS._named(ol, "w").copy_(w)
        for c, (ph, _) in enumerate(cases):
            if ph == 2:
                QS._named(ol, f"ap{c}").copy_(ap_in)
                QS._named(ol, f"tp{c}").copy_(tp_in)
                QS._named(ol, f"pre{c}").copy_(pre)
        return ol
    ol, _ = QS._run(build)
    ap, tp = R.masked_pool(xatt, w), R.masked_pool(text, w)
    for c, (ph, nr) in enumerate(cases):
        tag = f"pool_gate_ln D{D} L{L} phase{ph} no_round{nr}"
        if ph != 2:
            QS._check(tag + " att_pooled", QS._named(ol, f"ap{c}").cpu(), ap, "f32", GATES["ln"])
            QS._check(tag + " txt_pooled", QS._named(ol, f"tp{c}").cpu(), tp, "f32", GATES["ln"])
        if ph == 1:
            QS._check(tag + " cat", QS._named(ol, f"cat{c}").cpu(), torch.cat([ap, tp], -1), FORMS[nr], GATES["ln"])
            continue
        f = ap + tp if ph == 0 else R.gate_mix(ap_in, tp_in, pre)
        want = R.layernorm(f, prm["g1"], prm["b1"])
        QS._check(tag + " fused", QS._named(ol, f"fused{c}").cpu(), want, "f32", GATES["ln"])
        if nr == 2:
            QS._check(tag + " fused fp16", QS._named(ol, f"cat{c}").cpu(), want, "f16", GATES["ln"])


# (embed_dim, heads): head_dim 16 and 64, and 64 at the widest embedding
HEADS = [(256, 16), (256, 4), (512, 8)]
ATTN_LENGTHS = [1, 20, 64, 65, 128, 512]


def _attn(ol, kind, name, D, H, B, L, T, q, kv, out, nr, mask=None, weights=None, qpk=1, self_attn=False):
    i = dict(B=B, L=L, H=H, hd=D // H, no_round=nr)
    if kind == "self_attn":
        ol._op("self_attn", name, dict(i, ld_qkv=3 * D), dict(qkv=q, mask=mask, out=out))
        return
    i.update(T=T, q_per_kv=qpk)
    i.update(dict(ld_q=3 * D, ld_kv=3 * D, k_off=D, v_off=2 * D) if self_attn else dict(ld_q=D, ld_kv=2 * D, k_off=0, v_off=D))
    p = dict(q=q, kv=kv, out=out, weights=weights)
    if kind == "attn_chunked":
        p["mask"] = mask
    ol._op(kind, name, i, p)


@pytest.mark.parametrize("L", ATTN_LENGTHS)
@pytest.mark.parametrize("D,H", HEADS, ids=lambda v: str(v))
def test_self_attention_matches_fp64(D, H, L):
    """Every mask shape of test_gpu_long_questions.py (a fully masked row last), each output form at unit and x8 input
    scale, through attn_chunked_kernel and, for L <= 64, attn_mma_kernel."""
    kinds = LQ.MASK_KINDS
    B = len(kinds)
    mask = torch.stack([LQ.key_mask(k, L) for k in kinds])
    ops = ["attn_chunked"] + (["self_attn"] if L <= 64 else [])
    cases = [(op, nr, sc) for op in ops for nr in (0, 1, 2) for sc in (1.0, 8.0)]
    g = torch.Generator().manual_seed(7000 + D + H + L)
    inputs = [torch.randn(B * L, 3 * D, generator=g) * sc for _, _, sc in cases]

    def build(device):
        ol = P.OpList(QS._weights(device), device)
        m = ol._buf("mask", torch.int32, B, L)
        for c, (op, nr, _) in enumerate(cases):
            qkv = ol._buf(f"qkv{c}", torch.float32, B * L, 3 * D)
            out = ol._buf(f"out{c}", torch.float16 if nr == 2 else torch.float32, B * L, D)
            _attn(ol, op, f"attn{c}", D, H, B, L, L, qkv, qkv, out, nr, mask=m, self_attn=True)
        ol.commit()
        QS._named(ol, "mask").copy_(mask)
        for c, x in enumerate(inputs):
            QS._named(ol, f"qkv{c}").copy_(x)
        return ol
    ol, _ = QS._run(build)
    for c, (op, nr, sc) in enumerate(cases):
        x = inputs[c].view(B, L, 3 * D)
        want, _ = MW.attention(x[..., :D], x[..., D:2 * D], x[..., 2 * D:], H, mask)
        assert bool(torch.isnan(want[-1]).all()) and not bool(torch.isnan(want[:-1]).any())
        got = QS._named(ol, f"out{c}").view(B, L, D)
        QS._check(f"{op} hd{D // H} D{D} L{L} x{sc:g}", got, want, FORMS[nr], GATES["attn"] if sc == 1 else LQ.GATE_X8)


@pytest.mark.parametrize("L", ATTN_LENGTHS)
@pytest.mark.parametrize("D,H", HEADS, ids=lambda v: str(v))
def test_cross_attention_matches_fp64(D, H, L):
    """49 image tokens, 2 images, 1 / 2 / 5 questions per image, every output form, weights and their row sums."""
    T, Bi = 49, 2
    ops = ["attn_chunked"] + (["cross_attn"] if L <= 64 else [])
    cases = [(op, qpk, nr) for op in ops for qpk, nr in ((1, 0), (2, 1), (5, 2))]
    g = torch.Generator().manual_seed(8000 + D + H + L)
    data = [(torch.randn(Bi * qpk * L, D, generator=g), torch.randn(Bi * T, 2 * D, generator=g)) for _, qpk, _ in cases]

    def build(device):
        ol = P.OpList(QS._weights(device), device)
        for c, (op, qpk, nr) in enumerate(cases):
            B = Bi * qpk
            q = ol._buf(f"q{c}", torch.float32, B * L, D)
            kv = ol._buf(f"kv{c}", torch.float32, Bi * T, 2 * D)
            out = ol._buf(f"out{c}", torch.float16 if nr == 2 else torch.float32, B * L, D)
            w = ol._buf(f"w{c}", torch.float32, B, H, L, T)
            _attn(ol, op, f"x{c}", D, H, B, L, T, q, kv, out, nr, weights=w, qpk=qpk)
        ol.commit()
        for c, (q, kv) in enumerate(data):
            QS._named(ol, f"q{c}").copy_(q)
            QS._named(ol, f"kv{c}").copy_(kv)
        return ol
    ol, _ = QS._run(build)
    for c, (op, qpk, nr) in enumerate(cases):
        B = Bi * qpk
        q, kv = data[c]
        kv = kv.view(Bi, T, 2 * D)
        want, wref = MW.attention(q.view(B, L, D), kv[..., :D], kv[..., D:], H, None, qpk)
        tag = f"{op} cross hd{D // H} D{D} L{L} x{qpk}"
        QS._check(tag, QS._named(ol, f"out{c}").view(B, L, D), want, FORMS[nr], GATES["attn"])
        w = QS._named(ol, f"w{c}").cpu()
        QS._check(tag + " weights", w, wref, "f32", GATES["attn"])
        rows = (w.double().sum(dim=-1) - 1).abs().max().item()
        assert rows <= ROW_SUM_GATE, f"{tag}: a weight row sums to 1 +- {rows:.2e}"


@pytest.mark.skipif(DRY, reason="the launchers' refusals are the library's; the emulator does not model them")
@pytest.mark.parametrize("kind", ["self_hd8", "cross_hd128", "chunked_hd8", "chunked_hd128", "layernorm_D160",
                                  "layernorm_D576", "pool_D96", "pool_D576"])
def test_launchers_refuse_other_widths(kind):
    """Head widths other than 16 / 32 / 64 and LayerNorm / fusion-tail widths outside 128 .. 512 in steps of 64 are
    errors, and nothing is launched."""
    from vqa_b200.runtime import Plan, VqaError, launch_count
    op, n = kind.split("_")
    val = int(n[2:] if n.startswith("hd") else n[1:])
    B, L = 2, 20
    W = QS._weights("cuda", g=torch.ones(576), b=torch.zeros(576))
    ol = P.OpList(W, "cuda")
    if op in ("self", "cross", "chunked"):
        D, H = 256, 256 // val
        q = ol._buf("q", torch.float32, B * L, 3 * D)
        kv = ol._buf("kv", torch.float32, B * 49, 2 * D)
        out = ol._buf("out", torch.float32, B * L, D)
        kind_ = {"self": "self_attn", "cross": "cross_attn", "chunked": "attn_chunked"}[op]
        _attn(ol, kind_, "x", D, H, B, L, 49, q, kv if op != "self" else q, out, 1, self_attn=op == "self")
    elif op == "layernorm":
        out = ol._buf("out", torch.float32, 4, val)
        ol._op("layernorm", "x", dict(rows=4, D=val, ld_src=val, mode=0, round_tf32=0),
               dict(src=ol._buf("src", torch.float32, 4, val), gamma=W.buf("g"), beta=W.buf("b"), dst=out), dict(eps=1e-5))
    else:
        out = ol._buf("out", torch.float32, B, val)
        ol._op("pool_gate_ln", "x", dict(B=B, L=L, D=val, use_gate=0, phase=0, no_round=1),
               dict(xatt=ol._buf("xa", torch.float32, B * L, val), text=ol._buf("tx", torch.float32, B * L, val),
                    gamma=W.buf("g"), beta=W.buf("b"), fused=out, att_pooled=ol._buf("ap", torch.float32, B, val),
                    txt_pooled=ol._buf("tp", torch.float32, B, val)), dict(eps=1e-5))
    ol.commit()
    QS._named(ol, "out").fill_(7.0)
    plan = Plan(ol.ops, 0)
    torch.cuda.synchronize()
    n0 = launch_count()
    with pytest.raises(VqaError):
        plan.run([0] * 6, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert launch_count() == n0, "a kernel was launched"
    assert bool((QS._named(ol, "out") == 7.0).all()), "the output was written"


# ============================================================================ 2. question side, layer by layer
# (config, max_question_length, L, questions, images, mask dtype, precision, fully masked question)
E2E = [(name, 20, 20, 6, 3, "i64", "bf16", True) for name in MW.CONFIGS]
E2E += [(name, 20, 17, 4, 2, "f32", "tf32", False) for name in MW.CONFIGS]
E2E += [("a", 128, 128, 4, 2, "bool", "bf16", True), ("b", 128, 100, 3, 3, "i64", "bf16", False),
        ("c", 128, 128, 3, 1, "f32", "tf32", True), ("e", 65, 65, 5, 5, "i64", "bf16", False)]


@pytest.mark.parametrize("case", E2E, ids=lambda c: f"{c[0]}-maxlen{c[1]}-L{c[2]}-B{c[3]}-img{c[4]}-{c[5]}-{c[6]}"
                         + ("-empty" if c[7] else ""))
def test_question_side_layers_match_fp64(case):
    name, maxL, L, B, Bi, dtype, precision, empty = case
    ids, mask = QS._questions(maxL, L, B, dtype, empty, 17 * maxL + L + ord(name), 10000)
    prog, sd, ext = LP.make_case(MW.ctor(name, max_question_length=maxL), B, L=L, n_images=Bi, precision=precision,
                                 device=DEV, seed=maxL + L + ord(name), ids=ids, mask=mask)
    if not DRY:
        LP.poison(prog)
    rep = QS._parity(prog, sd, ext, f"config {name} {MW.CONFIGS[name]} L {L} B {B} images {Bi} {dtype} {precision}",
                     imgs=sorted({0, Bi - 1}))
    if empty:
        assert bool(torch.isnan(ext[P.EXT["logits"]][1]).all()) and not bool(torch.isnan(ext[P.EXT["logits"]][0]).any())
    assert any(r.module == "text.3" for r in rep.rows) and any(r.module == "x.1" for r in rep.rows)


# ============================================================================ 3. API
def _model(name, precision="bf16", maxL=20):
    from vqa_b200.model import VQAModel
    from vqa_b200.synth import randomise_state
    torch.manual_seed(0)
    model = VQAModel(**MW.ctor(name, max_question_length=maxL), precision=precision).eval()
    sd = randomise_state(model.state_dict(), 1)
    model.load_state_dict(sd, strict=True)
    return model.cuda(), sd


@needs_gpu
@pytest.mark.parametrize("precision", ["bf16", "tf32"])
@pytest.mark.parametrize("name", list(MW.CONFIGS))
def test_model_api_at_each_width(name, precision, tmp_path):
    from vqa_b200.model import load_vqa_model
    from vqa_b200.synth import synth_batch
    D, H, F = MW.CONFIGS[name]
    model, sd = _model(name, precision)
    _, img, ids, mask = synth_batch(9, 31 + ord(name))
    img, ids, mask = img.cuda(), ids.cuda(), mask.cuda()
    with torch.no_grad():
        logits, aux = model(img, ids, mask, return_aux=True)
        cached = model.answer(model.encode_images(img), ids, mask)
    assert torch.equal(cached, logits), "encode_images + answer differs from forward"
    assert [tuple(w.shape) for w in aux["cross_attention_weights"]] == [(9, H, 20, 49)] * 2
    want, waux = O.vqa_forward(sd, img.cpu(), ids.cpu(), mask.cpu(), num_heads=H, return_aux=True)
    err = float((logits.cpu() - want).abs().max() / want.abs().max())
    print(f"WORST config {name} {precision} logits rel err {err:.3e}")
    assert err <= LOGIT_REL_TOL[precision]
    for got, ref in zip(aux["cross_attention_weights"], waux["cross_attention_weights"]):
        werr = float((got.cpu().double() - ref.double()).abs().max())
        assert werr <= (5e-2 if precision == "bf16" else 1e-3), f"cross-attention weights differ by {werr:.2e}"
    idx, probs = model.predict(img, ids, mask, top_k=5)
    ref_p, ref_i = torch.softmax(logits, dim=1).topk(5, dim=1)
    assert torch.equal(idx, ref_i) and torch.allclose(probs, ref_p, rtol=2e-5, atol=1e-7)
    path = str(tmp_path / "ckpt.pt")
    torch.save({"config": model.config, "model_state_dict": model.state_dict(), "epoch": 1}, path)
    again = load_vqa_model(path, "cuda").eval()
    again.precision = precision
    with torch.no_grad():
        assert torch.equal(again(img, ids, mask)[0], logits), "a reloaded checkpoint answers differently"


@needs_gpu
def test_inference_api_with_a_non_default_checkpoint(tmp_path):
    from PIL import Image
    from vqa_b200 import VQAInference
    from vqa_b200.synth import synth_images_u8
    from vqa_b200.text import Tokenizer
    model, sd = _model("c")
    ckpt = tmp_path / "model.pt"
    torch.save({"config": model.config, "model_state_dict": sd}, ckpt)
    words = [f"w{i}" for i in range(40)]
    tok = Tokenizer(max_length=20)
    tok.build_vocab([" ".join(words)], min_freq=1)
    tok.save(str(tmp_path / "question_vocab.json"))
    qs = ["w1 w2 w3", " ".join(words[:15]), "w7"]
    imgs = [Image.fromarray(synth_images_u8(1, 70 + i)[0].numpy(), "RGB") for i in range(3)]
    inf = VQAInference(checkpoint_path=str(ckpt), question_vocab_path=str(tmp_path / "question_vocab.json"))
    inf.load()
    assert inf.model.config["embed_dim"] == 512 and inf.model.config["num_attention_heads"] == 8
    single = [inf.predict(im, q, top_k=3) for im, q in zip(imgs, qs)]
    batch = inf.predict_batch(imgs, qs, top_k=3)
    for s, b in zip(single, batch):
        assert [a["index"] for a in s["answers"]] == [a["index"] for a in b["answers"]]
    ids, mask = inf.preprocess_question(qs[1])
    u8 = inf.preprocess_image_u8(imgs[1]).cpu()
    want, _ = O.vqa_forward(sd, O.preprocess_u8(u8.unsqueeze(0)), ids, mask, num_heads=8)
    assert single[1]["answers"][0]["index"] == int(want.argmax(1))


# ============================================================================ 4. schedule
@needs_gpu
def test_whole_plan_and_graph_match_serial_at_config_c():
    import test_gpu_schedule as GS
    ids, mask = QS._questions(20, 20, 6, "i64", True, 9, 10000)
    prog = GS._case("config c: embed_dim 512, head_dim 64, FFN 2048, fully masked question",
                    ctor=MW.ctor("c"), B=6, L=20, ids=ids, mask=mask, masked_rows=(1,))[0]
    assert prog.cfg["embed_dim"] == 512
