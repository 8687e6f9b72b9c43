"""Questions of 65 to 512 tokens: attn_chunked_kernel (VQA_OP_ATTN_CHUNKED, keys streamed in chunks of 64) against fp64,
the whole question side layer by layer, the public API and the concurrent schedule at such lengths.

1. The kernel against softmax(QK^T/sqrt(32) + mask) V in fp64 (tests/question_ref.py) on its own fp32 inputs: self-
   attention at lengths on both sides of every chunk and query-block boundary up to 512 (L <= 64 too: the kernel is
   correct there, the program just does not pick it), the seven mask shapes of test_gpu_question_side.py plus keys valid
   only in the last chunk, only in the first chunk and one valid key per chunk (a row with no valid key in some chunk
   must stay finite; a fully masked row is NaN at exactly the reference's elements), every output form at input scale 1
   and x8; cross-attention over 49 image tokens with 1, 2 and 5 questions per image, weights and their row sums; the
   launcher's refusals.  Gates: GATES of test_gpu_question_side.py, except at input scale x8 (below).
2. The whole question side through tests/layer_parity.py at max_question_length 65, 128 and 512 (token counts over
   several 128-row tiles, i64 / f32 / bool masks, bf16 and tf32, a fully masked question, 1 image x 16 questions of 128
   tokens, the cached path).
3. The API at max_question_length 128 and 512: logits against the fp32 oracle, predict, encode_images + answer, batch
   invariance, CUDA graphs, the pipelined path, attention maps, and VQAInference with a 128-token vocabulary.
4. The two-lane schedule at L = 128: whole-plan runs and graph replays on a poisoned workspace equal the serial run.

VQA_DRY=1 runs parts 1 and 2 on the CPU emulator instead of the library; parts 3 and 4 need the GPU.

Worst error measured on B200 (1000 W power limit), over every length, by check and output form (fp32 / tf32 / fp16):

    self-attention, randn inputs       2.00e-6 / 7.19e-7 / 6.24e-7   (gate GATES["attn"] = 5e-6)
    self-attention, inputs x8          2.86e-5 / 1.97e-5 / 2.72e-5   (L = 257, 127; at L <= 64 1.42e-5 like attn_mma_kernel)
    cross-attention output             1.75e-6 / 5.80e-7 / 6.52e-7   weights 1.70e-6, row sums 1 +- 2.5e-7

The x8 error grows with the number of keys (a larger largest score among more keys, its fp32 rounding amplified by the
near one-hot softmax), so x8 has its own gate at 2.8x the worst; GATES["attn_x8"] (4e-5) would leave 1.4x.  End to end
(layer_parity.GATES classes), worst over the cases of part 2: linear 1.76e-3 (bf16) / 1.17e-5 (tf32), fp32 4.60e-7;
logits of part 3 within 2.4e-3 of the fp32 oracle.
"""
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

from conftest import REPO  # noqa: E402
import attn_chunked_support  # noqa: E402,F401  (emulator op and access table of the new kind)
import layer_parity as LP  # noqa: E402
import question_ref as R  # noqa: E402
import test_gpu_question_side as QS  # noqa: E402
from vqa_b200 import program as P  # noqa: E402

sys.path.insert(0, REPO)
from oracle import vqa_oracle as O  # noqa: E402

DRY, DEV = QS.DRY, QS.DEV
H, D = QS.H, QS.D
GATES, FORMS, ROW_SUM_GATE = QS.GATES, QS.FORMS, QS.ROW_SUM_GATE
GATE_X8 = 8e-5                # 2.86e-5 measured (self-attention, inputs x8, L = 257)
LOGIT_REL_TOL = 2e-2          # test_gpu_model.py: bf16 logits within 2e-2 max-abs relative error of the fp32 oracle
needs_gpu = pytest.mark.skipif(DRY, reason="runs the library itself (engine, graphs, streams)")


# ============================================================================ 1. the kernel
SELF_LENGTHS = [1, 33, 64, 65, 96, 127, 128, 129, 191, 192, 193, 255, 256, 257, 383, 511, 512]
CHUNK_KINDS = ("last_chunk", "first_chunk", "per_chunk")
MASK_KINDS = QS.MASK_KINDS[:-1] + CHUNK_KINDS + ("none",)


def key_mask(kind, L):
    if kind not in CHUNK_KINDS:
        return QS.key_mask(kind, L)
    m = torch.zeros(L, dtype=torch.int32)
    if kind == "last_chunk":                     # every earlier chunk fully masked
        m[(L - 1) // 64 * 64:] = 1
    elif kind == "first_chunk":                  # every later chunk fully masked
        m[:64] = 1
    else:                                        # one valid key per chunk, at a different place in each
        for c in range(0, L, 64):
            m[c + (c // 64 * 23) % min(64, L - c)] = 1
    return m


def _attn_op(ol, name, B, L, T, q, kv, out, nr, mask=None, weights=None, qpk=1, self_attn=False):
    i = dict(B=B, L=L, H=H, hd=32, T=T, no_round=nr, q_per_kv=qpk)
    i.update(dict(ld_q=3 * D, ld_kv=3 * D, k_off=D, v_off=2 * D) if self_attn else dict(ld_q=D, ld_kv=2 * D, k_off=0, v_off=D))
    ol._op("attn_chunked", name, i, dict(q=q, kv=kv, mask=mask, out=out, weights=weights))


@pytest.mark.parametrize("L", SELF_LENGTHS)
def test_chunked_self_attention_matches_fp64(L):
    """One pair per mask shape (10 pairs), each output form at unit and x8 input scale."""
    B = len(MASK_KINDS)
    mask = torch.stack([key_mask(k, L) for k in MASK_KINDS])
    cases = [(nr, sc) for nr in (0, 1, 2) for sc in (1.0, 8.0)]
    g = torch.Generator().manual_seed(1000 + L)
    inputs = [torch.randn(B * L, 3 * D, generator=g) * sc for _, sc in cases]

    def build(device):
        ol = P.OpList(QS._weights(device), device)
        m = ol._buf("mask", torch.int32, B, L)
        for c, (nr, _) in enumerate(cases):
            qkv = ol._buf(f"qkv{c}", torch.float32, B * L, 3 * D)
            out = ol._buf(f"out{c}", torch.float16 if nr == 2 else torch.float32, B * L, D)
            _attn_op(ol, f"attn{c}", B, L, L, qkv, qkv, out, nr, mask=m, self_attn=True)
        ol.commit()
        QS._named(ol, "mask").copy_(mask)
        for c, x in enumerate(inputs):
            QS._named(ol, f"qkv{c}").copy_(x)
        return ol
    ol, _ = QS._run(build)
    for c, (nr, sc) in enumerate(cases):
        x = inputs[c].view(B, L, 3 * D)
        want, _ = R.attention(x[..., :D], x[..., D:2 * D], x[..., 2 * D:], H, mask)
        got = QS._named(ol, f"out{c}").view(B, L, D)
        assert bool(torch.isnan(want[-1]).all()) and not bool(torch.isnan(want[:-1]).any())
        QS._check(f"chunked self L{L} x{sc:g}", got, want, FORMS[nr], GATES["attn"] if sc == 1 else GATE_X8)


@pytest.mark.parametrize("L", [65, 128, 512])
def test_chunked_cross_attention_matches_fp64(L):
    """49 image tokens, 2 images, 1 / 2 / 5 questions per image, every output form, weights and their row sums."""
    T, Bi = 49, 2
    cases = [(qpk, nr) for qpk, nr in ((1, 0), (2, 1), (5, 2))]
    g = torch.Generator().manual_seed(2000 + L)
    data = [(torch.randn(Bi * qpk * L, D, generator=g), torch.randn(Bi * T, 2 * D, generator=g)) for qpk, _ in cases]

    def build(device):
        ol = P.OpList(QS._weights(device), device)
        for c, (qpk, nr) in enumerate(cases):
            B = Bi * qpk
            q = ol._buf(f"q{c}", torch.float32, B * L, D)
            kv = ol._buf(f"kv{c}", torch.float32, Bi * T, 2 * D)
            out = ol._buf(f"out{c}", torch.float16 if nr == 2 else torch.float32, B * L, D)
            w = ol._buf(f"w{c}", torch.float32, B, H, L, T)
            _attn_op(ol, f"x{c}", B, L, T, q, kv, out, nr, weights=w, qpk=qpk)
        ol.commit()
        for c, (q, kv) in enumerate(data):
            QS._named(ol, f"q{c}").copy_(q)
            QS._named(ol, f"kv{c}").copy_(kv)
        return ol
    ol, _ = QS._run(build)
    for c, (qpk, nr) in enumerate(cases):
        B = Bi * qpk
        q, kv = data[c]
        kv = kv.view(Bi, T, 2 * D)
        want, wref = R.attention(q.view(B, L, D), kv[..., :D], kv[..., D:], H, None, qpk)
        tag = f"chunked cross L{L} x{qpk}"
        QS._check(tag, QS._named(ol, f"out{c}").view(B, L, D), want, FORMS[nr], GATES["attn"])
        w = QS._named(ol, f"w{c}").cpu()
        QS._check(tag + " weights", w, wref, "f32", GATES["attn"])
        rows = (w.double().sum(dim=-1) - 1).abs().max().item()
        print(f"WORST {tag} row sums {rows:.3e}")
        assert rows <= ROW_SUM_GATE, f"{tag}: a weight row sums to 1 +- {rows:.2e}"


@pytest.mark.skipif(DRY, reason="the launcher's refusals are the library's; the emulator does not model them")
@pytest.mark.parametrize("kind", ["L513", "T513", "weights_T65", "batch_not_multiple"])
def test_chunked_launcher_refuses_out_of_envelope(kind):
    """513 queries, 513 keys, weights over more than one chunk and a batch that is not a multiple of q_per_kv are
    errors, and nothing is launched."""
    from vqa_b200.runtime import Plan, VqaError, launch_count
    B, L, T, qpk, wts = {"L513": (2, 513, 49, 1, False), "T513": (2, 20, 513, 1, False),
                         "weights_T65": (2, 20, 65, 1, True), "batch_not_multiple": (5, 100, 49, 2, False)}[kind]
    ol = P.OpList(QS._weights("cuda"), "cuda")
    q = ol._buf("q", torch.float32, B * L, D)
    kv = ol._buf("kv", torch.float32, B * T, 2 * D)
    out = ol._buf("out", torch.float32, B * L, D)
    w = ol._buf("w", torch.float32, B, H, L, T) if wts else None
    _attn_op(ol, "x", B, L, T, q, kv, out, 1, weights=w, qpk=qpk)
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


# ============================================================================ 2. whole question side
# (max_question_length, L, questions, images, mask dtype, precision, fully masked question); T = 325, 512, 700, 1536, 600
E2E = [
    (65, 65, 5, 1, "i64", "bf16", True),
    (128, 128, 4, 2, "f32", "bf16", False),
    (128, 100, 7, 7, "bool", "tf32", True),
    (512, 512, 3, 3, "i64", "bf16", True),
    (512, 300, 2, 1, "f32", "tf32", False),
    (128, 128, 16, 1, "i64", "bf16", False),          # 1 image x 16 questions of 128 tokens
]


@pytest.mark.parametrize("case", E2E, ids=lambda c: f"maxlen{c[0]}-L{c[1]}-B{c[2]}-img{c[3]}-{c[4]}-{c[5]}"
                         + ("-empty" if c[6] else ""))
def test_long_question_side_layers_match_fp64(case):
    maxL, L, B, Bi, dtype, precision, empty = case
    ids, mask = QS._questions(maxL, L, B, dtype, empty, 31 * maxL + L, 10000)
    prog, sd, ext = LP.make_case(dict(max_question_length=maxL), B, L=L, n_images=Bi, precision=precision, device=DEV,
                                 seed=maxL + L, ids=ids, mask=mask)
    assert prog.Bi == Bi and sum(op.kind == "attn_chunked" for op in prog.ops) == 6
    if not DRY:
        LP.poison(prog)
    rep = QS._parity(prog, sd, ext, f"maxlen {maxL} L {L} B {B} images {Bi} {dtype} {precision}", imgs=sorted({0, Bi - 1}))
    if empty:
        assert bool(torch.isnan(ext[P.EXT["logits"]][1]).all()) and not bool(torch.isnan(ext[P.EXT["logits"]][0]).any())
    assert any(r.module == "text.3" for r in rep.rows)


def test_long_cached_question_side_matches_fp64():
    """Image side of 2 images, then 6 questions of 128 tokens per image against the cached K/V."""
    maxL, L, B, Bi = 128, 128, 12, 2
    ids, mask = QS._questions(maxL, L, B, "i64", True, 11, 10000)
    prog, sd, ext = LP.make_case(dict(max_question_length=maxL), B, L=L, n_images=Bi, device=DEV, seed=3, ids=ids,
                                 mask=mask, side="question")
    img = P.Program(prog.W, prog.cfg, Bi, 1, "nchw_f32", P.MASK_NONE, n_images=Bi, device=DEV, side="image")
    img_ext = [ext[P.EXT["images"]]] + [None] * 5
    QS._run(lambda device: img, img_ext)
    for l in range(img.n_cross_layers):
        ext[P.EXT[f"kv{l}"]] = img.tensor(f"x.{l}.kv").reshape(-1)
    QS._parity(prog, sd, ext, "cached: 2 images x 6 questions of 128 tokens",
               image_projected=img.tensor("image_projected").view(Bi, 49, D).clone())


# ============================================================================ 3. API
def _model(maxL):
    from vqa_b200.model import VQAModel
    from vqa_b200.synth import randomise_state
    torch.manual_seed(0)
    model = VQAModel(max_question_length=maxL).eval()
    sd = randomise_state(model.state_dict(), 1)
    model.load_state_dict(sd, strict=True)
    return model.cuda(), sd


def _inputs(B, L, seed):
    from vqa_b200.synth import synth_batch
    _, img, _, _ = synth_batch(B, seed)
    ids, mask = QS._questions(L, L, B, "i64", False, seed, 10000)
    return img, ids, mask


@needs_gpu
@pytest.mark.parametrize("maxL", [128, 512])
def test_model_api_at_long_questions(maxL):
    model, sd = _model(maxL)
    img, ids, mask = _inputs(33, maxL, 7 + maxL)
    with torch.no_grad():
        full, _ = model(img.cuda(), ids.cuda(), mask.cuda())
        for b in (1, 7):                         # batch invariance, bit for bit
            part, _ = model(img[:b].cuda(), ids[:b].cuda(), mask[:b].cuda())
            assert torch.equal(part, full[:b]), f"batch {b}"
        cached = model.answer(model.encode_images(img[:7].cuda()), ids[:7].cuda(), mask[:7].cuda())
    assert torch.equal(cached, full[:7]), "encode_images + answer differs from forward"
    want, _ = O.vqa_forward(sd, img[:7], ids[:7], mask[:7])
    err = float((full[:7].cpu() - want).abs().max() / want.abs().max())
    print(f"WORST maxlen {maxL} logits rel err {err:.3e}")
    assert err <= LOGIT_REL_TOL
    idx, _ = model.predict(img[:7].cuda(), ids[:7].cuda(), mask[:7].cuda(), top_k=5)
    assert torch.equal(idx, full[:7].topk(5, dim=1).indices)
    maps = model.get_attention_maps(img[:3].cuda(), ids[:3].cuda(), mask[:3].cuda())
    assert tuple(maps["cross_attention_spatial"].shape) == (3, maxL, 7, 7)
    assert [tuple(w.shape) for w in maps["cross_attention"]] == [(3, H, maxL, 49)] * 2      # one per cross layer


@needs_gpu
def test_inference_api_with_a_128_token_vocabulary(tmp_path):
    from PIL import Image
    from vqa_b200 import VQAInference
    from vqa_b200.synth import synth_batch, synth_images_u8
    from vqa_b200.text import Tokenizer
    model, sd = _model(128)
    ckpt = tmp_path / "model.pt"
    torch.save({"config": model.config, "model_state_dict": sd}, ckpt)
    words = [f"w{i}" for i in range(60)]
    tok = Tokenizer(max_length=128)
    tok.build_vocab([" ".join(words)], min_freq=1)
    tok.save(str(tmp_path / "question_vocab.json"))
    long_q = " ".join(words[i % 60] for i in range(110))        # 110 words: longer than the engine's former 64 tokens
    qs = [long_q, "w1 w2 w3", " ".join(words[:90])]
    imgs = [Image.fromarray(synth_images_u8(1, 40 + i)[0].numpy(), "RGB") for i in range(3)]
    results = {}
    for cache in (0, 4):
        inf = VQAInference(checkpoint_path=str(ckpt), question_vocab_path=str(tmp_path / "question_vocab.json"),
                           image_cache_size=cache)
        inf.load()
        assert inf.tokenizer.max_length == 128 and inf.model.config["max_question_length"] == 128
        ids, mask = inf.preprocess_question(long_q)
        assert tuple(ids.shape) == (1, 128) and int(mask.sum()) == 112
        single = [inf.predict(im, q, top_k=3) for im, q in zip(imgs, qs)]
        batch = inf.predict_batch(imgs, qs, top_k=3)
        shared = inf.predict_questions(imgs[0], qs, top_k=3)
        again = inf.predict(imgs[0], long_q, top_k=3)           # image cache hit when the cache is on
        if cache:
            assert inf.cache_hits > 0
        results[cache] = single
        for s, b in zip(single, batch):
            assert [a["index"] for a in s["answers"]] == [a["index"] for a in b["answers"]]
        assert [a["index"] for a in shared[0]["answers"]] == [a["index"] for a in single[0]["answers"]]
        assert [a["index"] for a in again["answers"]] == [a["index"] for a in single[0]["answers"]]
        u8 = inf.preprocess_image_u8(imgs[0]).cpu()
        want, _ = O.vqa_forward(sd, O.preprocess_u8(u8.unsqueeze(0)), ids, mask)
        assert single[0]["answers"][0]["index"] == int(want.argmax(1))
    assert [[a["index"] for a in r["answers"]] for r in results[0]] == [[a["index"] for a in r["answers"]] for r in results[4]]


@needs_gpu
def test_graph_and_pipelined_predict_at_128_tokens():
    from vqa_b200 import VQAInference
    from vqa_b200.synth import synth_batch
    model, _ = _model(128)
    inf = VQAInference()
    inf.load()
    inf.model = model                             # _run takes token tensors: the tokenizer plays no part
    batches = []
    for i in range(5):
        u8, _, _, _ = synth_batch(6, 60 + i)
        ids, mask = QS._questions(128, 128, 6, "i64", False, 60 + i, 10000)
        batches.append((u8.pin_memory(), ids.pin_memory(), mask.pin_memory()))
    runs = {}
    for graph in (True, False):
        inf.use_cuda_graph = graph
        runs[graph] = [inf._run(u8, ids, mask, 4) for u8, ids, mask in batches]
    for (a_idx, a_p), (b_idx, b_p) in zip(runs[True], runs[False]):
        assert torch.equal(a_idx, b_idx) and torch.equal(a_p, b_p)
    inf.use_cuda_graph = True
    outs = list(inf.predict_tensors_pipelined(batches, top_k=4))
    for (idx, probs), (ridx, rprobs) in zip(outs, runs[False]):
        assert torch.equal(idx, ridx) and torch.equal(probs, rprobs)


# ============================================================================ 4. schedule
@needs_gpu
def test_whole_plan_and_graph_match_serial_at_128_tokens():
    import test_gpu_schedule as GS
    ids, mask = QS._questions(128, 128, 6, "i64", True, 5, 10000)
    prog = GS._case("maxlen 128, fully masked question", ctor=dict(max_question_length=128), B=6, L=128, ids=ids,
                    mask=mask, masked_rows=(1,))[0]
    assert sum(op.kind == "attn_chunked" for op in prog.ops) == 6
