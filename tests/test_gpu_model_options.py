"""The model options of tests/model_options_support.py on the GPU, against fp64.

1. Every entry: the poisoned layer-parity walk of test_gpu_layer_parity.py (every module against its fp64 reference,
   every pad exactly 0) in bf16 at B = 3 with top-k min(5, num_answers); tf32 for se_reduction 1 and 3, no cross layer
   and no text layer; bf16 at B = 256 for se_reduction 1 and no cross layer.
2. Whole-plan and CUDA-graph runs against the fp64-checked serial run, bit for bit (test_gpu_schedule.py), for no cross
   layer, no text and no cross layer, and se_reduction 1.
3. The API: logits against the fp32 oracle, predict and VQAInference.predict against the exact rank order of the model's
   own logits, the image cache at 0 and 8 cross layers and its refusal at 9.
4. softmax_topk_kernel at 10 001 to 50 000 answers against the exact references of tests/topk_ref.py (the launcher's
   refusal above 50 000 is in tests/test_gpu_topk.py).
"""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

import model_options_support as MO  # noqa: E402
import test_gpu_layer_parity as GLP  # noqa: E402
import test_gpu_schedule as GS  # noqa: E402
import test_gpu_topk as GT  # noqa: E402
from oracle import vqa_oracle as O  # noqa: E402
from topk_ref import ROW_KINDS, make_row, ref_order  # noqa: E402

DRY = bool(os.environ.get("VQA_DRY"))
DEV = "cpu" if DRY else "cuda"
needs_gpu = pytest.mark.skipif(DRY, reason="runs the library itself (engine, graphs, streams)")
LOGIT_REL_TOL = 2e-2          # test_gpu_model.py: bf16 logits within 2e-2 max-abs relative error of the fp32 oracle


def _env(name, monkeypatch):
    for k, v in MO.ENV.get(name, {}).items():
        monkeypatch.setenv(k, v)


# ============================================================================ 1. layer parity
def _parity(name, B, precision, monkeypatch, seed=5):
    _env(name, monkeypatch)
    MO.relax_spatial_gate(name, monkeypatch)
    prog, sd, ext = MO.make_case(name, B, DEV, seed=seed, precision=precision)
    rep = GLP._check(prog, sd, ext, title=f"{name} {precision} B={B}")
    n_text = MO.MATRIX[name].get("num_transformer_layers", 4)
    assert sum(r.module.startswith("text.") and r.module[5:].isdigit() for r in rep.rows) == n_text
    assert sum(r.module.startswith("x.") and r.output == "x.q" for r in rep.rows) == MO.n_cross(name)
    return prog, rep


@pytest.mark.parametrize("name", list(MO.MATRIX))
def test_layers_bf16_b3(name, monkeypatch):
    prog, rep = _parity(name, 3, "bf16", monkeypatch)
    N = prog.cfg["num_answers"]
    if prog.top_k:
        assert any(r.module == "topk" for r in rep.rows)
    if N % 4:
        assert any(op.kind == "copy_rows" for op in prog.ops)


@pytest.mark.parametrize("name", ["se1", "se3", "cross0", "text0"])
def test_layers_tf32_b3(name, monkeypatch):
    _parity(name, 3, "tf32", monkeypatch, seed=6)


@pytest.mark.parametrize("name", ["se1", "cross0"])
def test_layers_bf16_b256(name, monkeypatch):
    _parity(name, 2 if DRY else 256, "bf16", monkeypatch, seed=7)


# ============================================================================ 2. schedule
@pytest.mark.parametrize("name", ["cross0", "text0_cross0", "se1"])
def test_whole_plan_and_graph_match_serial(name, monkeypatch):
    _env(name, monkeypatch)
    B = 2 if DRY else 16
    ids, mask = MO.questions(name, B, 21)
    kw = {} if ids is None else dict(ids=ids, mask=mask)
    prog = GS._case(name, ctor=MO.MATRIX[name], B=B, seed=21, top_k=MO.top_k(name), **kw)[0]
    assert prog.n_cross_layers == MO.n_cross(name)


# ============================================================================ 3. API
def _model(name, precision="bf16"):
    from vqa_b200.model import VQAModel
    from vqa_b200.synth import randomise_state
    torch.manual_seed(0)
    model = VQAModel(**MO.MATRIX[name], precision=precision).eval()
    sd = randomise_state(model.state_dict(), 1)
    model.load_state_dict(sd, strict=True)
    return model.cuda(), sd


def _inputs(name, B, seed):
    from vqa_b200.synth import synth_batch
    cfg = {**dict(vocab_size=10000, max_question_length=20), **MO.MATRIX[name]}
    u8, img, ids, mask = synth_batch(B, seed, max_len=cfg["max_question_length"], vocab=max(cfg["vocab_size"], 5))
    qi, qm = MO.questions(name, B, seed)
    if qi is not None:
        ids, mask = qi, qm
    return u8, img, ids, mask


API = ["cross0", "text0", "se1", "answers1", "answers3", "answers20000"]


@needs_gpu
@pytest.mark.parametrize("name", API)
def test_model_api_against_the_oracle(name):
    """Logits within the bf16 gate of the fp32 oracle; the argmax equals the oracle's wherever the oracle's top two are
    further apart than twice the largest logit error; predict's winners are the exact rank order of the logits."""
    model, sd = _model(name)
    u8, img, ids, mask = _inputs(name, 9, 40)
    with torch.no_grad():
        logits = model(img.cuda(), ids.cuda(), mask.cuda())[0].cpu()
    want, _ = O.vqa_forward(sd, img, ids, mask, num_heads=model.config["num_attention_heads"])
    assert tuple(logits.shape) == tuple(want.shape) == (9, model.config["num_answers"])
    amax = float(want.abs().max())
    err = float((logits - want).abs().max()) / amax
    print(f"WORST {name} logits rel err {err:.3e}")
    assert err <= LOGIT_REL_TOL
    if want.shape[1] > 1:
        top2 = want.topk(2, dim=1).values
        clear = (top2[:, 0] - top2[:, 1]) > 2 * err * amax
        assert bool(clear.any())
        assert torch.equal(logits.argmax(1)[clear], want.argmax(1)[clear])
    k = MO.top_k(name)
    idx, probs = model.predict(u8.cuda(), ids.cuda(), mask.cuda(), top_k=k)
    with torch.no_grad():
        lu8 = model(u8.cuda(), ids.cuda(), mask.cuda())[0].cpu()
    assert torch.equal(idx.cpu(), ref_order(lu8, k))
    GT._check_probs(f"{name} predict k={k}", idx, probs, lu8)


def _inference(name, tmp_path, **kw):
    from vqa_b200 import VQAInference
    model, sd = _model(name)
    ckpt = tmp_path / f"{name}.pt"
    torch.save({"config": model.config, "model_state_dict": sd}, ckpt)
    return VQAInference(checkpoint_path=str(ckpt), **kw)


@needs_gpu
@pytest.mark.parametrize("name", API)
def test_inference_predict_against_the_rank_order(name, tmp_path):
    from PIL import Image
    from vqa_b200.synth import synth_images_u8
    inf = _inference(name, tmp_path)
    inf.load()
    img = Image.fromarray(synth_images_u8(1, 50)[0].numpy(), "RGB")
    q = "what color is this"
    k = MO.top_k(name)
    out = inf.predict(img, q, top_k=5)
    ids, mask = inf.preprocess_question(q)
    with torch.no_grad():
        lg = inf.model(inf.preprocess_image_u8(img).unsqueeze(0).cuda(), ids.cuda(), mask.cuda())[0].cpu()
    assert [a["index"] for a in out["answers"]] == ref_order(lg, k)[0].tolist()
    GT._check_probs(f"{name} VQAInference k={k}", ref_order(lg, k), torch.tensor([[a["probability"] for a in out["answers"]]]), lg)


@needs_gpu
@pytest.mark.parametrize("name", ["cross0", "cross8"])
def test_image_cache_round_trip(name, tmp_path):
    """encode_images + answer equal forward bit for bit; VQAInference with an image cache gives predict's answers on a
    miss and on a hit."""
    from PIL import Image
    from vqa_b200.synth import synth_images_u8
    model, _ = _model(name)
    u8, img, ids, mask = _inputs(name, 6, 60)
    img, ids, mask = img.cuda(), ids.cuda(), mask.cuda()
    with torch.no_grad():
        logits = model(img, ids, mask)[0]
        cache = model.encode_images(img)
        assert cache.n_images == 6 and len(cache.kv) == MO.n_cross(name)
        assert torch.equal(model.answer(cache, ids, mask), logits)
        one = model.encode_images(img[:2])
        assert one.n_images == 2
        assert torch.equal(model.answer(one, ids, mask), model(img[:2], ids, mask)[0])
        sel = cache.select([4, 4, 1])
        assert sel.n_images == 3 and torch.equal(model.answer(sel, ids[:3], mask[:3]), model(img[[4, 4, 1]], ids[:3], mask[:3])[0])
    plain = _inference(name, tmp_path)
    cached = _inference(name, tmp_path, image_cache_size=4)
    pic = Image.fromarray(synth_images_u8(1, 61)[0].numpy(), "RGB")
    want = plain.predict(pic, "what is this", top_k=5)
    for _ in range(2):
        got = cached.predict(pic, "what is this", top_k=5)
        assert got["answers"] == want["answers"]
    assert cached.cache_info()["hits"] == 1 and cached.cache_info()["misses"] == 1


@needs_gpu
def test_image_cache_refuses_nine_cross_layers(tmp_path):
    model, _ = _model("cross9")
    _, img, ids, mask = _inputs("cross9", 2, 62)
    with torch.no_grad():
        assert model(img.cuda(), ids.cuda(), mask.cuda())[0].shape == (2, 1000)     # forward runs
        with pytest.raises(NotImplementedError, match="8 cross-attention layers"):
            model.encode_images(img.cuda())
    inf = _inference("cross9", tmp_path, image_cache_size=4)
    with pytest.raises(NotImplementedError, match="8 cross-attention layers"):
        inf.load()
    _inference("cross9", tmp_path).load()          # without the cache the model loads


# ============================================================================ 4. top-k kernel
@needs_gpu
@pytest.mark.parametrize("N", [10001, 20000, 50000])
@pytest.mark.parametrize("k", [1, 5, 128])
def test_softmax_topk_kernel_on_large_heads(N, k):
    logits = torch.stack([make_row(kind, N, 1000 * N + 17 * k + r) for r, kind in enumerate(ROW_KINDS)])
    idx, probs = GT._run_softmax_topk(logits, k)
    want = ref_order(logits, k)
    bad = [ROW_KINDS[r] for r in range(len(ROW_KINDS)) if not torch.equal(idx[r].cpu(), want[r])]
    assert not bad, f"N={N} k={k}: winners differ from the rank order on rows {bad}"
    GT._check_probs(f"softmax_topk N={N} k={k}", idx, probs, logits)
