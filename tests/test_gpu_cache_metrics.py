"""SURVEY 8f rows f2 (image cache that outlives a call) and f4 (device-resident accuracy counters) on the GPU."""
import sys

import pytest
import torch
from PIL import Image

pytestmark = pytest.mark.gpu

from conftest import REPO  # noqa: E402

sys.path.insert(0, REPO)
from vqa_b200 import VQAInference  # noqa: E402
from vqa_b200.engine import ImageCache  # noqa: E402
from vqa_b200.metrics import VQAAccuracy, compute_confusion_matrix, evaluate  # noqa: E402
from vqa_b200.model import VQAModel  # noqa: E402
from vqa_b200.runtime import VqaError, accuracy_update, launch_count  # noqa: E402
from vqa_b200.synth import randomise_state, synth_batch, synth_images_u8  # noqa: E402


@pytest.fixture(scope="module")
def model():
    torch.manual_seed(0)
    m = VQAModel().eval()
    m.load_state_dict(randomise_state(m.state_dict(), 1))
    return m.cuda()


# ----------------------------------------------------------------------------- f2: encode_images / answer
@pytest.mark.parametrize("fmt", ["nchw_f32", "hwc_u8"])
def test_encode_then_answer_is_bit_identical_to_forward(model, fmt):
    u8, img, ids, mask = synth_batch(6, 321)
    images = (u8 if fmt == "hwc_u8" else img).cuda()
    ids, mask = ids.cuda(), mask.cuda()
    with torch.no_grad():
        want, _ = model(images, ids, mask)
        cache = model.encode_images(images)
        assert isinstance(cache, ImageCache) and cache.n_images == 6 and len(cache.kv) == 2
        assert cache.kv[0].shape == (6, 49, 512) and cache.nbytes == 2 * 6 * 49 * 512 * 4
        n0 = launch_count()
        got = model.answer(cache, ids, mask)
        n_question_side = launch_count() - n0
    assert torch.equal(got, want)
    # the question side launches no backbone kernel: far fewer launches than a whole forward
    n0 = launch_count()
    with torch.no_grad():
        model(images, ids, mask)
    assert 0 < n_question_side < launch_count() - n0 - 20


def test_cache_outlives_calls_select_and_sharing(model):
    u8, img, ids, mask = synth_batch(8, 99)
    img, ids, mask = img.cuda(), ids.cuda(), mask.cuda()
    with torch.no_grad():
        cache = model.encode_images(img[:2])                       # two images, kept
        # other work in between must not disturb the cache (entries are copies, not workspace views)
        model(img[4:8], ids[4:8], mask[4:8])
        model.encode_images(img[2:4])
        # image 0 answers questions 0..3, image 1 answers 4..7
        got = model.answer(cache, ids, mask)
        want, _ = model(img[:2], ids, mask)
        assert torch.equal(got, want)
        # arbitrary question -> image assignment through select()
        pick = torch.tensor([1, 0, 0, 1, 1, 1, 0, 1])
        got = model.answer(cache.select(pick), ids, mask)
        want, _ = model(img[:2][pick.cuda()], ids, mask)
        assert torch.equal(got, want)
        both = ImageCache.cat([cache.select([1]), cache.select([0])])
        assert torch.equal(both.kv[1][0], cache.kv[1][1]) and both.n_images == 2
    with pytest.raises(ValueError):
        model.answer(cache.select([0, 1, 0]), ids, mask)           # 3 images do not divide 8 questions
    with pytest.raises(ValueError):
        model.answer(ImageCache([cache.kv[0]]), ids, mask)         # wrong number of layers
    with pytest.raises(VqaError):
        model.answer(ImageCache([t.cpu() for t in cache.kv]), ids.cpu(), mask.cpu())


def test_inference_lru_cache():
    torch.manual_seed(0)
    plain = VQAInference()
    plain.load()
    cached = VQAInference(image_cache_size=2)
    cached.model, cached.tokenizer, cached.answer_vocab = plain.model, plain.tokenizer, plain.answer_vocab
    cached._is_loaded = True
    imgs = [Image.fromarray(synth_images_u8(1, 40 + i)[0].numpy(), "RGB") for i in range(3)]
    imgs[2] = imgs[2].resize((300, 260))
    qs = ["what is this", "how many are there", "what color is this"]
    for im in imgs[:2]:
        for q in qs:
            a, b = plain.predict(im, q, top_k=4), cached.predict(im, q, top_k=4)
            assert [x["index"] for x in a["answers"]] == [x["index"] for x in b["answers"]]
            assert all(abs(x["probability"] - y["probability"]) < 1e-6 for x, y in zip(a["answers"], b["answers"]))
    info = cached.cache_info()
    assert info["misses"] == 2 and info["hits"] == 4 and info["size"] == 2 and info["bytes"] == 2 * 2 * 49 * 512 * 4
    cached.predict(imgs[2], qs[0])                                  # third image evicts the least recently used one
    assert cached.cache_info()["size"] == 2 and cached.image_key(imgs[0]) not in cached._image_cache
    # explicit encode / answer: many questions against one entry
    entry = cached.encode_image(imgs[2])
    res = cached.answer(entry, qs, top_k=3)
    ref = plain.predict_questions(imgs[2], qs, top_k=3)
    assert [[a["index"] for a in r["answers"]] for r in res] == [[a["index"] for a in r["answers"]] for r in ref]
    assert cached.answer(entry, []) == []
    assert cached.image_key(b"abc") == cached.image_key(bytearray(b"abc")) != cached.image_key(b"abd")


# ----------------------------------------------------------------------------- f4: accuracy counters
def _reference_update(logits, targets):
    """utils/metrics.py:70-91 on the host."""
    top1 = int((logits.argmax(-1) == targets).sum())
    top5 = int((logits.topk(5, -1).indices == targets.unsqueeze(1)).any(-1).sum())
    return top1, top5


@pytest.mark.parametrize("B,N", [(1, 1000), (7, 37), (256, 1000), (1000, 3129)])
def test_accuracy_kernel_matches_reference_update(B, N):
    g = torch.Generator().manual_seed(B * 7 + N)
    logits = torch.randn(B, N, generator=g)
    # make hits likely: half the targets are the argmax, a quarter lie in the top 5, the rest random / unknown (-1)
    top = logits.topk(5, -1).indices
    targets = torch.randint(0, N, (B,), generator=g)
    sel = torch.rand(B, generator=g)
    targets = torch.where(sel < 0.5, top[:, 0], targets)
    targets = torch.where((sel >= 0.5) & (sel < 0.75), top[:, 3], targets)
    targets = torch.where(sel > 0.95, torch.full_like(targets, -1), targets)
    want1, want5 = _reference_update(logits, targets)
    counters = torch.zeros(3, dtype=torch.int64, device="cuda")
    pred = torch.empty(B, dtype=torch.int64, device="cuda")
    rank = torch.empty(B, dtype=torch.int32, device="cuda")
    accuracy_update(logits.cuda(), targets.cuda(), counters, k=5, pred_out=pred, rank_out=rank)
    accuracy_update(logits.cuda(), targets.cuda(), counters, k=5)          # counters accumulate
    assert counters.tolist() == [2 * want1, 2 * want5, 2 * B]
    assert torch.equal(pred.cpu(), logits.argmax(-1))
    order = logits.argsort(dim=-1, descending=True, stable=True)
    want_rank = torch.where(targets >= 0, (order == targets.unsqueeze(1)).float().argmax(-1), torch.full_like(targets, N))
    assert torch.equal(rank.cpu().long(), want_rank)


def test_accuracy_ties_strided_logits_and_index_form():
    # ties go to the lower index (argmax / stable topk order)
    logits = torch.zeros(4, 8)
    targets = torch.tensor([0, 4, 5, 7])
    c = torch.zeros(3, dtype=torch.int64, device="cuda")
    accuracy_update(logits.cuda(), targets.cuda(), c, k=5)
    assert c.tolist() == [1, 2, 4]
    # logits as a column slice of a wider matrix (row pitch > N)
    wide = torch.randn(9, 64)
    t = torch.randint(0, 40, (9,))
    c.zero_()
    accuracy_update(wide.cuda()[:, :40], t.cuda(), c, k=5)
    assert c.tolist()[:2] == list(_reference_update(wide[:, :40], t))
    for n in (38, 5, 3):                      # 16-byte row pitch, N not a multiple of 4: vector body + scalar tail
        c.zero_()
        tn = t % n
        accuracy_update(wide.cuda()[:, :n], tn.cuda(), c, k=2)
        want1 = int((wide[:, :n].argmax(-1) == tn).sum())
        want2 = int((wide[:, :n].topk(2, -1).indices == tn.unsqueeze(1)).any(-1).sum())
        assert c.tolist() == [want1, want2, 9]
    # the [B] form of update(): indices, top-1 only
    c.zero_()
    accuracy_update(torch.tensor([3, 1, 2], device="cuda"), torch.tensor([3, 0, 2], device="cuda"), c)
    assert c.tolist() == [2, 0, 3]
    with pytest.raises(VqaError):
        accuracy_update(torch.randn(2, 4), torch.zeros(2, dtype=torch.long), c)       # CPU tensors: no CPU path
    with pytest.raises(ValueError):
        accuracy_update(torch.randn(2, 4, device="cuda"), torch.zeros(3, dtype=torch.long, device="cuda"), c)


def test_vqa_accuracy_class_and_evaluate_loop(model):
    acc = VQAAccuracy()
    assert acc.compute() == {"accuracy": 0.0, "accuracy_top5": 0.0, "correct": 0, "total": 0}
    g = torch.Generator().manual_seed(5)
    want1 = want5 = total = 0
    types_right, types_seen = {}, {}
    for step in range(3):
        logits = torch.randn(33, 1000, generator=g)
        targets = torch.where(torch.rand(33, generator=g) < 0.4, logits.argmax(-1), torch.randint(0, 1000, (33,), generator=g))
        qt = [("yes/no", "number", "other")[i % 3] for i in range(33)] if step != 1 else None
        acc.update(logits.cuda(), targets.cuda(), qt)
        a, b = _reference_update(logits, targets)
        want1, want5, total = want1 + a, want5 + b, total + 33
        if qt:
            for t, ok in zip(qt, (logits.argmax(-1) == targets).tolist()):
                types_seen[t] = types_seen.get(t, 0) + 1
                types_right[t] = types_right.get(t, 0) + int(ok)
    m = acc.compute()
    assert (m["correct"], m["total"]) == (want1, total)
    assert m["accuracy"] == want1 / total and m["accuracy_top5"] == want5 / total
    assert m["per_type"] == {t: types_right[t] / types_seen[t] for t in types_seen}
    assert str(acc).startswith("Accuracy: ")
    acc.reset()
    assert acc.compute()["total"] == 0

    # Evaluator.evaluate on the fused forward: same numbers as computing them from the logits on the host
    batches = []
    for i in range(3):
        u8, img, ids, mask = synth_batch(5, 700 + i)
        batches.append({"images": img, "token_ids": ids, "attention_mask": mask})
    with torch.no_grad():
        all_logits = torch.cat([model(b["images"].cuda(), b["token_ids"].cuda(), b["attention_mask"].cuda())[0].cpu()
                                for b in batches])
    answers = torch.where(torch.arange(15) % 2 == 0, all_logits.argmax(-1), all_logits.topk(3, -1).indices[:, 2])
    for i, b in enumerate(batches):
        b["answers"] = answers[5 * i: 5 * i + 5]
    res = evaluate(model, batches)
    assert res["total_samples"] == 15 and res["correct"] == 8 and res["accuracy"] == 8 / 15 and res["accuracy_top5"] == 1.0
    assert len(res["per_class_accuracy"]) == 100 and sum(e["count"] for e in res["common_errors"]) == 7
    conf = compute_confusion_matrix(all_logits.argmax(-1), answers, 1000)
    assert int(conf.sum()) == 15 and int(conf.diag().sum()) == 8


def test_accuracy_counters_match_reference_golden():
    """f4 against the REAL reference: tests/golden/metrics_golden.json was written by running utils/metrics.py's
    VQAAccuracy (update :56-105, compute :107-134) on the seeded inputs of tests/golden/metrics_inputs.py
    (tests/golden/make_metrics_golden.py); the device-resident counters must reproduce every number."""
    import json
    import os
    import sys
    from conftest import GOLDEN
    sys.path.insert(0, GOLDEN)
    import metrics_inputs as MI
    from vqa_b200.metrics import VQAAccuracy
    with open(os.path.join(GOLDEN, "metrics_golden.json")) as f:
        golden = json.load(f)
    assert [(g["B"], g["N"], g["seed"]) for g in golden] == MI.CASES
    for g in golden:
        logits, targets, qtypes = MI.make(g["B"], g["N"], g["seed"])
        acc = VQAAccuracy()
        acc.update(logits.cuda(), targets.cuda(), qtypes)
        acc.update(logits.flip(0).cuda(), targets.flip(0).cuda(), list(reversed(qtypes)))
        res = acc.compute()
        assert (res["correct"], res["total"]) == (g["correct"], g["total"]), g
        assert res["accuracy"] == pytest.approx(g["accuracy"], abs=1e-12)
        assert res["accuracy_top5"] == pytest.approx(g["accuracy_top5"], abs=1e-12)
        assert set(res["per_type"]) == set(g["per_type"])
        for t, v in g["per_type"].items():
            assert res["per_type"][t] == pytest.approx(v, abs=1e-12), (g["seed"], t)
        idx = VQAAccuracy()
        idx.update(logits.argmax(-1).cuda(), targets.cuda())
        r1 = idx.compute()
        assert [r1["correct"], round(r1["accuracy_top5"] * r1["total"]), r1["total"]] == g["index_form"]


def _special_rows(N):
    """(logits [R, N], targets [R]): rows with NaN, +-inf and signed zeros, each with the targets that probe them."""
    nan, inf = float("nan"), float("inf")
    base = torch.randn(N, generator=torch.Generator().manual_seed(N))
    rows, targets = [], []

    def add(row, *ts):
        for t in ts:
            rows.append(row)
            targets.append(t)

    add(torch.full((N,), nan), 0, 1, 3, N - 1)                        # all NaN: only index 0 is the argmax
    r = base.clone()
    r[5] = nan
    add(r, 5, 2)                                                      # a NaN target: rank 0
    r = base.clone()
    r[[N - 3, 9]] = nan
    add(r, N - 3, 9, int(base.argmax()))                              # two NaNs; the finite maximum ranks third
    r = torch.zeros(N)
    r[[0, 2, 3]] = torch.tensor([0.1, 0.3, 0.2])
    r[[1, 4]] = nan
    add(r, 1, 2, 4)                                                   # pred is the first NaN, not the largest finite value
    r = base.clone()
    r[[4, 11]] = inf
    r[[2, 6]] = -inf
    add(r, 11, 4, 6, 2)                                               # +inf ties go to the lower index; -inf ranks last
    r = torch.full((N,), -1.0)
    r[8], r[3] = -0.0, 0.0
    add(r, 8, 3)                                                      # -0.0 ties +0.0
    add(torch.full((N,), -inf), 0, N - 1)
    add(base, -1, N)                                                  # unknown answers: never correct, still counted
    return torch.stack(rows), torch.tensor(targets)


@pytest.mark.parametrize("N", [37, 40, 1000])
def test_accuracy_kernel_follows_argmax_on_nan_and_inf_rows(N):
    """Rank order NaN > +inf > finite > -inf, equal keys to the lower index: pred_out is torch.argmax (the first NaN of a
    row that has one), rank_out is the exact rank, and top-1 / top-k hits follow from the rank.  N = 37 reads the row
    with scalar loads, N = 40 and 1000 with 16-byte loads."""
    from topk_ref import ref_rank
    logits, targets = _special_rows(N)
    B = logits.shape[0]
    for k in (1, 2, 5):
        c = torch.zeros(3, dtype=torch.int64, device="cuda")
        pred = torch.full((B,), -7, dtype=torch.int64, device="cuda")
        rank = torch.full((B,), -7, dtype=torch.int32, device="cuda")
        accuracy_update(logits.cuda(), targets.cuda(), c, k=k, pred_out=pred, rank_out=rank)
        want_rank = ref_rank(logits, targets)
        assert torch.equal(pred.cpu(), torch.argmax(logits, dim=1))
        assert torch.equal(rank.cpu().long(), want_rank)
        valid = (targets >= 0) & (targets < N)
        assert c.tolist() == [int((valid & (want_rank == 0)).sum()), int((valid & (want_rank < k)).sum()), B]
        assert c.tolist()[0] == int((torch.argmax(logits, dim=1) == targets).sum())


def test_evaluate_with_a_fully_masked_question(model):
    """A question whose mask is all zero has a NaN logit row (as in the reference); evaluate() must count it the way
    torch.argmax does and never report a predicted index outside the answer range."""
    batches = []
    for i in range(2):
        u8, img, ids, mask = synth_batch(4, 900 + i)
        batches.append({"images": img, "token_ids": ids, "attention_mask": mask})
    batches[1]["attention_mask"][2] = 0
    with torch.no_grad():
        logits = torch.cat([model(b["images"].cuda(), b["token_ids"].cuda(), b["attention_mask"].cuda())[0].cpu()
                            for b in batches])
    assert bool(torch.isnan(logits[6]).all()) and int(torch.isnan(logits).any(1).sum()) == 1
    answers = logits.nan_to_num(nan=-1.0).argmax(-1)                  # right for every finite row
    answers[6] = 3                                                    # wrong for the NaN row (argmax 0)
    for i, b in enumerate(batches):
        b["answers"] = answers[4 * i: 4 * i + 4]
    res = evaluate(model, batches)
    assert res["total_samples"] == 8 and res["correct"] == int((logits.argmax(-1) == answers).sum()) == 7
    assert res["common_errors"] == [{"predicted_idx": 0, "target_idx": 3, "count": 1}]
