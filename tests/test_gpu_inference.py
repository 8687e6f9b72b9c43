"""VQAInference (predict API) on the GPU: result schema, parity with the oracle, batching, CUDA graph."""
import sys

import numpy as np
import pytest
import torch
from PIL import Image

pytestmark = pytest.mark.gpu

from conftest import REPO  # noqa: E402

sys.path.insert(0, REPO)
from oracle import vqa_oracle as O  # noqa: E402
from vqa_b200 import VQAInference  # noqa: E402
from vqa_b200.synth import synth_images_u8  # noqa: E402


@pytest.fixture(scope="module")
def engine():
    torch.manual_seed(0)
    inf = VQAInference()
    inf.load()
    return inf


def _oracle_topk(inf, u8, question, k):
    sd = {n: t.detach().cpu() for n, t in inf.model.state_dict().items()}
    ids, mask = inf.preprocess_question(question)
    logits, _ = O.vqa_forward(sd, O.preprocess_u8(u8.unsqueeze(0)), ids, mask)
    return O.predict_topk(logits, k)


@pytest.mark.parametrize("graph", [True, False])
def test_predict_schema_and_parity(engine, graph):
    engine.use_cuda_graph = graph
    u8 = synth_images_u8(1, 7)[0]
    q = "What COLOR is this, really?!  don't know"
    out = engine.predict(Image.fromarray(u8.numpy(), "RGB"), q, top_k=5)
    assert set(out) == {"question", "answers", "top_answer", "confidence"} and out["question"] == q
    assert len(out["answers"]) == 5 and set(out["answers"][0]) == {"answer", "probability", "index"}
    idx, probs = _oracle_topk(engine, u8, q, 5)
    assert out["answers"][0]["index"] == int(idx[0, 0])
    assert out["top_answer"] == f"answer_{int(idx[0, 0])}" and out["confidence"] == out["answers"][0]["probability"]
    np.testing.assert_allclose([a["probability"] for a in out["answers"]], probs[0].numpy(), rtol=2e-2, atol=1e-5)
    ids, mask = engine.preprocess_question(q)
    assert ids.tolist()[0][:9] == [2, 4, 7, 5, 6, 1, 1, 1, 3] and int(mask.sum()) == 9   # default 13-word tokenizer


def test_predict_batch_and_resize(engine):
    engine.use_cuda_graph = True
    imgs = [Image.fromarray(synth_images_u8(1, 10 + i)[0].numpy(), "RGB") for i in range(3)]
    imgs[1] = imgs[1].resize((320, 200))   # goes through the PIL antialiased bilinear resize
    qs = ["what is this", "how many are there", "where is what type"]
    res = engine.predict_batch(imgs, qs, top_k=3)
    assert [r["question"] for r in res] == qs and all(len(r["answers"]) == 3 for r in res)
    for im, q, r in zip(imgs, qs, res):
        u8 = engine.preprocess_image_u8(im).cpu()          # non-224 inputs come back from the device-side resize
        idx, _ = _oracle_topk(engine, u8, q, 3)
        assert r["answers"][0]["index"] == int(idx[0, 0])
    single = engine.predict(imgs[0], qs[0], top_k=3)
    assert single["answers"][0]["index"] == res[0]["answers"][0]["index"]
    with pytest.raises(ValueError):
        engine.predict_batch(imgs, qs[:2])
    info = engine.get_model_info()
    assert info["num_answers"] == 1000 and info["vocab_size"] == 13 and info["parameters"]["total"] == 19310316


@pytest.mark.parametrize("lanes,graph", [(2, True), (1, True), (2, False)])
def test_pipelined_throughput_path_matches_single_calls(engine, lanes, graph):
    """Two compute lanes (own stream + own plan workspace each) overlap consecutive batches; results must come back in
    order and equal the one-call path bit for bit, also when slots and lanes are reused (11 batches over 4 slots)."""
    from vqa_b200.synth import synth_batch
    engine.pipeline_lanes, engine.use_cuda_graph = lanes, graph
    batches = []
    for i in range(11):
        u8, _, ids, mask = synth_batch(6, 50 + i)
        batches.append((u8.pin_memory(), ids.pin_memory(), mask.pin_memory()))
    outs = list(engine.predict_tensors_pipelined(batches, top_k=4))
    assert len(outs) == 11
    outs2 = list(engine.predict_tensors_pipelined(batches[::-1], top_k=4))      # second call reuses the captured slots
    assert all(torch.equal(a[0], b[0]) for a, b in zip(outs, outs2[::-1]))
    engine.pipeline_lanes = 3
    engine.use_cuda_graph = False
    for (u8, ids, mask), (idx, probs) in zip(batches, outs):
        ridx, rprobs = engine._run(u8, ids, mask, 4)
        assert torch.equal(idx, ridx) and torch.equal(probs, rprobs)


@pytest.mark.parametrize("hw", [(300, 400), (100, 160), (333, 211), (224, 500), (640, 224), (17, 23), (1080, 1920), (225, 223),
                                (300, 3), (301, 3), (1000, 3), (205, 2), (225, 2), (2000, 5), (70000, 5), (1, 300), (300, 1),
                                (3000, 4000), (1, 1), (66000, 700)])
def test_device_resize_is_bit_exact_with_pil(engine, hw):
    """vqa_resize_bilinear_u8 (csrc/resize.cu) against PIL.Image.resize(BILINEAR) itself: every byte equal.  (301, 3) ..
    (70000, 5) take Pillow's vertical-first order (height > 100 * width); 66 000 rows exceed a grid's 65 535 y-blocks."""
    from vqa_b200.runtime import resize_bilinear_u8
    rng = np.random.default_rng(hw[0] * 7919 + hw[1])
    img = rng.integers(0, 256, (hw[0], hw[1], 3), dtype=np.uint8)
    want = np.asarray(Image.fromarray(img, "RGB").resize((224, 224), Image.BILINEAR))
    got = resize_bilinear_u8(torch.from_numpy(img).cuda(), 224, 224).cpu().numpy()
    assert got.shape == (224, 224, 3) and np.array_equal(got, want)


def test_device_resize_matches_golden_and_host_path(engine):
    import os
    from conftest import GOLDEN
    g = np.load(os.path.join(GOLDEN, "preprocess.npz"))
    for name in ("down", "up", "odd"):
        im = Image.fromarray(g[f"{name}.u8"], "RGB")
        dev = engine.preprocess_image_u8(im)                        # CUDA kernels
        host = engine.preprocess_image_u8(im, device_resize=False)  # PIL on the host
        assert dev.is_cuda and not host.is_cuda
        assert np.array_equal(dev.cpu().numpy(), g[f"{name}.resized_u8"]) and torch.equal(dev.cpu(), host)
    tall = Image.fromarray(np.random.default_rng(3).integers(0, 256, (1000, 3, 3), dtype=np.uint8), "RGB")
    dev = engine.preprocess_image_u8(tall)                          # vertical pass first, as Pillow does
    assert dev.is_cuda and torch.equal(dev.cpu(), engine.preprocess_image_u8(tall, device_resize=False))
    im = Image.fromarray(g["down.u8"], "RGB")
    engine.gpu_resize = True
    a = engine.predict(im, "what is this", top_k=5)
    engine.gpu_resize = False
    b = engine.predict(im, "what is this", top_k=5)
    engine.gpu_resize = True
    assert a == b


def test_predict_questions_shares_the_image(engine):
    """One image, many questions: same dicts as predict() per question."""
    engine.use_cuda_graph = True
    im = Image.fromarray(synth_images_u8(1, 21)[0].numpy(), "RGB")
    qs = ["what is this", "what color is this", "how many are there", "where is this", "is there what type"]
    res = engine.predict_questions(im, qs, top_k=4)
    assert [r["question"] for r in res] == qs
    for q, r in zip(qs, res):
        single = engine.predict(im, q, top_k=4)
        assert [a["index"] for a in r["answers"]] == [a["index"] for a in single["answers"]]
        np.testing.assert_allclose([a["probability"] for a in r["answers"]],
                                   [a["probability"] for a in single["answers"]], rtol=1e-5, atol=1e-7)
    assert engine.predict_questions(im, []) == []


def test_micro_batcher_in_front_of_the_real_engine():
    """SURVEY 8f row f3 on hardware (VERDICT r1): 20 concurrent clients through ``MicroBatcher`` in front of the real
    ``VQAInference`` -- every client gets exactly what ``predict`` returns for its pair, the batches are padded to
    [1, 2, 4, 8] so at most four CUDA graphs (and plan workspaces) exist afterwards (api/inference.py:255-323 behind
    api/main.py:224-267's batch endpoint)."""
    import threading
    from vqa_b200.batcher import MicroBatcher
    torch.manual_seed(0)
    inf = VQAInference()
    inf.load()
    imgs = [Image.fromarray(synth_images_u8(1, 100 + i)[0].numpy(), "RGB") for i in range(20)]
    imgs[3] = imgs[3].resize((300, 180))
    qs = [("what is this", "how many are there", "where is what type", "what color is this")[i % 4] + " " * (i % 3)
          for i in range(20)]
    want = [inf.predict(im, q, top_k=3) for im, q in zip(imgs, qs)]
    before = set(inf._graphs)
    out = [None] * 20
    with MicroBatcher(inf, max_batch=8, max_wait_ms=20, pad_to=[1, 2, 4, 8]) as mb:
        def client(i):
            out[i] = mb.predict(imgs[i], qs[i], top_k=3, timeout=60)
        threads = [threading.Thread(target=client, args=(i,)) for i in range(20)]
        [t.start() for t in threads]
        [t.join() for t in threads]
        assert mb.requests == 20 and mb.batches < 20
    for o, w in zip(out, want):
        assert o["question"] == w["question"] and [a["index"] for a in o["answers"]] == [a["index"] for a in w["answers"]]
        np.testing.assert_allclose([a["probability"] for a in o["answers"]], [a["probability"] for a in w["answers"]],
                                   rtol=1e-5, atol=1e-7)
    new = set(inf._graphs) - before
    assert {k[0] for k in new} <= {1, 2, 4, 8} and len(new) <= 4, new


def test_plan_and_graph_caches_are_bounded():
    """VERDICT r1 weak #10: predict_batch with varying batch sizes must not grow device memory without limit."""
    torch.manual_seed(0)
    inf = VQAInference(max_graphs=3)
    inf.load()
    inf.model.engine().max_plans = 3
    img = Image.fromarray(synth_images_u8(1, 5)[0].numpy(), "RGB")
    first = inf.predict_batch([img], ["what is this"], top_k=2)
    for b in (2, 3, 5, 6, 7):
        inf.predict_batch([img] * b, ["what is this"] * b, top_k=2)
        assert len(inf._graphs) <= 3 and len(inf.model.engine()._plans) <= 3
    torch.cuda.synchronize()
    again = inf.predict_batch([img], ["what is this"], top_k=2)          # evicted shape: rebuilt, same answer
    assert again[0]["answers"] == first[0]["answers"]
    with pytest.raises(IndexError):                                       # tokenizer id beyond the model's vocabulary
        inf.model.config["vocab_size"] = 5
        try:
            inf.preprocess_question("what color is this")
        finally:
            inf.model.config["vocab_size"] = 10000
