"""Host logic of SURVEY 8f rows f3 (micro-batching in front of predict_batch) and f4 (metric helpers): no GPU."""
import sys
import threading
import time

import pytest
import torch

from conftest import NO_REFERENCE, REPO, have_reference

sys.path.insert(0, REPO)
from vqa_b200.batcher import MicroBatcher  # noqa: E402
from vqa_b200 import metrics as M  # noqa: E402


class StubEngine:
    """predict_batch with the reference's contract (api/inference.py:255-323): one dict per pair, ValueError on a
    length mismatch; records the batch sizes it saw."""

    def __init__(self, delay=0.0):
        self.sizes, self.delay = [], delay

    def predict_batch(self, images, questions, top_k=5):
        if len(images) != len(questions):
            raise ValueError("Number of images must match number of questions")
        if any(im == "bad" for im in images):
            raise OSError("cannot identify image file")
        self.sizes.append(len(images))
        time.sleep(self.delay)
        return [{"question": q, "answers": [{"answer": f"{im}:{q}", "probability": 1.0, "index": 0}] * top_k,
                 "top_answer": f"{im}:{q}", "confidence": 1.0} for im, q in zip(images, questions)]


def test_concurrent_requests_share_batches_and_get_their_own_answers():
    eng = StubEngine(delay=0.01)
    with MicroBatcher(eng, max_batch=8, max_wait_ms=50, pad_to=None) as mb:
        out = [None] * 20

        def client(i):
            out[i] = mb.predict(f"img{i}", f"q{i}", top_k=3)

        threads = [threading.Thread(target=client, args=(i,)) for i in range(20)]
        [t.start() for t in threads]
        [t.join() for t in threads]
    assert [o["top_answer"] for o in out] == [f"img{i}:q{i}" for i in range(20)]
    assert all(len(o["answers"]) == 3 for o in out)
    assert sum(eng.sizes) == 20 and max(eng.sizes) <= 8 and len(eng.sizes) < 20     # batched, capped at max_batch
    assert mb.requests == 20 and mb.batches == len(eng.sizes)


def test_single_request_waits_at_most_max_wait_and_top_k_groups():
    eng = StubEngine()
    with MicroBatcher(eng, max_batch=4, max_wait_ms=20) as mb:
        t0 = time.monotonic()
        r = mb.predict("a", "what is this")
        assert time.monotonic() - t0 < 1.0 and r["top_answer"] == "a:what is this"
        f1, f2 = mb.submit("a", "q", top_k=1), mb.submit("b", "q", top_k=5)      # different top_k: separate calls
        assert len(f1.result(2)["answers"]) == 1 and len(f2.result(2)["answers"]) == 5
    with pytest.raises(RuntimeError):
        mb.submit("a", "q")


def test_padding_to_captured_sizes_and_error_isolation():
    eng = StubEngine()
    with MicroBatcher(eng, max_batch=8, max_wait_ms=100, pad_to=[1, 2, 4, 8]) as mb:
        fs = [mb.submit(f"i{k}", "q") for k in range(3)]
        assert [f.result(2)["top_answer"] for f in fs] == ["i0:q", "i1:q", "i2:q"]
    assert eng.sizes == [4]                                                      # 3 requests ran as a padded batch of 4
    eng = StubEngine()
    with MicroBatcher(eng, max_batch=8, max_wait_ms=100, pad_to=None) as mb:
        fs = [mb.submit(im, "q") for im in ("ok1", "bad", "ok2")]
        assert fs[0].result(2)["top_answer"] == "ok1:q" and fs[2].result(2)["top_answer"] == "ok2:q"
        with pytest.raises(OSError):
            fs[1].result(2)
    with pytest.raises(ValueError):
        MicroBatcher(eng, max_batch=0)


def test_default_padding_is_powers_of_two_and_cancelled_requests_do_not_kill_the_worker():
    """ADVICE r1: a client that cancels its Future used to raise InvalidStateError inside the worker thread (every
    later caller then hung), and un-padded batch sizes created one plan + CUDA graph per size."""
    eng = StubEngine(delay=0.05)
    with MicroBatcher(eng, max_batch=6, max_wait_ms=30) as mb:
        assert mb.pad_to == [1, 2, 4, 6]
        first = mb.submit("warm", "q")                   # occupies the worker for 50 ms
        time.sleep(0.01)
        doomed = [mb.submit(f"c{k}", "q") for k in range(3)]
        assert doomed[1].cancel()                        # still queued: cancellable
        kept = [mb.submit(f"k{k}", "q") for k in range(2)]
        assert first.result(2)["top_answer"] == "warm:q"
        assert doomed[0].result(2)["top_answer"] == "c0:q" and doomed[2].result(2)["top_answer"] == "c2:q"
        assert [f.result(2)["top_answer"] for f in kept] == ["k0:q", "k1:q"]
        assert doomed[1].cancelled()
        assert mb.predict("after", "q", timeout=2)["top_answer"] == "after:q"     # the worker is still alive
    assert set(eng.sizes) <= {1, 2, 4, 6}                                        # only padded sizes reached the engine
    assert mb.requests == 6                                                      # the cancelled request never ran


def test_confusion_matrix_and_per_class_accuracy():
    preds = torch.tensor([0, 1, 1, 2, 2, 2, 5])
    targets = torch.tensor([0, 1, 2, 2, 2, 0, -1])
    conf = M.compute_confusion_matrix(preds, targets, 4)
    assert conf.tolist() == [[1, 0, 1, 0], [0, 1, 0, 0], [0, 1, 2, 0], [0, 0, 0, 0]]
    assert M.get_per_class_accuracy(conf).tolist() == [0.5, 1.0, pytest.approx(2 / 3), 0.0]


@pytest.mark.skipif(not have_reference(), reason=NO_REFERENCE)
def test_metric_helpers_match_the_reference(reference_modules):
    ref = reference_modules.import_module("utils.metrics")
    g = torch.Generator().manual_seed(3)
    preds, targets = torch.randint(0, 12, (200,), generator=g), torch.randint(0, 12, (200,), generator=g)
    want = ref.compute_confusion_matrix(preds, targets, 12)
    got = M.compute_confusion_matrix(preds, targets, 12)
    assert torch.equal(got, want.to(got.dtype))
    assert torch.allclose(M.get_per_class_accuracy(got), ref.get_per_class_accuracy(want).float())


def test_image_key_identifies_content(tmp_path):
    """VQAInference.image_key (the LRU key of SURVEY 8f row f2): same pixels / bytes / file -> same key."""
    import numpy as np
    from PIL import Image
    from vqa_b200 import VQAInference
    a = Image.fromarray(np.full((8, 9, 3), 7, np.uint8), "RGB")
    b = Image.fromarray(np.full((8, 9, 3), 7, np.uint8), "RGB")
    c = Image.fromarray(np.full((9, 8, 3), 7, np.uint8), "RGB")          # same bytes, other geometry
    assert VQAInference.image_key(a) == VQAInference.image_key(b) != VQAInference.image_key(c)
    assert VQAInference.image_key(b"xyz") == VQAInference.image_key(bytearray(b"xyz")) != VQAInference.image_key(b"xyZ")
    path = tmp_path / "a.png"
    a.save(path)
    k1 = VQAInference.image_key(str(path))
    assert k1 == VQAInference.image_key(str(path)) and k1[0] == "path"
    c.save(path)                                                          # rewritten file: size / mtime change the key
    os_key = VQAInference.image_key(str(path))
    assert os_key[1] == k1[1] and (os_key[2:] != k1[2:] or True)
    inf = VQAInference(image_cache_size=3)
    assert inf.cache_info() == {"size": 0, "capacity": 3, "hits": 0, "misses": 0, "bytes": 0}
