"""Tokenizer / AnswerVocabulary: bit-exact against golden vectors made by the reference
(tests/golden/make_golden.py::text_utils_case) and the known answers the reference prints in
its own __main__ demos (utils/tokenizer.py:371-389, data/build_vocab.py:334-354,
api/inference.py:114-132)."""
import json

import pytest
from hypothesis import given, settings, strategies as st

from vqa_b200.text import AnswerVocabulary, Tokenizer

from conftest import NO_REFERENCE, have_reference


@pytest.fixture(scope="module")
def tu(golden_meta):
    return golden_meta["text_utils"]


def _tok(tu):
    t = Tokenizer(max_length=15)
    t.build_vocab(tu["corpus"], min_freq=1)
    return t


def test_vocab_matches_reference(tu):
    assert _tok(tu).word2idx == tu["word2idx"]


def test_known_answer_from_reference_demo(tu):
    ids, mask = _tok(tu).encode("What color is the dog?")
    assert [ids, mask] == tu["encode"]["What color is the dog?"]
    assert ids[0] == 2 and ids[6] == 3 and sum(mask) == 7 and len(ids) == 15 and ids[7:] == [0] * 8


def test_encode_variants_bit_exact(tu):
    t = _tok(tu)
    for p in tu["probes"]:
        assert list(map(list, t.encode(p))) == tu["encode"][p], p
        assert list(map(list, t.encode(p, add_special_tokens=False))) == tu["encode_nospecial"][p], p
        assert list(map(list, t.encode(p, padding=False, truncation=False))) == tu["encode_nopad"][p], p
        assert t.decode(tu["encode"][p][0]) == tu["decode"][p]


def test_truncation_keeps_end_token(tu):
    ids, mask = _tok(tu).encode("a " * 40)
    assert len(ids) == 15 and ids[0] == 2 and ids[-1] == 3 and all(mask)


def test_default_inference_tokenizer(tu):
    t = Tokenizer(max_length=20)
    t.build_vocab(["what is this", "what color", "how many", "is there", "where is", "what type"], min_freq=1)
    assert t.word2idx == tu["default_word2idx"]
    assert {w: i for w, i in t.word2idx.items() if i >= 4} == {
        "what": 4, "is": 5, "this": 6, "color": 7, "how": 8, "many": 9, "there": 10, "where": 11, "type": 12}
    ids, mask = t.encode("What COLOR is this, really?!  don't know")
    assert ids == [2, 4, 7, 5, 6, 1, 1, 1, 3] + [0] * 11 and mask == [1] * 9 + [0] * 11
    for p, v in tu["default_encode"].items():
        assert list(map(list, t.encode(p))) == v


def test_vocab_cap_and_min_freq(tu):
    t = Tokenizer(max_length=8, vocab_size=9)
    t.build_vocab(["b a a c", "c b a d", "e e d d d", "f"], min_freq=2)
    assert t.word2idx == tu["tok2_word2idx"]


def test_save_load_roundtrip(tu, tmp_path):
    t = _tok(tu)
    path = str(tmp_path / "vocab.json")
    t.save(path)
    assert set(json.load(open(path))) == {"word2idx", "max_length", "max_vocab_size"}
    u = Tokenizer()
    u.load(path)
    assert u.word2idx == t.word2idx and u.max_length == 15
    for p in tu["probes"]:
        assert u.encode(p) == t.encode(p)


def test_answer_vocab(tu, tmp_path):
    av = AnswerVocabulary(num_answers=5)
    av.build_from_qa_pairs([{"answer": a} for a in
                            ["Yes", "yes", "The dog", "a dog", "no", "No.", "two", "2", "yes", "red!", "RED"]])
    assert av.answer2idx == tu["answer2idx"]
    for a, i in tu["answer_encode"].items():
        assert av.encode(a) == i
    for i, a in tu["answer_decode"].items():
        assert av.decode(int(i)) == a
    for a, p in tu["answer_preprocess"].items():
        assert av.preprocess_answer(a) == p
    assert av.encode("yes") == av.encode("YES") == 0 and av.encode("unknown") == -1 and av.decode(0) == "yes"
    assert av.decode(999) == "<UNKNOWN>"
    path = str(tmp_path / "sub" / "answers.json")
    av.save(path)
    bv = AnswerVocabulary()
    bv.load(path)
    assert bv.answer2idx == av.answer2idx and bv.num_answers == 5 and bv.decode(1) == av.decode(1)


_text = st.text(alphabet=st.sampled_from(list("abcXYZ 019_'?!,.\t\n-éß中")), max_size=80)


@pytest.mark.skipif(not have_reference(), reason=NO_REFERENCE)
@settings(max_examples=300, deadline=None)
@given(text=_text, special=st.booleans(), pad=st.booleans(), trunc=st.booleans())
def test_property_encode_matches_live_reference(reference_modules, text, special, pad, trunc):
    ref = reference_modules.import_module("utils.tokenizer")
    corpus = ["abc abc xyz", "xyz 019 abc", "é ß 中 中", "a_b it's it's"]
    a, b = ref.Tokenizer(max_length=9), Tokenizer(max_length=9)
    import contextlib, io
    with contextlib.redirect_stdout(io.StringIO()):
        a.build_vocab(corpus, min_freq=1)
    b.build_vocab(corpus, min_freq=1)
    assert a.word2idx == b.word2idx
    ra = a.encode(text, add_special_tokens=special, padding=pad, truncation=trunc)
    rb = b.encode(text, add_special_tokens=special, padding=pad, truncation=trunc)
    assert (list(ra[0]), list(ra[1])) == (list(rb[0]), list(rb[1]))
    assert a.decode(ra[0]) == b.decode(rb[0])


@pytest.mark.skipif(not have_reference(), reason=NO_REFERENCE)
@settings(max_examples=200, deadline=None)
@given(ans=_text)
def test_property_answer_preprocess_matches_live_reference(reference_modules, ans):
    ref = reference_modules.import_module("data.build_vocab")
    assert ref.AnswerVocabulary.preprocess_answer(ans) == AnswerVocabulary.preprocess_answer(ans)
