"""Models whose embed_dim, head count or FFN width differ from the reference defaults, on the CPU: the envelope
``VQAModel`` accepts, the default model's programs unchanged op for op, the embedding fold at widths that are not
perfect squares, layer parity on the emulator and the two-lane schedule at every width the GPU tests run."""
import hashlib
import math
import sys

import pytest
import torch
import torch.nn.functional as F

from conftest import REPO

sys.path.insert(0, REPO)
import attn_chunked_support  # noqa: E402,F401  (emulator op and access table of the chunked kind)
import layer_parity as LP  # noqa: E402
import model_widths_support as MW  # noqa: E402
import schedule as S  # noqa: E402
import test_schedule_cpu as TS  # noqa: E402
from vqa_b200 import program as P  # noqa: E402
from vqa_b200.model import VQAModel  # noqa: E402

# (embed_dim, heads, ffn_hidden_dim, accepted)
ENVELOPE = [
    (256, 8, 1024, True),       # the reference defaults
    (128, 2, 64, True), (128, 8, 4096, True), (192, 12, 192, True), (192, 3, 768, True), (320, 5, 1280, True),
    (384, 6, 1536, True), (448, 28, 448, True), (512, 32, 2048, True), (512, 8, 64, True), (256, 4, 1024, True),
    (32, 4, 128, False),        # reproduce_issue.py's toy model: embed_dim and head_dim 8 outside the envelope
    (256, 32, 1024, False),     # head_dim 8
    (256, 2, 1024, False),      # head_dim 128
    (512, 4, 2048, False),      # head_dim 128
    (576, 9, 1024, False),      # embed_dim above 512
    (64, 2, 256, False),        # embed_dim below 128
    (160, 5, 640, False),       # embed_dim not a multiple of 64
    (256, 8, 1000, False),      # FFN width not a multiple of 64
    (256, 8, 4160, False),      # FFN width above 4096
    (256, 8, 0, False),
    (192, 4, 768, False),       # head_dim 48
    (240, 5, 960, False),       # head_dim 48, embed_dim not a multiple of 64
]


@pytest.mark.parametrize("D,H,F,ok", ENVELOPE, ids=lambda v: str(v))
def test_envelope(D, H, F, ok):
    model = VQAModel(vocab_size=50, num_answers=7, embed_dim=D, num_attention_heads=H, ffn_hidden_dim=F,
                     num_transformer_layers=1, num_cross_layers=1)
    if ok:
        model._check_supported()
        return
    with pytest.raises(NotImplementedError) as e:
        model._check_supported()
    assert "embed_dim 128..512" in str(e.value) and "{16, 32, 64}" in str(e.value)


def test_envelope_keeps_the_question_length_limit():
    VQAModel(**MW.ctor("c", max_question_length=512))._check_supported()
    with pytest.raises(NotImplementedError):
        VQAModel(**MW.ctor("c", max_question_length=513))._check_supported()


# sha256 (first 16 hex digits) of [(kind, name, lane, sorted integer fields)] of the default model's programs, as the
# parent commit of the width support built them: the default model must run exactly the ops it ran before
DEFAULT_DIGESTS = {
    ("bf16", "both", 1): "fdf5a01e287c4bd2",
    ("bf16", "both", 7): "3401bbdf9e646e90",
    ("bf16", "both", 256): "daf762c8406ac786",
    ("bf16", "image", 1): "f2d7e883e275a2dc",
    ("bf16", "image", 7): "3edb9b24597d5312",
    ("bf16", "image", 256): "d64de7097c2fa2d2",
    ("bf16", "question", 1): "1df6f463443aa626",
    ("bf16", "question", 7): "6896bcf179db4add",
    ("bf16", "question", 256): "60ac7a9ccc1954cb",
    ("tf32", "both", 1): "6e014fcea782d23c",
    ("tf32", "both", 7): "1aae7d92cc70ba61",
    ("tf32", "both", 256): "85bc939990e9feeb",
    ("tf32", "image", 1): "4354d986b0ad38f4",
    ("tf32", "image", 7): "217360e0e6ec5014",
    ("tf32", "image", 256): "8ea2c6637735af10",
    ("tf32", "question", 1): "ae996262599b6d6b",
    ("tf32", "question", 7): "82e7357d3d56e2ec",
    ("tf32", "question", 256): "498c9d5bed62bc3a",
}


def _digest(prog):
    rows = [(op.kind, op.name, op.lane, tuple(sorted(op.i.items()))) for op in prog.ops]
    return hashlib.sha256(repr(rows).encode()).hexdigest()[:16]


@pytest.mark.parametrize("key", list(DEFAULT_DIGESTS), ids=lambda k: "-".join(map(str, k)))
def test_default_programs_are_unchanged(key, monkeypatch):
    for var in ("VQA_CHAIN", "VQA_FUSE_LN", "VQA_FUSED_TOPK", "VQA_SMALL_M", "VQA_WIDE_CONV", "VQA_PAIR_BN"):
        monkeypatch.delenv(var, raising=False)
    precision, side, B = key
    prog, _, _ = LP.make_case({}, B, device="meta", precision=precision, side=side)
    assert _digest(prog) == DEFAULT_DIGESTS[key]


@pytest.mark.parametrize("name", list(MW.CONFIGS))
@pytest.mark.parametrize("precision", ["bf16", "tf32"])
def test_programs_follow_the_widths(name, precision):
    D, H, F = MW.CONFIGS[name]
    prog, _, _ = LP.make_case(MW.ctor(name, max_question_length=20), 3, device="meta", precision=precision)
    chain = precision == "bf16" and D == 256
    assert any(op.kind == "mlp_chain" for op in prog.ops) == chain
    assert any(op.kind == "embed" and "gamma" in op.p for op in prog.ops) == (D == 256)   # fused embed + LayerNorm
    for op in prog.ops:
        if op.kind in ("layernorm", "pool_gate_ln", "embed"):
            assert op.i["D"] == D, op.name
        if op.kind in ("self_attn", "cross_attn", "attn_chunked"):
            assert (op.i["H"], op.i["hd"]) == (H, D // H), op.name
        if op.kind == "gemm":
            assert op.i["Npad"] % op.i["BN"] == 0, op.name
    for buf, shape in (("text.x", (3 * 20, D)), ("x.q", (3 * 20, D)), ("fused", (3, D)), ("fusion.cat", (3, 2 * D)),
                       ("head.h0", (3, 2 * D)), ("head.h1", (3, D)), ("x.0.kv", (3 * 49, 2 * D)),
                       ("aux.xattn.0", (3, H, 20, 49))):
        assert prog.named[buf][2] == shape, buf
    if not chain:
        assert prog.named["text.hid"][2] == (3 * 20, max(F, 4 * D))   # text FFN and the cross layers' 4 * D FFN
        fc = [op for op in prog.ops if op.kind == "gemm" and op.name in ("text.0.fc1", "x.0.fc1")]
        assert [op.i["N"] for op in fc] == [F, 4 * D]


@pytest.mark.parametrize("D", [128, 192, 320, 448, 512])
def test_embedding_fold_is_the_reference_product(D):
    """Scaling the table once at load time gives the bits of the reference's F.embedding(ids, emb) * math.sqrt(D)."""
    assert math.isqrt(D) ** 2 != D
    torch.manual_seed(D)
    model = VQAModel(vocab_size=97, num_answers=5, embed_dim=D, num_attention_heads=D // 64, ffn_hidden_dim=64,
                     num_transformer_layers=1, num_cross_layers=1)
    sd = model.state_dict()
    W = P.build_weights(sd, model.config, "cpu")
    ids = torch.randint(0, 97, (4, 20))
    emb = sd["text_encoder.token_embedding.weight"].float()
    assert torch.equal(W.tensor("text.emb")[ids], F.embedding(ids, emb) * math.sqrt(D))


def _masked(B, L):
    m = torch.zeros(B, L, dtype=torch.int64)
    m[0, : (2 * L) // 3] = 1
    m[1] = 0                                     # a fully masked question: NaN end to end
    m[2, L - L // 3:] = 1
    return m


@pytest.mark.parametrize("L", [20, 65])
@pytest.mark.parametrize("name", list(MW.CONFIGS))
def test_layer_parity_on_the_emulator(name, L):
    B = 3
    ids = torch.randint(0, 10000, (B, L), generator=torch.Generator().manual_seed(L))
    prog, sd, ext = LP.make_case(MW.ctor(name, max_question_length=L), B, ids=ids, mask=_masked(B, L))
    rep = LP.check_on_emulator(prog, sd, ext, title=f"config {name} L {L}")
    print(rep.table())
    assert not rep.failures(), rep.table()
    assert {"text.0", "x.1"} <= {r.module for r in rep.rows}
    logits = ext[P.EXT["logits"]]
    assert bool(torch.isnan(logits[1]).all()) and not bool(torch.isnan(logits[[0, 2]]).any())


@pytest.mark.parametrize("name", list(MW.CONFIGS))
@pytest.mark.parametrize("kw", [dict(), dict(side="question", B=4, n_images=2), dict(precision="tf32", L=65)],
                         ids=["whole", "question_side", "tf32_L65"])
def test_schedule_at_each_width(name, kw, monkeypatch):
    kw = dict(kw)
    L = kw.pop("L", 20)
    monkeypatch.setitem(TS.CASES, f"width_{name}", dict(ctor=MW.ctor(name, max_question_length=L), L=L, **kw))
    TS.test_schedule_orders_every_conflict(f"width_{name}", monkeypatch)


@pytest.mark.parametrize("name", ["c", "e"])
def test_access_table_matches_the_emulator_at_other_widths(name, monkeypatch):
    monkeypatch.setitem(TS.CASES, f"width_{name}", dict(ctor=MW.ctor(name)))
    TS.test_access_table_matches_the_emulator(f"width_{name}", monkeypatch)
