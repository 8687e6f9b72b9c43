"""Questions longer than 64 tokens (max_question_length 65-512), on the CPU: the program runs every self- and
cross-attention of such a question as attn_chunked (keys streamed in chunks of 64) and nothing else changes; every
program of at most 64 tokens keeps attn_mma_kernel's self_attn / cross_attn; layer parity on the emulator; the two-lane
schedule; the model's envelope."""
import sys

import pytest
import torch

from conftest import REPO

sys.path.insert(0, REPO)
import layer_parity as LP  # noqa: E402
import attn_chunked_support  # noqa: E402,F401  (emulator op and access table of the new kind)
import schedule as S  # noqa: E402
import test_schedule_cpu as TS  # noqa: E402
from vqa_b200 import program as P  # noqa: E402
from vqa_b200.model import VQAModel  # noqa: E402

D = 256


def _prog(L, device="meta", **kw):
    kw.setdefault("B", 2)
    prog, _, _ = LP.make_case(dict(max_question_length=L), L=L, device=device, **kw)
    return prog


def _attn_names(prog):
    n_text = sum(1 for op in prog.ops if op.name.startswith("text.") and op.name.endswith(".attn"))
    return [f"text.{i}.attn" for i in range(n_text)] + [f"x.{l}.attn" for l in range(prog.n_cross_layers)]


@pytest.mark.parametrize("L", [65, 128, 512])
@pytest.mark.parametrize("side", ["both", "question"])
def test_long_programs_use_chunked_attention_at_exactly_the_attention_ops(L, side):
    kw = dict(side=side, B=4, n_images=2) if side == "question" else {}
    prog = _prog(L, **kw)
    names = _attn_names(prog)
    assert len(names) == 4 + 2
    assert [op.name for op in prog.ops if op.kind == "attn_chunked"] == names
    assert not any(op.kind in ("self_attn", "cross_attn") for op in prog.ops)
    for op in prog.ops:
        if op.kind != "attn_chunked":
            continue
        i, p = op.i, op.p
        assert (i["B"], i["L"], i["H"], i["hd"], i["no_round"]) == (prog.B, L, 8, 32, prog.out_mode)
        if op.name.startswith("text."):          # packed qkv rows, the key mask
            assert p["q"] is p["kv"] is prog.named["text.qkv"][0] and p["mask"] is prog.named["mask_i32"][0]
            assert (i["T"], i["ld_q"], i["ld_kv"], i["k_off"], i["v_off"], i["q_per_kv"]) == (L, 3 * D, 3 * D, D, 2 * D, 1)
            assert p["out"] is prog.named["text.ctx"][0]
        else:                                    # 49 image tokens, no mask, q_per_kv questions per image
            assert p["mask"] is None and p["out"] is prog.named["x.ctx"][0]
            assert (i["T"], i["ld_q"], i["ld_kv"], i["k_off"], i["v_off"], i["q_per_kv"]) == (49, D, 2 * D, 0, D,
                                                                                              prog.B // prog.Bi)
            if side == "both":
                assert p["weights"] is prog.named[f"aux.xattn.{op.name.split('.')[1]}"][0]


@pytest.mark.parametrize("side", ["both", "question"])
def test_only_the_attention_kind_differs_from_a_64_token_program(side):
    """Same op names, lanes, JOIN flags and the same kinds elsewhere as at L = 64: the layer-parity walker and the
    schedule checker find the modules by name."""
    kw = dict(side=side, B=4, n_images=2) if side == "question" else {}
    short, long_ = _prog(64, **kw), _prog(65, **kw)
    assert [(op.name, op.lane) for op in short.ops] == [(op.name, op.lane) for op in long_.ops]
    swap = {"self_attn": "attn_chunked", "cross_attn": "attn_chunked"}
    assert [swap.get(op.kind, op.kind) for op in short.ops] == [op.kind for op in long_.ops]
    assert sorted(short.named) == sorted(long_.named)


@pytest.mark.parametrize("case", list(TS.CASES))
def test_programs_up_to_64_tokens_keep_the_single_warp_kernel(case, monkeypatch):
    prog, _ = TS._build(monkeypatch, "meta", **TS.CASES[case])
    assert prog.L <= 64
    assert not any(op.kind == "attn_chunked" for op in prog.ops)
    if prog.side != "image":
        assert sum(op.kind in ("self_attn", "cross_attn") for op in prog.ops) == len(_attn_names(prog))


@pytest.mark.parametrize("L", [1, 20, 33, 63, 64])
def test_every_length_up_to_64_keeps_the_single_warp_kernel(L):
    prog = _prog(L)
    assert not any(op.kind == "attn_chunked" for op in prog.ops)
    assert [op.name for op in prog.ops if op.kind in ("self_attn", "cross_attn")] == _attn_names(prog)


def _masked(B, L, empty=1):
    """i64 mask: prefix, left-padded and holes rows, one fully masked question."""
    m = torch.zeros(B, L, dtype=torch.int64)
    m[0, : (2 * L) // 3] = 1
    m[2 % B, L - L // 3:] = 1
    if B > 3:
        m[3, 0::5] = 1
    m[empty] = 0
    return m


@pytest.mark.parametrize("L", [65, 128])
def test_layer_parity_on_the_emulator(L):
    B = 3
    ids = torch.randint(0, 10000, (B, L), generator=torch.Generator().manual_seed(L))
    prog, sd, ext = LP.make_case(dict(max_question_length=L), B, ids=ids, mask=_masked(B, L))
    assert any(op.kind == "attn_chunked" for op in prog.ops)
    rep = LP.check_on_emulator(prog, sd, ext, title=f"maxlen {L}")
    print(rep.table())
    assert not rep.failures(), rep.table()
    assert {"text.0", "x.1"} <= {r.module for r in rep.rows}
    logits = ext[P.EXT["logits"]]
    assert bool(torch.isnan(logits[1]).all()) and not bool(torch.isnan(logits[[0, 2]]).any())


@pytest.mark.parametrize("kw", [dict(), dict(side="image"), dict(side="question", B=4, n_images=2)],
                         ids=["whole", "image_side", "question_side"])
def test_schedule_at_128_tokens(kw):
    prog = _prog(128, **kw)
    problems = [str(h) for h in S.hazards(prog)] + S.unwritten_reads(prog)
    problems += [f"{name} is allocated but no op reads or writes it" for name in S.untouched_buffers(prog)]
    assert not problems, "\n".join(problems)


def test_access_table_of_the_chunked_kind_matches_the_emulator(monkeypatch):
    monkeypatch.setitem(TS.CASES, "len65", dict(ctor=dict(max_question_length=65), L=65))
    TS.test_access_table_matches_the_emulator("len65", monkeypatch)


def test_envelope_is_512_tokens():
    VQAModel(max_question_length=512)._check_supported()
    with pytest.raises(NotImplementedError):
        VQAModel(max_question_length=513)._check_supported()
