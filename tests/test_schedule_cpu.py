"""The two-lane schedule against the data flow of the op list (tests/schedule.py), on the CPU.

For every program of the matrix below: no two ops on different lanes touch one allocation without an order between them
(one of them writing), every workspace byte an op reads was written by an op ordered before it (apart from the
zero-at-commit regions of ``schedule.ALLOW``), and every allocation is used.  The access table itself is checked against
the CPU emulator op by op: an op changes no byte outside the fields it declares as written, and it writes the same bytes
when everything outside its declared reads and writes is poisoned.  Mutations of the lanes and of the allow-list must
fail and name the ops and the buffer.

The static checks build their programs on the "meta" device (offsets only), so B = 257 costs nothing; the emulator check
runs the programs of at most two images (the access table depends on the op kind and the form of the op, not on the
batch size).
"""
import sys

import pytest
import torch

from conftest import REPO

sys.path.insert(0, REPO)
import emulator as E  # noqa: E402
import layer_parity as LP  # noqa: E402
import schedule as S  # noqa: E402
from vqa_b200 import program as P  # noqa: E402

ANS3129 = dict(vocab_size=20000, num_answers=3129, num_transformer_layers=1, num_cross_layers=3, se_reduction=4)
SWITCHES = {"VQA_FUSED_TOPK": "1", "VQA_CHAIN": "0", "VQA_FUSE_LN": "0", "VQA_STEM_TWO_ROW": "0",
            "VQA_PHASE_WINDOWS": "0", "VQA_SE_EPILOGUE": "1", "VQA_SHIFT_FUSED": "1"}

CASES = {
    **{f"bf16_b{B}": dict(B=B) for B in (1, 2, 7, 257)},
    **{f"tf32_b{B}": dict(B=B, precision="tf32") for B in (1, 2, 7, 257)},
    "u8_b2": dict(in_fmt="hwc_u8"),
    "u8_b257": dict(B=257, in_fmt="hwc_u8"),
    "mask_none": dict(mask_kind="none"),
    "mask_f32": dict(mask_kind="f32"),
    "tf32_u8_mask_f32": dict(precision="tf32", in_fmt="hwc_u8", mask_kind="f32"),
    "img1_q16_len64": dict(ctor=dict(max_question_length=64), B=16, L=64, n_images=1),
    "side_image": dict(side="image"),
    "side_question": dict(side="question", B=4, n_images=2),
    "side_question_tf32": dict(side="question", B=4, n_images=2, precision="tf32"),
    "ablate": dict(ctor=LP.ABLATE, mask_kind="none"),
    "nospatial": dict(ctor=LP.NOSPATIAL, mask_kind="f32"),
    "cross3_answers3129": dict(ctor=ANS3129),
    "topk0": dict(top_k=0),
    "topk9": dict(top_k=9),
    "no_window": dict(window=False),
    "tf32_no_window": dict(window=False, precision="tf32"),
    **{f"env_{k[4:]}_{v}": dict(env={k: v}) for k, v in SWITCHES.items()},
}
EMULATED = [k for k, c in CASES.items() if c.get("B", 2) <= 2 or c.get("n_images") == 1]


def _build(monkeypatch, device, ctor=None, env=(), **kw):
    for k, v in dict(env).items():
        monkeypatch.setenv(k, v)
    kw.setdefault("B", 2)
    prog, sd, ext = LP.make_case(ctor or {}, device=device, **kw)
    if prog.side == "question":          # the cached image side: K/V of every cross-attention layer
        g = torch.Generator().manual_seed(3)
        for l in range(prog.n_cross_layers):
            ext[P.EXT[f"kv{l}"]] = torch.randn(prog.Bi * 49 * 2 * prog.cfg["embed_dim"], generator=g).to(device)
    return prog, ext


def test_access_table_names_every_pointer_field():
    for kind, spec in P.FIELDS.items():
        tables = S.ACCESS[kind].values() if kind == "pool_gate_ln" else [S.ACCESS[kind]]
        for t in tables:
            assert set(t) == set(spec["p"]), (kind, sorted(set(t) ^ set(spec["p"])))


@pytest.mark.parametrize("case", list(CASES))
def test_schedule_orders_every_conflict(case, monkeypatch):
    prog, _ = _build(monkeypatch, "meta", **CASES[case])
    print(f"{case}: {len(prog.ops)} ops; per op, the other lane's ops it may run alongside")
    print(S.overlap_table(prog))
    problems = [str(h) for h in S.hazards(prog)] + S.unwritten_reads(prog)
    problems += [f"{name} is allocated but no op reads or writes it" for name in S.untouched_buffers(prog)]
    assert not problems, "\n".join(problems)
    # The side lane forks at its first op, after the caller's stream has been handed the whole image side up to the
    # projector: the text encoder may overlap the projector and the K/V projections, never the backbone.
    hb, stream = S.happens_before(prog.ops, 1)
    side = [k for k in range(len(prog.ops)) if stream[k]]
    if side:
        fork = side[0]
        assert all((hb[fork] >> j) & 1 for j in range(fork)), "the fork must follow every op issued before it"


def _poison_ext(ext, keep):
    """Output slots the op does not read: NaN / -1, so that a read of them shows."""
    for name in ("logits", "top_idx", "top_probs"):
        t = ext[P.EXT[name]]
        if t is not None and "ext:" + name not in keep:
            t.fill_(-1 if not t.dtype.is_floating_point else float("nan"))


def _bytes(t):
    return t.reshape(-1).view(torch.uint8)


def _first_outside(changed, ranges):
    """First True byte of ``changed`` outside ``ranges`` (None if there is none); clears ``changed`` inside them."""
    for lo, hi in ranges:
        changed[lo:hi] = False
    idx = changed.nonzero()
    return None if idx.numel() == 0 else int(idx[0])


@pytest.mark.parametrize("case", EMULATED)
def test_access_table_matches_the_emulator(case, monkeypatch):
    prog, ext = _build(monkeypatch, "cpu", **CASES[case])
    lay = S.Layout(prog)
    emu = E.Emulator(prog)
    ws = prog.ws.tensor
    name = lambda off: lay.alloc_of(P.Buf(prog.ws, off, 0)).name
    for k, op in enumerate(prog.ops):
        acc = lay.accesses(op)
        wr = [(a.lo, a.hi) for a in acc if a.writes and a.lo is not None]
        rw = [(a.lo, a.hi) for a in acc if a.lo is not None]
        ext_keys = {a.key for a in acc if a.lo is None}
        ext_w = {a.key for a in acc if a.writes and a.lo is None}
        before = ws.clone()
        ext_before = [None if t is None else t.clone() for t in ext]
        emu.run(ext, k, k + 1)
        after = ws.clone()
        ext_after = [None if t is None else t.clone() for t in ext]
        off = _first_outside(after != before, wr)
        assert off is None, f"{op.name} changes bytes outside its declared writes, first in {name(off)}"
        for key, s in P.EXT.items():
            if s < len(ext) and ext[s] is not None and "ext:" + key not in ext_w:
                assert torch.equal(_bytes(ext[s]), _bytes(ext_before[s])), f"{op.name} writes {key}, not declared"
        # the same op with every workspace byte and output slot it does not declare poisoned
        ws.fill_(0xFF)
        for lo, hi in rw:
            ws[lo:hi] = before[lo:hi]
        for s, t in enumerate(ext_before):
            if t is not None:
                ext[s].copy_(t)
        _poison_ext(ext, ext_keys)
        emu.run(ext, k, k + 1)
        for lo, hi in wr:
            d = (ws[lo:hi] != after[lo:hi]).nonzero()
            assert d.numel() == 0, (f"{op.name} writes other bytes to {name(lo)} when its undeclared inputs are "
                                    f"poisoned (first at byte {int(d[0])}): it reads more than it declares")
        for key in ext_w:
            s = P.EXT[key[4:]]
            assert torch.equal(_bytes(ext[s]), _bytes(ext_after[s])), f"{op.name}: {key} differs under poison"
        ws.copy_(after)
        for s, t in enumerate(ext_after):
            if t is not None:
                ext[s].copy_(t)


# ----------------------------------------------------------------------------- mutations
def _op(prog, name):
    return next(op for op in prog.ops if op.name == name)


def _failures(prog, allow=None):
    return [str(h) for h in S.hazards(prog)] + S.unwritten_reads(prog, allow)


def test_missing_join_before_the_first_attention_is_named(monkeypatch):
    prog, _ = _build(monkeypatch, "meta")
    _op(prog, "x.0.attn").lane &= ~P.LANE_JOIN
    msg = "\n".join(_failures(prog))
    print(msg)
    assert "x.0.q [side, w] and x.0.attn [main, r] both touch x.qp unordered" in msg, msg
    assert "JOIN is missing on x.0.attn" in msg


def test_missing_join_on_the_side_lane_kv_projection_is_named(monkeypatch):
    prog, _ = _build(monkeypatch, "meta")
    first = next(op for op in prog.ops if op.lane & 1 and op.name.startswith("x.1."))
    assert first.name == "x.1.kv" and first.lane & P.LANE_JOIN
    first.lane &= ~P.LANE_JOIN
    msg = "\n".join(_failures(prog))
    print(msg)
    assert "proj.ln [main, w] and x.1.kv [side, r] both touch x.1.imgn unordered" in msg, msg
    assert "JOIN is missing on x.1.kv" in msg


def test_side_lane_output_on_a_main_lane_input_is_named(monkeypatch):
    prog, _ = _build(monkeypatch, "meta")
    op = _op(prog, "x.0.q")
    assert op.lane & 1
    op.p["out"] = prog.named["x.0.imgn"][0]          # the K/V projection of layer 0 reads it on the main lane
    msg = "\n".join(str(h) for h in S.hazards(prog))
    print(msg)
    assert "x.0.q [side, w] and proj.ln [main, w] both touch x.0.imgn unordered" in msg, msg
    assert "x.0.q [side, w] and x.0.kv [main, r] both touch x.0.imgn unordered" in msg, msg


def test_stem_guard_rows_are_a_zero_contract(monkeypatch):
    """The tf32 stem reads the guard rows of stem_in that nothing but the commit-time zero fill writes."""
    prog, _ = _build(monkeypatch, "meta", precision="tf32")
    assert not S.unwritten_reads(prog)
    allow = [a for a in S.ALLOW if a[0] != "stem_in guard rows"]
    msg = "\n".join(S.unwritten_reads(prog, allow))
    print(msg)
    assert msg.startswith("stem.conv.a0 reads bytes [0, ") and "of stem_in" in msg, msg
    assert all(line.startswith("stem.conv.a0 ") for line in msg.splitlines()), msg
