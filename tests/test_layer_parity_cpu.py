"""Layer-by-layer parity on the CPU emulator (tests/layer_parity.py): every module of the program against an fp64
restatement of its reference module, and host-side mutations of the op list that the checker must catch and charge to
the mutated module.  The same checker runs on the GPU in tests/test_gpu_layer_parity.py."""
import sys

import pytest
import torch

from conftest import REPO

sys.path.insert(0, REPO)
import layer_parity as LP  # noqa: E402
from vqa_b200 import program as P  # noqa: E402


@pytest.mark.parametrize("name,kw", [
    ("default", dict(ctor={})),
    ("ablate", dict(ctor=LP.ABLATE, mask_kind="none")),
    ("nospatial", dict(ctor=LP.NOSPATIAL)),
    ("cross3_len64", dict(ctor=dict(num_cross_layers=3, max_question_length=64), in_fmt="hwc_u8", mask_kind="f32")),
    ("tf32", dict(ctor={}, precision="tf32")),
    ("no_window", dict(ctor={}, window=False)),
])
def test_every_layer_matches_fp64_reference_on_emulator(name, kw):
    prog, sd, ext = LP.make_case(B=2, **kw)
    rep = LP.check_on_emulator(prog, sd, ext, title=name)
    print(rep.table())
    assert not rep.failures(), rep.table()
    kinds = {r.module for r in rep.rows}
    n_conv = sum(1 for op in prog.ops if op.name.endswith((".conv1", ".conv2")))
    assert n_conv == 16 and all(op.name in kinds for op in prog.ops if op.name.endswith((".conv1", ".conv2")))
    assert sum(1 for r in rep.rows if r.cls == "pads") >= 2 + 16 + 3     # stem_in, s1.in, every .mid / .out, stage tails


def _op(prog, name):
    return next(op for op in prog.ops if op.name == name)


def _swap_taps(prog):
    op = _op(prog, "s3.b0.conv1")                 # stride-2 block entry: taps of one phase window
    op.i["tap_rel0"], op.i["tap_rel1"] = op.i["tap_rel1"], op.i["tap_rel0"]


def _mask_last_row(prog):
    _op(prog, "s3.b0.conv1").i["mH"] -= 1


def _mask_last_col(prog):
    _op(prog, "s4.b1.conv2").i["mW"] -= 1


def _shift_bias(prog):
    # one channel of the BN-folded bias of s1.b1.conv1 moved by 1 % of the layer's output range (max |y| = 7.5 here);
    # a 1 % change of the bias value itself (~5e-3) is below the bf16 weight-rounding floor of a layer
    b = prog.W.tensor("s1.b1.conv1.b")
    c = int(b.abs().argmax())
    b[c] += 0.075 * torch.sign(b[c])


def _ln_eps(prog):
    _op(prog, "proj.ln").f["eps"] = 1e-3


def _shift_key_mask(prog):
    op = _op(prog, "text.0.attn")                 # every query sees the key mask one token to the left
    m = op.p["mask"]
    op.p["mask"] = P.Buf(m.arena, m.offset + 4, m.nbytes, m.name)


def _empty_question_case():
    """Three questions of 20 tokens; the second is fully masked, which the reference turns into NaN (SURVEY T5)."""
    mask = torch.ones(3, 20, dtype=torch.int64)
    mask[1] = 0
    mask[2, 5:] = 0
    return LP.make_case({}, B=3, mask=mask)


def test_checker_matches_nan_positions():
    """Where the fp64 reference is NaN the program must be NaN at exactly those elements; a key mask read one question
    to the left moves the NaN to another question, and the checker charges that to the first encoder layer only."""
    prog, sd, ext = _empty_question_case()
    rep = LP.check_on_emulator(prog, sd, ext, title="fully masked question")
    assert not rep.failures(), rep.table()
    logits = ext[P.EXT["logits"]]
    assert bool(torch.isnan(logits[1]).all()) and not bool(torch.isnan(logits[[0, 2]]).any())

    prog, sd, ext = _empty_question_case()
    op = _op(prog, "text.0.attn")
    m = op.p["mask"]
    op.p["mask"] = P.Buf(m.arena, m.offset + 4 * prog.L, m.nbytes, m.name)
    rep = LP.check_on_emulator(prog, sd, ext, title="key mask shifted by one question")
    print(rep.table())
    assert rep.failing_modules() == ["text.0"], rep.table()


@pytest.mark.parametrize("mutate,module", [
    (_swap_taps, "s3.b0.conv1"),
    (_mask_last_row, "s3.b0.conv1"),
    (_mask_last_col, "s4.b1.conv2"),
    (_shift_bias, "s1.b1.conv1"),
    (_ln_eps, "proj"),
    (_shift_key_mask, "text.0"),
])
def test_checker_names_a_mutated_module(mutate, module):
    """Each module is checked on the upstream state the program produced, so a subtle error in one layer fails that
    layer and no other."""
    prog, sd, ext = LP.make_case({}, B=2)
    mutate(prog)
    rep = LP.check_on_emulator(prog, sd, ext, title=mutate.__name__)
    print(rep.table())
    assert rep.failing_modules() == [module], rep.table()
