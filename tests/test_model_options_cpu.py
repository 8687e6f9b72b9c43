"""The model options of tests/model_options_support.py on the CPU: the two-lane schedule of every entry, emulator layer
parity, and the API's refusals for what the engine still does not run.

The schedule check is test_schedule_cpu.py's (``schedule.hazards``, ``unwritten_reads``, ``untouched_buffers``) on the
"meta" device, for bf16 and tf32 at B = 2 and 257, and for the image-side and question-side programs the entry allows.
A model without cross-attention layers has no attention op to join the lanes before the fusion tail, which reads the
text encoder's output; its first fusion op carries the join.
"""
import functools
import sys

import pytest
import torch

from conftest import REPO

sys.path.insert(0, REPO)
import layer_parity as LP  # noqa: E402
import model_options_support as MO  # noqa: E402
import schedule as S  # noqa: E402
from vqa_b200 import program as P  # noqa: E402
from vqa_b200.model import _SUPPORTED, VQAModel  # noqa: E402
from vqa_b200.synth import randomise_state  # noqa: E402

NAMES = list(MO.MATRIX)


@functools.lru_cache(maxsize=4)
def _weights(name, precision):
    torch.manual_seed(0)
    model = VQAModel(**MO.MATRIX[name]).eval()
    return P.build_weights(randomise_state(model.state_dict(), 1), model.config, "meta", precision=precision), model.config


def _program(name, precision, B, side, monkeypatch):
    for k, v in MO.ENV.get(name, {}).items():
        monkeypatch.setenv(k, v)
    W, cfg = _weights(name, precision)
    n_images = 1 if side == "question" else None
    return P.Program(W, cfg, B, cfg["max_question_length"], "nchw_f32", P.MASK_I64, want_aux=side == "both",
                     top_k=MO.top_k(name) if side != "image" else 0, device="meta", n_images=n_images, side=side)


def _problems(prog):
    out = [str(h) for h in S.hazards(prog)] + S.unwritten_reads(prog)
    return out + [f"{n} is allocated but no op reads or writes it" for n in S.untouched_buffers(prog)]


SIDES = [(name, side) for name in NAMES for side in ("both", "image", "question")
         if not (side == "question" and MO.n_cross(name) > P.MAX_CACHED_LAYERS)]


@pytest.mark.parametrize("precision", ["bf16", "tf32"])
@pytest.mark.parametrize("name,side", SIDES)
def test_schedule_orders_every_conflict(name, side, precision, monkeypatch):
    for B in ((2, 257) if side == "both" else (2,)):
        prog = _program(name, precision, B, side, monkeypatch)
        problems = _problems(prog)
        assert not problems, f"{name} {side} {precision} B={B}:\n" + "\n".join(problems)


def test_cross0_fusion_tail_joins_the_text_lane(monkeypatch):
    """Without cross layers the fusion tail's first op waits for the side lane (no buffer of the cross layers is
    allocated); dropping that join is named: the text encoder's final norm and the pool race on text_features."""
    for name in ("cross0", "text0_cross0"):
        prog = _program(name, "bf16", 2, "both", monkeypatch)
        assert not any(n.startswith("x.") for n in prog.named), sorted(n for n in prog.named if n.startswith("x."))
        op = next(o for o in prog.ops if o.name == "fusion.pool")
        assert op.lane == P.LANE_JOIN
        op.lane &= ~P.LANE_JOIN
        msg = "\n".join(_problems(prog))
        print(msg)
        assert "text.lnf [side, w] and fusion.pool [main, r] both touch text_features unordered" in msg, msg
        assert "JOIN is missing on fusion.pool" in msg, msg
        assert "fusion.pool.text reads" in msg and "of text_features" in msg, msg


def test_programs_with_cross_layers_keep_their_joins(monkeypatch):
    """The tail join is added only where no cross-attention op joined the lanes."""
    for name in ("cross1", "nogate_cross2", "se1"):
        prog = _program(name, "bf16", 2, "both", monkeypatch)
        joins = [o.name for o in prog.ops if o.lane & P.LANE_JOIN]
        assert not any(n.startswith("fusion.") for n in joins), joins
        assert "x.0.attn" in joins


@pytest.mark.parametrize("name", NAMES)
def test_layers_on_the_emulator(name, monkeypatch):
    for k, v in MO.ENV.get(name, {}).items():
        monkeypatch.setenv(k, v)
    MO.relax_spatial_gate(name, monkeypatch)
    prog, sd, ext = MO.make_case(name, 2, "cpu", seed=11)
    LP.poison(prog)
    rep = LP.check_on_emulator(prog, sd, ext, title=name)
    print(rep.table())
    assert not rep.failures(), rep.table()
    n_text = MO.MATRIX[name].get("num_transformer_layers", 4)
    assert sum(r.module.startswith("text.") and r.module[5:].isdigit() for r in rep.rows) == n_text
    assert sum(r.module.startswith("x.") and r.output == "x.q" for r in rep.rows) == MO.n_cross(name)


# ----------------------------------------------------------------------------- refusals
def test_encode_images_refuses_more_cached_layers_than_slots():
    """Nine cross layers: forward runs, but the question side reads K/V from one slot per layer (8).  encode_images
    refuses before it builds an engine (here there is no GPU to build one on) and names the limit."""
    model = VQAModel(**MO.MATRIX["cross9"]).eval()
    with pytest.raises(NotImplementedError, match="at most 8|up to 8"):
        model.encode_images(torch.zeros(1, 3, 224, 224))
    assert model._engine is None


@pytest.mark.parametrize("N,ok", [(50000, True), (50001, False), (100000, False)])
def test_plan_for_refuses_top_k_beyond_the_kernel_limit(N, ok, monkeypatch):
    """predict (top_k >= 1) on a head the top-k kernel cannot hold raises ValueError in plan_for, before any program is
    built; forward (top_k = 0) has no limit.  (An Engine needs a GPU; here one is assembled without its weights, and
    building a program stops the call.)"""
    from vqa_b200.engine import MAX_TOP_K_ANSWERS, Engine
    assert MAX_TOP_K_ANSWERS == 50000
    eng = Engine.__new__(Engine)
    eng.cfg = dict(num_answers=N, max_question_length=20)
    eng._plans, eng.window, eng.max_plans, eng.weights, eng.device = {}, True, 16, None, torch.device("cpu")
    built = []

    def no_build(*a, **k):
        built.append(k["top_k"] if "top_k" in k else a[7])
        raise RuntimeError("stop: a program would be built")
    monkeypatch.setattr(P, "Program", no_build)
    for k in (1, 5, 0):
        if ok or k == 0:
            with pytest.raises(RuntimeError, match="stop"):
                eng.plan_for(2, 20, "nchw_f32", P.MASK_I64, False, k)
        else:
            with pytest.raises(ValueError, match="50000"):
                eng.plan_for(2, 20, "nchw_f32", P.MASK_I64, False, k)
    assert built == ([1, 5, 0] if ok else [0])


def test_supported_states_every_remaining_limit():
    from vqa_b200.engine import MAX_TOP_K_ANSWERS
    for needle in ("512", str(MAX_TOP_K_ANSWERS), f"{P.MAX_CACHED_LAYERS} cross-attention layers", "se_reduction",
                   "Layer counts (0 included)", "image cache"):
        assert needle in _SUPPORTED, needle
