"""The concurrent schedule against the serial one, bit for bit, on a poisoned workspace.

The fp64 layer checks (tests/test_gpu_layer_parity.py, tests/layer_parity.py) run a plan in op ranges, serially, on one
stream.  The product runs it whole: the side lane on the plan's side stream with fork / join events, kernels overlapping
through programmatic dependent launch, plans replayed from CUDA graphs, several slots in flight on several streams.  Here
each case

  1. poisons the workspace (0xFF bytes: NaN in fp32, bf16 and fp16; ``layer_parity.poison``), walks the plan serially
     under the fp64 gates of ``layer_parity.Checker`` and snapshots every workspace byte and the outputs (input set A);
     the same, op by op without the gates, for a second seeded input set B;
  2. re-poisons and runs the whole plan: every byte equals A's serial snapshot (NaN rows of a fully masked question too);
  3. runs the whole plan on B and then on A again without re-poisoning: a kernel that read the previous run's
     intermediate, or a byte that no op of the run writes, shows as a difference;
  4. captures the whole plan (both lanes) in a CUDA graph the way VQAInference does and replays it with A, B and A.

Three slots with their own workspaces run different inputs concurrently on three streams, and the pipelined predict path
with its defaults (3 lanes, 6 input slots) reuses every slot with new batches.  Every sequence runs once; nothing repeats
to provoke a race.  Under VQA_DRY=1 the CPU emulator stands in for the library (small batches, no graphs, no slots), so
the Python side can be rehearsed without a GPU.
"""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

import emulator as E  # noqa: E402
import layer_parity as LP  # noqa: E402
from vqa_b200 import program as P  # noqa: E402
from vqa_b200.synth import synth_batch  # noqa: E402

DRY = bool(os.environ.get("VQA_DRY"))
DEV = "cpu" if DRY else "cuda"
OUTS = ("logits", "top_idx", "top_probs")


def _b(B):
    return min(B, 2) if DRY else B


class Runner:
    """One program on libvqa_b200 (the CPU emulator under VQA_DRY)."""

    def __init__(self, prog, ext):
        self.prog, self.ext = prog, ext
        if DRY:
            self.emu = E.Emulator(prog)
        else:
            from vqa_b200.runtime import Plan
            self.plan = Plan(prog.ops, 0)
            self.ptrs = [0 if t is None else t.data_ptr() for t in ext]

    def kernel_name(self, k):
        return "" if DRY else self.plan.kernel_name(k)

    def serial(self, first, last):
        """Ops [first, last) on the current stream (partial ranges never use the side lane), then a device sync."""
        if DRY:
            self.emu.run(self.ext, first, last)
        else:
            self.plan.run(self.ptrs, torch.cuda.current_stream().cuda_stream, first, last)
            torch.cuda.synchronize()

    def op_by_op(self):
        for k in range(len(self.prog.ops)):
            self.serial(k, k + 1)

    def whole(self, stream=None):
        """The whole plan: two lanes, programmatic dependent launch.  No sync."""
        if DRY:
            self.emu.run(self.ext)
        else:
            self.plan.run(self.ptrs, (stream or torch.cuda.current_stream()).cuda_stream)

    def snapshot(self):
        return self.prog.ws.tensor.clone(), {n: self.ext[P.EXT[n]].clone() for n in OUTS}

    def compare(self, tag, snap):
        if not DRY:
            torch.cuda.synchronize()
        ws, outs = snap
        cur = self.prog.ws.tensor
        bad = []
        if not torch.equal(cur, ws):
            diff = cur != ws
            covered = 0
            for b in self.prog.ws._bufs:
                n = int(diff[b.offset: b.offset + b.nbytes].sum())
                covered += n
                if n:
                    bad.append(f"{b.name} ({n} of {b.nbytes} B)")
            rest = int(diff.sum()) - covered
            if rest:
                bad.append(f"{rest} B outside every allocation")
        for n in OUTS:
            a, b = self.ext[P.EXT[n]], outs[n]
            if not torch.equal(a.reshape(-1).view(torch.uint8), b.reshape(-1).view(torch.uint8)):
                bad.append(f"output {n}")
        assert not bad, f"{tag}: differs from the serial run in " + ", ".join(bad)


def _inputs(prog, ext, seed, masked_rows=()):
    """A second seeded input set of the shapes and types ``ext`` holds."""
    cfg = prog.cfg
    u8, img, ids, mask = synth_batch(prog.B, seed, max_len=prog.L, vocab=cfg["vocab_size"])
    out = {"images": (u8 if prog.in_fmt == "hwc_u8" else img)[:prog.Bi], "ids": ids}
    m = ext[P.EXT["mask"]]
    if m is not None:
        mask = mask.to(m.dtype)
        mask[list(masked_rows)] = 0
        out["mask"] = mask
    return out


def _current(ext):
    return {n: ext[P.EXT[n]].clone() for n in ("images", "ids", "mask") if ext[P.EXT[n]] is not None}


def _set(ext, inputs):
    for n, t in inputs.items():
        ext[P.EXT[n]].copy_(t)


def _serial_checked(run, sd, imgs=None, title="", image_projected=None):
    LP.poison(run.prog)
    rep = LP.Checker(run.prog, sd, run.ext, run.serial, imgs=imgs, kernel_name=run.kernel_name, title=title,
                     image_projected=image_projected).run()
    assert not rep.failures(), rep.table()
    return run.snapshot()


def _serial_plain(run, inputs):
    _set(run.ext, inputs)
    LP.poison(run.prog)
    run.op_by_op()
    return run.snapshot()


def _concurrent(run, title, snap_a, a, snap_b, b):
    """Whole-plan runs and graph replays against the serial snapshots of input sets a and b."""
    _set(run.ext, a)
    LP.poison(run.prog)
    run.whole()
    run.compare(f"{title}: whole plan, A", snap_a)
    for tag, inp, snap in (("B after A", b, snap_b), ("A after B", a, snap_a)):
        _set(run.ext, inp)
        run.whole()
        run.compare(f"{title}: whole plan, {tag} (no re-poison)", snap)
    if DRY:
        return
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        run.whole()
    for tag, inp, snap in (("A", a, snap_a), ("B", b, snap_b), ("A again", a, snap_a)):
        _set(run.ext, inp)
        graph.replay()
        run.compare(f"{title}: graph replay, {tag}", snap)


def _case(title, ctor=None, seed=5, imgs=None, masked_rows=(), **kw):
    prog, sd, ext = LP.make_case(ctor or {}, device=DEV, seed=seed, **kw)
    run = Runner(prog, ext)
    a = _current(ext)
    snap_a = _serial_checked(run, sd, imgs=imgs, title=title)
    b = _inputs(prog, ext, seed + 1000, masked_rows)
    snap_b = _serial_plain(run, b)
    _concurrent(run, title, snap_a, a, snap_b, b)
    return prog, sd, run, snap_a, a


@pytest.mark.parametrize("B", [256, 1, 257])
def test_whole_plan_matches_serial_bf16(B):
    _case(f"bf16 B={_b(B)}", B=_b(B), seed=4242 + B)


def test_whole_plan_matches_serial_uint8_1024():
    B = _b(1024)
    g = torch.Generator().manual_seed(11)
    imgs = sorted({0, B - 1} | set((1 + torch.randperm(B - 2, generator=g)[:14]).tolist())) if B > 16 else None
    _case(f"bf16 u8 B={B}", B=B, in_fmt="hwc_u8", seed=777, imgs=imgs)


def test_whole_plan_matches_serial_tf32():
    _case("tf32", B=_b(256), precision="tf32", seed=99)


def test_whole_plan_matches_serial_one_image_sixteen_questions():
    prog = _case("1 image x 16 questions", ctor=dict(max_question_length=64), B=16, L=64, n_images=1, seed=77)[0]
    assert prog.Bi == 1


def test_whole_plan_matches_serial_three_cross_layers_masked_question():
    """3 cross layers (the side lane projects K/V of layers 1 and 2), 3129 answers (padded logits + copy_rows), and a
    fully masked question, whose NaN logits must come out in the same bits."""
    B = 3
    _, _, ids, mask = synth_batch(B, 5, max_len=20, vocab=20000)
    mask[1] = 0
    prog, _, run, _, _ = _case("3 cross layers, 3129 answers", ctor=dict(vocab_size=20000, num_answers=3129,
                               num_transformer_layers=1, num_cross_layers=3, se_reduction=4), B=B, ids=ids, mask=mask,
                               masked_rows=(1,))
    assert any(op.kind == "copy_rows" for op in prog.ops)
    logits = run.ext[P.EXT["logits"]]
    assert bool(torch.isnan(logits[1]).all()) and not bool(torch.isnan(logits[[0, 2]]).any())


@pytest.mark.parametrize("env", ["VQA_FUSED_TOPK=1", "VQA_CHAIN=0"])
def test_whole_plan_matches_serial_switches(env, monkeypatch):
    k, v = env.split("=")
    monkeypatch.setenv(k, v)
    prog = _case(env, B=_b(256), seed=31)[0]
    if k == "VQA_FUSED_TOPK":
        assert any(op.p.get("topk_cnt") is not None for op in prog.ops)
    else:
        assert not any(op.kind == "mlp_chain" for op in prog.ops)


def test_encode_images_and_answer_match_serial():
    """The image side alone (side="image") and the question side against its K/V (side="question")."""
    Bi, B = _b(64), _b(256)
    B -= B % Bi
    prog_i, sd, ext_i = LP.make_case({}, Bi, device=DEV, seed=61, side="image")
    run_i = Runner(prog_i, ext_i)
    a_i, b_i = _current(ext_i), _inputs(prog_i, ext_i, 62)
    snap_bi = _serial_plain(run_i, b_i)
    snap_ai = _serial_plain(run_i, a_i)
    _concurrent(run_i, "image side", snap_ai, a_i, snap_bi, b_i)

    _set(ext_i, a_i)
    run_i.whole()
    if not DRY:
        torch.cuda.synchronize()
    prog_q, sd_q, ext_q = LP.make_case({}, B, device=DEV, seed=63, n_images=Bi, side="question")
    for l in range(prog_q.n_cross_layers):
        ext_q[P.EXT[f"kv{l}"]] = prog_i.tensor(f"x.{l}.kv").reshape(-1).clone()
    run_q = Runner(prog_q, ext_q)
    a_q = _current(ext_q)
    img = prog_i.tensor("image_projected").view(Bi, 49, -1).clone()
    snap_aq = _serial_checked(run_q, sd_q, title="question side", image_projected=img)
    b_q = _inputs(prog_q, ext_q, 64)
    b_q.pop("images", None)
    snap_bq = _serial_plain(run_q, b_q)
    _concurrent(run_q, "question side", snap_aq, a_q, snap_bq, b_q)


@pytest.mark.skipif(DRY, reason="streams and slots need the GPU")
def test_three_slots_on_three_streams():
    """Three plans (own workspaces), different inputs, issued back to back on three streams with no sync between."""
    B = 256
    prog, sd, ext = LP.make_case({}, B, device=DEV, seed=7)
    runs = [Runner(prog, ext)]
    for slot in (1, 2):
        p = P.Program(prog.W, prog.cfg, B, prog.L, prog.in_fmt, prog.mask_dtype, want_aux=True, top_k=prog.top_k,
                      device=DEV)
        e = [None if t is None else t.clone() for t in ext]
        runs.append(Runner(p, e))
    inputs = [_inputs(prog, ext, 7 + 100 * s) for s in range(3)]
    snaps = [_serial_plain(r, inp) for r, inp in zip(runs, inputs)]
    for r in runs:
        LP.poison(r.prog)
    streams = [torch.cuda.Stream() for _ in runs]
    for r, s in zip(runs, streams):
        s.wait_stream(torch.cuda.current_stream())
        r.whole(s)
    torch.cuda.synchronize()
    for slot, (r, snap) in enumerate(zip(runs, snaps)):
        r.compare(f"slot {slot}", snap)


@pytest.mark.skipif(DRY, reason="VQAInference runs on the GPU only")
def test_pipelined_predict_reuses_every_slot():
    """predict_tensors_pipelined with its defaults (3 lanes, 6 input slots, one CUDA graph per slot) over 9 distinct
    batches, so slots 0-2 are refilled with new data: each result equals predict on that batch alone, bit for bit."""
    from vqa_b200 import VQAInference
    torch.manual_seed(0)
    inf = VQAInference()
    inf.load()
    assert inf.pipeline_lanes == 3 and not getattr(inf, "pipeline_slots", 0) and inf.use_cuda_graph
    batches = []
    for i in range(9):
        u8, _, ids, mask = synth_batch(6, 900 + i)
        batches.append((u8.pin_memory(), ids.pin_memory(), mask.pin_memory()))
    outs = list(inf.predict_tensors_pipelined(batches, top_k=5))
    assert len(outs) == 9
    inf.use_cuda_graph = False
    for i, ((u8, ids, mask), (idx, probs)) in enumerate(zip(batches, outs)):
        ridx, rprobs = inf._run(u8, ids, mask, 5)
        assert torch.equal(idx, ridx) and torch.equal(probs, rprobs), f"batch {i} (slot {i % 6})"
