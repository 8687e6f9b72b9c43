"""Layer-by-layer parity of libvqa_b200 at the shapes the product runs (tests/layer_parity.py): every module of the
forward -- ingest, stem, each convolution, each block output, each stage tail with its SE scale and spatial map, the
projector, each K/V projection, the embedding, each text layer, the final norm, each cross layer with its attention
weights, pools / gate / output norm, head and top-k -- against an fp64 restatement of its reference module applied to
the module's own inputs as the GPU left them, plus every pad cell of every padded-flat grid exactly 0.

The fp64 references run on the same device (torch, fp64), one module at a time between op ranges of the plan; the whole
file takes about 15 s on a B200.  Worst max|err| / max|ref| measured on B200 (1000 W), per class:

    case             ingest   conv (backbone)  linear   fp32      channel mean
    bf16 B=256       2.95e-3  4.29e-3          6.56e-4  2.48e-7   8.69e-3
    bf16 u8 B=1024   2.95e-3  4.54e-3          6.31e-4  1.91e-7   8.60e-3
    tf32 B=256       3.69e-4  6.49e-4          1.10e-5  2.91e-7   1.07e-3

The gates (tests/layer_parity.py) sit at 2-3x the worst over every case.
"""
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

import layer_parity as LP  # noqa: E402

DRY = bool(os.environ.get("VQA_DRY"))     # CPU-only rehearsal of the test's Python side: the emulator stands in
DEV = "cpu" if DRY else "cuda"


def _check(prog, sd, ext, imgs=None, title=""):
    if DRY:
        rep = LP.check_on_emulator(prog, sd, ext, imgs=imgs, title=title)
    else:
        from vqa_b200.runtime import Plan
        plan = Plan(prog.ops, 0)
        ptrs = [0 if t is None else t.data_ptr() for t in ext]
        stream = torch.cuda.current_stream().cuda_stream

        def runner(first, last):
            plan.run(ptrs, stream, first, last)
            torch.cuda.synchronize()
        rep = LP.Checker(prog, sd, ext, runner, imgs=imgs, kernel_name=plan.kernel_name, title=title).run()
    print(rep.table())
    print("worst", title, {c: f"{rep.worst(c):.2e}" for c in ("ingest", "conv", "linear", "fp32")},
          f"chan {max((r.chan for r in rep.rows if r.chan is not None), default=0.0):.2e}")
    assert not rep.failures(), rep.table()
    return rep


@pytest.mark.parametrize("B", [1, 7, 255, 256, 257])
def test_layers_bf16_fp32_nchw(B):
    """bf16 mode, fp32 NCHW images.  256 is the benchmark shape; 255 and 257 end in a partial last tile and land on
    different persistent-walker counts and cluster tails."""
    prog, sd, ext = LP.make_case({}, B, device=DEV, seed=4242 + B)
    _check(prog, sd, ext, title=f"bf16 B={B}")


def test_layers_uint8_1024():
    """uint8 HWC images with the normalisation on the GPU, 1024 per call.  The backbone is checked on the first and last
    image and 14 seeded others; pads, projector, K/V and the text / fusion / head side on every image and pair."""
    B = 1024
    prog, sd, ext = LP.make_case({}, B, in_fmt="hwc_u8", device=DEV, seed=777)
    g = torch.Generator().manual_seed(11)
    imgs = sorted({0, B - 1} | set((1 + torch.randperm(B - 2, generator=g)[:14]).tolist()))
    _check(prog, sd, ext, imgs=imgs, title="bf16 u8 B=1024")


def test_layers_tf32_256():
    """precision="tf32": fp32 activations and tf32 operands in the backbone, 3xTF32 Linears, at the benchmark shape."""
    prog, sd, ext = LP.make_case({}, 256, precision="tf32", device=DEV, seed=99)
    _check(prog, sd, ext, title="tf32 B=256")


def test_layers_one_image_sixteen_questions():
    """One image answering 16 questions of 64 tokens: the image side runs once, its K/V serve every question."""
    prog, sd, ext = LP.make_case(dict(max_question_length=64), 16, L=64, n_images=1, device=DEV, seed=77)
    assert prog.Bi == 1
    _check(prog, sd, ext, title="1 image x 16 questions")


@pytest.mark.parametrize("name,kw", [
    ("ablate", dict(ctor=LP.ABLATE, mask_kind="none")),
    ("nospatial", dict(ctor=LP.NOSPATIAL, mask_kind="f32")),
    ("answers3129", dict(ctor=dict(vocab_size=20000, num_answers=3129, num_transformer_layers=1, num_cross_layers=3,
                                   se_reduction=4))),
])
def test_layers_model_variants(name, kw):
    """No attention / gating, no spatial attention, and an odd 3129-answer head (padded logits + copy_rows)."""
    prog, sd, ext = LP.make_case(B=3, device=DEV, seed=5, **kw)
    if name == "answers3129":
        assert any(op.kind == "copy_rows" for op in prog.ops)
    _check(prog, sd, ext, title=name)
