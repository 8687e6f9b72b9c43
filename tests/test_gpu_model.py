"""End-to-end parity of the sm_100a VQAModel with the oracle / golden vectors of the reference."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from conftest import GOLDEN, REPO  # noqa: E402
import layer_parity as LP  # noqa: E402

sys.path.insert(0, REPO)
from oracle import vqa_oracle as O  # noqa: E402
from vqa_b200.model import VQAModel, create_vqa_model, load_vqa_model  # noqa: E402
from vqa_b200.synth import randomise_state, synth_batch  # noqa: E402

# BASELINE.json north_star: bf16 mode, logits within 2e-2 max-abs relative error
LOGIT_REL_TOL = 2e-2


def rel_err(got, want):
    return float((got - want).abs().max() / want.abs().max())


def make(meta, precision="bf16"):
    torch.manual_seed(meta["seed_weights"])
    model = VQAModel(**meta["ctor"], precision=precision).eval()
    sd = model.state_dict()
    if meta["randomise"]:
        sd = randomise_state(sd, 1)
        model.load_state_dict(sd, strict=True)
    u8, img, ids, mask = synth_batch(meta["batch"], meta["seed_inputs"], max_len=meta["max_len"], vocab=meta["vocab"])
    return model.cuda(), sd, u8, img, ids, mask


@pytest.mark.parametrize("case", ["default_b4", "plain_b2", "ablate_b3", "nospatial_b2"])
def test_forward_matches_reference_golden(golden_meta, case):
    meta = golden_meta[case]
    model, sd, u8, img, ids, mask = make(meta)
    g = np.load(os.path.join(GOLDEN, f"{case}.npz"))
    with torch.no_grad():
        logits, aux = model(img.cuda(), ids.cuda(), mask.cuda(), return_aux=True)
    torch.cuda.synchronize()
    assert logits.dtype == torch.float32 and tuple(logits.shape) == g["logits"].shape
    errs = {"logits": rel_err(logits.cpu(), torch.from_numpy(g["logits"]))}
    for k in ("image_features", "text_features", "fused", "image_projected", "attended_pooled", "text_pooled"):
        errs[k] = rel_err(aux[k].cpu(), torch.from_numpy(g[k]))
    for i, w in enumerate(aux["cross_attention_weights"]):
        errs[f"xattn{i}"] = rel_err(w.cpu(), torch.from_numpy(g[f"cross_attention_weights_{i}"]))
    print(case, {k: f"{v:.2e}" for k, v in errs.items()})
    assert errs["logits"] <= LOGIT_REL_TOL, errs
    assert errs["image_features"] <= 5e-2, errs      # bf16 backbone, 17 conv layers deep
    assert errs["text_features"] <= 1e-2 and errs["fused"] <= 5e-2, errs
    # every aux tensor of models/vqa_model.py:301-309 is gated, not only the ones the logits depend on most
    assert errs["image_projected"] <= 5e-2 and errs["attended_pooled"] <= 5e-2 and errs["text_pooled"] <= 1e-2, errs
    assert all(v <= 5e-2 for k, v in errs.items() if k.startswith("xattn")), errs
    top_idx, top_p = model.predict(img.cuda(), ids.cuda(), mask.cuda(), top_k=5)
    assert top_idx.dtype == torch.int64 and tuple(top_idx.shape) == (meta["batch"], 5)
    assert np.array_equal(top_idx[:, 0].cpu().numpy(), g["top_indices"][:, 0])
    np.testing.assert_allclose(top_p.cpu().numpy(), g["top_probs"], rtol=2e-2, atol=1e-4)


@pytest.mark.parametrize("case", ["default_b4", "plain_b2", "ablate_b3", "nospatial_b2"])
def test_backbone_stage_taps_match_golden(golden_meta, case):
    """VERDICT r1: logits barely see the image (SURVEY T11), so a backbone bug could hide behind the logit gate.  The
    golden files hold strided samples of the reference's own stem / stage outputs (models/cnn_backbone.py:267-279,
    349-354, taken through the reference modules by tests/golden/make_golden.py); the CUDA path's buffers after the
    fused stem+pool, after every stage's residual blocks and after every stage's attention are checked against them."""
    meta = golden_meta[case]
    model, sd, u8, img, ids, mask = make(meta)
    g = np.load(os.path.join(GOLDEN, f"{case}.npz"))
    with torch.no_grad():
        _, _, _, prog = model.engine().run(img.cuda(), ids.cuda(), mask.cuda())
    torch.cuda.synchronize()
    got = {"stem": LP.grid_nchw(prog, "s1.in", 56, 56)[0]}
    for s, hw in enumerate((56, 28, 14, 7), start=1):
        got[f"stage{s}.blocks"] = LP.grid_nchw(prog, f"s{s}.b1.out", hw, hw)[0]
        if s < 4:
            got[f"stage{s}"] = LP.phases_nchw(prog, f"s{s + 1}.in", hw, hw)[0]
        else:
            got[f"stage{s}"] = LP.grid_nchw(prog, prog.feat_name, hw, hw)[0]
    errs = {}
    for k, v in got.items():
        v = v.float().cpu()
        want = torch.from_numpy(g[f"tap.{k}.sample"])
        sample = v.flatten()[::997]
        assert sample.shape == want.shape, (k, sample.shape, want.shape)
        errs[k] = float((sample - want).abs().max() / want.abs().max())
    print(case, {k: f"{v:.2e}" for k, v in errs.items()})
    assert errs["stem"] <= 1.5e-2, errs                       # one bf16 convolution + pool
    assert all(v <= 5e-2 for v in errs.values()), errs        # up to 17 bf16 convolutions deep


def test_batch256_fp32_nchw_matches_oracle():
    """BASELINE configs[1] at its own size: 256 pairs, fp32 NCHW images, 20-token questions, against the fp32 oracle."""
    torch.manual_seed(0)
    model = VQAModel().eval()
    sd = randomise_state(model.state_dict(), 1)
    model.load_state_dict(sd, strict=True)
    model = model.cuda()
    _, img, ids, mask = synth_batch(256, 4242)
    with torch.no_grad():
        got, aux = model(img.cuda(), ids.cuda(), mask.cuda(), return_aux=True)
    want, waux = O.vqa_forward(sd, img, ids, mask, return_aux=True)
    got = got.cpu()
    errs = {"logits": rel_err(got, want)}
    for k in ("image_features", "text_features", "fused", "image_projected", "attended_pooled", "text_pooled"):
        errs[k] = rel_err(aux[k].cpu(), waux[k])
    agree = float((got.argmax(1) == want.argmax(1)).float().mean())
    print("B=256", {k: f"{v:.2e}" for k, v in errs.items()}, f"top-1 agreement {agree:.4f}")
    assert errs["logits"] <= LOGIT_REL_TOL and errs["image_features"] <= 5e-2 and errs["text_features"] <= 1e-2, errs
    assert errs["fused"] <= 5e-2 and errs["image_projected"] <= 5e-2 and errs["attended_pooled"] <= 5e-2, errs
    assert agree >= 0.98            # 256 pairs: the 99 % gate is checked on 10 000 pairs below
    # every row of the big batch equals the same pair run in a small batch (tiles / CTAs do not leak between images)
    with torch.no_grad():
        small, _ = model(img[100:104].cuda(), ids[100:104].cuda(), mask[100:104].cuda())
    assert torch.equal(small.cpu(), got[100:104])


def test_batch1024_uint8_matches_oracle_sample():
    """BASELINE configs[2] per GPU: 1024 uint8 HWC images + questions in one step, GPU preprocessing included; the
    oracle (fp32 CPU) checks every 16th pair."""
    torch.manual_seed(0)
    model = VQAModel().eval()
    sd = model.state_dict()
    model = model.cuda()
    u8, img, ids, mask = synth_batch(1024, 777)
    with torch.no_grad():
        got, _ = model(u8.cuda(), ids.cuda(), mask.cuda())
        idx, probs = model.predict(u8.cuda(), ids.cuda(), mask.cuda(), top_k=5)
    got = got.cpu()
    pick = torch.arange(0, 1024, 16)
    want, _ = O.vqa_forward(sd, O.preprocess_u8(u8[pick]), ids[pick], mask[pick])
    err = rel_err(got[pick], want)
    agree = float((got[pick].argmax(1) == want.argmax(1)).float().mean())
    print(f"B=1024 u8: logits rel err {err:.2e}, top-1 agreement on the 64-pair sample {agree:.3f}")
    assert err <= LOGIT_REL_TOL and agree >= 0.95
    assert torch.equal(idx[:, 0].cpu(), got.argmax(1))
    wi, wp = O.predict_topk(got, 5)
    assert torch.equal(idx.cpu(), wi)
    np.testing.assert_allclose(probs.cpu().numpy(), wp.numpy(), rtol=1e-4, atol=1e-7)


def test_fully_masked_row_and_weighted_float_mask():
    """ADVICE r1.  (1) An all-zero mask row makes the reference's self-attention softmax NaN (models/text_encoder.py:244)
    and its logits NaN; predict(top_k=5) must return that (NaN probabilities) without faulting -- the top-k kernel used
    to index shared memory with 0x7fffffff on a NaN row -- also under CUDA-graph replay, and the other rows stay right.
    (2) The masked mean pools weigh tokens with attention_mask.float() (models/fusion.py:303-313): a float mask with
    weights other than 0 / 1 must match the oracle, not a binarised mask."""
    torch.manual_seed(0)
    model = VQAModel().eval()
    sd = model.state_dict()
    model = model.cuda()
    _, img, ids, mask = synth_batch(6, 31)
    dead = mask.clone()
    dead[2] = 0
    x, t, m = img.cuda(), ids.cuda(), dead.cuda()
    idx, probs = model.predict(x, t, m, top_k=5)
    torch.cuda.synchronize()
    want, _ = O.vqa_forward(sd, img, ids, dead)
    assert bool(torch.isnan(want[2]).all()) and bool(torch.isnan(probs[2]).all())
    assert bool(((idx[2] >= 0) & (idx[2] < 1000)).all()) and len(set(idx[2].tolist())) == 5
    live = [0, 1, 3, 4, 5]
    assert torch.equal(idx[live, 0].cpu(), want[live].argmax(1))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gi, gp = model.predict(x, t, m, top_k=5)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(gi.cpu(), idx.cpu()) and bool(torch.isnan(gp[2]).all())
    with torch.no_grad():
        ok, _ = model(x, t, mask.cuda())                      # the context survived: a normal forward still works
    assert rel_err(ok.cpu(), O.vqa_forward(sd, img, ids, mask)[0]) <= LOGIT_REL_TOL
    # (2) weighted float mask
    wmask = mask.float() * (0.25 + 0.5 * (torch.arange(mask.shape[1]) % 3).float()).view(1, -1)   # per-token weights
    with torch.no_grad():
        got, aux = model(x, t, wmask.cuda(), return_aux=True)
    want, waux = O.vqa_forward(sd, img, ids, wmask, return_aux=True)
    assert rel_err(got.cpu(), want) <= LOGIT_REL_TOL
    assert rel_err(aux["text_pooled"].cpu(), waux["text_pooled"]) <= 1e-2
    binar, _ = O.vqa_forward(sd, img, ids, mask)
    assert rel_err(want, binar) > 1e-3                        # the weights do matter in the reference
    with pytest.raises(ValueError):
        model.predict(x, t, m, top_k=0)
    with pytest.raises(ValueError):
        model.predict(x, t, m, top_k=1001)


@pytest.mark.parametrize("case", ["default_b4", "plain_b2", "ablate_b3", "nospatial_b2"])
def test_tf32_tolerance_mode_within_1e_3(golden_meta, case):
    """BASELINE.json: "in fp32-accumulate TF32 mode, logits must be within 1e-3" (max-abs relative) of the fp32
    reference.  precision="tf32": fp32 activations and tf32 operands in the backbone, 3xTF32 Linears in the tail."""
    meta = golden_meta[case]
    model, sd, u8, img, ids, mask = make(meta, precision="tf32")
    g = np.load(os.path.join(GOLDEN, f"{case}.npz"))
    with torch.no_grad():
        logits, aux = model(img.cuda(), ids.cuda(), mask.cuda(), return_aux=True)
        logits_u8, _ = model(u8.cuda(), ids.cuda(), mask.cuda())
    errs = {"logits": rel_err(logits.cpu(), torch.from_numpy(g["logits"])),
            "image_features": rel_err(aux["image_features"].cpu(), torch.from_numpy(g["image_features"])),
            "text_features": rel_err(aux["text_features"].cpu(), torch.from_numpy(g["text_features"])),
            "fused": rel_err(aux["fused"].cpu(), torch.from_numpy(g["fused"]))}
    print("tf32", case, {k: f"{v:.2e}" for k, v in errs.items()})
    assert errs["logits"] <= 1e-3, errs
    assert errs["image_features"] <= 2e-3 and errs["text_features"] <= 1e-4 and errs["fused"] <= 1e-3, errs
    assert torch.equal(logits_u8, logits)
    assert np.array_equal(logits.argmax(1).cpu().numpy(), g["top_indices"][:, 0])


def test_large_answer_and_word_vocabularies():
    """VQA-v2-sized head (3129 answers: wider than the epilogue's 2048-entry bias table) and a 20k-word embedding."""
    torch.manual_seed(0)
    model = VQAModel(vocab_size=20000, num_answers=3129, num_transformer_layers=1, num_cross_layers=3, se_reduction=4).eval()
    sd = randomise_state(model.state_dict(), 1)
    model.load_state_dict(sd, strict=True)
    model = model.cuda()
    u8, img, ids, mask = synth_batch(3, 5, vocab=20000)
    with torch.no_grad():
        logits, _ = model(img.cuda(), ids.cuda(), mask.cuda())
    want, _ = O.vqa_forward(sd, img, ids, mask)
    assert tuple(logits.shape) == (3, 3129) and rel_err(logits.cpu(), want) <= LOGIT_REL_TOL
    assert torch.equal(logits.argmax(1).cpu(), want.argmax(1))


def test_one_image_many_questions():
    """BASELINE configs[4]: one image, 16 questions of 64 tokens on VQAModel(max_question_length=64); the backbone,
    projector and K/V projections run once per image.  Must equal the plain forward on the repeated image bit for
    bit, and match the fp32 oracle within the bf16 gate."""
    torch.manual_seed(0)
    model = VQAModel(max_question_length=64).eval()
    sd = randomise_state(model.state_dict(), 1)
    model.load_state_dict(sd, strict=True)
    model = model.cuda()
    u8, img, ids, mask = synth_batch(16, 77, max_len=64)
    one = img[:1]
    with torch.no_grad():
        shared, aux = model(one.cuda(), ids.cuda(), mask.cuda(), return_aux=True)
        plain, _ = model(one.repeat(16, 1, 1, 1).cuda(), ids.cuda(), mask.cuda())
        two, _ = model(img[:2].cuda(), ids.cuda(), mask.cuda())          # 2 images x 8 questions
        plain2, _ = model(img[:2].repeat_interleave(8, dim=0).cuda(), ids.cuda(), mask.cuda())
    assert tuple(shared.shape) == (16, 1000) and tuple(aux["image_features"].shape) == (1, 512, 7, 7)
    assert torch.equal(shared, plain) and torch.equal(two, plain2)
    want, _ = O.vqa_forward(sd, one.repeat(16, 1, 1, 1), ids, mask)
    assert rel_err(shared.cpu(), want) <= LOGIT_REL_TOL
    idx, probs = model.predict(one.cuda(), ids.cuda(), mask.cuda(), top_k=3)
    assert tuple(idx.shape) == (16, 3)
    with pytest.raises(ValueError):
        model(img[:3].cuda(), ids.cuda(), mask.cuda())                    # 16 questions over 3 images


def test_uint8_input_equals_normalised_input(golden_meta):
    model, sd, u8, img, ids, mask = make(golden_meta["plain_b2"])
    with torch.no_grad():
        a, _ = model(img.cuda(), ids.cuda(), mask.cuda())
        b, _ = model(u8.cuda(), ids.cuda(), mask.cuda())
    assert torch.equal(a, b)  # same fp32 normalisation arithmetic, same bf16 rounding


def test_mask_variants_and_padding_invariance(golden_meta):
    model, sd, u8, img, ids, mask = make(golden_meta["plain_b2"])
    x, t, m = img.cuda(), ids.cuda(), mask.cuda()
    with torch.no_grad():
        a, _ = model(x, t, m)
        b, _ = model(x, t, m.float())
        c, _ = model(x, t, m.int())
        d, _ = model(x, torch.where(m == 0, torch.full_like(t, 17), t), m)
        e, _ = model(x, t, m.bool())
        f, _ = model(x, t, m.to(torch.uint8))
        full, _ = model(x, t, None)
        want_full, _ = O.vqa_forward(sd, img, ids, None)
    assert torch.equal(a, b) and torch.equal(a, c) and torch.equal(a, d) and torch.equal(a, e) and torch.equal(a, f)
    assert rel_err(full.cpu(), want_full) <= LOGIT_REL_TOL
    # a uint8 mask is read as weights, like the same values in fp32 (the masked mean pools weigh tokens by the mask)
    w = mask * (1 + torch.arange(mask.shape[1]) % 3).view(1, -1)       # values 0..3
    with torch.no_grad():
        wu, _ = model(x, t, w.to(torch.uint8).cuda())
        wf, _ = model(x, t, w.float().cuda())
    assert torch.equal(wu, wf)
    assert rel_err(wu.cpu(), O.vqa_forward(sd, img, ids, w.float())[0]) <= LOGIT_REL_TOL


def test_top1_agreement_10000_pairs():
    """BASELINE.json: >= 99 % top-1 agreement with the fp32 reference over 10 000 pairs (plain seeded random init;
    SURVEY 8d: 40 batches of 250 with seeds 1234 + i).  The fp32 oracle runs on the host cores (about a minute)."""
    torch.manual_seed(0)
    model = VQAModel().eval()
    sd = model.state_dict()
    model = model.cuda()
    agree = n = 0
    worst = 0.0
    for b in range(40):
        _, img, ids, mask = synth_batch(250, 1234 + b)
        with torch.no_grad():
            got, _ = model(img.cuda(), ids.cuda(), mask.cuda())
        want, _ = O.vqa_forward(sd, img, ids, mask)
        got = got.cpu()
        agree += int((got.argmax(1) == want.argmax(1)).sum())
        n += 250
        worst = max(worst, rel_err(got, want))
    print(f"top-1 agreement {agree}/{n} = {100.0 * agree / n:.2f}%  worst logit rel err {worst:.2e}")
    assert worst <= LOGIT_REL_TOL
    assert agree / n >= 0.99


def test_batch_sizes_and_lengths():
    torch.manual_seed(0)
    model = VQAModel().eval()
    sd = model.state_dict()
    model = model.cuda()
    for B, L in ((1, 20), (5, 7), (33, 20), (130, 1)):
        _, img, ids, mask = synth_batch(B, 99 + B, max_len=L)
        with torch.no_grad():
            got, _ = model(img.cuda(), ids.cuda(), mask.cuda())
        want, _ = O.vqa_forward(sd, img, ids, mask)
        assert rel_err(got.cpu(), want) <= LOGIT_REL_TOL, (B, L)
    with pytest.raises(RuntimeError):
        _, img, ids, mask = synth_batch(1, 1, max_len=21)
        model(img.cuda(), ids.cuda(), mask.cuda())  # L > max_question_length, like the reference's PE buffer


def test_api_surface_and_errors(tmp_path):
    torch.manual_seed(0)
    model = create_vqa_model(vocab_size=300, num_answers=20, use_attention=False)
    assert model.config["use_se_attention"] is False and model.num_answers == 20
    with pytest.raises(Exception):
        model.eval()(torch.zeros(1, 3, 224, 224), torch.zeros(1, 20, dtype=torch.long))  # CPU tensors: no fallback
    model = model.cuda()
    with pytest.raises(NotImplementedError):
        model.train()(torch.zeros(1, 3, 224, 224).cuda(), torch.zeros(1, 20, dtype=torch.long).cuda())
    model.eval()
    path = str(tmp_path / "ckpt.pt")
    torch.save({"config": model.config, "model_state_dict": model.state_dict(), "epoch": 3}, path)
    again = load_vqa_model(path, "cuda")
    _, img, ids, mask = synth_batch(2, 5, vocab=300)
    with torch.no_grad():
        a, _ = model(img.cuda(), ids.cuda(), mask.cuda())
        b, _ = again.eval()(img.cuda(), ids.cuda(), mask.cuda())
    assert torch.equal(a, b)
    maps = model.get_attention_maps(img.cuda(), ids.cuda(), mask.cuda())
    assert tuple(maps["cross_attention_spatial"].shape) == (2, 20, 7, 7)
    with pytest.raises(NotImplementedError):
        VQAModel(embed_dim=32, num_attention_heads=4).cuda().eval()(img.cuda(), ids.cuda())


def test_batch_invariance_across_tile_shapes():
    """A pair's logits do not depend on the batch it arrives in: small batches pick smaller convolution tiles (128-row
    sub-tiles, single CTAs, 64-column tiles; program.py::gemm) and every batch size lands on a different mix of tile
    shapes and persistent-grid sizes, but none of that may change the order in which K is accumulated.  Bit-exact."""
    torch.manual_seed(0)
    model = VQAModel().eval()
    sd = randomise_state(model.state_dict(), 1)
    model.load_state_dict(sd, strict=True)
    model = model.cuda()
    _, img, ids, mask = synth_batch(130, 31337)
    img, ids, mask = img.cuda(), ids.cuda(), mask.cuda()
    with torch.no_grad():
        full, _ = model(img, ids, mask)
        for b in (1, 2, 3, 5, 8, 13, 24, 33, 48, 65, 96):
            part, _ = model(img[:b], ids[:b], mask[:b])
            assert torch.equal(part, full[:b]), f"batch {b}: max diff {float((part - full[:b]).abs().max()):.3e}"
            if b < 60:                                         # the same pairs at the END of a batch of their own
                tail, _ = model(img[130 - b:], ids[130 - b:], mask[130 - b:])
                assert torch.equal(tail, full[130 - b:]), f"tail batch {b}"
