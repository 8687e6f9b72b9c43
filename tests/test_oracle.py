"""The oracle (oracle/vqa_oracle.py) against the golden vectors produced by the real
reference, and against the live reference where it is importable.  Also pins the parameter
container: seeded construction must reproduce the reference's random init bit-for-bit."""
import os
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN, NO_REFERENCE, REPO, have_reference

sys.path.insert(0, REPO)
from oracle import vqa_oracle as O  # noqa: E402
from vqa_b200.model import VQAModel  # noqa: E402
from vqa_b200.synth import randomise_state, state_fingerprint, synth_batch  # noqa: E402

CASES = ["default_b4", "plain_b2", "ablate_b3", "nospatial_b2"]


def build_case(meta):
    torch.manual_seed(meta["seed_weights"])
    model = VQAModel(**meta["ctor"]).eval()
    sd = model.state_dict()
    if meta["randomise"]:
        sd = randomise_state(sd, seed=1)
    _, images, ids, mask = synth_batch(meta["batch"], meta["seed_inputs"], max_len=meta["max_len"],
                                       vocab=meta["vocab"])
    return model, sd, images, ids, mask


@pytest.mark.parametrize("case", CASES)
def test_seeded_init_fingerprint(golden_meta, case):
    meta = golden_meta[case]
    model, sd, *_ = build_case(meta)
    assert len(sd) == meta["state_keys"]
    fp = state_fingerprint(sd)
    for k, v in meta["fingerprint"].items():
        assert fp[k] == pytest.approx(v, rel=1e-12, abs=1e-12), k
    assert model.get_num_parameters() == meta["num_parameters"]


def test_default_parameter_counts(golden_meta):
    n = golden_meta["default_b4"]["num_parameters"]
    assert n["total"] == 19310316 and golden_meta["default_b4"]["state_keys"] == 225


@pytest.mark.parametrize("case", CASES)
def test_oracle_matches_golden(golden_meta, case):
    meta = golden_meta[case]
    _, sd, images, ids, mask = build_case(meta)
    g = np.load(os.path.join(GOLDEN, f"{case}.npz"))
    taps = {}
    heads = meta["ctor"].get("num_attention_heads", 8)
    logits, aux = O.vqa_forward(sd, images, ids, mask, num_heads=heads, return_aux=True, taps=taps)
    tol = dict(rtol=1e-4, atol=2e-5)  # fp32 CPU vs fp32 CPU, different op order only
    np.testing.assert_allclose(logits.numpy(), g["logits"], **tol)
    for k in ("image_features", "text_features", "fused", "image_projected", "attended_pooled", "text_pooled"):
        np.testing.assert_allclose(aux[k].numpy(), g[k], err_msg=k, **tol)
    _, enc_pooled = O.text_encoder(sd, ids, mask, heads)
    np.testing.assert_allclose(enc_pooled.numpy(), g["text_pooled_encoder"], **tol)
    for i, w in enumerate(aux["cross_attention_weights"]):
        np.testing.assert_allclose(w.numpy(), g[f"cross_attention_weights_{i}"], **tol)
    names = {"stem": "image_encoder.stem"}
    for s in (1, 2, 3, 4):
        names[f"stage{s}.blocks"] = f"image_encoder.stage{s}.blocks"
        names[f"stage{s}"] = f"image_encoder.stage{s}"
    for gk, ok in names.items():
        np.testing.assert_allclose(taps[ok].flatten()[::997].numpy(), g[f"tap.{gk}.sample"], err_msg=gk, **tol)
        v64 = taps[ok].double()
        mom = np.array([float(v64.sum()), float(v64.abs().sum()), float((v64 * v64).sum()), float(v64.max())])
        np.testing.assert_allclose(mom, g[f"tap.{gk}.moments"], rtol=1e-4, err_msg=gk)
    idx, probs = O.predict_topk(logits, 5)
    assert np.array_equal(idx.numpy(), g["top_indices"])
    np.testing.assert_allclose(probs.numpy(), g["top_probs"], rtol=1e-4)


def test_oracle_preprocess_identity_224():
    g = np.load(os.path.join(GOLDEN, "preprocess.npz"))
    out = O.preprocess_u8(torch.from_numpy(g["id224.u8"]).unsqueeze(0))[0]
    np.testing.assert_allclose(out.numpy(), g["id224.out"], rtol=0, atol=1e-6)
    assert np.array_equal(g["id224.resized_u8"], g["id224.u8"])  # PIL resize is the identity at 224x224


def test_mask_dtype_and_padding_invariance(golden_meta):
    """SURVEY T6: long/float masks agree; ids at masked positions never influence logits."""
    meta = golden_meta["plain_b2"]
    _, sd, images, ids, mask = build_case(meta)
    a, _ = O.vqa_forward(sd, images, ids, mask)
    b, _ = O.vqa_forward(sd, images, ids, mask.float())
    assert torch.equal(a, b)
    ids2 = torch.where(mask == 0, torch.full_like(ids, 17), ids)
    c, _ = O.vqa_forward(sd, images, ids2, mask)
    assert torch.equal(a, c)


@pytest.mark.skipif(not have_reference(), reason=NO_REFERENCE)
def test_oracle_matches_live_reference(reference_modules):
    ref = reference_modules.import_module("models.vqa_model")
    torch.manual_seed(11)
    rm = ref.VQAModel().eval()
    sd = randomise_state(rm.state_dict(), seed=3)
    rm.load_state_dict(sd)
    torch.manual_seed(11)
    mine = VQAModel()
    assert list(mine.state_dict().keys()) == list(rm.state_dict().keys())
    mine.load_state_dict(sd, strict=True)
    _, images, ids, mask = synth_batch(2, 5)
    with torch.no_grad():
        want, waux = rm(images, ids, mask, return_aux=True)
    got, gaux = O.vqa_forward(sd, images, ids, mask, return_aux=True)
    torch.testing.assert_close(got, want, rtol=1e-4, atol=2e-5)
    torch.testing.assert_close(gaux["image_features"], waux["image_features"], rtol=1e-4, atol=2e-5)
    # None mask path
    with torch.no_grad():
        want2, _ = rm(images, ids, None)
    got2, _ = O.vqa_forward(sd, images, ids, None)
    torch.testing.assert_close(got2, want2, rtol=1e-4, atol=2e-5)


@pytest.mark.skipif(not have_reference(), reason=NO_REFERENCE)
def test_seeded_construction_is_bit_identical_to_reference(reference_modules):
    ref = reference_modules.import_module("models.vqa_model")
    for kw in ({}, dict(use_se_attention=False, use_spatial_attention=False, use_gating=False,
                        num_transformer_layers=1, num_cross_layers=3, vocab_size=50, num_answers=7)):
        torch.manual_seed(123)
        a = ref.VQAModel(**kw).state_dict()
        ra = torch.rand(3)
        torch.manual_seed(123)
        m = VQAModel(**kw)
        b = m.state_dict()
        rb = torch.rand(3)
        assert list(a.keys()) == list(b.keys())
        assert all(torch.equal(a[k], b[k]) for k in a)
        assert torch.equal(ra, rb)  # RNG stream consumed identically
        assert m.config == ref.VQAModel(**kw).config
