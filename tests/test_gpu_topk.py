"""softmax_topk_kernel (csrc/kernels_misc.cu) and the model's top-k outputs against the exact references of
tests/topk_ref.py: winners must equal the stable rank order exactly, probabilities the fp64 softmax to 2e-5 relative,
with NaN exactly where the fp64 softmax has NaN."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from topk_ref import ROW_KINDS, make_row, ref_order, ref_softmax  # noqa: E402
from vqa_b200 import program as P  # noqa: E402
from vqa_b200.runtime import Plan, VqaError  # noqa: E402

PROB_RTOL = 2e-5


def _check_probs(tag, got_i, got_p, logits):
    """got_p [B, k] against the fp64 softmax of ``logits`` at the winners; returns the worst relative error."""
    want = torch.gather(ref_softmax(logits), 1, got_i.cpu())
    got = got_p.cpu().double()
    assert torch.equal(torch.isnan(got), torch.isnan(want)), f"{tag}: NaN pattern differs"
    ok = ~torch.isnan(want)
    rel = ((got - want).abs() / want.abs().clamp_min(1e-300))[ok & (want != 0)]
    worst = float(rel.max()) if rel.numel() else 0.0
    assert bool((got[ok & (want == 0)] == 0).all()), f"{tag}: nonzero probability where the softmax is 0"
    print(f"{tag}: worst probability rel err {worst:.3e}")
    assert worst <= PROB_RTOL, f"{tag}: worst relative probability error {worst:.3e}"
    return worst


def _topk_plan(B, N, k):
    """A Plan of one softmax_topk op over the logits / top_idx / top_probs slots."""
    W = P.Weights("cuda")
    W.add("unused", torch.zeros(4), torch.float32)
    W.finalize()
    ol = P.OpList(W, "cuda")
    ol._op("softmax_topk", "topk", dict(B=B, N=N, k=k, ld=N),
           dict(logits=P.ExtRef(P.EXT["logits"]), idx=P.ExtRef(P.EXT["top_idx"]), probs=P.ExtRef(P.EXT["top_probs"])))
    ol.commit()
    return Plan(ol.ops, 0)


def _topk_ext(logits, k):
    B = logits.shape[0]
    return [None, None, None, logits.cuda(), torch.full((B, k), -7, dtype=torch.int64, device="cuda"),
            torch.full((B, k), -7.0, device="cuda")]


def _run_softmax_topk(logits, k):
    """One softmax_topk op through an OpList / Plan, on ``logits`` [B, N] (fp32, CPU)."""
    plan = _topk_plan(*logits.shape, k)
    ext = _topk_ext(logits, k)
    plan.run([0 if t is None else t.data_ptr() for t in ext], torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return ext[4], ext[5]


SHAPES = [(N, k) for N in (9, 37, 256, 257, 1000, 3129, 10000) for k in (1, 5, 9, 16, 17, 64, 128) if k <= N]
SHAPES += [(37, 37), (128, 128)]


@pytest.mark.parametrize("N,k", SHAPES)
def test_softmax_topk_kernel_is_exact_on_every_row_kind(N, k):
    logits = torch.stack([make_row(kind, N, 1000 * N + 17 * k + r) for r, kind in enumerate(ROW_KINDS)])
    idx, probs = _run_softmax_topk(logits, k)
    want = ref_order(logits, k)
    bad = [ROW_KINDS[r] for r in range(len(ROW_KINDS)) if not torch.equal(idx[r].cpu(), want[r])]
    assert not bad, f"N={N} k={k}: winners differ from the rank order on rows {bad}"
    _check_probs(f"softmax_topk N={N} k={k}", idx, probs, logits)


def test_softmax_topk_launcher_refuses_bad_sizes_and_heads_over_50000():
    """k = 129, k > N and N = 50 001 (one above the largest row the kernel keeps in shared memory) are refused, nothing
    is launched and the outputs are not written."""
    from vqa_b200.runtime import launch_count
    for N, k in ((300, 129), (8, 9), (50001, 5)):
        plan = _topk_plan(2, N, k)
        ext = _topk_ext(torch.randn(2, N), k)
        torch.cuda.synchronize()
        n0 = launch_count()
        with pytest.raises(VqaError, match="N<=50000"):
            plan.run([0 if t is None else t.data_ptr() for t in ext], torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert launch_count() == n0, f"N={N} k={k}: a kernel was launched"
        assert bool((ext[4] == -7).all()) and bool((ext[5] == -7.0).all()), f"N={N} k={k}: the outputs were written"


def test_model_top_k_paths_agree_with_the_fp64_reference(monkeypatch):
    """Default VQAModel: the fused top-8 epilogue (opt-in), softmax_topk_kernel at k = 9 and k = 128, and the
    predict API at top_k = 50 all pick the stable rank order of the model's own logits.  One question is fully
    masked, so its logit row is NaN (as in the reference) and its winners are 0..k-1 with NaN probabilities."""
    from PIL import Image

    from vqa_b200 import VQAInference
    from vqa_b200.model import VQAModel
    from vqa_b200.synth import randomise_state, synth_batch
    torch.manual_seed(0)
    model = VQAModel().eval()
    model.load_state_dict(randomise_state(model.state_dict(), 1))
    model = model.cuda()
    u8, _, ids, mask = synth_batch(6, 77)
    mask[4] = 0
    u8, ids, mask = u8.cuda(), ids.cuda(), mask.cuda()
    with torch.no_grad():
        logits = model(u8, ids, mask)[0].cpu()
    assert bool(torch.isnan(logits[4]).all()) and bool(torch.isfinite(logits[[0, 1, 2, 3, 5]]).all())
    monkeypatch.setenv("VQA_FUSED_TOPK", "1")
    model.invalidate_engine()
    i8, p8 = model.predict(u8, ids, mask, top_k=8)
    assert any(op.kind == "gemm" and op.i.get("topk") for op in model.engine().last_plan[0].ops), "top-8 not fused"
    monkeypatch.delenv("VQA_FUSED_TOPK")
    model.invalidate_engine()
    i9, p9 = model.predict(u8, ids, mask, top_k=9)
    i128, p128 = model.predict(u8, ids, mask, top_k=128)
    assert any(op.kind == "softmax_topk" for op in model.engine().last_plan[0].ops)
    for tag, i, p, k in (("fused k=8", i8, p8, 8), ("kernel k=9", i9, p9, 9), ("kernel k=128", i128, p128, 128)):
        assert torch.equal(i.cpu(), ref_order(logits, k)), tag
        assert torch.equal(i[:, :8].cpu(), i8.cpu()), tag
        _check_probs(f"model {tag}", i, p, logits)

    inf = VQAInference()
    inf.load()
    img = Image.fromarray(u8[0].cpu().numpy(), "RGB")
    q = "what color is this"
    out = inf.predict(img, q, top_k=50)
    qids, qmask = inf.preprocess_question(q)
    with torch.no_grad():
        lg = inf.model(inf.preprocess_image_u8(img).unsqueeze(0).cuda(), qids.cuda(), qmask.cuda())[0].cpu()
    assert [a["index"] for a in out["answers"]] == ref_order(lg, 50)[0].tolist()
    got_p = torch.tensor([[a["probability"] for a in out["answers"]]])
    _check_probs("VQAInference.predict k=50", ref_order(lg, 50), got_p, lg)

