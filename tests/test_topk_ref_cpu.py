"""The selection references of tests/topk_ref.py against torch.argmax, torch.topk and torch.softmax, wherever torch's
answer is defined: NaN positions compare as sets because torch.topk promises no order among them."""
import pytest
import torch

from topk_ref import ROW_KINDS, make_row, ref_order, ref_rank, ref_softmax


@pytest.mark.parametrize("N", [9, 37, 300])
def test_references_agree_with_torch(N):
    rows = torch.stack([make_row(kind, N, 7 * N + i) for i, kind in enumerate(ROW_KINDS)])
    extra = torch.tensor([[0.0, -0.0, 1.0, -1.0, 1.0] + [-2.0] * (N - 5)])           # -0.0 ties +0.0, 1.0 ties 1.0
    rows = torch.cat([rows, extra])
    order = ref_order(rows, N)
    assert torch.equal(order[:, 0], torch.argmax(rows, dim=1))                      # argmax: the first NaN, else first max
    assert torch.equal(order[-1, :4], torch.tensor([2, 4, 0, 1]))
    for r in range(rows.shape[0]):
        row = rows[r]
        assert sorted(order[r].tolist()) == list(range(N))
        nn = int(torch.isnan(row).sum())
        for k in (1, 5, 9):
            if k > N or nn > k:
                continue
            tv, ti = torch.topk(row, k)
            assert set(ti[:nn].tolist()) == set(order[r, :nn].tolist())
            assert torch.equal(tv[nn:], row[order[r, nn:k]])                        # same values, in the same order
        ranks = ref_rank(row.expand(N, N), order[r])
        assert torch.equal(ranks, torch.arange(N))
    assert torch.equal(ref_rank(rows[:2], torch.tensor([-1, N])), torch.tensor([N, N]))
    want = torch.softmax(rows.double(), dim=-1)
    got = ref_softmax(rows)
    assert torch.equal(torch.isnan(got), torch.isnan(want))
    torch.testing.assert_close(got, want, rtol=1e-12, atol=0, equal_nan=True)
    for kind in ("pos_inf", "one_nan", "all_nan", "all_neg_inf"):
        assert bool(torch.isnan(got[ROW_KINDS.index(kind)]).all()), kind
