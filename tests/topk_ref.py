"""Exact CPU references for the kernels that select from logit rows (softmax_topk_kernel, the fused top-k epilogue of the
head GEMM, accuracy_kernel).

Rank order: NaN > +inf > finite > -inf; equal keys (NaN against NaN, -0.0 against +0.0) go to the lower index.  That is
torch.argmax's and torch.topk's order with ties made deterministic.  Everything here sorts integers and fp64 values
in numpy, so it shares no code with torch's or the library's selection.
"""
from __future__ import annotations

import numpy as np
import torch


def _rank_keys(x: np.ndarray):
    """(class, value) per element: class 3 NaN, 2 +inf, 1 finite, 0 -inf; value the fp64 logit for finite ones."""
    x = np.asarray(x, dtype=np.float64)
    cls = np.where(np.isnan(x), 3, np.where(x == np.inf, 2, np.where(x == -np.inf, 0, 1)))
    val = np.where(cls == 1, x, 0.0) + 0.0          # + 0.0 turns -0.0 into +0.0
    return cls, val


def ref_order(logits, k: int) -> torch.Tensor:
    """int64 [B, k]: the first k indices of each row of ``logits`` [B, N] in rank order (a stable sort)."""
    x = torch.as_tensor(logits).detach().cpu().double().numpy()
    B, N = x.shape
    out = np.empty((B, k), dtype=np.int64)
    idx = np.arange(N)
    for b in range(B):
        cls, val = _rank_keys(x[b])
        out[b] = np.lexsort((idx, -val, -cls))[:k]   # last key is primary: class desc, value desc, index asc
    return torch.from_numpy(out)


def ref_rank(logits, targets) -> torch.Tensor:
    """int64 [B]: how many entries of each row rank before the target's; N for a target outside [0, N)."""
    x = torch.as_tensor(logits).detach().cpu().double().numpy()
    t = torch.as_tensor(targets).cpu().numpy()
    B, N = x.shape
    order = ref_order(torch.from_numpy(x), N).numpy()
    out = np.full(B, N, dtype=np.int64)
    for b in range(B):
        if 0 <= t[b] < N:
            out[b] = int(np.nonzero(order[b] == t[b])[0][0])
    return torch.from_numpy(out)


def ref_softmax(logits) -> torch.Tensor:
    """fp64 softmax over the last dimension; a row with a NaN, a +inf or only -inf is all NaN, as torch.softmax gives."""
    x = torch.as_tensor(logits).detach().cpu().double()
    m = x.max(dim=-1, keepdim=True).values            # NaN when the row holds one
    e = torch.exp(x - m)
    return e / e.sum(dim=-1, keepdim=True)


ROW_KINDS = ("random", "tied_max", "neg_inf_col", "pos_inf", "one_nan", "three_nans", "nan_and_inf", "all_nan",
             "all_neg_inf", "all_equal")


def make_row(kind: str, N: int, seed: int) -> torch.Tensor:
    """fp32 [N] logit row of one kind.  tied_max puts the row maximum at columns 3, 43 and 259 (different warps of a
    256-thread block, the same thread for 3 and 259); the special entries sit at the first, middle and last columns."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(N, generator=g) * 3
    nan, inf = float("nan"), float("inf")
    if kind == "tied_max":
        x[[c for c in (3, 43, 259) if c < N]] = float(x.max()) + 1
    elif kind == "neg_inf_col":
        x[N // 2] = -inf
    elif kind == "pos_inf":
        x[N - 1] = inf
    elif kind == "one_nan":
        x[N // 3] = nan
    elif kind == "three_nans":
        x[[N - 1, N // 2, 1]] = nan
    elif kind == "nan_and_inf":
        x[0], x[N - 2] = inf, nan
    elif kind == "all_nan":
        x[:] = nan
    elif kind == "all_neg_inf":
        x[:] = -inf
    elif kind == "all_equal":
        x[:] = 0.5
    else:
        assert kind == "random", kind
    return x
