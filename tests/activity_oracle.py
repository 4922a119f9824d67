"""Test-side restatement of the activity-matched binarisation (sdrm_b200/sparsify.py activity_matched_device, kernel K12) in
NumPy, straight from the rule: equal-sparsity row counts from np.quantile, a stable rank of the rows by count, the real
activities at the rank's quantile, and per row a stable descending sort of the scores in K7's order."""
import numpy as np
import torch


def as_float32(S):
    """Host float32 copy of a score matrix (bfloat16 scores widened exactly)."""
    if isinstance(S, torch.Tensor):
        return S.detach().float().cpu().numpy()
    return np.asarray(S, dtype=np.float32)


def order_keys(S):
    """int64 keys whose order is K7's order of the scores: NaN as -inf, -0.0 equal to +0.0."""
    x = as_float32(S).copy()
    x[np.isnan(x)] = -np.inf
    x = x + np.float32(0.0)                      # -0.0 -> +0.0
    u = x.view(np.uint32).astype(np.int64)
    return np.where(u & 0x80000000, (~u) & 0xFFFFFFFF, u | 0x80000000)


def topk_dense(S, k):
    """bool [M, I]: row j keeps its k[j] highest scores, ties to the lower item index."""
    keys = order_keys(S)
    m, n = keys.shape
    order = np.argsort(-keys, axis=1, kind="stable")
    rank = np.empty_like(order)
    np.put_along_axis(rank, order, np.broadcast_to(np.arange(n), (m, n)), axis=1)
    return rank < np.asarray(k, dtype=np.int64)[:, None]


def equal_sparsity_counts(S, sparsity):
    x = as_float32(S)
    thr = np.quantile(x.flatten(), sparsity)
    return (x >= thr).sum(axis=1).astype(np.int64)


def targets(counts, activity):
    c = np.asarray(counts, dtype=np.int64)
    a = np.sort(np.asarray(activity, dtype=np.int64))
    m, n = len(c), len(a)
    rank = np.empty(m, dtype=np.int64)
    rank[np.argsort(c, kind="stable")] = np.arange(m)
    return a[((2 * rank + 1) * n) // (2 * m)]


def activity_matched(S, sparsity, activity):
    """(dense bool rows, per-row targets) of activity_matched_device(S, sparsity, activity)."""
    k = targets(equal_sparsity_counts(S, sparsity), activity)
    return topk_dense(S, k), k
