"""Top-K recommendation on the device: the k best items of every user row, with the items the user has already interacted with
excluded, by the K7 kernel (sdrm_recommend_topk, include/sdrm_b200.h).  The history is a CSR pair (indptr int64[users + 1],
indices int32[nnz]); no dense mask is built.  There is no CPU fallback.
"""
import operator

import torch

from . import _lib

MAX_K = 256
MAX_ITEMS = 1 << 20
_TOO_FEW, _BAD_INDEX, _BAD_INDPTR = 1, 2, 4   # enum sdrm_recommend_status


def check_history(history_indptr, history_indices, users):
    """Dtype and shape checks of a CSR history for `users` rows (no device access).  Returns (indptr, indices) contiguous."""
    if not isinstance(history_indptr, torch.Tensor) or not isinstance(history_indices, torch.Tensor):
        raise TypeError("history_indptr and history_indices must be torch tensors")
    if history_indptr.dtype != torch.int64:
        raise TypeError(f"history_indptr must be int64, got {history_indptr.dtype}")
    if history_indices.dtype != torch.int32:
        raise TypeError(f"history_indices must be int32, got {history_indices.dtype}")
    if history_indptr.dim() != 1 or history_indptr.numel() != users + 1:
        raise ValueError(f"history_indptr must have users + 1 = {users + 1} entries, got shape {tuple(history_indptr.shape)}")
    if history_indices.dim() != 1:
        raise ValueError(f"history_indices must be 1-D, got shape {tuple(history_indices.shape)}")
    return history_indptr.contiguous(), history_indices.contiguous()


def check_k(k, n_items):
    """Returns k as a Python int.  Any integer type is accepted (numpy integers included); bools and floats are not."""
    if isinstance(k, bool):
        raise TypeError(f"k must be an integer, got {k!r}")
    try:
        k = operator.index(k)
    except TypeError:
        raise TypeError(f"k must be an integer, got {k!r}") from None
    if not 1 <= k <= min(MAX_K, n_items):
        raise ValueError(f"k={k} must lie in [1, {min(MAX_K, n_items)}] (at most {MAX_K}, at most the {n_items} items)")
    return k


def recommend_topk(logits, history_indptr, history_indices, k):
    """logits: CUDA float32 or bfloat16 [users, items] (rows may be strided; columns must be contiguous).
    history_indptr int64[users + 1], history_indices int32[nnz]: row u's seen items are
    history_indices[history_indptr[u]:history_indptr[u + 1]] (duplicates allowed), on the logits' device.

    Returns (values [users, k] in the logits' dtype, indices int64 [users, k]): per row the k highest logits among the items
    outside the row's history, by descending score, ties to the lower item index.  NaN ranks as -inf (its value is returned as
    -inf) and -0.0 as +0.0.  Raises ValueError when k > 256, k > items, a row has fewer than k items left after the exclusion,
    or the history is malformed (indptr not non-decreasing within [0, nnz], an index outside [0, items)); the check reads one
    status word back from the device, so the call synchronises with the current stream."""
    if not isinstance(logits, torch.Tensor):
        raise TypeError("logits must be a torch tensor")
    if logits.dtype not in (torch.float32, torch.bfloat16):
        raise TypeError(f"logits must be float32 or bfloat16, got {logits.dtype}")
    if logits.dim() != 2:
        raise ValueError(f"logits must be 2-D [users, items], got shape {tuple(logits.shape)}")
    users, n_items = logits.shape
    indptr, indices = check_history(history_indptr, history_indices, users)
    if n_items < 1 or n_items > MAX_ITEMS:
        raise ValueError(f"logits must have between 1 and {MAX_ITEMS} items, got {n_items}")
    k = check_k(k, n_items)
    if (n_items > 1 and logits.stride(1) != 1) or (users > 1 and logits.stride(0) < n_items):
        raise ValueError("logits must have unit column stride and rows that do not overlap (a row-strided view is fine); "
                         "call .contiguous() first")
    dev = logits.device
    if dev.type != "cuda":
        raise _lib.SdrmError("recommend_topk needs CUDA tensors (no CPU fallback)")
    if indptr.device != dev or indices.device != dev:
        raise ValueError(f"history_indptr and history_indices must be on {dev} like the logits")
    values = torch.empty((users, k), dtype=logits.dtype, device=dev)
    idx = torch.empty((users, k), dtype=torch.int64, device=dev)
    if users == 0:
        return values, idx
    ld = logits.stride(0) if users > 1 else n_items
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    lib = _lib.load()
    with torch.cuda.device(dev):
        fn = lib.sdrm_recommend_topk if logits.dtype == torch.float32 else lib.sdrm_recommend_topk_bf16
        _lib.check(fn(_lib.ptr(logits), users, n_items, ld, _lib.ptr(indptr), _lib.ptr(indices) if indices.numel() else None,
                      indices.numel(), k, _lib.ptr(values), _lib.ptr(idx), _lib.ptr(status), _lib.stream_ptr()),
                   "sdrm_recommend_topk")
        st = int(status.item())
    if st & _BAD_INDPTR:
        raise ValueError(f"history_indptr must be non-decreasing within [0, {indices.numel()}] (the number of history entries)")
    if st & _BAD_INDEX:
        raise ValueError(f"history_indices has entries outside [0, {n_items})")
    if st & _TOO_FEW:
        raise ValueError(f"k={k} exceeds the number of items left after excluding the history in at least one row")
    return values, idx
