"""Fidelity audit of binary rows: how closely synthetic user x item rows resemble the real rows, with no downstream evaluator.
Item popularity and user activity come from the popcounts of the operand images; the pairwise item correlation (the phi
coefficient of every item pair in each set, compared over all pairs) is computed by the K9 kernel (sdrm_fidelity_*,
include/sdrm_b200.h) as an exact integer product on the tensor cores with the sums fused into its epilogue; each item's nearest
items by Jaccard similarity come from K8 (privacy.py) on the same item-major images.  Nothing dense goes through the host.  There
is no CPU fallback.

    rep = compare(real_csr, synthetic_bits, k=10)
    rep.summary()   # item frequencies, user activity, phi correlation difference, item-neighbour recall

Accepted row sets (either side) are those of privacy.nearest_rows: sparsify.PackedMatrix, scipy CSR, torch sparse CSR,
training.DeviceCSR, and dense 0/1 torch or NumPy arrays (nonzero = 1).  For sparse input a stored value != 0 is an interaction;
explicit stored zeros are not, and a repeated column counts once.
"""
import math

import numpy as np
import torch

from . import _lib, privacy
from .privacy import NearestRows

MAX_USERS = 1 << 20
MAX_ITEMS = 1 << 20
SUM_KEYS = ("S_dd", "S_r", "S_s", "S_rr", "S_ss", "S_rs")   # the order of sdrm_fidelity_pair_stats' d_sums_out


class FidelityReport:
    """What compare() computed (device tensors): item_ones_* int32 [items] and user_ones_* int32 [users] of the real and the
    synthetic set; sums float64 [6] over the item pairs i < j, in SUM_KEYS order (d = phiR - phiS): sum d^2, sum phiR,
    sum phiS, sum phiR^2, sum phiS^2, sum phiR phiS; neighbours_real / neighbours_synth: NearestRows of every item's k nearest
    items in each set (None when compare ran with k=None)."""

    def __init__(self, item_ones_real, item_ones_synth, user_ones_real, user_ones_synth, sums, neighbours_real=None,
                 neighbours_synth=None):
        self.item_ones_real = torch.as_tensor(item_ones_real)
        self.item_ones_synth = torch.as_tensor(item_ones_synth)
        self.user_ones_real = torch.as_tensor(user_ones_real)
        self.user_ones_synth = torch.as_tensor(user_ones_synth)
        self.sums = torch.as_tensor(sums, dtype=torch.float64)
        self.neighbours_real = neighbours_real
        self.neighbours_synth = neighbours_synth

    def summary(self):
        """Host-side metrics (dict of Python numbers; NaN where a metric is undefined):
        users_real, users_synth, items; ones_per_user_real / _synth (mean of the user ones); activity_ks (two-sample
        Kolmogorov-Smirnov statistic of the two user-ones samples); item_freq_pearson / item_freq_spearman (correlation of the
        item frequencies a / U between the sets; Spearman with average ranks for ties); item_tv (1/2 sum |pR - pS|, p = a / sum a);
        item_coverage (share of the items present in the real rows that the synthetic rows hold too); phi_pcd (sqrt(2 S_dd): the
        Frobenius norm of phiR - phiS off the diagonal), phi_rmse (sqrt(S_dd / P), P = I (I - 1) / 2 pairs), phi_corr (Pearson
        correlation of phiR and phiS over the pairs); neighbour_recall_at_k (per item, the share of its real nearest items with
        c > 0 that are among its synthetic nearest items with c > 0, averaged over the items that have any)."""
        ar = self.item_ones_real.cpu().numpy().astype(np.float64)
        as_ = self.item_ones_synth.cpu().numpy().astype(np.float64)
        ur = self.user_ones_real.cpu().numpy().astype(np.float64)
        us = self.user_ones_synth.cpu().numpy().astype(np.float64)
        s_dd, s_r, s_s, s_rr, s_ss, s_rs = (float(v) for v in self.sums.cpu().tolist())
        n_items, n_r, n_s = len(ar), len(ur), len(us)
        nan = float("nan")
        out = {"users_real": n_r, "users_synth": n_s, "items": n_items,
               "ones_per_user_real": float(ur.mean()) if n_r else nan,
               "ones_per_user_synth": float(us.mean()) if n_s else nan,
               "activity_ks": _ks_statistic(ur, us) if n_r and n_s else nan}
        fr, fs = ar / max(n_r, 1), as_ / max(n_s, 1)
        out["item_freq_pearson"] = _pearson(fr, fs)
        out["item_freq_spearman"] = _pearson(_average_ranks(fr), _average_ranks(fs))
        tr, ts = ar.sum(), as_.sum()
        out["item_tv"] = float(0.5 * np.abs(ar / tr - as_ / ts).sum()) if tr > 0 and ts > 0 else nan
        present = ar > 0
        out["item_coverage"] = float((as_[present] > 0).mean()) if present.any() else nan
        P = n_items * (n_items - 1) / 2
        out["phi_pcd"] = math.sqrt(2.0 * s_dd)
        out["phi_rmse"] = math.sqrt(s_dd / P) if P > 0 else nan
        var_r, var_s = P * s_rr - s_r * s_r, P * s_ss - s_s * s_s
        out["phi_corr"] = (P * s_rs - s_r * s_s) / math.sqrt(var_r * var_s) if P >= 2 and var_r > 0 and var_s > 0 else nan
        out["neighbour_recall_at_k"] = _neighbour_recall(self.neighbours_real, self.neighbours_synth)
        return out


def _ks_statistic(x, y):
    """sup |F_x - F_y| of the two empirical distribution functions (scipy.stats.ks_2samp's statistic)."""
    x, y = np.sort(x), np.sort(y)
    pts = np.concatenate([x, y])
    return float(np.max(np.abs(np.searchsorted(x, pts, side="right") / len(x) - np.searchsorted(y, pts, side="right") / len(y))))


def _average_ranks(x):
    """1-based ranks, ties given their average rank (scipy.stats.rankdata's default)."""
    order = np.argsort(x, kind="stable")
    _, first, counts = np.unique(x[order], return_index=True, return_counts=True)
    ranks = np.empty(len(x), dtype=np.float64)
    ranks[order] = np.repeat(first + (counts + 1) / 2.0, counts)
    return ranks


def _pearson(x, y):
    if len(x) < 2:
        return float("nan")
    dx, dy = x - x.mean(), y - y.mean()
    den = math.sqrt(float((dx * dx).sum()) * float((dy * dy).sum()))
    return float((dx * dy).sum()) / den if den > 0 else float("nan")


def _neighbour_recall(real, synth):
    if real is None or synth is None:
        return float("nan")
    ir, cr = real.index.cpu().numpy(), real.intersection.cpu().numpy()
    is_, cs = synth.index.cpu().numpy(), synth.intersection.cpu().numpy()
    keep_r, keep_s = cr > 0, cs > 0   # J = 0 entries are index-ordered ties, not neighbours
    hit = ((ir[:, :, None] == is_[:, None, :]) & keep_r[:, :, None] & keep_s[:, None, :]).any(2)
    n_r = keep_r.sum(1)
    rows = n_r > 0
    if not rows.any():
        return float("nan")
    return float((hit.sum(1)[rows] / n_r[rows]).mean())


def _item_image(x, kind, users, n_items, dev):
    """(item-major uint8 0/1 image [items, pitch(users)], item ones int32 [items], user ones int32 [users]) on `dev`."""
    lib = _lib.load()
    pitch = int(lib.sdrm_privacy_image_pitch(users))
    img = torch.empty((n_items, pitch), dtype=torch.uint8, device=dev)
    item_ones = torch.empty(n_items, dtype=torch.int32, device=dev)
    user_ones = torch.empty(users, dtype=torch.int32, device=dev)
    if kind == "bits":
        bits = x.bits.to(dev)
        if users > 1 and bits.stride(1) != 1:
            bits = bits.contiguous()
        _lib.check(lib.sdrm_fidelity_item_image_bits(_lib.ptr(bits), bits.stride(0) if users > 1 else bits.shape[1], users,
                                                     n_items, _lib.ptr(img), pitch, _lib.ptr(item_ones), _lib.ptr(user_ones),
                                                     _lib.stream_ptr()),
                   "sdrm_fidelity_item_image_bits")
        return img, item_ones, user_ones
    indptr, indices, values = privacy._csr_arrays(x, kind, users, dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    nnz = indices.numel()
    _lib.check(lib.sdrm_fidelity_item_image_csr(_lib.ptr(indptr), _lib.ptr(indices) if nnz else None,
                                                _lib.ptr(values) if values is not None and nnz else None, nnz, users, n_items,
                                                _lib.ptr(img), pitch, _lib.ptr(item_ones), _lib.ptr(user_ones),
                                                _lib.ptr(status), _lib.stream_ptr()),
               "sdrm_fidelity_item_image_csr")
    privacy._raise_csr_status(status, nnz, n_items)
    return img, item_ones, user_ones


def _pair_stats(r_img, r_item_ones, r_users, s_img, s_item_ones, s_users, n_items):
    """K9 on prepared item-major images: float64 [6] in SUM_KEYS order."""
    lib = _lib.load()
    dev = r_img.device
    sums = torch.empty(6, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        ws_bytes = int(lib.sdrm_fidelity_workspace_bytes(n_items))
        if ws_bytes == 0:
            _lib.check(-1, "sdrm_fidelity_workspace_bytes")
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.check(lib.sdrm_fidelity_pair_stats(_lib.ptr(r_img), _lib.ptr(r_item_ones), r_users, r_img.shape[1],
                                                _lib.ptr(s_img), _lib.ptr(s_item_ones), s_users, s_img.shape[1], n_items,
                                                _lib.ptr(sums), _lib.ptr(ws), ws_bytes, _lib.stream_ptr()),
                   "sdrm_fidelity_pair_stats")
    return sums


def compare(real, synthetic, k=10):
    """Fidelity of `synthetic` rows to `real` rows over the same items.  Returns a FidelityReport (device tensors; summary() for
    the metrics).  k: the number of nearest items per item (by Jaccard similarity over the users, K8) behind
    neighbour_recall_at_k, at most min(16, items - 1); k=None skips that search (neighbour_recall_at_k is then NaN), as sets
    with fewer than two items require.

    Raises ValueError for row sets with different numbers of columns, more than 2^20 columns or users (or none), k outside its
    range, or malformed sparse input (indptr, indices out of range); TypeError for other input types.  Sparse input is checked
    on the device, so the call synchronises with the current stream."""
    rk, ur, ir = privacy._kind(real)
    sk, us, is_ = privacy._kind(synthetic)
    if ir != is_:
        raise ValueError(f"real and synthetic rows must have the same number of columns, got {ir} and {is_}")
    if not 1 <= ir <= MAX_ITEMS:
        raise ValueError(f"rows must have between 1 and {MAX_ITEMS} columns, got {ir}")
    for name, u in (("real", ur), ("synthetic", us)):
        if not 1 <= u <= MAX_USERS:
            raise ValueError(f"the {name} set must have between 1 and {MAX_USERS} rows, got {u}")
    if k is not None:
        k = privacy.check_k(k, ir, exclude_same_index=True)
    devs = {d for d in (privacy._device_of(real), privacy._device_of(synthetic)) if d is not None and d.type == "cuda"}
    if len(devs) > 1:
        raise ValueError(f"real and synthetic rows are on different devices: {sorted(map(str, devs))}")
    if not torch.cuda.is_available():
        raise _lib.SdrmError("fidelity.compare needs a CUDA device (no CPU fallback)")
    dev = devs.pop() if devs else torch.device("cuda", torch.cuda.current_device())
    with torch.cuda.device(dev):
        r_img, r_items, r_users = _item_image(real, rk, ur, ir, dev)
        s_img, s_items, s_users = _item_image(synthetic, sk, us, ir, dev)
        sums = _pair_stats(r_img, r_items, ur, s_img, s_items, us, ir)
        nb_r = nb_s = None
        if k is not None:
            nb_r = NearestRows(*privacy._search(r_img, r_items, r_img, r_items, ur, k, exclude_same_index=True), r_items)
            nb_s = NearestRows(*privacy._search(s_img, s_items, s_img, s_items, us, k, exclude_same_index=True), s_items)
    return FidelityReport(r_items, s_items, r_users, s_users, sums, nb_r, nb_s)
