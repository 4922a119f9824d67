"""CPU tests of the fidelity audit (sdrm_b200/fidelity.py): the test oracle against a per-pair loop, summary() against scipy,
and every argument error that needs no device."""
import ctypes
import math

import numpy as np
import pytest
import scipy.stats
import torch

from fidelity_oracle import pair_sums, phi_matrix, report
from privacy_oracle import random_rows
from sdrm_b200.fidelity import FidelityReport, compare
from sdrm_b200.privacy import NearestRows


def _loop_sums(R, S):
    """Per pair, straight from the definition, in Python floats."""
    def phi(X, i, j):
        U = X.shape[0]
        a, b = int(X[:, i].sum()), int(X[:, j].sum())
        c = int((X[:, i] * X[:, j]).sum())
        vi, vj = a * (U - a), b * (U - b)
        return 0.0 if vi == 0 or vj == 0 else (U * c - a * b) / (math.sqrt(vi) * math.sqrt(vj))
    out = [0.0] * 6
    I = R.shape[1]
    for i in range(I):
        for j in range(i + 1, I):
            r, s = phi(R, i, j), phi(S, i, j)
            for n, v in enumerate(((r - s) ** 2, r, s, r * r, s * s, r * s)):
                out[n] += v
    return out


@pytest.mark.parametrize("seed,ur,us,items,density", [(0, 9, 14, 7, 0.4), (1, 12, 5, 5, 0.3), (2, 30, 6, 3, 0.5), (3, 11, 11, 40, 0.1)])
def test_oracle_matches_per_pair_loop(seed, ur, us, items, density):
    rng = np.random.default_rng(seed)
    R, S = random_rows(rng, ur, items, density), random_rows(rng, us, items, density)
    R[:, 0] = 0          # constant items: all-zero in the real set, all-one in the synthetic set
    S[:, 1] = 1
    got = pair_sums(R, S)
    ref = _loop_sums(R, S)
    assert torch.allclose(got, torch.tensor(ref, dtype=torch.float64), rtol=1e-12, atol=1e-12)
    # phi is the Pearson correlation of the item columns where both are non-constant
    X = R.astype(np.float64)
    ph = phi_matrix(R).numpy()
    for i in range(items):
        for j in range(items):
            if X[:, i].std() > 0 and X[:, j].std() > 0:
                assert ph[i, j] == pytest.approx(np.corrcoef(X[:, i], X[:, j])[0, 1], abs=1e-12)


def test_oracle_single_item():
    R, S = np.ones((4, 1), dtype=np.uint8), np.zeros((3, 1), dtype=np.uint8)
    assert torch.equal(pair_sums(R, S), torch.zeros(6, dtype=torch.float64))
    s = report(R, S).summary()
    assert s["items"] == 1 and s["phi_pcd"] == 0.0
    assert math.isnan(s["phi_rmse"]) and math.isnan(s["phi_corr"]) and math.isnan(s["neighbour_recall_at_k"])
    assert math.isnan(s["item_tv"])   # the synthetic set has no ones
    assert s["item_coverage"] == 0.0


def test_summary_against_scipy():
    rng = np.random.default_rng(4)
    R, S = random_rows(rng, 40, 25, 0.2), random_rows(rng, 33, 25, 0.15)
    R[:, 3] = 0
    rep = report(R, S, k=3)
    s = rep.summary()
    ur, us = R.sum(1), S.sum(1)
    ar, as_ = R.sum(0).astype(np.float64), S.sum(0).astype(np.float64)
    assert s["users_real"] == 40 and s["users_synth"] == 33 and s["items"] == 25
    assert s["ones_per_user_real"] == pytest.approx(ur.mean()) and s["ones_per_user_synth"] == pytest.approx(us.mean())
    assert s["activity_ks"] == pytest.approx(scipy.stats.ks_2samp(ur, us).statistic, abs=1e-15)
    assert s["item_freq_pearson"] == pytest.approx(scipy.stats.pearsonr(ar / 40, as_ / 33)[0], abs=1e-12)
    assert s["item_freq_spearman"] == pytest.approx(scipy.stats.spearmanr(ar / 40, as_ / 33)[0], abs=1e-12)
    assert s["item_tv"] == pytest.approx(0.5 * np.abs(ar / ar.sum() - as_ / as_.sum()).sum(), abs=1e-15)
    assert s["item_coverage"] == pytest.approx(((ar > 0) & (as_ > 0)).sum() / (ar > 0).sum())
    pr, ps = phi_matrix(R).numpy(), phi_matrix(S).numpy()
    iu = np.triu_indices(25, 1)
    d = pr[iu] - ps[iu]
    assert s["phi_pcd"] == pytest.approx(np.linalg.norm(pr - ps - np.diag(np.diag(pr - ps))), rel=1e-12)
    assert s["phi_rmse"] == pytest.approx(np.sqrt(np.mean(d * d)), rel=1e-12)
    assert s["phi_corr"] == pytest.approx(scipy.stats.pearsonr(pr[iu], ps[iu])[0], abs=1e-12)
    # neighbour recall from the lists, by hand
    rec = []
    for i in range(25):
        nr = {int(j) for j, c in zip(rep.neighbours_real.index[i], rep.neighbours_real.intersection[i]) if c > 0}
        ns = {int(j) for j, c in zip(rep.neighbours_synth.index[i], rep.neighbours_synth.intersection[i]) if c > 0}
        if nr:
            rec.append(len(nr & ns) / len(nr))
    assert s["neighbour_recall_at_k"] == pytest.approx(np.mean(rec), abs=1e-15)


def test_summary_ties_and_degenerate_sums():
    # Spearman with tied frequencies: average ranks
    rep = FidelityReport(np.array([2, 2, 0, 5]), np.array([1, 3, 3, 0]), np.array([3, 6]), np.array([4, 3]), np.zeros(6))
    s = rep.summary()
    assert s["item_freq_spearman"] == pytest.approx(scipy.stats.spearmanr([1, 1, 0, 2.5], [.5, 1.5, 1.5, 0])[0], abs=1e-12)
    assert math.isnan(s["phi_corr"])            # zero variance
    assert s["phi_pcd"] == 0.0 and s["phi_rmse"] == 0.0
    # an item set with no real neighbour of c > 0: recall undefined
    nb = NearestRows(np.array([[1], [0]]), np.array([[0], [0]]), np.array([[3], [3]]), np.array([1, 2]))
    rep2 = FidelityReport(np.array([1, 2]), np.array([1, 2]), np.array([1, 2]), np.array([1, 2]), np.zeros(6), nb, nb)
    assert math.isnan(rep2.summary()["neighbour_recall_at_k"])


def test_argument_errors_before_any_launch():
    X = np.zeros((3, 10), dtype=np.int64)
    with pytest.raises(ValueError, match="same number of columns"):
        compare(X, np.zeros((4, 11)))
    with pytest.raises(ValueError):
        compare(X, np.zeros((4, 10)), k=10)          # k <= items - 1
    with pytest.raises(ValueError):
        compare(X, np.zeros((4, 10)), k=17)
    with pytest.raises(ValueError):
        compare(np.zeros((3, 1)), np.zeros((4, 1)), k=1)   # one item: only k=None
    with pytest.raises(TypeError):
        compare(X, np.zeros((4, 10)), k=2.0)
    with pytest.raises(TypeError):
        compare(X, [[0, 1]], k=None)
    with pytest.raises(TypeError):
        compare(torch.zeros(3, 10).to_sparse_coo(), X, k=None)
    with pytest.raises(ValueError, match="rows"):
        compare(np.zeros((0, 10)), X, k=None)
    sp = __import__("scipy.sparse", fromlist=["csr_matrix"])
    wide = sp.csr_matrix((2, (1 << 20) + 1))
    with pytest.raises(ValueError, match="columns"):
        compare(wide, wide, k=None)
    tall = sp.csr_matrix(((1 << 20) + 1, 10))
    with pytest.raises(ValueError, match="rows"):
        compare(X, tall, k=None)


def test_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from sdrm_b200 import _lib
    with pytest.raises(_lib.SdrmError):
        compare(np.eye(4), np.eye(4), k=2)


def test_c_abi_host_checks():
    from sdrm_b200 import _lib
    from sdrm_b200.csrc import build
    build.build()
    lib = _lib.load()
    # 300 items: 3 tiles a side, 6 upper-triangle tiles of 6 doubles, after the 256-byte header and 32 bytes of statistics per
    # item (rounded up to 256 bytes)
    assert lib.sdrm_fidelity_workspace_bytes(300) == 256 + 9728 + 6 * 6 * 8
    assert lib.sdrm_fidelity_workspace_bytes(128) == 256 + 128 * 32 + 1 * 6 * 8
    assert lib.sdrm_fidelity_workspace_bytes(0) == 0 and lib.sdrm_fidelity_workspace_bytes((1 << 20) + 1) == 0
    buf = ctypes.create_string_buffer(1 << 16)
    p = ctypes.c_void_p((ctypes.addressof(buf) + 15) // 16 * 16)
    odd = ctypes.c_void_p(p.value + 8)
    pitch = lib.sdrm_privacy_image_pitch   # the images take K8's pitch, over the users
    assert pitch(938) == 1024

    def stats(ur=4, us=5, items=10, pr=None, ps=None, img=p, ws=1 << 15):
        return lib.sdrm_fidelity_pair_stats(img, p, ur, pitch(ur) if pr is None else pr, p, p, us, pitch(us) if ps is None else ps,
                                            items, p, p, ws, None)
    assert lib.sdrm_fidelity_pair_stats(None, p, 4, 128, p, p, 5, 128, 10, p, p, 1 << 15, None) == -1
    assert stats(ur=(1 << 20) + 1, pr=(1 << 20) + 128) == -2
    assert stats(us=0, ps=128) == -2
    assert stats(items=(1 << 20) + 1) == -2
    assert stats(pr=256) == -1                     # pitch must be K8's pitch of the users
    assert stats(img=odd) == -1                    # misaligned image
    assert stats(ws=16) == -5
    assert lib.sdrm_fidelity_item_image_bits(p, 0, 4, 40, p, 128, p, p, None) == -1        # words_ld < 2
    assert lib.sdrm_fidelity_item_image_bits(p, 2, 4, 40, p, 256, p, p, None) == -1        # bad pitch
    assert lib.sdrm_fidelity_item_image_bits(p, 2, 0, 40, p, 128, p, p, None) == -2        # no users
    assert lib.sdrm_fidelity_item_image_csr(p, p, None, 1, 4, 10, p, 64, p, p, p, None) == -1    # bad pitch
    assert lib.sdrm_fidelity_item_image_csr(None, p, None, 1, 4, 10, p, 128, p, p, p, None) == -1
    assert lib.sdrm_fidelity_item_image_csr(p, p, None, 1, 4, (1 << 20) + 1, p, 128, p, p, p, None) == -2
