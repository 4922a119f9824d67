"""CPU tests of the nearest-rows audit (sdrm_b200/privacy.py): the test oracle against exact fractions, summary() against NumPy,
and every argument error that needs no device."""
import ctypes
from fractions import Fraction

import numpy as np
import pytest
import torch

from privacy_oracle import nearest_oracle, random_rows
from sdrm_b200 import privacy
from sdrm_b200.privacy import NearestRows, nearest_rows


def _brute(Q, R, k, exclude=False):
    """Per row: sort the references by (exact Fraction J descending, index ascending)."""
    out = []
    for i, q in enumerate(Q):
        cands = []
        for j, r in enumerate(R):
            if exclude and i == j:
                continue
            c = int(np.sum((q != 0) & (r != 0)))
            u = int(np.sum(q != 0) + np.sum(r != 0)) - c
            cands.append((Fraction(1) if u == 0 else Fraction(c, u), -j, c, u))
        cands.sort(reverse=True)
        out.append([(-t[1], t[2], t[3]) for t in cands[:k]])
    return out


@pytest.mark.parametrize("exclude", [False, True])
@pytest.mark.parametrize("seed,n,m,items,density", [(0, 9, 14, 7, 0.4), (1, 12, 12, 5, 0.3), (2, 6, 30, 3, 0.5), (3, 11, 11, 40, 0.1)])
def test_oracle_matches_exact_fractions(seed, n, m, items, density, exclude):
    rng = np.random.default_rng(seed)
    Q, R = random_rows(rng, n, items, density), random_rows(rng, m, items, density)
    Q[0] = 0                 # an empty query row (u = 0 against empty references: J = 1)
    R[1] = 0
    R[3] = R[2]              # duplicate references: equal J, tie to the lower index
    Q[1] = R[4]              # an exact copy
    k = min(5, m - 1)
    idx, c, u = nearest_oracle(Q, R, k, exclude_same_index=exclude)
    ref = _brute(Q, R, k, exclude)
    for i in range(n):
        assert [(int(idx[i, e]), int(c[i, e]), int(u[i, e])) for e in range(k)] == ref[i], i


def test_oracle_query_offset_exclusion():
    rng = np.random.default_rng(5)
    R = random_rows(rng, 20, 9, 0.4)
    full = nearest_oracle(R, R, 3, exclude_same_index=True)
    part = nearest_oracle(R[7:15], R, 3, exclude_same_index=True, q_index_offset=7)
    for a, b in zip(full, part):
        assert torch.equal(a[7:15], b)


def test_summary_against_numpy():
    idx = np.array([[3, 1], [0, 2], [5, 4], [2, 0]])
    c = np.array([[4, 2], [0, 0], [3, 1], [1, 1]], dtype=np.int32)
    u = np.array([[4, 5], [0, 3], [6, 7], [2, 2]], dtype=np.int32)
    res = NearestRows(idx, c, u, np.array([4, 0, 5, 2], dtype=np.int32))
    j = np.where(u == 0, 1.0, c / np.maximum(u, 1))
    assert np.array_equal(res.jaccard.numpy(), j)
    assert np.array_equal(res.hamming.numpy(), u - c)
    s = res.summary()
    d1, d2 = 1 - j[:, 0], 1 - j[:, 1]
    assert s["rows"] == 4
    assert s["dcr_mean"] == pytest.approx(d1.mean(), abs=0, rel=1e-15)
    for key, q in (("dcr_p5", 0.05), ("dcr_p50", 0.5), ("dcr_p95", 0.95)):
        assert s[key] == pytest.approx(np.quantile(d1, q), abs=1e-15)
    assert s["exact_copies"] == 2 and s["exact_copy_share"] == 0.5     # rows 0 (4 of 4) and 1 (both empty)
    ratio = np.array([0.0, 0.0, 0.5 / (1 - 1 / 7), 0.5 / 0.5])          # row 1: d1 = 0, d2 = 1
    assert s["nndr_median"] == pytest.approx(np.median(ratio), rel=1e-15)


def test_summary_k1_and_nndr_zero_distance():
    res = NearestRows(np.zeros((2, 1), dtype=np.int64), np.array([[2], [1]]), np.array([[2], [3]]), np.array([2, 1]))
    s = res.summary()
    assert "nndr_median" not in s and s["exact_copies"] == 1
    res2 = NearestRows(np.zeros((1, 2), dtype=np.int64), np.array([[3, 3]]), np.array([[3, 3]]), np.array([3]))
    assert res2.summary()["nndr_median"] == 1.0      # d1 = d2 = 0: ratio 1


def test_check_k_integer_types():
    assert privacy.check_k(np.int64(3), 10) == 3
    assert privacy.check_k(np.uint8(16), 100) == 16
    with pytest.raises(TypeError):
        privacy.check_k(True, 10)
    with pytest.raises(TypeError):
        privacy.check_k(2.0, 10)
    for k, m, ex in ((0, 10, False), (17, 100, False), (6, 5, False), (5, 5, True), (1, 1, True)):
        with pytest.raises(ValueError):
            privacy.check_k(k, m, ex)
    assert privacy.check_k(4, 5, True) == 4


def test_argument_errors_before_any_launch():
    Q = np.zeros((3, 10), dtype=np.int64)
    with pytest.raises(ValueError, match="same number of columns"):
        nearest_rows(Q, np.zeros((4, 11)), k=1)
    with pytest.raises(ValueError):
        nearest_rows(Q, np.zeros((4, 10)), k=5)
    with pytest.raises(ValueError):
        nearest_rows(Q, np.zeros((4, 10)), k=4, exclude_same_index=True)
    with pytest.raises(TypeError):
        nearest_rows(Q, np.zeros((4, 10)), k=1.0)
    with pytest.raises(TypeError):
        nearest_rows(Q, [[0, 1]], k=1)
    with pytest.raises(TypeError):
        nearest_rows(torch.zeros(3, 10).to_sparse_coo(), Q, k=1)
    with pytest.raises(ValueError):
        nearest_rows(np.zeros((2, 3, 10)), Q, k=1)
    wide = __import__("scipy.sparse", fromlist=["csr_matrix"]).csr_matrix((2, (1 << 20) + 1))
    with pytest.raises(ValueError, match="columns"):
        nearest_rows(wide, wide, k=1)


def test_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from sdrm_b200 import _lib
    with pytest.raises(_lib.SdrmError):
        nearest_rows(np.eye(4), np.eye(4), k=1)


def test_c_abi_host_checks():
    from sdrm_b200 import _lib
    from sdrm_b200.csrc import build
    build.build()
    lib = _lib.load()
    assert lib.sdrm_privacy_image_pitch(1) == 128 and lib.sdrm_privacy_image_pitch(128) == 128
    assert lib.sdrm_privacy_image_pitch(129) == 256 and lib.sdrm_privacy_image_pitch(0) == 0
    # explicit split: 2 CTAs per query tile x 2 lists per CTA x 300 rows x 8 entries of 16 bytes, after a 256-byte header
    assert lib.sdrm_privacy_workspace_bytes(300, 1000, 8, 2) == 256 + 2 * 2 * 300 * 8 * 16
    assert lib.sdrm_privacy_workspace_bytes(300, 1000, 5, 1) == 256 + 1 * 2 * 300 * 8 * 16   # k rounds up to a compiled list
    assert lib.sdrm_privacy_workspace_bytes(300, 1000, 17, 1) == 0
    assert lib.sdrm_privacy_workspace_bytes(300, 1000, 1, 99) == 256 + 4 * 2 * 300 * 1 * 16   # at most one split per tile
    buf = ctypes.create_string_buffer(4096)
    p = ctypes.c_void_p((ctypes.addressof(buf) + 15) // 16 * 16)
    args = dict(n=4, m=4, items=10, pitch=128, k=1)

    def call(**kw):
        a = {**args, **kw}
        return lib.sdrm_privacy_nearest(p, p, a["n"], p, p, a["m"], a["items"], a["pitch"], a["k"], 0, 0, 1, p, p, p, p, 4096,
                                        None)
    assert lib.sdrm_privacy_nearest(None, p, 4, p, p, 4, 10, 128, 1, 0, 0, 1, p, p, p, p, 4096, None) == -1
    assert call(k=17) == -2 and call(k=5) == -2
    assert call(items=(1 << 20) + 1, pitch=(1 << 20) + 128) == -2
    assert call(pitch=256) == -1
    assert call(n=0) == -1
    assert lib.sdrm_privacy_image_bits(p, 0, 4, 40, p, 128, p, None) == -1      # words_ld < 2
    assert lib.sdrm_privacy_image_csr(p, p, None, 1, 4, 10, p, 64, p, p, None) == -1   # bad pitch
