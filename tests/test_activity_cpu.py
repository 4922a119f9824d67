"""CPU tests of the activity-matched binarisation's host side: row_activity, activity_targets against the NumPy oracle, and the
command-line flags of main.py --binarise and synthesize --activity-from."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

import activity_oracle as oracle
from sdrm_b200.sparsify import activity_targets, row_activity


def test_row_activity_sparse_explicit_zeros_and_duplicates():
    # row 0: columns 1, 3 (3 stored twice); row 1: an explicit zero only; row 2: column 0 twice, one of them zero; row 3: empty
    rows = np.array([0, 0, 0, 1, 2, 2])
    cols = np.array([1, 3, 3, 2, 0, 0])
    vals = np.array([1.0, 2.0, 5.0, 0.0, 0.0, 1.0])
    coo = sp.coo_matrix((vals, (rows, cols)), shape=(4, 5))
    csr = sp.csr_matrix((vals, cols, np.array([0, 3, 4, 6, 6])), shape=(4, 5))   # duplicates kept as stored
    assert csr.nnz == 6
    for m in (coo, csr, csr.tocsc()):
        a = row_activity(m)
        assert a.dtype == np.int64 and a.tolist() == [2, 0, 1, 0]


def test_row_activity_dense():
    d = np.array([[0, 1, 1], [0, 0, 0], [1, 1, 1]])
    assert row_activity(d).tolist() == [2, 0, 3]
    assert row_activity(d.astype(np.float32)).tolist() == [2, 0, 3]
    with pytest.raises(ValueError):
        row_activity(np.zeros(3))


@pytest.mark.parametrize("seed", range(5))
def test_targets_permutation_when_sizes_match(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 300))
    c = rng.integers(0, 20, size=n)
    a = rng.integers(0, 50, size=n)
    k = activity_targets(torch.as_tensor(c), a, n_cols=50)
    assert k.dtype == torch.int64 and k.device.type == "cpu"
    assert np.array_equal(np.sort(k.numpy()), np.sort(a))
    assert np.array_equal(k.numpy(), oracle.targets(c, a))


@pytest.mark.parametrize("m,n", [(7, 3), (3, 7), (100, 1), (1, 100), (1, 1), (250, 97)])
def test_targets_formula_and_monotone(m, n):
    rng = np.random.default_rng(m * 1000 + n)
    c = rng.integers(0, 5, size=m)
    a = rng.integers(0, 40, size=n)
    k = activity_targets(torch.as_tensor(c), a).numpy()
    a_sorted = np.sort(a)
    rank = np.empty(m, dtype=np.int64)
    rank[np.lexsort((np.arange(m), c))] = np.arange(m)
    assert np.array_equal(k, a_sorted[((2 * rank + 1) * n) // (2 * m)])
    order = np.lexsort((np.arange(m), c))
    assert np.all(np.diff(k[order]) >= 0)                      # monotone in (c, row index)
    if m == 1:
        assert k.tolist() == [a_sorted[n // 2]]
    if n == 1:
        assert np.all(k == a[0])


def test_targets_ties_go_by_row_index():
    c = torch.tensor([3, 1, 3, 1, 3])
    a = np.array([10, 20, 30, 40, 50])
    # ranks: row 1 -> 0, row 3 -> 1, row 0 -> 2, row 2 -> 3, row 4 -> 4
    assert activity_targets(c, a).tolist() == [30, 10, 40, 20, 50]


def test_targets_int32_inputs_and_tensor_activity():
    c = torch.tensor([2, 0, 1], dtype=torch.int32)
    assert activity_targets(c, torch.tensor([5, 1, 3], dtype=torch.int32)).tolist() == [5, 1, 3]


def test_targets_errors():
    c = torch.tensor([1, 2, 3])
    with pytest.raises(ValueError):
        activity_targets(c, np.array([], dtype=np.int64))
    with pytest.raises(ValueError):
        activity_targets(c, np.array([1, -1, 2]))
    with pytest.raises(ValueError):
        activity_targets(c, np.array([1, 6, 2]), n_cols=5)
    assert activity_targets(c, np.array([1, 5, 2]), n_cols=5).tolist() == [1, 2, 5]
    with pytest.raises(ValueError):
        activity_targets(c, np.array([1.5, 2.0]))
    with pytest.raises(ValueError):
        activity_targets(c.reshape(3, 1), np.array([1, 2]))


def test_main_binarise_flag():
    import main as cli
    p = cli.build_parser()
    assert p.parse_args([]).binarise == "equal-sparsity"
    assert p.parse_args(["--binarise", "activity"]).binarise == "activity"
    assert p.parse_args(["--binarise", "equal-sparsity"]).binarise == "equal-sparsity"
    with pytest.raises(SystemExit):
        p.parse_args(["--binarise", "quantile"])


def test_synthesize_activity_from_flag(tmp_path):
    from sdrm_b200.synthesize import load_activity, parse_args
    base = ["--generator", "g.pt", "--users", "5", "--out", "x.npz"]
    assert parse_args(base).activity_from is None
    assert parse_args(base + ["--activity-from", "real.npz"]).activity_from == "real.npz"
    real = sp.csr_matrix(np.array([[1, 0, 1], [0, 0, 0], [1, 1, 1]], dtype=np.float32))
    path = str(tmp_path / "real.npz")
    sp.save_npz(path, real)
    assert load_activity(path, 3).tolist() == [2, 0, 3]
    with pytest.raises(ValueError):
        load_activity(path, 4)
