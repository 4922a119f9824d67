"""GPU tests of the device SVD evaluator: compute_mf_results_gpu against evaluators.compute_mf_results itself (sklearn on dense
rows), the scored block against sklearn's, every synthetic input kind, run-to-run identity, the adm shape against the CSR
oracle, and kernel K11 alone against a torch fp64 product."""
import numpy as np
import pandas as pd
import pytest
import torch

import svd_oracle as orc
from sdrm_b200 import evaluators, metrics, svd
from sdrm_b200.sparsify import SparseRows, threshold_pack

pytestmark = pytest.mark.gpu

# (n_train, n_test, n_synth, n_items, density, synthetic density): the evaluator's shapes with random rows
SHAPES = {
    "ml-100k": (843, 95, 843, 1008, 0.0575, 0.1007),    # 1 781 x 1 008 with only_synthetic=False
    "alb": (1200, 152, 1200, 729, 0.03, 0.05),           # 2 552 x 729
    "wide": (400, 100, 400, 1008, 0.06, 0.1),            # 900 x 1 008: rows < items, sklearn transposes
    "adm": (9500, 1179, 9500, 8582, 0.00115, 0.002),     # 20 179 x 8 582
}


def _state():
    s = np.random.get_state()
    return s[0], s[1].copy(), s[2:]


def _same_state(a, b):
    return a[0] == b[0] and (a[1] == b[1]).all() and a[2:] == b[2:]


def _close(block, ref, tol=1e-9):
    got = block.cpu().numpy()
    fin = np.isfinite(ref)
    assert (np.isfinite(got) == fin).all() and (got[~fin] == ref[~fin]).all()
    diff = np.abs(got[fin] - ref[fin]).max() / np.abs(ref[fin]).max()
    assert diff <= tol, diff
    return diff


def _per_row_equal(a, b):
    for k in evaluators.K_LIST:
        for x, y in zip(a[k], b[k]):
            np.testing.assert_array_equal(x, y)


@pytest.mark.parametrize("only_synthetic", [False, True])
@pytest.mark.parametrize("shape", ["ml-100k", "alb", "wide"])
def test_matches_compute_mf_results(shape, only_synthetic):
    train, testing, synth = orc.random_case(2024, *SHAPES[shape])
    dense = synth.toarray()
    np.random.seed(1)
    rec_ref, ndcg_ref = evaluators.compute_mf_results(train, testing, synthetic_data=pd.DataFrame(dense),
                                                      only_synthetic=only_synthetic)
    state_ref = _state()
    np.random.seed(2)
    rec, ndcg = evaluators.compute_mf_results_gpu(train, testing, dense, only_synthetic=only_synthetic)
    assert _same_state(state_ref, _state())
    np.testing.assert_array_equal(rec, rec_ref)
    np.testing.assert_array_equal(ndcg, ndcg_ref)

    ref, valid = orc.sklearn_block(train, testing, dense, only_synthetic)
    block, valid_gpu = evaluators.mf_scores_gpu(train, testing, dense, only_synthetic)
    assert (valid != valid_gpu).nnz == 0
    _close(block, ref)
    _per_row_equal(metrics.recall_ndcg_multi_k(block, valid, evaluators.K_LIST),
                   metrics.recall_ndcg_multi_k(ref, valid, evaluators.K_LIST))


@pytest.mark.parametrize("only_synthetic", [False, True])
def test_input_kinds_agree_and_repeat_bit_identically(only_synthetic):
    train, testing, synth = orc.random_case(7, *SHAPES["ml-100k"])
    dense = synth.toarray()
    packed = threshold_pack(torch.from_numpy(dense.astype(np.float32)).cuda(), 0.5)
    assert (packed.numpy() == dense).all()
    rows = packed.to_sparse()
    kinds = {"packed": packed, "sparse rows": rows, "dense": dense, "frame": pd.DataFrame(dense), "csr": synth}
    blocks = {}
    for name, x in kinds.items():
        np.random.seed(3)
        blocks[name] = evaluators.mf_scores_gpu(train, testing, x, only_synthetic)[0]
    again = evaluators.mf_scores_gpu(train, testing, packed, only_synthetic)[0]
    for name, b in blocks.items():
        assert torch.equal(b, blocks["dense"]), name
    assert torch.equal(again, blocks["packed"])
    res = [evaluators.compute_mf_results_gpu(train, testing, x, only_synthetic) for x in (packed, rows, dense)]
    for r in res[1:]:
        np.testing.assert_array_equal(r[0], res[0][0])
        np.testing.assert_array_equal(r[1], res[0][1])


def test_adm_shape_against_csr_oracle():
    """Dense sklearn takes minutes at this shape; the CSR oracle runs sklearn's steps on scipy products."""
    train, testing, synth = orc.random_case(11, *SHAPES["adm"])
    np.random.seed(1)
    ref, valid = orc.csr_block(train, testing, synth, False)
    state_ref = _state()
    np.random.seed(2)
    block, _ = evaluators.mf_scores_gpu(train, testing, synth, False)
    assert _same_state(state_ref, _state())
    _close(block, ref)
    _per_row_equal(metrics.recall_ndcg_multi_k(block, valid, evaluators.K_LIST),
                   metrics.recall_ndcg_multi_k(ref, valid, evaluators.K_LIST))


def _rows_on_device(csr):
    return SparseRows(torch.from_numpy(csr.indptr.astype(np.int64)).cuda(), torch.from_numpy(csr.indices.astype(np.int32)).cuda(),
                      csr.shape[1])


@pytest.mark.parametrize("w", [1, 20, 30, 32])
def test_k11_against_torch(w):
    rng = np.random.default_rng(w)
    csr = orc.random_rows(rng, 300, 6000, 0.01).tolil()
    csr[5, :] = 0                                   # empty rows, at the start, in the middle and at the end
    csr[0, :] = 0
    csr[299, :] = 0
    csr[17, rng.choice(6000, 5000, replace=False)] = 1      # a 5 000-entry row: about 20 chunks of 256
    csr[18, :300] = 1                                       # a row crossing chunk boundaries
    csr = csr.tocsr()
    csr.sort_indices()
    rows = _rows_on_device(csr)
    wide = torch.randn(6000, 40, dtype=torch.float64, device="cuda")
    x = wide[:, 3:3 + w]                            # row stride 40 > w
    y = svd.spmm(rows, x)
    ref = torch.from_numpy(csr.toarray().astype(np.float64)).cuda() @ x
    assert y.shape == (300, w)
    torch.testing.assert_close(y, ref, rtol=1e-12, atol=1e-12)
    assert (y[[0, 5, 299]] == 0).all()
    assert torch.equal(svd.spmm(rows, x), y)        # fixed summation order


def test_k11_status_word():
    """An out-of-range index is reported in the status word and contributes nothing; an inconsistent indptr pair is reported and
    its row is written as 0.  Neither faults."""
    lib_rows = SparseRows(torch.tensor([0, 3, 5, 8], dtype=torch.int64, device="cuda"),
                          torch.tensor([0, 1, 9, 2, 3, -4, 4, 5], dtype=torch.int32, device="cuda"), 6)
    x = torch.arange(12, dtype=torch.float64, device="cuda").reshape(6, 2)
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    y = svd.spmm(lib_rows, x, status)
    assert int(status.item()) == 1
    expect = torch.stack([x[0] + x[1], x[2] + x[3], x[4] + x[5]])
    assert torch.equal(y, expect)
    with pytest.raises(ValueError, match="outside the item range"):
        svd.spmm(lib_rows, x)
    bad = SparseRows(torch.tensor([0, 3, 2, 5], dtype=torch.int64, device="cuda"),
                     torch.tensor([0, 1, 2, 3, 4], dtype=torch.int32, device="cuda"), 6)
    status.zero_()
    y = svd.spmm(bad, x, status)
    assert int(status.item()) == 2 and (y[1] == 0).all()
    with pytest.raises(ValueError, match="indptr"):
        svd.spmm(bad, x)


def test_randomized_svd_shape_checks_on_device():
    train, testing, synth = orc.random_case(5, *SHAPES["wide"])
    M = _rows_on_device(synth)
    with pytest.raises(ValueError, match="transpose"):
        svd.randomized_svd(M, M)
    with pytest.raises(ValueError):
        svd.spmm(M, torch.zeros(1008, 33, dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        svd.spmm(M, torch.zeros(1008, 30, dtype=torch.float32, device="cuda"))
