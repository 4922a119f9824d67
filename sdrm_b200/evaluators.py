"""Downstream consumers of the synthetic rows.

The SVD evaluator comes twice.  compute_mf_results is the reference's sklearn code on dense host rows; the end-to-end
Recall@10 parity check is measured against it, so it stays the default.  compute_mf_results_gpu computes the same randomized
truncated SVD on the device (sdrm_b200.svd: the products on kernel K11) from CSR rows, with the same seeds and row bookkeeping.
The Keras MLP and NeuMF evaluators are out of scope as kernels (SURVEY.md §2 rows 7-9) and are loaded lazily from the user's
reference checkout if it is importable.  Metrics go through the K3 top-k kernel (sdrm_b200.metrics).
"""
import importlib

import numpy as np
import torch

from . import metrics
from .data import split_train_test_proportion_from_csr_matrix

K_LIST = [1, 3, 5, 10, 20, 50]


def compute_mf_results(training_dataset, testing_dataset, synthetic_data=None, nnmf=False, only_synthetic=False):
    """TruncatedSVD(20, n_iter=100) recommender on [train | synthetic] + visible validation part
    (reference: svd_benchmark.compute_mf_results, svd_benchmark.py:17-70; same seeds, same row bookkeeping)."""
    from sklearn.decomposition import NMF, TruncatedSVD
    test_data, valid_data = split_train_test_proportion_from_csr_matrix(testing_dataset, batch_size=1000, random_seed=123)
    synth = None if synthetic_data is None else np.asarray(synthetic_data)
    head = synth if only_synthetic else training_dataset.toarray()
    training_data = np.concatenate([head, test_data.toarray()], axis=0)
    combined = training_data if (only_synthetic and synth is not None) else np.concatenate([training_data, synth], axis=0)
    mf = NMF(n_components=15, max_iter=50) if nnmf else TruncatedSVD(n_components=20, n_iter=100)
    recon = mf.inverse_transform(mf.fit_transform(combined))
    masked = metrics.mask_training_examples(sparse_training_set=training_data, dense_matrix=recon[:training_data.shape[0]].copy())
    lo = head.shape[0]
    block = masked[lo: lo + valid_data.shape[0]]
    both = metrics.recall_ndcg_multi_k(block, valid_data, K_LIST)   # one pass over the scores for all six cut-offs
    recall = [np.round(np.nanmean(both[k][0]), 4) for k in K_LIST]
    ndcg = [np.round(np.nanmean(both[k][1]), 4) for k in K_LIST]
    return np.array(recall), np.array(ndcg)


def mf_scores_gpu(training_dataset, testing_dataset, synthetic_data, only_synthetic=False):
    """The scored block of compute_mf_results_gpu: reconstructed scores of the visible test rows with their own items at -inf,
    a CUDA float64 tensor [V, items], and valid_data (the held-out parts, scipy CSR).  Within rounding of the block
    compute_mf_results scores.

    Rows are assembled on the device in compute_mf_results' order, [head; test_data] (only_synthetic) or
    [train; test_data; synthetic] with head = synthetic or train, without a dense host matrix.  Every argument is checked
    before NumPy's global RandomState is touched; afterwards it has been consumed exactly as compute_mf_results consumes it."""
    from scipy.sparse import csr_matrix

    from . import svd
    if synthetic_data is None:
        raise ValueError("compute_mf_results_gpu needs synthetic_data")
    if type(testing_dataset) is not csr_matrix:
        raise TypeError("Input data is not of type csr_matrix")
    s_rows, n_items = svd.rows_shape(synthetic_data)
    shapes = {"synthetic_data": n_items, "testing_dataset": testing_dataset.shape[1]}
    if not only_synthetic:
        t_rows, shapes["training_dataset"] = svd.rows_shape(training_dataset)
    if len(set(shapes.values())) != 1:
        raise ValueError(f"item counts differ: {shapes}")
    n_test = int(np.count_nonzero(np.diff(testing_dataset.indptr) >= 2))   # users the split keeps
    svd.check_shape((s_rows if only_synthetic else t_rows + s_rows) + n_test, n_items)
    synth = _binary_rows(synthetic_data)
    train = None if only_synthetic else _binary_rows(training_dataset)
    dev = svd._device()

    test_data, valid_data = split_train_test_proportion_from_csr_matrix(testing_dataset, batch_size=1000, random_seed=123)
    test = svd.device_rows(test_data, dev)
    synth = svd.device_rows(synth, dev)
    parts = [synth, test] if only_synthetic else [svd.device_rows(train, dev), test, synth]
    M = svd.vstack_rows(parts)
    VT, _ = svd.randomized_svd(M, svd.transpose_rows(M))
    block = svd.spmm(test, VT.T) @ VT
    seen = torch.repeat_interleave(torch.arange(test.shape[0], device=dev), test.indptr.diff(), output_size=test.nnz)
    block[seen, test.indices.long()] = -np.inf
    return block, valid_data


def _binary_rows(x):
    """Host rows validated and made canonical CSR now (before any random draw); device rows as they are."""
    from . import svd
    return x if isinstance(x, (svd.PackedMatrix, svd.SparseRows)) else svd.binary_csr_host(x)


def compute_mf_results_gpu(training_dataset, testing_dataset, synthetic_data, only_synthetic=False):
    """compute_mf_results (TruncatedSVD(20, n_iter=100), nnmf=False) on the device: same return value (recall[6], ndcg[6]),
    same consumption of NumPy's global RandomState.  synthetic_data: a PackedMatrix, SparseRows, scipy sparse matrix,
    ndarray or DataFrame of 0/1 rows; training_dataset: scipy CSR (unused when only_synthetic).  Raises ValueError for
    values other than 0 and 1, differing item counts and the shapes sdrm_b200.svd does not support."""
    block, valid_data = mf_scores_gpu(training_dataset, testing_dataset, synthetic_data, only_synthetic)
    both = metrics.recall_ndcg_multi_k(block, valid_data, K_LIST)
    recall = [np.round(np.nanmean(both[k][0]), 4) for k in K_LIST]
    ndcg = [np.round(np.nanmean(both[k][1]), 4) for k in K_LIST]
    return np.array(recall), np.array(ndcg)


def _external(module, fn):
    try:
        return getattr(importlib.import_module(module), fn)
    except Exception as exc:  # TensorFlow / the reference checkout is not part of this package
        raise RuntimeError(f"evaluator {module}.{fn} is outside the B200 hot path and is not bundled; put the reference "
                           f"checkout on PYTHONPATH to use it ({exc})")


def compute_mlp_results(*args, **kwargs):
    return _external("mlp_benchmark", "compute_mlp_results")(*args, **kwargs)


def compute_neuralcf_results(*args, **kwargs):
    return _external("neural_cf_benchmark_pt", "compute_neuralcf_results")(*args, **kwargs)
