"""NumPy / scipy oracles of the SVD evaluator's scored block (evaluators.compute_mf_results up to the metrics call).

sklearn_block: the dense sklearn path itself (TruncatedSVD(20, n_iter=100) on the dense 0/1 matrix), as compute_mf_results runs it.
csr_block:     the same randomized SVD restated on scipy CSR products: sklearn's steps (same single draw from NumPy's global
               RandomState, same LU normaliser, same final QR and SVD) with the products summed in another order.  It scales
               to shapes where the dense path takes minutes.
Both return (block [V, items] float64 with each test row's own items at -inf, valid_data).
"""
import numpy as np
import scipy.linalg as sla
import scipy.sparse as sp

from sdrm_b200.data import split_train_test_proportion_from_csr_matrix

K, P, N_ITER = 20, 10, 100


def _dense(x):
    if sp.issparse(x):
        return x.toarray()
    return x.to_numpy() if hasattr(x, "to_numpy") else np.asarray(x)


def _mask(block, test_data):
    block[test_data.nonzero()] = -np.inf
    return block


def sklearn_block(train, testing, synth, only_synthetic=False):
    from sklearn.decomposition import TruncatedSVD
    test_data, valid_data = split_train_test_proportion_from_csr_matrix(testing, batch_size=1000, random_seed=123)
    synth = _dense(synth)
    head = synth if only_synthetic else train.toarray()
    training_data = np.concatenate([head, test_data.toarray()], axis=0)
    combined = training_data if only_synthetic else np.concatenate([training_data, synth], axis=0)
    mf = TruncatedSVD(n_components=K, n_iter=N_ITER)
    recon = mf.inverse_transform(mf.fit_transform(combined))
    lo = head.shape[0]
    return _mask(recon[lo: lo + valid_data.shape[0]].copy(), test_data), valid_data


def randomized_components(M, k=K, p=P, n_iter=N_ITER):
    """sklearn's _randomized_svd(M, k, n_oversamples=p, n_iter, power_iteration_normalizer='LU') components, M scipy CSR."""
    m, n = M.shape
    A = M.T.tocsr() if m < n else M
    At = A.T.tocsr()
    Q = np.random.normal(size=(A.shape[1], k + p))
    for _ in range(n_iter):
        Q = sla.lu(A @ Q, permute_l=True, check_finite=False)[0]
        Q = sla.lu(At @ Q, permute_l=True, check_finite=False)[0]
    Q = sla.qr(A @ Q, mode="economic", check_finite=False)[0]
    B = (At @ Q).T
    Uh, s, Vt = sla.svd(B, full_matrices=False, check_finite=False, lapack_driver="gesdd")
    return (Q @ Uh)[:, :k].T if m < n else Vt[:k]


def csr_block(train, testing, synth, only_synthetic=False):
    test_data, valid_data = split_train_test_proportion_from_csr_matrix(testing, batch_size=1000, random_seed=123)
    synth = sp.csr_matrix(synth if sp.issparse(synth) else _dense(synth), dtype=np.float64)
    test_data = sp.csr_matrix(test_data, dtype=np.float64)
    head = synth if only_synthetic else sp.csr_matrix(train, dtype=np.float64)
    M = sp.vstack([head, test_data] + ([] if only_synthetic else [synth]), format="csr")
    VT = randomized_components(M)
    return _mask((test_data @ VT.T) @ VT, test_data), valid_data


def random_rows(rng, n, n_items, density):
    """n seeded random 0/1 rows over n_items, each entry 1 with probability about `density`, as canonical int64 CSR."""
    counts = rng.binomial(n_items, density, size=n)
    keys = np.unique(np.repeat(np.arange(n, dtype=np.int64), counts) * n_items + rng.integers(0, n_items, int(counts.sum())))
    return sp.csr_matrix((np.ones(keys.size, dtype=np.int64), (keys // n_items, keys % n_items)), shape=(n, n_items))


def random_case(seed, n_train, n_test, n_synth, n_items, density, synth_density=None):
    """(train, testing, synthetic) seeded random 0/1 rows as CSR; the split skips test rows with fewer than 2 items."""
    rng = np.random.default_rng(seed)
    return (random_rows(rng, n_train, n_items, density), random_rows(rng, n_test, n_items, density),
            random_rows(rng, n_synth, n_items, synth_density or density))
