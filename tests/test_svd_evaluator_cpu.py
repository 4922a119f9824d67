"""CPU tests of the device SVD evaluator (evaluators.compute_mf_results_gpu, sdrm_b200.svd, K11): the CSR oracle against sklearn,
the random state the evaluator leaves behind, the host-side row assembly and every argument check, which all run before
anything reaches a device."""
import ctypes

import numpy as np
import pandas as pd
import pytest
import scipy.sparse as sp
import torch

import svd_oracle as orc
from sdrm_b200 import evaluators, svd
from sdrm_b200.sparsify import SparseRows

# (n_train, n_test, n_synth, n_items, density): rows > items, and rows < items (sklearn transposes)
SHAPES = {"tall": (150, 60, 150, 120, 0.08), "wide": (40, 30, 40, 260, 0.06)}


def _max_rel(a, b):
    fin = np.isfinite(b)
    assert (np.isfinite(a) == fin).all() and (a[~fin] == b[~fin]).all()
    return np.abs(a[fin] - b[fin]).max() / np.abs(b[fin]).max()


@pytest.mark.parametrize("only_synthetic", [False, True])
@pytest.mark.parametrize("shape", sorted(SHAPES))
def test_csr_oracle_matches_sklearn(shape, only_synthetic):
    train, testing, synth = orc.random_case(7, *SHAPES[shape])
    np.random.seed(99)
    ref, valid_ref = orc.sklearn_block(train, testing, synth.toarray(), only_synthetic)
    state_ref = np.random.get_state()
    np.random.seed(99)
    got, valid = orc.csr_block(train, testing, synth, only_synthetic)
    state = np.random.get_state()
    assert _max_rel(got, ref) <= 1e-12
    assert (valid != valid_ref).nnz == 0
    assert state[0] == state_ref[0] and (state[1] == state_ref[1]).all() and state[2:] == state_ref[2:]
    # sklearn's draw is the only one after the split's re-seed: the state does not depend on the seed before the call
    np.random.seed(5)
    orc.csr_block(train, testing, synth, only_synthetic)
    assert (np.random.get_state()[1] == state_ref[1]).all()


def test_oracle_transposes_like_sklearn():
    """rows < items: the components come from U of the transposed problem; rows > items: from Vt."""
    for shape in SHAPES:
        train, testing, synth = orc.random_case(3, *SHAPES[shape])
        M = sp.vstack([train, testing, synth], format="csr").astype(np.float64)
        from sklearn.utils.extmath import randomized_svd
        np.random.seed(4)
        _, _, vt_ref = randomized_svd(M, 20, n_oversamples=10, n_iter=100, random_state=None, flip_sign=False)
        np.random.seed(4)
        vt = orc.randomized_components(M)
        assert np.abs(np.abs((vt * vt_ref).sum(axis=1)) - 1).max() < 1e-10   # each component equal up to its sign


def test_binary_csr_host_inputs():
    dense = np.array([[0, 1, 0, 1], [0, 0, 0, 0], [1, 1, 0, 0]])
    for x in (dense, dense.astype(bool), dense.astype(np.float32), pd.DataFrame(dense), sp.csr_matrix(dense),
              sp.coo_matrix(dense)):
        csr = svd.binary_csr_host(x)
        assert csr.has_canonical_format and csr.dtype == np.int64 and (csr.toarray() == dense).all()
    # explicit stored zeros are no interaction; duplicates of a 0 stay 0
    z = sp.csr_matrix((np.array([1.0, 0.0, 1.0]), np.array([3, 1, 0]), np.array([0, 2, 2, 3])), shape=(3, 4))
    csr = svd.binary_csr_host(z)
    assert csr.nnz == 2 and (csr.toarray() == z.toarray()).all()


@pytest.mark.parametrize("bad", [np.array([[0, 2], [1, 0]]), np.array([[0.5, 1.0]]), np.array([[-1, 0]]),
                                 pd.DataFrame([[1, 3]]), sp.csr_matrix(np.array([[0, 1, 7]])),
                                 sp.coo_matrix((np.ones(2), (np.array([0, 0]), np.array([1, 1]))), shape=(1, 3)),  # 1 + 1
                                 np.array([["a", "b"]])])
def test_non_binary_values_raise(bad):
    with pytest.raises(ValueError):
        svd.binary_csr_host(bad)


def test_vstack_and_transpose_rows_cpu():
    rng = np.random.default_rng(0)
    dense = [(rng.random((r, 37)) < 0.2).astype(np.int64) for r in (5, 0, 11, 3)]
    dense[2][4] = 0                                              # an empty row in the middle
    blocks = [sp.csr_matrix(d) for d in dense]
    parts = [SparseRows(torch.from_numpy(b.indptr.astype(np.int64)), torch.from_numpy(b.indices.astype(np.int32)), 37)
             for b in blocks]
    M = svd.vstack_rows(parts)
    ref = sp.vstack(blocks, format="csr")
    assert (M.indptr.numpy() == ref.indptr).all() and (M.indices.numpy() == ref.indices).all() and M.shape == ref.shape
    Mt = svd.transpose_rows(M)
    ref_t = ref.T.tocsr()
    ref_t.sort_indices()
    assert Mt.shape == (37, 19) and Mt.indices.dtype == torch.int32
    assert (Mt.indptr.numpy() == ref_t.indptr).all() and (Mt.indices.numpy() == ref_t.indices).all()
    with pytest.raises(ValueError, match="item counts"):
        svd.vstack_rows([parts[0], SparseRows(parts[0].indptr, parts[0].indices, 38)])


def test_check_shape():
    svd.check_shape(30, 30)
    svd.check_shape(10 ** 6, 20000)
    with pytest.raises(ValueError, match="minimum of 2"):
        svd.check_shape(100, 1)
    with pytest.raises(ValueError, match="n_components"):
        svd.check_shape(100, 19)
    for m, n in ((29, 500), (500, 29), (10, 25)):
        with pytest.raises(ValueError):
            svd.check_shape(m, n)
    with pytest.raises(ValueError, match="2\\^31"):
        svd.check_shape(100, 2 ** 31)


def _state():
    s = np.random.get_state()
    return s[0], s[1].copy(), s[2:]


def _same_state(a, b):
    return a[0] == b[0] and (a[1] == b[1]).all() and a[2:] == b[2:]


@pytest.mark.parametrize("case", ["non-binary synth", "non-binary train", "items differ (synth)", "items differ (train)",
                                  "too few items", "too few rows", "type synth", "type testing", "no synth"])
def test_compute_mf_results_gpu_rejects_before_any_draw(case):
    train, testing, synth = orc.random_case(1, 60, 40, 60, 50, 0.1)
    only = False
    if case == "non-binary synth":
        synth = synth * 2
    elif case == "non-binary train":
        train = train * 3
    elif case == "items differ (synth)":
        synth = synth[:, :-1]
    elif case == "items differ (train)":
        train = train[:, :-1]
    elif case == "too few items":
        train, testing, synth = orc.random_case(1, 60, 40, 60, 19, 0.3)
    elif case == "too few rows":
        train, testing, synth = orc.random_case(1, 0, 10, 15, 50, 0.2)
        only = True
    elif case == "type synth":
        synth = torch.from_numpy(synth.toarray())
    elif case == "type testing":
        testing = testing.tocoo()
    elif case == "no synth":
        synth = None
    np.random.seed(11)
    before = _state()
    with pytest.raises((ValueError, TypeError)):
        evaluators.compute_mf_results_gpu(train, testing, synth, only_synthetic=only)
    assert _same_state(before, _state())


def test_types_raise_type_error():
    train, testing, synth = orc.random_case(1, 60, 40, 60, 50, 0.1)
    for bad in (synth.toarray().tolist(), torch.from_numpy(synth.toarray()), "rows"):
        with pytest.raises(TypeError):
            evaluators.compute_mf_results_gpu(train, testing, bad)
    with pytest.raises(ValueError, match="2-D"):
        evaluators.compute_mf_results_gpu(train, testing, synth.toarray()[0])


def test_no_nnmf_argument():
    with pytest.raises(TypeError):
        evaluators.compute_mf_results_gpu(None, None, None, nnmf=True)


def test_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from sdrm_b200 import _lib
    train, testing, synth = orc.random_case(1, 60, 40, 60, 50, 0.1)
    with pytest.raises(_lib.SdrmError):
        evaluators.compute_mf_results_gpu(train, testing, synth)


@pytest.fixture(scope="module")
def lib():
    from sdrm_b200 import _lib
    from sdrm_b200.csrc import build
    build.build()
    return _lib.load()


def test_c_abi_host_checks(lib):
    """Bad arguments return SDRM_ERR_BAD_ARG (-1), SDRM_ERR_UNSUPPORTED (-2) or SDRM_ERR_WORKSPACE (-5) before any launch."""
    ws = lib.sdrm_spmm_binary_workspace_bytes
    assert ws(0, 30) == 0 and ws(1, 30) == 2 * 30 * 8 and ws(256, 30) == 2 * 30 * 8 and ws(257, 1) == 2 * 2 * 8
    assert ws(100, 0) == 0 and ws(100, 33) == 0
    buf = ctypes.create_string_buffer(4096)
    p = ctypes.c_void_p((ctypes.addressof(buf) + 15) // 16 * 16)
    f = lib.sdrm_spmm_binary
    #        indptr ind rows nnz  x  n_x w  ldx  y  ldy status ws  bytes stream
    assert f(p, p, -1, 10, p, 8, 30, 30, p, 30, p, p, 4096, None) == -1
    assert f(p, p, 4, -1, p, 8, 30, 30, p, 30, p, p, 4096, None) == -1
    assert f(p, p, 4, 10, p, 8, 0, 30, p, 30, p, p, 4096, None) == -1
    assert f(p, p, 4, 10, p, 8, 30, 29, p, 30, p, p, 4096, None) == -1           # ldx < w
    assert f(p, p, 4, 10, p, 8, 30, 30, p, 29, p, p, 4096, None) == -1           # ldy < w
    assert f(p, p, 4, 10, p, 8, 33, 33, p, 33, p, p, 4096, None) == -2           # w > 32
    assert f(p, p, 0, 10, p, 8, 30, 30, p, 30, p, p, 4096, None) == -1           # entries without rows
    assert f(None, p, 4, 10, p, 8, 30, 30, p, 30, p, p, 4096, None) == -1 and b"null" in lib.sdrm_last_error()
    assert f(p, None, 4, 10, p, 8, 30, 30, p, 30, p, p, 4096, None) == -1
    assert f(p, p, 4, 10, None, 8, 30, 30, p, 30, p, p, 4096, None) == -1
    assert f(p, p, 4, 10, p, 8, 30, 30, None, 30, p, p, 4096, None) == -1
    assert f(p, p, 4, 10, p, 8, 30, 30, p, 30, None, p, 4096, None) == -1
    assert f(p, p, 4, 10, p, 8, 30, 30, p, 30, p, None, 4096, None) == -1
    assert f(p, p, 4, 10, p, 8, 30, 30, p, 30, p, p, 8, None) == -5
    assert f(None, None, 0, 0, None, 0, 30, 30, None, 30, None, None, 0, None) == 0   # zero rows: nothing to do


def test_main_and_e2e_flags():
    import main as cli
    assert cli.build_parser().parse_args([]).svd_on_gpu is False
    assert cli.build_parser().parse_args(["--svd-on-gpu"]).svd_on_gpu is True
