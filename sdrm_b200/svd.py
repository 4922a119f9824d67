"""Randomized truncated SVD of binary rows on the device: what sklearn's TruncatedSVD(n_components=20, n_iter=100) computes for
the SVD evaluator (evaluators.compute_mf_results), with every product of the sparse matrix on kernel K11.

sklearn 1.9 (utils/extmath.py: _randomized_svd, _randomized_range_finder) on M (m x n), k = 20, p = 10:

    A = M.T if m < n else M
    Q = np.random.normal(size=(A.shape[1], k + p))          # the global RandomState: the only draw
    n_iter times: Q = normalise(A @ Q); Q = normalise(A.T @ Q)
    Q = qr(A @ Q); B = Q.T @ A; Uh, s, Vt = svd(B)
    components (k x n) = Vt[:k], or (Q @ Uh)[:, :k].T when transposed

Here M and M.T are CSR on the device (`SparseRows`), A @ Q, A.T @ Q and B = (A.T @ Q).T are K11 products
(`sdrm_spmm_binary`), and the 30-column algebra is torch plumbing.  The normaliser is a reduced QR where sklearn uses LU with
permute_l: only the span of Q matters, so the components agree within rounding, up to a sign per component that
X @ VT.T @ VT cancels.

Supported: binary rows (stored values 0 or 1), 2 <= n < 2^31 items, fewer than 2^31 rows, and min(m, n) >= k + p.  sklearn
itself rejects fewer than 2 items and k > n; the last condition is this module's (sklearn's power iterations shrink Q below
k + p columns there).  Every other shape raises ValueError before anything reaches the device.

No CPU fallback: the products need a CUDA device.
"""
import numpy as np
import scipy.sparse as sp
import torch

from . import _lib
from .sparsify import PackedMatrix, SparseRows

N_COMPONENTS, N_OVERSAMPLES, N_ITER = 20, 10, 100
MAX_WIDTH = 32                      # K11's widest X
_INT32_LIMIT = 2 ** 31 - 1


def _device():
    if not torch.cuda.is_available():
        raise _lib.SdrmError("the SVD evaluator's products need a CUDA device (sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


# --------------------------------------------------------------------------------------------------
# binary rows from what the callers hold
# --------------------------------------------------------------------------------------------------
def rows_shape(x):
    """(rows, items) of a PackedMatrix, SparseRows, scipy sparse matrix, 2-D ndarray or DataFrame; TypeError for anything else."""
    if isinstance(x, (PackedMatrix, SparseRows)) or sp.issparse(x):
        return tuple(int(s) for s in x.shape)
    if _is_frame(x) or isinstance(x, np.ndarray):
        if x.ndim != 2:
            raise ValueError(f"binary rows must be 2-D, got shape {x.shape}")
        return tuple(int(s) for s in x.shape)
    raise TypeError(f"binary rows must be a PackedMatrix, SparseRows, scipy sparse matrix, ndarray or DataFrame, "
                    f"got {type(x).__name__}")


def _is_frame(x):
    return type(x).__name__ == "DataFrame" and hasattr(x, "to_numpy")


def binary_csr_host(x):
    """Host rows (scipy sparse, ndarray or DataFrame) as a canonical scipy CSR of int64 ones, the way the dense evaluator sees
    them: duplicates summed, explicit zeros dropped.  A value other than 0 or 1 raises ValueError."""
    rows_shape(x)
    if sp.issparse(x):
        csr = sp.csr_matrix(x, copy=True)
        csr.sum_duplicates()
        data = csr.data
    else:
        a = x.to_numpy() if _is_frame(x) else x
        if a.dtype == object or a.dtype.kind not in "biuf":
            raise ValueError(f"binary rows must hold numbers, got dtype {a.dtype}")
        nz = a != 0
        data = a[nz]
        csr = sp.csr_matrix((np.ones(int(nz.sum()), dtype=np.int64), np.nonzero(nz)[1],
                             np.concatenate([[0], np.cumsum(nz.sum(axis=1))])), shape=a.shape)
    if data.size and not np.all((data == 0) | (data == 1)):
        bad = data[(data != 0) & (data != 1)][0]
        raise ValueError(f"the SVD evaluator takes binary rows; found the value {bad!r}")
    if sp.issparse(x):
        csr.eliminate_zeros()
        csr = sp.csr_matrix((np.ones(csr.nnz, dtype=np.int64), csr.indices, csr.indptr), shape=csr.shape)
    return csr


def device_rows(x, device=None):
    """Binary rows as SparseRows on the device.  A PackedMatrix goes through K10 (PackedMatrix.to_sparse), SparseRows are used
    as they are, host rows are validated by binary_csr_host and uploaded (indptr int64, indices int32)."""
    if isinstance(x, PackedMatrix):
        return x.to_sparse()
    if isinstance(x, SparseRows):
        return x
    dev = device or _device()
    csr = binary_csr_host(x)
    return SparseRows(torch.from_numpy(csr.indptr.astype(np.int64)).to(dev),
                      torch.from_numpy(csr.indices.astype(np.int32)).to(dev), csr.shape[1])


def vstack_rows(parts):
    """Row blocks over the same items stacked in order (one SparseRows; indices stay ascending within each row)."""
    n_cols = {p.n_cols for p in parts}
    if len(n_cols) != 1:
        raise ValueError(f"row blocks over different item counts: {sorted(n_cols)}")
    indptr, off = [parts[0].indptr[:1]], 0
    for p in parts:
        indptr.append(p.indptr[1:] + off)
        off += p.nnz
    return SparseRows(torch.cat(indptr), torch.cat([p.indices for p in parts]), n_cols.pop())


def transpose_rows(rows):
    """The CSR of the transpose: a stable sort of the column indices keeps each column's rows ascending."""
    m, n = rows.shape
    if m > _INT32_LIMIT:
        raise ValueError(f"{m} rows do not fit the int32 indices of the transpose")
    dev = rows.indices.device
    cols, order = torch.sort(rows.indices.long(), stable=True)
    indptr = torch.searchsorted(cols, torch.arange(n + 1, device=dev))
    row_of = torch.repeat_interleave(torch.arange(m, device=dev), rows.indptr.diff(), output_size=rows.nnz)
    return SparseRows(indptr, row_of[order].to(torch.int32), m)


# --------------------------------------------------------------------------------------------------
# K11 and the randomized SVD
# --------------------------------------------------------------------------------------------------
def spmm(rows, x, status=None):
    """Y = rows @ x for binary SparseRows [m, n] and a CUDA fp64 x [n, w], w <= 32, with kernel K11 (fixed summation order:
    bit-identical from call to call).  `status` (int32[1], zeroed) collects K11's status bits without a synchronisation;
    without it the call reads them back and raises ValueError on a bad index or indptr."""
    m, n = rows.shape
    if x.dtype != torch.float64 or x.dim() != 2 or x.shape[0] != n or not 1 <= x.shape[1] <= MAX_WIDTH:
        raise ValueError(f"x must be float64 [{n}, w] with 1 <= w <= {MAX_WIDTH}, got {x.dtype} {tuple(x.shape)}")
    if x.stride(1) != 1:
        x = x.contiguous()
    lib = _lib.load()
    w = x.shape[1]
    y = torch.empty((m, w), dtype=torch.float64, device=x.device)
    own = status is None
    if own:
        status = torch.zeros(1, dtype=torch.int32, device=x.device)
    ws_bytes = lib.sdrm_spmm_binary_workspace_bytes(rows.nnz, w)
    ws = torch.empty(max(1, (ws_bytes + 7) // 8), dtype=torch.float64, device=x.device)
    _lib.check(lib.sdrm_spmm_binary(_lib.ptr(rows.indptr), _lib.ptr(rows.indices), m, rows.nnz, _lib.ptr(x), n, w,
                                    x.stride(0) if n else w, _lib.ptr(y), w, _lib.ptr(status), _lib.ptr(ws), ws_bytes,
                                    _lib.stream_ptr()), "sdrm_spmm_binary")
    if own:
        check_status(status)
    return y


def check_status(status):
    """Raise ValueError if K11 flagged a bad index or indptr (one read-back)."""
    bits = int(status.item())
    if bits:
        what = [s for b, s in ((1, "an index outside the item range"), (2, "an inconsistent indptr")) if bits & b]
        raise ValueError(f"sdrm_spmm_binary: the rows hold {' and '.join(what)} (status {bits})")


def check_shape(m, n, n_components=N_COMPONENTS, n_oversamples=N_OVERSAMPLES):
    """ValueError for the shapes sklearn rejects and for those this module does not support (see the module docstring)."""
    if n < 2:
        raise ValueError(f"Found array with {n} feature(s) (shape=({m}, {n})) while a minimum of 2 is required.")
    if n_components > n:
        raise ValueError(f"n_components({n_components}) must be <= n_features({n}).")
    if min(m, n) < n_components + n_oversamples:
        raise ValueError(f"the device SVD needs min(rows, items) >= n_components + n_oversamples = "
                         f"{n_components + n_oversamples}, got {m} x {n}")
    if n > _INT32_LIMIT or m > _INT32_LIMIT:
        raise ValueError(f"the device SVD needs fewer than 2^31 rows and items, got {m} x {n}")
    if n_components + n_oversamples > MAX_WIDTH:
        raise ValueError(f"n_components + n_oversamples = {n_components + n_oversamples} exceeds K11's {MAX_WIDTH} columns")


def _orth(y):
    return torch.linalg.qr(y, mode="reduced").Q.contiguous()


def randomized_svd(M, Mt, n_components=N_COMPONENTS, n_oversamples=N_OVERSAMPLES, n_iter=N_ITER):
    """sklearn's _randomized_svd(M, n_components, n_oversamples, n_iter, random_state=None) on the device for binary M [m, n]
    given with its transpose Mt (SparseRows).  Draws np.random.normal once from NumPy's global RandomState, like sklearn.
    Returns (components fp64 [n_components, n], singular values fp64 [n_components]), both on the device; a component may
    differ from sklearn's by its sign."""
    m, n = M.shape
    check_shape(m, n, n_components, n_oversamples)
    if Mt.shape != (n, m) or Mt.nnz != M.nnz:
        raise ValueError(f"Mt {Mt.shape} with {Mt.nnz} ones is not the transpose of M {M.shape} with {M.nnz} ones")
    dev = M.indptr.device
    transpose = m < n
    A, At = (Mt, M) if transpose else (M, Mt)
    Q = torch.from_numpy(np.random.normal(size=(A.shape[1], n_components + n_oversamples))).to(dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    for _ in range(n_iter):
        Q = _orth(spmm(A, Q, status))
        Q = _orth(spmm(At, Q, status))
    Q = _orth(spmm(A, Q, status))
    B = spmm(At, Q, status).T                       # Q.T @ A
    Uh, s, Vt = torch.linalg.svd(B, full_matrices=False)
    check_status(status)
    VT = (Q @ Uh)[:, :n_components].T if transpose else Vt[:n_components]
    return VT.contiguous(), s[:n_components]
