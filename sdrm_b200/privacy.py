"""Memorisation audit of binary rows: for every query row (e.g. a synthetic user), its nearest reference rows (e.g. the real users
the generator was trained on) by Jaccard similarity, found by the K8 kernel (sdrm_privacy_*, include/sdrm_b200.h).  The
intersection counts are an exact integer product on the tensor cores and the top-k is fused into its epilogue; nothing dense
goes through the host.  There is no CPU fallback.

    res = nearest_rows(synthetic_bits, real_csr, k=2)
    res.summary()   # distance to the closest record (DCR = 1 - J), exact copies, nearest-neighbour distance ratio

Accepted row sets (either side): sparsify.PackedMatrix (bit-packed rows, e.g. sample_ddpm_sharded(gather="bits")), scipy CSR,
torch sparse CSR, training.DeviceCSR, and dense 0/1 torch or NumPy arrays (nonzero = 1).  For sparse input a stored value != 0
is an interaction; explicit stored zeros are not, and a repeated column counts once.
"""
import operator

import numpy as np
import torch

from . import _lib

MAX_K = 16
MAX_ITEMS = 1 << 20
_BAD_INDEX, _BAD_INDPTR = 1, 2   # enum sdrm_privacy_status


class NearestRows:
    """Per query row the k nearest reference rows, best first (highest J, ties to the lower reference index).
    index int64 [n, k]; intersection c and union u int32 [n, k]; query_ones int32 [n] (the ones of each query row)."""

    def __init__(self, index, intersection, union, query_ones):
        self.index = torch.as_tensor(index)
        self.intersection = torch.as_tensor(intersection)
        self.union = torch.as_tensor(union)
        self.query_ones = torch.as_tensor(query_ones)

    @property
    def k(self):
        return self.index.shape[1]

    @property
    def jaccard(self):
        """float64 [n, k]: c / u, and 1 where u = 0 (two empty rows)."""
        c, u = self.intersection.double(), self.union.double()
        return torch.where(u == 0, torch.ones_like(u), c / u.clamp_min(1))

    @property
    def hamming(self):
        """int32 [n, k]: u - c, the number of columns in which the two rows differ."""
        return self.union - self.intersection

    def summary(self):
        """Distance to the closest record, DCR = 1 - J of the nearest reference row: mean and 5 / 50 / 95 % quantiles (NumPy's
        linear interpolation); exact copies = rows whose nearest reference row has Hamming distance 0, as a count and a share;
        with k >= 2 the median nearest-neighbour distance ratio DCR_1 / DCR_2 (taken as 1 where DCR_2 = 0)."""
        dcr = 1.0 - self.jaccard.cpu().numpy()
        ham = self.hamming.cpu().numpy()
        n = dcr.shape[0]
        out = {"rows": n}
        d1 = dcr[:, 0] if n else np.zeros(0)
        q = np.quantile(d1, [0.05, 0.5, 0.95]) if n else [float("nan")] * 3
        out.update(dcr_mean=float(d1.mean()) if n else float("nan"), dcr_p5=float(q[0]), dcr_p50=float(q[1]),
                   dcr_p95=float(q[2]))
        copies = int((ham[:, 0] == 0).sum()) if n else 0
        out.update(exact_copies=copies, exact_copy_share=copies / n if n else float("nan"))
        if self.k >= 2:
            d2 = dcr[:, 1]
            ratio = np.divide(d1, d2, out=np.ones_like(d1), where=d2 > 0)
            out["nndr_median"] = float(np.median(ratio)) if n else float("nan")
        return out


def check_k(k, m, exclude_same_index=False):
    """k as a Python int in [1, min(16, m)] (m - 1 with exclude_same_index).  Any integer type is accepted (numpy integers
    included); bools and floats are not."""
    if isinstance(k, bool):
        raise TypeError(f"k must be an integer, got {k!r}")
    try:
        k = operator.index(k)
    except TypeError:
        raise TypeError(f"k must be an integer, got {k!r}") from None
    cand = m - 1 if exclude_same_index else m
    hi = min(MAX_K, cand)
    if not 1 <= k <= hi:
        raise ValueError(f"k={k} must lie in [1, {hi}] (at most {MAX_K}, at most the {cand} candidate reference rows"
                         f"{' left after excluding the same index' if exclude_same_index else ''})")
    return k


def _kind(x):
    """(kind, rows, n_cols) of an accepted row set, without touching a device."""
    from .sparsify import PackedMatrix
    from .training import DeviceCSR
    if isinstance(x, PackedMatrix):
        return "bits", int(x.bits.shape[0]), int(x.n_cols)
    if isinstance(x, DeviceCSR):
        return "device_csr", int(x.shape[0]), int(x.shape[1])
    if isinstance(x, torch.Tensor):
        if x.layout == torch.sparse_csr:
            return "torch_csr", int(x.shape[0]), int(x.shape[1])
        if x.layout != torch.strided:
            raise TypeError(f"torch sparse input must be in CSR layout, got {x.layout} (call .to_sparse_csr())")
        if x.dim() != 2:
            raise ValueError(f"dense rows must be 2-D [rows, items], got shape {tuple(x.shape)}")
        return "dense", int(x.shape[0]), int(x.shape[1])
    try:
        import scipy.sparse as sp
        if sp.issparse(x):
            if x.ndim != 2:
                raise ValueError("sparse rows must be 2-D")
            return "scipy", int(x.shape[0]), int(x.shape[1])
    except ImportError:
        pass
    if isinstance(x, np.ndarray):
        if x.ndim != 2:
            raise ValueError(f"dense rows must be 2-D [rows, items], got shape {x.shape}")
        return "dense", int(x.shape[0]), int(x.shape[1])
    raise TypeError(f"unsupported row set {type(x).__name__}: pass a PackedMatrix, scipy / torch CSR, DeviceCSR or a dense "
                    "0/1 array")


def _device_of(x):
    from .sparsify import PackedMatrix
    from .training import DeviceCSR
    if isinstance(x, PackedMatrix):
        return x.bits.device
    if isinstance(x, DeviceCSR):
        return x.device
    if isinstance(x, torch.Tensor):
        return x.device
    return None


def _csr_device(indptr, indices, values, rows, dev):
    """CSR arrays (any integer / value dtypes; values None = every stored entry is an interaction) as the prep kernels take
    them: int64 indptr and indices, float32 values or None, contiguous on `dev`."""
    indptr = torch.as_tensor(indptr).to(device=dev, dtype=torch.int64).contiguous()
    indices = torch.as_tensor(indices).to(device=dev, dtype=torch.int64).contiguous()
    if values is not None:
        values = torch.as_tensor(values).to(dev)
        if values.dtype != torch.float32:
            values = (values != 0).to(torch.float32)   # exact: a tiny nonzero would round to 0.0 in a float32 cast
        values = values.contiguous()
    if indptr.dim() != 1 or indptr.numel() != rows + 1:
        raise ValueError(f"CSR indptr must have rows + 1 = {rows + 1} entries, got shape {tuple(indptr.shape)}")
    if values is not None and values.numel() != indices.numel():
        raise ValueError("CSR values and indices must have the same length")
    return indptr, indices, values


def _csr_arrays(x, kind, rows, dev):
    """The CSR arrays of a sparse or dense row set (every kind but "bits")."""
    if kind == "device_csr":
        return _csr_device(x.indptr, x.indices, x.values, rows, dev)
    if kind == "torch_csr":
        return _csr_device(x.crow_indices(), x.col_indices(), x.values(), rows, dev)
    if kind == "scipy":
        x = x.tocsr()
        return _csr_device(torch.from_numpy(x.indptr.astype(np.int64)), torch.from_numpy(x.indices.astype(np.int64)),
                           torch.from_numpy(np.asarray(x.data != 0, dtype=np.float32)), rows, dev)
    t = torch.as_tensor(np.ascontiguousarray(x)) if isinstance(x, np.ndarray) else x
    csr = (t.to(dev) != 0).to(torch.float32).to_sparse_csr()   # dense rows: nonzero = 1
    return _csr_device(csr.crow_indices(), csr.col_indices(), None, rows, dev)


def _raise_csr_status(status, nnz, n_cols):
    """ValueError for the sdrm_privacy_status bits a CSR prep kernel set (reading them synchronises with the stream)."""
    st = int(status.item())
    if st & _BAD_INDPTR:
        raise ValueError(f"CSR indptr must be non-decreasing within [0, {nnz}] (the number of stored entries)")
    if st & _BAD_INDEX:
        raise ValueError(f"CSR indices has entries outside [0, {n_cols})")


def _csr_image(indptr, indices, values, rows, n_cols, dev):
    """Operand image from CSR arrays (any integer / value dtypes; values None = every stored entry is an interaction)."""
    lib = _lib.load()
    indptr, indices, values = _csr_device(indptr, indices, values, rows, dev)
    pitch = int(lib.sdrm_privacy_image_pitch(n_cols))
    img = torch.empty((rows, pitch), dtype=torch.uint8, device=dev)
    ones = torch.empty(rows, dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    nnz = indices.numel()
    _lib.check(lib.sdrm_privacy_image_csr(_lib.ptr(indptr), _lib.ptr(indices) if nnz else None,
                                          _lib.ptr(values) if values is not None and nnz else None, nnz, rows, n_cols,
                                          _lib.ptr(img), pitch, _lib.ptr(ones), _lib.ptr(status), _lib.stream_ptr()),
               "sdrm_privacy_image_csr")
    if rows:
        _raise_csr_status(status, nnz, n_cols)
    return img, ones


def _image(x, kind, rows, n_cols, dev):
    """(uint8 0/1 image [rows, pitch], int32 ones [rows]) of a row set on `dev`."""
    lib = _lib.load()
    if kind == "bits":
        bits = x.bits.to(dev)
        if rows > 1 and bits.stride(1) != 1:
            bits = bits.contiguous()
        pitch = int(lib.sdrm_privacy_image_pitch(n_cols))
        img = torch.empty((rows, pitch), dtype=torch.uint8, device=dev)
        ones = torch.empty(rows, dtype=torch.int32, device=dev)
        _lib.check(lib.sdrm_privacy_image_bits(_lib.ptr(bits), bits.stride(0) if rows else bits.shape[1], rows, n_cols,
                                               _lib.ptr(img), pitch, _lib.ptr(ones), _lib.stream_ptr()),
                   "sdrm_privacy_image_bits")
        return img, ones
    return _csr_image(*_csr_arrays(x, kind, rows, dev), rows, n_cols, dev)


def _search(q_img, q_ones, r_img, r_ones, n_items, k, exclude_same_index=False, q_index_offset=0, splits=0):
    """K8 on prepared images (splits: reference ranges per query tile, 0 = automatic; the result does not depend on it)."""
    lib = _lib.load()
    n, m = q_img.shape[0], r_img.shape[0]
    dev = q_img.device
    idx = torch.empty((n, k), dtype=torch.int64, device=dev)
    inter = torch.empty((n, k), dtype=torch.int32, device=dev)
    union = torch.empty((n, k), dtype=torch.int32, device=dev)
    if n == 0:
        return idx, inter, union
    with torch.cuda.device(dev):
        ws_bytes = int(lib.sdrm_privacy_workspace_bytes(n, m, k, splits))
        if ws_bytes == 0:
            _lib.check(-1, "sdrm_privacy_workspace_bytes")
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        _lib.check(lib.sdrm_privacy_nearest(_lib.ptr(q_img), _lib.ptr(q_ones), n, _lib.ptr(r_img), _lib.ptr(r_ones), m, n_items,
                                            q_img.shape[1], k, 1 if exclude_same_index else 0, q_index_offset, splits,
                                            _lib.ptr(idx), _lib.ptr(inter), _lib.ptr(union), _lib.ptr(ws), ws_bytes,
                                            _lib.stream_ptr()),
                   "sdrm_privacy_nearest")
    return idx, inter, union


def nearest_rows(query, reference, k=1, exclude_same_index=False, group=None):
    """For every row of `query`, the k rows of `reference` with the highest Jaccard similarity J = |q & r| / |q | r| (J = 1 for
    two empty rows), best first, ties to the lower reference index; compared exactly in integers.  Returns NearestRows (device
    tensors).

    exclude_same_index=True: query row i never takes reference row i (audit a set against itself: the real-vs-real baseline).
    group: a torch.distributed process group; rank r searches its distributed.shard_bounds block of the query rows against all
    reference rows and the results are all-gathered, so every rank returns all rows.

    Raises ValueError for row sets with different numbers of columns, more than 2^20 columns, k outside [1, min(16, m)]
    (m - 1 with exclude_same_index), or malformed sparse input (indptr, indices out of range); TypeError for other input types.
    Sparse input is checked on the device, so the call synchronises with the current stream."""
    qk, n, nq = _kind(query)
    rk, m, nr = _kind(reference)
    if nq != nr:
        raise ValueError(f"query and reference must have the same number of columns, got {nq} and {nr}")
    if not 1 <= nq <= MAX_ITEMS:
        raise ValueError(f"rows must have between 1 and {MAX_ITEMS} columns, got {nq}")
    k = check_k(k, m, exclude_same_index)
    devs = {d for d in (_device_of(query), _device_of(reference)) if d is not None and d.type == "cuda"}
    if len(devs) > 1:
        raise ValueError(f"query and reference are on different devices: {sorted(map(str, devs))}")
    if not torch.cuda.is_available():
        raise _lib.SdrmError("nearest_rows needs a CUDA device (no CPU fallback)")
    dev = devs.pop() if devs else torch.device("cuda", torch.cuda.current_device())
    with torch.cuda.device(dev):
        q_img, q_ones = _image(query, qk, n, nq, dev)
        r_img, r_ones = _image(reference, rk, m, nr, dev)
        if group is None:
            return NearestRows(*_search(q_img, q_ones, r_img, r_ones, nq, k, exclude_same_index), q_ones)
        import torch.distributed as dist

        from .distributed import shard_bounds
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        lo, hi = shard_bounds(n, rank, world)
        part = _search(q_img[lo:hi], q_ones[lo:hi], r_img, r_ones, nq, k, exclude_same_index, lo)
        cap = shard_bounds(n, 0, world)[1]

        def gather(t):
            padded = t.new_zeros((cap,) + tuple(t.shape[1:]))
            padded[: t.shape[0]] = t
            parts = [torch.empty_like(padded) for _ in range(world)]
            dist.all_gather(parts, padded, group=group)
            return torch.cat([p[: shard_bounds(n, r, world)[1] - shard_bounds(n, r, world)[0]] for r, p in enumerate(parts)])

        return NearestRows(*(gather(t) for t in part), q_ones)
