"""Equal-sparsity thresholding of synthetic score matrices on the GPU (SURVEY.md §8f-1).

Reference (main.py:177-185, 259-262; hyperparameter_search.py:162-166):

    threshold = np.quantile(S.flatten(), SPARSITY)
    S_equal_sparsity = pd.DataFrame((S >= threshold).astype(int))
    lower = (S <= np.quantile(S.flatten(), 1 - SPARSITY))            # NeuMF negatives

The reference does this on the host after `.cpu().numpy()` (a full partition of n*I floats; 80 GB at the scale-up
shape).  Here the matrix stays in HBM: an exact radix select (three histogram passes of kernel K4, `sdrm_key_histogram`)
finds the two order statistics NumPy interpolates between, the interpolation itself is done with NumPy's own rule so the
threshold is bit-identical to `np.quantile`, and `sdrm_threshold_pack` emits one bit per score.  When the rows are
sharded over several GPUs the 2048-bin histograms are summed with one all-reduce per pass (the only exchange step), so
every rank derives the SAME global threshold the single-process reference would.

bfloat16 score matrices (sample_ddpm(..., out_dtype=torch.bfloat16)) take the same path at 2 bytes per score.  Their scores
are ranked and compared as float32 values, so the threshold is np.quantile(S.astype(np.float32).flatten(), q) bit for bit and
the bits are S >= thr.  The float32 key of a bfloat16 score has its low 16 bits fixed by the sign, so two histogram passes
(11 + 5 bits) pin it instead of three.

No CPU fallback: a CPU tensor raises.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib

_DIGITS = ((11, 21), (11, 10), (10, 0))   # (bits, shift): 11 + 11 + 10 = 32
_DIGITS_BF16 = ((11, 21), (5, 16))         # bfloat16 scores: the low 16 key bits follow from the sign bit


# --------------------------------------------------------------------------------------------------
# NumPy's quantile rule (method='linear'), restated so that it can be applied to order statistics found elsewhere
# --------------------------------------------------------------------------------------------------
def quantile_plan(n_total, q, dtype=np.float32):
    """Which order statistics np.quantile(a.flatten(), q) reads for an array of n_total values of `dtype`, and the weight.

    Returns (previous_index, next_index, gamma) with gamma a NumPy scalar of the dtype NumPy computes it in.
    Follows numpy/lib/_function_base_impl.py (quantile, _quantile, _get_indexes, _get_gamma): since NumPy 2.0 a Python
    float `q` is first cast to the array's float dtype, so for float32 scores the virtual index (n-1)*q is a float32.
    """
    if n_total < 1:
        raise ValueError("quantile of an empty matrix")
    if isinstance(q, (int, float)) and np.dtype(dtype).kind == "f" and np.lib.NumpyVersion(np.__version__) >= "2.0.0":
        qa = np.asanyarray(q, dtype=dtype)
    else:
        qa = np.asanyarray(q)
    if not (0.0 <= float(qa) <= 1.0):
        raise ValueError("Quantiles must be in the range [0, 1]")
    virtual = np.asanyarray((n_total - 1) * qa)
    prev = np.floor(virtual)
    nxt = prev + 1
    if virtual >= n_total - 1:
        prev_i = nxt_i = n_total - 1
    elif virtual < 0:
        prev_i = nxt_i = 0
    else:
        prev_i, nxt_i = int(prev), int(nxt)
    gamma = np.asanyarray(virtual - prev, dtype=virtual.dtype)
    return prev_i, nxt_i, gamma[()]


def lerp(a, b, t):
    """numpy.lib._function_base_impl._lerp on scalars: a + (b-a) t, or b - (b-a)(1-t) when t >= 0.5."""
    a, b, t = np.asanyarray(a), np.asanyarray(b), np.asanyarray(t)
    diff = np.subtract(b, a)
    out = np.asanyarray(np.add(a, diff * t))
    if t >= 0.5:
        out = np.asanyarray(np.subtract(b, diff * (1 - t)).astype(out.dtype))
    return out[()]


def key_to_float(key):
    """Inverse of the device's order-preserving key map (sparsify.cu: score_key)."""
    key = int(key) & 0xFFFFFFFF
    u = (key ^ 0x80000000) if (key & 0x80000000) else (~key & 0xFFFFFFFF)
    return np.array([u], dtype=np.uint32).view(np.float32)[0]


def float_to_key(x):
    u = int(np.array([x], dtype=np.float32).view(np.uint32)[0])
    return (~u & 0xFFFFFFFF) if (u & 0x80000000) else (u | 0x80000000)


def select_ranks(hist_fn, ranks, digits=_DIGITS):
    """Exact radix select.  hist_fn(prefix, prefix_bits, shift, bits) -> int64 array of global digit counts.
    Returns the float32 order statistic for every 0-based rank in `ranks` (histograms shared between ranks).
    digits=_DIGITS_BF16 for bfloat16 scores: the key bits below the last digit are 0 for a positive score, all ones else."""
    cache = {}
    out = []
    for r in ranks:
        prefix, pbits, rem = 0, 0, int(r)
        for bits, shift in digits:
            k = (prefix, pbits)
            if k not in cache:
                cache[k] = np.cumsum(np.asarray(hist_fn(prefix, pbits, shift, bits), dtype=np.int64)[: 1 << bits])
            cum = cache[k]
            if rem >= cum[-1]:
                raise ValueError("rank beyond the number of scores")
            b = int(np.searchsorted(cum, rem, side="right"))
            if b:
                rem -= int(cum[b - 1])
            prefix, pbits = (prefix << bits) | b, pbits + bits
        low = 32 - pbits
        if low:
            prefix = (prefix << low) | (0 if (prefix >> (pbits - 1)) & 1 else (1 << low) - 1)
        out.append(key_to_float(prefix))
    return out


# --------------------------------------------------------------------------------------------------
# device entry points
# --------------------------------------------------------------------------------------------------
def _check(scores):
    if not isinstance(scores, torch.Tensor) or scores.device.type != "cuda":
        raise _lib.SdrmError("sparsify: scores must be a CUDA tensor (no CPU fallback)")
    if scores.dtype not in (torch.float32, torch.bfloat16) or scores.dim() != 2 or scores.stride(1) != 1:
        raise ValueError("scores must be float32 or bfloat16 [rows, items] with unit column stride")


def _bf16(scores):
    return scores.dtype == torch.bfloat16


def _world(group):
    import torch.distributed as dist
    if group is None or not dist.is_available() or not dist.is_initialized():
        return None
    return dist


def device_histogram_fn(scores, group=None):
    """hist_fn for select_ranks backed by kernel K4; sums over `group` (pass dist.group.WORLD) when rows are sharded."""
    _check(scores)
    lib = _lib.load()
    dist = _world(group)
    rows, n_cols = scores.shape

    def hist_fn(prefix, prefix_bits, shift, bits):
        h = torch.zeros(2048, dtype=torch.int64, device=scores.device)
        entry = lib.sdrm_key_histogram_bf16 if _bf16(scores) else lib.sdrm_key_histogram
        _lib.check(entry(_lib.ptr(scores), rows, n_cols, scores.stride(0) if rows else n_cols, prefix, prefix_bits,
                         shift, bits, _lib.ptr(h), _lib.stream_ptr()), "sdrm_key_histogram")
        if dist is not None:
            dist.all_reduce(h, group=group)
        return h.cpu().numpy()
    return hist_fn


def global_count(scores, group=None):
    n = scores.shape[0] * scores.shape[1]
    dist = _world(group)
    if dist is not None:
        t = torch.tensor([n], dtype=torch.int64, device=scores.device)
        dist.all_reduce(t, group=group)
        n = int(t.item())
    return n


def quantile_host_walk(scores, q, group=None):
    """The first implementation: histograms copied to the host between the passes and walked with NumPy (also the fallback of
    the device walk).  NaN scores are not looked for here (the device walk counts them; quantile_device handles that)."""
    _check(scores)
    n_total = global_count(scores, group)
    prev_i, nxt_i, gamma = quantile_plan(n_total, q, np.float32)
    ranks = [prev_i] if nxt_i == prev_i else [prev_i, nxt_i]
    vals = select_ranks(device_histogram_fn(scores, group), ranks, _DIGITS_BF16 if _bf16(scores) else _DIGITS)
    return lerp(vals[0], vals[-1], gamma)


def quantile_device(scores, q, group=None):
    """np.quantile(S.flatten(), q) for a float32 CUDA matrix (row-sharded over `group` if given), bit-identical to NumPy
    (NaN as soon as one score is NaN).  For a bfloat16 matrix: np.quantile(S.astype(np.float32).flatten(), q)."""
    _check(scores)
    state, g32 = _select_enqueue(scores, q, group)
    thr, fallback, nans = _read_state(state, g32)
    if nans:
        return np.float32(np.nan)
    return quantile_host_walk(scores, q, group) if fallback else thr


class PackedMatrix:
    """Bit-packed binary matrix on the device: bit j of word w of a row is column 32 w + j (little-endian bit order)."""

    def __init__(self, bits, n_cols, threshold, ones):
        self.bits, self.n_cols, self.threshold, self.ones = bits, n_cols, threshold, ones

    @property
    def shape(self):
        return (self.bits.shape[0], self.n_cols)

    def numpy(self, dtype=np.int64):
        """Dense 0/1 host array, like the reference's `(S >= threshold).astype(int)`; the D2H copy moves 1 bit per entry."""
        words = self.bits.cpu().numpy().view(np.uint32)
        dense = np.unpackbits(words.view(np.uint8), axis=1, bitorder="little")[:, : self.n_cols]
        return dense.astype(dtype)


def threshold_pack(scores, threshold, lower=False):
    """(S >= threshold) — or (S <= threshold) with lower=True — as a PackedMatrix (float32 or bfloat16 scores, compared as
    float32 values)."""
    _check(scores)
    lib = _lib.load()
    rows, n_cols = scores.shape
    wpr = (n_cols + 31) // 32
    bits = torch.empty((rows, wpr), dtype=torch.int32, device=scores.device)
    count = torch.zeros(1, dtype=torch.int64, device=scores.device)
    entry = lib.sdrm_threshold_pack_bf16 if _bf16(scores) else lib.sdrm_threshold_pack
    _lib.check(entry(_lib.ptr(scores), rows, n_cols, scores.stride(0) if rows else n_cols, float(threshold),
                                       1 if lower else 0, _lib.ptr(bits), wpr, _lib.ptr(count), _lib.stream_ptr()),
               "sdrm_threshold_pack")
    return PackedMatrix(bits, n_cols, threshold, count)


def _select_enqueue(scores, q, group):
    """Enqueue the device-side quantile selection (C ABI sdrm_select_*): three histogram passes (two for bfloat16 scores) with a
    one-block walk kernel between them (and one all-reduce of 2048 bins per pass when the rows are sharded); nothing is read
    back here."""
    lib = _lib.load()
    dist = _world(group)
    rows, n_cols = scores.shape
    n_total = global_count(scores, group)
    prev_i, nxt_i, gamma = quantile_plan(n_total, q, np.float32)
    dev = scores.device
    state = torch.zeros(lib.sdrm_select_state_bytes(), dtype=torch.uint8, device=dev)
    bf16 = _bf16(scores)
    n_digits = len(_DIGITS_BF16 if bf16 else _DIGITS)
    hist_entry, walk_entry = ((lib.sdrm_select_histogram_bf16, lib.sdrm_select_walk_bf16) if bf16
                              else (lib.sdrm_select_histogram, lib.sdrm_select_walk))
    hists = torch.zeros((n_digits, 2048), dtype=torch.int64, device=dev)
    st = _lib.stream_ptr()
    ld = scores.stride(0) if rows else n_cols
    _lib.check(lib.sdrm_select_begin(_lib.ptr(state), prev_i, nxt_i, st), "sdrm_select_begin")
    g32 = 1 if np.asarray(gamma).dtype == np.float32 else 0
    for d in range(n_digits):
        _lib.check(hist_entry(_lib.ptr(scores), rows, n_cols, ld, _lib.ptr(state), d, _lib.ptr(hists[d]), st),
                   "sdrm_select_histogram")
        if dist is not None:
            dist.all_reduce(hists[d], group=group)
            if d == 0:      # the NaN count of the other ranks (bytes 16..24 of the state)
                dist.all_reduce(state[16:24].view(torch.int64), group=group)
        _lib.check(walk_entry(_lib.ptr(hists[d]), _lib.ptr(state), d, float(gamma), g32, st), "sdrm_select_walk")
    return state, g32


def _read_state(state, g32):
    raw = state.cpu().numpy()          # the only synchronisation of the selection
    thr = raw[40:48].view(np.float64)[0]
    return (np.float32(thr) if g32 else np.float64(thr)), int(raw[28:32].view(np.uint32)[0]), int(raw[16:24].view(np.uint64)[0])


def _select_pack_device(scores, q, group, lower):
    """Quantile selection + bit packing enqueued back to back: ONE host read (the 56-byte state) at the end instead of a
    device->host histogram copy and a host walk per pass.  Returns None when the device walk flagged the rare case it does not
    handle (the two order statistics fall into different digit bins before the last digit): the caller takes the host walk."""
    lib = _lib.load()
    rows, n_cols = scores.shape
    state, g32 = _select_enqueue(scores, q, group)
    wpr = (n_cols + 31) // 32
    bits = torch.empty((rows, wpr), dtype=torch.int32, device=scores.device)
    count = torch.zeros(1, dtype=torch.int64, device=scores.device)
    entry = lib.sdrm_select_threshold_pack_bf16 if _bf16(scores) else lib.sdrm_select_threshold_pack
    _lib.check(entry(_lib.ptr(scores), rows, n_cols, scores.stride(0) if rows else n_cols, _lib.ptr(state),
                                              1 if lower else 0, _lib.ptr(bits), wpr, _lib.ptr(count), _lib.stream_ptr()),
               "sdrm_select_threshold_pack")
    thr, fallback, nans = _read_state(state, g32)
    if fallback and not nans:
        return None
    return PackedMatrix(bits, n_cols, thr, count)


def equal_sparsity_device(scores, sparsity, group=None, lower=False, host_walk=False):
    """The reference's equal-sparsity binarisation (main.py:177-185) without leaving the GPU.

    lower=False: S >= np.quantile(S.flatten(), sparsity);  lower=True: S <= np.quantile(S.flatten(), 1 - sparsity)
    (main.py:259-262).  With `group`, `scores` is this rank's row shard and the threshold is the GLOBAL quantile.
    A NaN score makes the threshold NaN (and every bit 0), like np.quantile.  host_walk=True forces the first implementation
    (histograms copied to the host between the passes), which is also the fallback of the device walk.

    bfloat16 scores (sample_ddpm(..., out_dtype=torch.bfloat16)): the reference's rule applied to the ROUNDED scores, i.e.
    thr = np.quantile(S.astype(np.float32).flatten(), q) and S >= thr.  Rounding to bfloat16 merges nearby scores, so the
    threshold often lands on a value many scores share, and every one of them is kept: the matrix can hold more ones than the
    binarisation of the float32 rows of the same seed (DESIGN.md section 3 gives the measured size of the effect).
    """
    _check(scores)
    q = (1 - sparsity) if lower else sparsity
    if not host_walk and scores.shape[0] > 0:
        pm = _select_pack_device(scores, q, group, lower)
        if pm is not None:
            return pm
    thr = quantile_host_walk(scores, q, group) if host_walk else quantile_device(scores, q, group)
    return threshold_pack(scores, thr, lower=lower)
