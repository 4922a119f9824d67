"""The kernels on one benchmark shard's data path at the shard's real size: 125 000 users x 20 000 items (bench.py cfg 5) is
2.5 x 10^9 scores, 10 GB of fp32 logits.  Rows past 53 687 sit beyond 2^32 bytes of fp32 and rows past 107 374 beyond 2^31
elements, so everything from there on depends on 64-bit offset arithmetic: K1's logits stores (contiguous and ld > I), K6's
stores, K4's sweeps and NaN count, K10, K3 and K7.  A 32-bit slip in any of them would corrupt only the last rows of every shard.

Each test compares a kernel with a plain reference of the same operation on 12-row slices that straddle those offsets, and checks
size-independent properties over the whole matrix with torch on the device in row chunks.  The big matrices are sampled once
(module fixture `shard`, freed at module teardown); peak device memory stays near 35 GB."""
import numpy as np
import pytest
import torch

from helpers import max_scaled_err, random_modules, rel_fro, state_dicts
from test_recommend_topk import reference_topk
from test_sampler_gpu import TOL, TOL_MAX, _engine

pytestmark = pytest.mark.gpu

# bench.py cfg 5, one of its 8 GPUs: rank 7's rows start at 7 x 125 000
N, I, H, L, T, NH, ND = 125_000, 20_000, 1000, 950, 178, 4, 1.0
ROW_OFFSET = 875_000
SEED = 0x5EED0C0FFEE5
# 12-row slices: first row; the 4 GiB fp32 byte offset (row 53 687); element 2^31 (row 107 374); a late wave; the ragged last
# tile (125 000 = 976 x 128 + 72: an odd 977th tile, so the last CTA pair holds a ghost tile)
STARTS = (0, 53_680, 107_368, 118_000, N - 12)
ROWS = 12
CHUNK = 4096       # rows per chunk of the torch references (a [4096, 20 000] int64 temporary is 655 MB)
NAN_AT = (120_000, I - 1)


def _chunks(n, rows=CHUNK):
    for a in range(0, n, rows):
        yield a, min(a + rows, n)


def _same_bits(a, b):
    """Bit-for-bit equality of two float tensors of one dtype (NaN equals NaN of the same payload, -0.0 differs from +0.0)."""
    as_int = torch.int32 if a.dtype == torch.float32 else torch.int16
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.view(as_int), b.view(as_int))


def _all_chunks(pred, n):
    return all(bool(pred(a, b)) for a, b in _chunks(n))


def _same_rows(x, y):
    """_same_bits in row chunks: torch.equal on a whole 10 GB matrix would allocate a 2.5 GB temporary."""
    return x.shape == y.shape and _all_chunks(lambda a, b: _same_bits(x[a:b], y[a:b]), x.shape[0])


def _noise(seed, row0, rows, L_, T_):
    from oracle import philox_ref
    return tuple(torch.from_numpy(t) for t in philox_ref.sampler_noise(seed, row0, rows, L_, T_))


@pytest.fixture(scope="module")
def model():
    diff, vae = random_modules(I, H, L, T, NH, seed=57, device="cuda")
    return diff, vae, state_dicts(diff, vae)


@pytest.fixture(scope="module")
def shard(model):
    """The shard's rows three times, from one engine: fp32 contiguous, fp32 into the [:, :I] view of a [N, I + 8] buffer filled with
    NaN (ld_logits = I + 8), and bfloat16."""
    diff, vae, _ = model
    eng = _engine(diff, vae, T, ND)
    lib = eng.lib
    m = {"eng": eng}
    m["fp32"] = eng.sample(N, row_offset=ROW_OFFSET, seed=SEED, check=True)
    m["flow"] = (lib.sdrm_last_cluster_size(eng.handle), lib.sdrm_last_resident_mode(eng.handle),
                 lib.sdrm_last_split_size(eng.handle))
    m["padded"] = torch.full((N, I + 8), float("nan"), device="cuda")
    eng.sample(N, row_offset=ROW_OFFSET, seed=SEED, out=m["padded"][:, :I], check=True)
    m["bf16"] = eng.sample(N, row_offset=ROW_OFFSET, seed=SEED, out=torch.empty((N, I), dtype=torch.bfloat16, device="cuda"),
                           check=True)
    yield m
    del eng
    m.clear()
    torch.cuda.empty_cache()
    print(f"\nshard-scale tests: peak device memory {torch.cuda.max_memory_allocated() / 2 ** 30:.1f} GiB")


def _matrix(shard, kind):
    return shard["padded"][:, :I] if kind == "strided" else shard[kind]


# ------------------------------------------------------------------------------------------------------------------------------
# D. K6 past 2^31 elements (runs first: its two 8.9 GB matrices are gone before the shard's matrices are sampled)
# ------------------------------------------------------------------------------------------------------------------------------
def test_k6_rows_past_2_31_elements():
    """cfg-3 widths (every width <= 64: the small-chain kernel) at 260 000 rows = 2.23 x 10^9 logits."""
    from oracle import sdrm_oracle as orc
    from sdrm_b200 import _lib
    n, I3, H3, L3, T3, nh3, nd3 = 260_000, 8582, 40, 40, 93, 5, 1.0
    diff, vae = random_modules(I3, H3, L3, T3, nh3, seed=58, device="cuda")
    dsd, vsd = state_dicts(diff, vae)
    eng = _engine(diff, vae, T3, nd3)
    seed, off = 0x6B6B6B6B, 3_000_000
    auto = eng.sample(n, row_offset=off, seed=seed, check=True)
    other = torch.full_like(auto, float("nan"))
    try:
        eng.set_option(_lib.OPT_ENGINE, 2)
        eng.sample(n, row_offset=off, seed=seed, out=other, check=True)
        assert _same_rows(auto, other)                    # the automatic choice is K6
        for start in (0, 125_110, 250_226, n - ROWS):     # fp32 4 GiB at row 125 115; element 2^31 at row 250 231
            xT, z, keep = _noise(seed, off + start, ROWS, L3, T3)
            ref = orc.sample_full(dsd, vsd, T3, nd3, xT, z, keep)
            got = auto[start:start + ROWS].cpu()
            fro, el = rel_fro(got, ref), max_scaled_err(got, ref)
            print(f"K6 cfg-3 n={n} rows {start}..{start + ROWS - 1}: rel-Frobenius {fro:.2e}, worst element {el:.2e}")
            assert fro < TOL and el < TOL_MAX, (start, fro, el)
        eng.set_option(_lib.OPT_ENGINE, 1)
        other.fill_(float("nan"))
        eng.sample(n, row_offset=off, seed=seed, out=other, check=True)
        assert eng.lib.sdrm_last_cluster_size(eng.handle) >= 1
        num = den = 0.0
        for a, b in _chunks(n, 16384):
            num += float((other[a:b].double() - auto[a:b].double()).square().sum())
            den += float(auto[a:b].double().square().sum())
        rel = (num / den) ** 0.5
        print(f"K1 vs K6 cfg-3 n={n}: rel-Frobenius {rel:.2e}")
        assert rel < 3e-4
    finally:
        eng.set_option(_lib.OPT_ENGINE, 0)
        del auto, other, eng
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------------------------------------
# B. Multi-resolution rows through the public call (rows sorted by chain length, written back through row ids)
# ------------------------------------------------------------------------------------------------------------------------------
def test_multires_rows_through_the_public_call(model):
    from oracle import sdrm_oracle as orc
    from sdrm_b200.train_SDRM import sample_ddpm
    diff, vae, (dsd, vsd) = model
    seed = 0xB0B0B0B0
    np.random.seed(59)
    t_np = np.random.randint(1, T, size=N)        # the draw the call makes itself ...
    np.random.seed(59)                             # ... replayed
    out = sample_ddpm(N, diff, vae, L, ND, timesteps="random", n_timesteps=T, seed=seed, row_offset=ROW_OFFSET)
    try:
        assert out.shape == (N, I) and _all_chunks(lambda a, b: torch.isfinite(out[a:b]).all(), N)
        for start in STARTS:
            xT, z, keep = _noise(seed, ROW_OFFSET + start, ROWS, L, T)
            ref = orc.sample_random(dsd, vsd, T, ND, xT, z, keep, t_np[start:start + ROWS])
            got = out[start:start + ROWS].cpu()
            fro, el = rel_fro(got, ref), max_scaled_err(got, ref)
            print(f"K1 random mode rows {start}..{start + ROWS - 1}: rel-Frobenius {fro:.2e}, worst element {el:.2e}")
            assert fro < TOL and el < TOL_MAX, (start, fro, el)
    finally:
        del out
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------------------------------------
# A. K1 fp32 rows at the benchmark shape
# ------------------------------------------------------------------------------------------------------------------------------
def test_k1_rows_match_oracle_across_the_int32_offsets(model, shard):
    from oracle import sdrm_oracle as orc
    _, _, (dsd, vsd) = model
    S = shard["fp32"]
    cluster, resident, split = shard["flow"]
    print(f"K1 cfg-5 n={N}: cluster {cluster}, resident {resident}, split {split}")
    assert (cluster, resident, split) == (2, 0, 0)     # CTA pairs, streaming tiles, no column split: the dead-buffer discard runs
    assert _all_chunks(lambda a, b: torch.isfinite(S[a:b]).all(), N)
    for start in STARTS:
        xT, z, keep = _noise(SEED, ROW_OFFSET + start, ROWS, L, T)
        got = S[start:start + ROWS].cpu()
        ref = orc.sample_full(dsd, vsd, T, ND, xT, z, keep)
        fro, el = rel_fro(got, ref), max_scaled_err(got, ref)
        line = f"K1 cfg-5 rows {start}..{start + ROWS - 1}: rel-Frobenius {fro:.2e}, worst element {el:.2e}"
        if start == 107_368:
            emu = rel_fro(got, orc.sample_bf16_emulated(dsd, vsd, T, ND, xT, z, keep))
            line += f", vs bf16 emulation {emu:.2e}"
            assert emu < 2e-4, emu                      # same rounding points: separates kernel bugs from bf16 effects
        print(line)
        assert fro < TOL and el < TOL_MAX, (start, fro, el)


def test_k1_launches_are_deterministic_and_flow_invariant(shard):
    """A second launch, a 1000-row shard around element 2^31, single CTAs and pairs without the dead-buffer discard (which runs
    over ~6.6 waves of row tiles in the default launch) all give the same bits."""
    from sdrm_b200 import _lib
    eng, S = shard["eng"], shard["fp32"]
    lib = eng.lib
    scratch = torch.full_like(S, float("nan"))
    try:
        eng.sample(N, row_offset=ROW_OFFSET, seed=SEED, out=scratch, check=True)
        assert _same_rows(scratch, S)
        part = eng.sample(1000, row_offset=ROW_OFFSET + 107_000, seed=SEED, check=True)
        assert _same_bits(part, S[107_000:108_000])     # rows depend only on (seed, global row id)
        del part
        for option, value, cluster in ((_lib.OPT_CLUSTER, 1, 1), (_lib.OPT_NO_DISCARD, 1, 2)):
            eng.set_option(option, value)
            scratch.fill_(float("nan"))
            eng.sample(N, row_offset=ROW_OFFSET, seed=SEED, out=scratch, check=True)
            eng.set_option(option, 0)
            assert lib.sdrm_last_cluster_size(eng.handle) == cluster
            assert _same_rows(scratch, S), (option, value)
    finally:
        eng.set_option(_lib.OPT_CLUSTER, 0)
        eng.set_option(_lib.OPT_NO_DISCARD, 0)
        del scratch
        torch.cuda.empty_cache()


def test_k1_strided_output_past_2_31(shard):
    """ld_logits = I + 8: the view holds the contiguous launch's bits and the 8 pad columns of every row stay NaN."""
    S, P = shard["fp32"], shard["padded"]
    assert _same_rows(P[:, :I], S)
    assert _all_chunks(lambda a, b: torch.isnan(P[a:b, I:]).all(), N)


# ------------------------------------------------------------------------------------------------------------------------------
# C. bfloat16 rows
# ------------------------------------------------------------------------------------------------------------------------------
def test_bf16_rows_are_the_rounded_fp32_rows(shard):
    S, B = shard["fp32"], shard["bf16"]
    assert _all_chunks(lambda a, b: _same_bits(B[a:b], S[a:b].to(torch.bfloat16)), N)


# ------------------------------------------------------------------------------------------------------------------------------
# E. K4 equal-sparsity thresholding on the 2.5 x 10^9-score matrices
# ------------------------------------------------------------------------------------------------------------------------------
def _count(S, pred):
    return sum(int(pred(S[a:b].float()).sum(dtype=torch.int64)) for a, b in _chunks(S.shape[0]))


def _reference_bits(S, thr, lower):
    """S >= thr (S <= thr) packed on the device: bit j of word w of a row is column 32 w + j (sparsify_oracle.pack_bits)."""
    rows, cols = S.shape
    assert cols % 32 == 0
    weights = torch.ones(32, dtype=torch.int64, device=S.device) << torch.arange(32, device=S.device)
    for a, b in _chunks(rows):
        x = S[a:b].float()
        hit = (x <= thr) if lower else (x >= thr)
        words = (hit.view(b - a, cols // 32, 32).to(torch.int64) * weights).sum(-1)
        yield a, b, torch.where(words >= 2 ** 31, words - 2 ** 32, words).to(torch.int32), int(hit.sum(dtype=torch.int64))


def _same_scalar(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype and a.tobytes() == b.tobytes()


@pytest.mark.parametrize("kind", ["fp32", "strided", "bf16"])
def test_k4_threshold_and_bits(shard, kind):
    """The two order statistics np.quantile interpolates are proven by counting (#(S < v) <= r < #(S <= v)), the threshold is
    NumPy's interpolation of them, and the bits are S >= thr (S <= thr).  `strided` is the fp32 rows in the [:, :I] view of a
    wider buffer: K4's non-contiguous sweep (row / column split of the flat index) past 2^31."""
    from sdrm_b200.sparsify import (_DIGITS, _DIGITS_BF16, device_histogram_fn, equal_sparsity_device, lerp, quantile_device,
                                    quantile_plan, select_ranks)
    S = _matrix(shard, kind)
    n = S.numel()
    digits = _DIGITS_BF16 if kind == "bf16" else _DIGITS
    for sparsity, lower in ((0.9424673, False), (0.99, False), (0.9424673, True)):
        q = (1 - sparsity) if lower else sparsity
        prev, nxt, gamma = quantile_plan(n, q)
        vals = select_ranks(device_histogram_fn(S), [prev, nxt], digits)
        for r, v in zip((prev, nxt), vals):
            assert _count(S, lambda x: x < float(v)) <= r < _count(S, lambda x: x <= float(v)), (kind, q, r, v)
        want = lerp(vals[0], vals[1], gamma)
        pm = equal_sparsity_device(S, sparsity, lower=lower)
        walked = equal_sparsity_device(S, sparsity, lower=lower, host_walk=True)
        print(f"K4 {kind} q={q:.7f}: ranks {prev}, {nxt}, threshold {want!r}, ones {int(pm.ones.item())}")
        assert _same_scalar(pm.threshold, want) and _same_scalar(walked.threshold, want), (pm.threshold, walked.threshold, want)
        assert _same_scalar(quantile_device(S, q), want)
        ones = 0
        for a, b, ref, hits in _reference_bits(S, float(want), lower):
            assert torch.equal(pm.bits[a:b], ref), (kind, q, a)
            assert torch.equal(walked.bits[a:b], ref), (kind, q, a)
            ones += hits
        assert int(pm.ones.item()) == ones == int(walked.ones.item())


@pytest.mark.parametrize("kind", ["fp32", "bf16"])
def test_k4_nan_past_2_31(shard, kind):
    """One NaN at element 2.4 x 10^9: np.quantile's answer is NaN, so the threshold is NaN and no bit is set."""
    from sdrm_b200.sparsify import equal_sparsity_device, quantile_device
    S = shard[kind]
    keep = S[NAN_AT].clone()
    S[NAN_AT] = float("nan")
    try:
        pm = equal_sparsity_device(S, 0.99)
        assert np.isnan(pm.threshold)
        assert int(pm.ones.item()) == 0 and int(torch.count_nonzero(pm.bits)) == 0
        assert np.isnan(quantile_device(S, 0.99))
    finally:
        S[NAN_AT] = keep
    assert not torch.isnan(S[NAN_AT[0]]).any()


# ------------------------------------------------------------------------------------------------------------------------------
# F. K10 on the real bits of the shard
# ------------------------------------------------------------------------------------------------------------------------------
def test_k10_csr_of_the_shard_bits(shard):
    from sdrm_b200.sparsify import equal_sparsity_device
    S = shard["fp32"]
    pm = equal_sparsity_device(S, 0.99)
    csr = pm.to_sparse()
    thr = float(pm.threshold)
    counts = torch.cat([(S[a:b] >= thr).sum(dim=1) for a, b in _chunks(N)])
    want = torch.cat([counts.new_zeros(1), counts.cumsum(0)])
    print(f"K10 fp32 sparsity 0.99: nnz {csr.nnz}, row counts {int(counts.min())}..{int(counts.max())}")
    assert csr.indptr.dtype == torch.int64 and torch.equal(csr.indptr, want)
    assert csr.nnz == int(pm.ones.item())
    for start in STARTS:
        lo, hi = int(csr.indptr[start]), int(csr.indptr[start + ROWS])
        ref = (S[start:start + ROWS] >= thr).nonzero()[:, 1].to(torch.int32)
        assert torch.equal(csr.indices[lo:hi], ref), start


# ------------------------------------------------------------------------------------------------------------------------------
# G. K3 top-k
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [10, 50, 100])
def test_k3_topk_of_the_shard(shard, k):
    """k = 100 takes two passes over a 10 GB working copy.  Slices: the stable descending argsort; whole matrix: sorted values,
    indices that point at them, and the scores above the k-th are exactly the listed ones before it."""
    from sdrm_b200.metrics import topk_device
    S = shard["fp32"]
    idx, vals = topk_device(S, k, return_values=True)
    for start in STARTS:
        x = S[start:start + ROWS].cpu().numpy()
        assert np.array_equal(idx[start:start + ROWS].cpu().numpy(), np.argsort(-x, axis=1, kind="stable")[:, :k]), start
    assert bool((vals[:, :-1] >= vals[:, 1:]).all())
    assert _same_bits(torch.gather(S, 1, idx.long()), vals)
    kth = vals[:, -1:]
    # (k - 1 of them unless the k-th ties with the (k-1)-th)
    assert _all_chunks(lambda a, b: torch.equal((S[a:b] > kth[a:b]).sum(dim=1), (vals[a:b] > kth[a:b]).sum(dim=1)), N)
    assert _all_chunks(lambda a, b: ((S[a:b] >= kth[a:b]).sum(dim=1) >= k).all(), N)


# ------------------------------------------------------------------------------------------------------------------------------
# H. K7 top-k recommendation, excluding the items of the shard's own binarised rows (~200 per row)
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["fp32", "bf16"])
def test_k7_recommend_with_exclusion(shard, kind):
    from sdrm_b200.recommend import recommend_topk
    from sdrm_b200.sparsify import equal_sparsity_device
    pm = equal_sparsity_device(shard["fp32"], 0.99)
    csr = pm.to_sparse()
    X = shard[kind]
    for k in (10, 256):
        vals, idx = recommend_topk(X, csr.indptr, csr.indices, k)
        for start in STARTS:
            ip = csr.indptr[start:start + ROWS + 1]
            ix = csr.indices[int(ip[0]):int(ip[-1])]
            rv, ri = reference_topk(X[start:start + ROWS], ip - ip[0], ix, k)
            assert torch.equal(idx[start:start + ROWS].cpu(), ri), (kind, k, start)
            assert _same_bits(vals[start:start + ROWS].cpu(), rv), (kind, k, start)
        word = pm.bits.gather(1, idx >> 5)
        assert not bool(((word >> (idx & 31)) & 1).any())            # no item of a row's history comes back
        v = vals.float()
        assert bool((v[:, :-1] >= v[:, 1:]).all())
