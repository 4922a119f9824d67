"""Top-K recommendation with seen-item exclusion (recommend.recommend_topk, K7 sdrm_recommend_topk[_bf16], sample_ddpm(topk=...)).

Reference: mask the history with -inf and take a stable descending sort (torch.topk's order with ties to the lower index); a second
stable sort on the exclusion flag keeps masked items behind genuine -inf logits.  NaN ranks as -inf and -0.0 as +0.0, as documented.
Results must match it exactly: same indices, same values.  The argument checks at the top run without a GPU.
"""
import numpy as np
import pytest
import torch

from sdrm_b200 import _lib
from sdrm_b200.recommend import MAX_K, recommend_topk

NEG_INF = float("-inf")


def reference_topk(logits, indptr, indices, k):
    """(values in the logits' dtype, int64 indices), on the CPU."""
    x = logits.detach().cpu().float()
    x = torch.where(torch.isnan(x), torch.full_like(x, NEG_INF), x) + 0.0
    users, n_items = x.shape
    indptr = indptr.cpu()
    rows = torch.repeat_interleave(torch.arange(users), indptr[1:] - indptr[:-1])
    excl = torch.zeros(users, n_items, dtype=torch.bool)
    excl[rows, indices.cpu().long()] = True
    x = x.masked_fill(excl, NEG_INF)
    order = torch.sort(x, dim=1, descending=True, stable=True).indices
    order = order.gather(1, torch.sort(excl.gather(1, order).to(torch.uint8), dim=1, stable=True).indices)
    idx = order[:, :k]
    assert not excl.gather(1, idx).any(), "fewer than k items left in a row"
    return x.gather(1, idx).to(logits.dtype), idx


def random_history(users, n_items, density, k, seed, full_rows=(), empty_rows=(), dup_rows=()):
    """CSR history (indptr int64, indices int32) with about `density` of the items per row; `full_rows` leave only k + 2 items
    (or k when fewer are left), `empty_rows` have none and `dup_rows` list every entry twice.  Row order inside a row is random."""
    rng = np.random.RandomState(seed)
    parts, counts = [], []
    for u in range(users):
        if u in empty_rows:
            h = np.zeros(0, np.int64)
        elif u in full_rows:
            h = rng.permutation(n_items)[: max(0, n_items - min(n_items, k + 2))]
        else:
            m = min(rng.binomial(n_items, density), n_items - k)
            h = rng.permutation(n_items)[:m]
        if u in dup_rows and h.size:
            h = rng.permutation(np.concatenate([h, h]))
        parts.append(h)
        counts.append(h.size)
    indptr = torch.from_numpy(np.concatenate([[0], np.cumsum(counts)]).astype(np.int64))
    indices = torch.from_numpy(np.concatenate(parts).astype(np.int32)) if parts else torch.zeros(0, dtype=torch.int32)
    return indptr, indices


def _check(logits, indptr, indices, k):
    vals, idx = recommend_topk(logits, indptr.cuda(), indices.cuda(), k)
    rv, ri = reference_topk(logits, indptr, indices, k)
    assert vals.dtype == logits.dtype and idx.dtype == torch.int64 and vals.shape == idx.shape == (logits.shape[0], k)
    assert torch.equal(idx.cpu(), ri)
    assert torch.equal(vals.cpu(), rv)
    return vals, idx


# ------------------------------------------------------------------------------------------------------------------------------
# argument checks (no GPU needed)
# ------------------------------------------------------------------------------------------------------------------------------
def _args(users=4, n_items=50, dtype=torch.float32):
    return torch.zeros(users, n_items, dtype=dtype), torch.zeros(users + 1, dtype=torch.int64), torch.zeros(0, dtype=torch.int32)


@pytest.mark.parametrize("dtype", [torch.float16, torch.float64, torch.int32])
def test_rejects_logit_dtypes(dtype):
    x, ip, ix = _args(dtype=dtype)
    with pytest.raises(TypeError, match="float32 or bfloat16"):
        recommend_topk(x, ip, ix, 5)


def test_rejects_history_dtypes():
    x, ip, ix = _args()
    with pytest.raises(TypeError, match="history_indptr must be int64"):
        recommend_topk(x, ip.int(), ix, 5)
    with pytest.raises(TypeError, match="history_indices must be int32"):
        recommend_topk(x, ip, ix.long(), 5)


@pytest.mark.parametrize("n", [0, 4, 6])
def test_rejects_mismatched_indptr_length(n):
    x, _, ix = _args()
    with pytest.raises(ValueError, match="users \\+ 1 = 5 entries"):
        recommend_topk(x, torch.zeros(n, dtype=torch.int64), ix, 5)


def test_rejects_bad_k():
    x, ip, ix = _args(n_items=300)
    for k in (0, -1, MAX_K + 1):
        with pytest.raises(ValueError, match=f"k={k} must lie in"):
            recommend_topk(x, ip, ix, k)
    x, ip, ix = _args(n_items=50)
    with pytest.raises(ValueError, match="k=51 must lie in \\[1, 50\\]"):
        recommend_topk(x, ip, ix, 51)
    with pytest.raises(TypeError):
        recommend_topk(x, ip, ix, 5.0)
    with pytest.raises(TypeError):
        recommend_topk(x, ip, ix, True)


def test_k_takes_any_integer_type():
    from sdrm_b200.recommend import check_k
    for k in (7, np.int32(7), np.int64(7), np.uint8(7), torch.tensor(7)):
        got = check_k(k, 50)
        assert got == 7 and type(got) is int
    x, ip, ix = _args()
    with pytest.raises(_lib.SdrmError, match="CUDA"):        # (past the argument checks: only the CPU tensors are wrong)
        recommend_topk(x, ip, ix, np.int64(5))


def test_rejects_shapes_and_layouts():
    x, ip, ix = _args()
    with pytest.raises(ValueError, match="2-D"):
        recommend_topk(x[0], ip, ix, 5)
    with pytest.raises(ValueError, match="unit column stride"):
        recommend_topk(torch.zeros(50, 4).t(), ip, ix, 5)


def test_rejects_cpu_tensors():
    x, ip, ix = _args()
    with pytest.raises(_lib.SdrmError, match="CUDA"):
        recommend_topk(x, ip, ix, 5)


def test_sample_ddpm_rejects_exclude_without_topk():
    from sdrm_b200.models import SDRM, VAE
    from sdrm_b200.train_SDRM import sample_ddpm
    diff, vae = SDRM(8, 5, 8, 1), VAE(12, 6, 8)
    with pytest.raises(ValueError, match="exclude= needs topk="):
        sample_ddpm(4, diff, vae, 8, 1.0, n_timesteps=5, exclude=_args()[1:])


def test_reference_orders_ties_and_drops_the_history():
    x = torch.tensor([[1.0, 3.0, 3.0, NEG_INF, 2.0, 3.0, float("nan"), -0.0, 0.0]])
    ip, ix = torch.tensor([0, 2], dtype=torch.int64), torch.tensor([2, 8], dtype=torch.int32)
    v, i = reference_topk(x, ip, ix, 7)
    assert i.tolist() == [[1, 5, 4, 0, 7, 3, 6]]
    assert v.tolist() == [[3.0, 3.0, 2.0, 1.0, 0.0, NEG_INF, NEG_INF]]


# ------------------------------------------------------------------------------------------------------------------------------
# the kernel against the reference
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("k", [1, 10, 100, MAX_K])
@pytest.mark.parametrize("n_items", [37, 255, 256, 257, 1000, 4099, 20011])
def test_matches_reference(n_items, k, dtype):
    if k > n_items:
        pytest.skip("k above the item count is an argument error")
    users = 70
    g = torch.Generator().manual_seed(n_items * 1000 + k)
    logits = torch.randn(users, n_items, generator=g).to(dtype)
    ip, ix = random_history(users, n_items, 0.05, k, seed=k + n_items, full_rows=(1, 7), empty_rows=(0, 5), dup_rows=(2, 7))
    _check(logits.cuda(), ip, ix, k)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_history_covering_all_but_k_items(dtype):
    n_items, k = 3000, 100
    logits = torch.randn(5, n_items, generator=torch.Generator().manual_seed(3)).to(dtype)
    rng = np.random.RandomState(3)
    rows = [rng.permutation(n_items)[: n_items - k] for _ in range(5)]
    ip = torch.tensor([0] + list(np.cumsum([r.size for r in rows])), dtype=torch.int64)
    ix = torch.from_numpy(np.concatenate(rows).astype(np.int32))
    vals, idx = _check(logits.cuda(), ip, ix, k)
    for u in range(5):   # exactly the items outside the history, best first
        assert sorted(idx[u].tolist()) == sorted(set(range(n_items)) - set(rows[u].tolist()))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("k", [1, 10, 100, MAX_K])
def test_tied_scores_go_to_the_lower_index(k, dtype):
    n_items, users = 3001, 12
    g = torch.Generator().manual_seed(k)
    logits = torch.randint(0, 4, (users, n_items), generator=g).float()   # heavy ties
    logits[0] = 1.0                                                       # one value only
    logits[1, ::7] = NEG_INF                                              # genuine -inf logits compete with nothing else ...
    logits[2] = NEG_INF                                                   # ... or with each other only
    logits[3, ::5] = float("nan")                                         # NaN ranks as -inf
    logits[4, ::2] = -0.0                                                 # -0.0 ties with +0.0
    logits[4, 1::2] = 0.0
    ip, ix = random_history(users, n_items, 0.02, k, seed=k, dup_rows=(0, 4))
    vals, idx = _check(logits.to(dtype).cuda(), ip, ix, k)
    # row 0: every score equal, so the k lowest item indices outside the history, in order
    seen = set(ix[ip[0]:ip[1]].tolist())
    assert idx[0].tolist() == [j for j in range(n_items) if j not in seen][:k]
    assert not torch.isnan(vals.float()).any()


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_single_user(dtype):
    logits = torch.randn(1, 777, generator=torch.Generator().manual_seed(9)).to(dtype)
    for k in (1, 10, 100, MAX_K):
        ip, ix = random_history(1, 777, 0.3, k, seed=k, dup_rows=(0,))
        _check(logits.cuda(), ip, ix, k)
    _check(logits[:, :5].contiguous().cuda(), torch.tensor([0, 0]), torch.zeros(0, dtype=torch.int32), 5)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_row_strided_views_and_rejected_layouts(dtype):
    users, n_items, k = 33, 1001, 50
    big = torch.randn(users * 2, n_items + 13, generator=torch.Generator().manual_seed(5)).to(dtype).cuda()
    ip, ix = random_history(users, n_items, 0.05, k, seed=5)
    _check(big[::2, 7:7 + n_items], ip, ix, k)           # row stride 2 (n_items + 13), start misaligned by 7 elements
    _check(big[:users, 3:3 + n_items], ip, ix, k)
    with pytest.raises(ValueError, match="unit column stride"):
        recommend_topk(big[:n_items, :users].t(), ip.cuda(), ix.cuda(), k)
    with pytest.raises(ValueError, match="unit column stride"):
        recommend_topk(big[0:1, :n_items].expand(users, n_items), ip.cuda(), ix.cuda(), k)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n_items", [380_000, 400_003])
def test_wide_rows_take_a_large_bitmap(n_items, dtype):
    """Bitmaps of 47 500 and 50 004 bytes: with the kernel's static shared memory both exceed the 48 KB a launch gets without
    the dynamic shared-memory opt-in (the first one only together with the static part)."""
    users, k = 3, MAX_K
    logits = torch.randn(users, n_items, generator=torch.Generator().manual_seed(11)).to(dtype)
    ip, ix = random_history(users, n_items, 0.01, k, seed=11, empty_rows=(1,))
    _check(logits.cuda(), ip, ix, k)


@pytest.mark.gpu
def test_no_users_and_outputs_on_the_current_device():
    vals, idx = recommend_topk(torch.zeros(0, 40, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda"),
                               torch.zeros(0, dtype=torch.int32, device="cuda"), 5)
    assert vals.shape == idx.shape == (0, 5) and vals.is_cuda and idx.is_cuda


@pytest.mark.gpu
def test_device_side_errors():
    logits = torch.randn(4, 60, device="cuda")
    ip = torch.tensor([0, 2, 2, 58, 60], dtype=torch.int64)
    ix = torch.cat([torch.tensor([1, 2]), torch.arange(56), torch.tensor([3, 4])]).int()
    recommend_topk(logits, ip.cuda(), ix.cuda(), 4)                       # row 2 keeps 4 items: fine
    with pytest.raises(ValueError, match="exceeds the number of items left"):
        recommend_topk(logits, ip.cuda(), ix.cuda(), 5)
    with pytest.raises(ValueError, match="outside \\[0, 60\\)"):
        recommend_topk(logits, ip.cuda(), torch.where(ix == 3, 60, ix).int().cuda(), 4)
    with pytest.raises(ValueError, match="outside \\[0, 60\\)"):
        recommend_topk(logits, ip.cuda(), torch.where(ix == 3, -1, ix).int().cuda(), 4)
    for bad in ([0, 2, 1, 58, 60], [0, 2, 2, 58, 61], [-1, 2, 2, 58, 60]):
        with pytest.raises(ValueError, match="non-decreasing"):
            recommend_topk(logits, torch.tensor(bad, dtype=torch.int64).cuda(), ix.cuda(), 4)
    with pytest.raises(ValueError, match="must be on"):
        recommend_topk(logits, ip, ix.cuda(), 4)


# ------------------------------------------------------------------------------------------------------------------------------
# sample_ddpm(topk=...) on every sampler flow and on strided DDPM / DDIM grids: the reference top-K of the same call's dense rows
# ------------------------------------------------------------------------------------------------------------------------------
GRIDS = {"full": {}, "strided": {"sampling_steps": 3}, "ddim": {"sampling_steps": 4, "eta": 0.5}}


@pytest.mark.gpu
@pytest.mark.parametrize("grid", list(GRIDS))
@pytest.mark.parametrize("multires", [False, True])
@pytest.mark.parametrize("kind", ["k1", "k6"])
def test_sample_ddpm_topk_on_every_flow(kind, multires, grid):
    from helpers import random_modules
    from sdrm_b200.train_SDRM import engine_for, sample_ddpm
    from test_sampler_edges_gpu import FLOWS, MODELS, _flows_of
    I, H, L, T, nh, nd = MODELS[kind]
    n, k = 300, 20
    diff, vae = random_modules(I, H, L, T, nh, seed=61, device="cuda")
    eng = engine_for(diff, torch.device("cuda", torch.cuda.current_device()))
    ip, ix = random_history(n, I, 0.05, k, seed=62, full_rows=(3,), empty_rows=(0,), dup_rows=(5,))
    exclude = (ip.cuda(), ix.cuda())
    kw = dict(GRIDS[grid], seed=0xBEEF, n_timesteps=T)
    if multires:
        kw.update(timesteps="random", t_rows=np.random.RandomState(63).randint(1, T, size=n))
    for flow in _flows_of(kind, multires):
        opts, (cluster, split, resident) = FLOWS[flow]
        try:
            for o, v in opts.items():
                eng.set_option(o, v)
            for dtype in (torch.float32, torch.bfloat16):
                dense = sample_ddpm(n, diff, vae, L, nd, out_dtype=dtype, **kw)
                (vals, idx), lat = sample_ddpm(n, diff, vae, L, nd, out_dtype=dtype, topk=k, exclude=exclude, return_latent=True,
                                               **kw)
                lib = eng.lib
                got = (lib.sdrm_last_cluster_size(eng.handle), lib.sdrm_last_split_size(eng.handle),
                       lib.sdrm_last_resident_mode(eng.handle))
                assert got[0] == cluster and split in (None, got[1]) and resident in (None, got[2]), (flow, got)
                assert lat.shape == (n, L)
                rv, ri = reference_topk(dense, ip, ix, k)
                assert torch.equal(idx.cpu(), ri), (flow, dtype)
                assert torch.equal(vals.cpu(), rv), (flow, dtype)
                v2, i2 = sample_ddpm(n, diff, vae, L, nd, out_dtype=dtype, topk=k, **kw)   # no history: plain top-K of the rows
                rv, ri = reference_topk(dense, torch.zeros(n + 1, dtype=torch.int64), torch.zeros(0, dtype=torch.int32), k)
                assert torch.equal(i2.cpu(), ri) and torch.equal(v2.cpu(), rv), (flow, dtype)
        finally:
            for o in opts:
                eng.set_option(o, 0)


@pytest.mark.gpu
def test_sample_ddpm_topk_arguments():
    from helpers import random_modules
    from sdrm_b200.train_SDRM import sample_ddpm
    from test_sampler_edges_gpu import MODELS
    I, H, L, T, nh, nd = MODELS["k6"]
    diff, vae = random_modules(I, H, L, T, nh, seed=64, device="cuda")
    with pytest.raises(ValueError, match="must lie in"):
        sample_ddpm(10, diff, vae, L, nd, n_timesteps=T, topk=MAX_K + 1)
    with pytest.raises(ValueError, match="users \\+ 1 = 11"):
        sample_ddpm(10, diff, vae, L, nd, n_timesteps=T, topk=5,
                    exclude=(torch.zeros(10, dtype=torch.int64, device="cuda"), torch.zeros(0, dtype=torch.int32, device="cuda")))
    with pytest.raises(ValueError, match="must be on"):
        sample_ddpm(10, diff, vae, L, nd, n_timesteps=T, topk=5,
                    exclude=(torch.zeros(11, dtype=torch.int64), torch.zeros(0, dtype=torch.int32)))
    v, i = sample_ddpm(0, diff, vae, L, nd, n_timesteps=T, topk=5)
    assert v.shape == i.shape == (0, 5) and i.dtype == torch.int64
    # the default output is unchanged by the new keywords
    a = sample_ddpm(50, diff, vae, L, nd, n_timesteps=T, seed=3)
    b = sample_ddpm(50, diff, vae, L, nd, n_timesteps=T, seed=3, topk=None, exclude=None)
    assert torch.equal(a, b) and a.shape == (50, I) and a.dtype == torch.float32
