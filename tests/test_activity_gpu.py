"""GPU tests of the activity-matched binarisation: K12 (sdrm_topk_pack) bit-exact against the NumPy oracle on every width edge and
score pattern, activity_matched_device against the rule, rows from the sampler, the sharded gathers (one process and two NCCL
ranks), main.py --binarise, synthesize --activity-from, and a cfg-5 shard at its real size."""
import os
import socket
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import scipy.sparse as sp
import torch

import activity_oracle as oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STAGED_COLS = {torch.float32: 20480, torch.bfloat16: 40960}   # the widest row K12 stages in shared memory (80 KB)


def _scores(rng, rows, n_cols, kind):
    """float32 host scores of one pattern."""
    if kind == "continuous":
        return rng.standard_normal((rows, n_cols)).astype(np.float32)
    if kind == "tied":
        return np.round(rng.standard_normal((rows, n_cols)) * 1.5).astype(np.float32) / 2
    if kind == "equal":
        return np.full((rows, n_cols), 0.25, dtype=np.float32)
    if kind == "zeros":   # -0.0 and +0.0 (equal scores), a few ones above them
        x = np.where(rng.random((rows, n_cols)) < 0.5, np.float32(-0.0), np.float32(0.0))
        x[rng.random((rows, n_cols)) < 0.1] = 1.0
        return x
    if kind == "special":
        x = rng.standard_normal((rows, n_cols)).astype(np.float32)
        pick = rng.random((rows, n_cols))
        x[pick < 0.1] = np.nan
        x[(pick >= 0.1) & (pick < 0.15)] = np.inf
        x[(pick >= 0.15) & (pick < 0.2)] = -np.inf
        x[(pick >= 0.2) & (pick < 0.25)] = -0.0
        x[(pick >= 0.25) & (pick < 0.3)] = 0.0
        return x
    raise ValueError(kind)


def _check_packed(pm, dense_want, k):
    rows, n_cols = dense_want.shape
    assert pm.threshold is None and pm.shape == (rows, n_cols)
    got = pm.numpy(np.int64).astype(bool)
    bad = np.nonzero((got != dense_want).any(axis=1))[0]
    assert bad.size == 0, f"rows {bad[:5]} differ"
    assert np.array_equal(got.sum(axis=1), np.asarray(k))
    assert int(pm.ones.item()) == int(np.sum(k))
    tail = n_cols % 32
    if tail and rows:
        last = pm.bits[:, -1].cpu().numpy().view(np.uint32)
        assert not np.any(last >> np.uint32(tail)), "padding bits must be 0"


def _ks_for(rng, rows, n_cols):
    base = [0, 1, n_cols]
    return np.array([base[i] if i < 3 else int(rng.integers(0, n_cols + 1)) for i in range(rows)], dtype=np.int64)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n_cols", [1, 31, 32, 33, 729, 1008, 8582, 20000, "staged", "staged+1", 1 << 20])
def test_topk_pack_against_oracle(dtype, n_cols):
    from sdrm_b200.sparsify import topk_pack
    if n_cols == "staged":
        n_cols = STAGED_COLS[dtype]
    elif n_cols == "staged+1":
        n_cols = STAGED_COLS[dtype] + 1
    rng = np.random.default_rng(n_cols * 7 + (dtype == torch.bfloat16))
    rows = 3 if n_cols >= (1 << 20) else 7
    kinds = ("continuous", "tied", "special") if n_cols >= (1 << 20) else ("continuous", "tied", "equal", "zeros", "special")
    for kind in kinds:
        host = _scores(rng, rows, n_cols, kind)
        S = torch.from_numpy(host).cuda().to(dtype)
        k = _ks_for(rng, rows, n_cols)
        want = oracle.topk_dense(S, k)
        _check_packed(topk_pack(S, torch.from_numpy(k).cuda()), want, k)
        _check_packed(topk_pack(S[:1], k[:1]), want[:1], k[:1])              # one row, k from the host
        _check_packed(topk_pack(S[:0], k[:0]), want[:0], k[:0])              # no row


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("n_cols", [33, 1008, 20000, 25000])
def test_topk_pack_strided_rows(dtype, n_cols):
    """A row slice of a wider matrix (unaligned row starts) and every other row of a taller one."""
    from sdrm_b200.sparsify import topk_pack
    rng = np.random.default_rng(n_cols)
    big = torch.from_numpy(_scores(rng, 40, n_cols + 11, "tied")).cuda().to(dtype)
    for view in (big[:, 3:3 + n_cols], big[::2, :n_cols], big[5:6, 1:1 + n_cols]):
        assert view.stride(1) == 1
        k = rng.integers(0, n_cols + 1, size=view.shape[0])
        _check_packed(topk_pack(view, torch.from_numpy(k).cuda()), oracle.topk_dense(view, k), k)


def test_topk_pack_errors():
    from sdrm_b200._lib import SdrmError
    from sdrm_b200.sparsify import topk_pack
    S = torch.randn(4, 50, device="cuda")
    for bad in ([0, 1, 51, 2], [0, -1, 3, 2], [2 ** 40, 0, 0, 0]):
        with pytest.raises(ValueError):
            topk_pack(S, torch.tensor(bad, device="cuda"))
    with pytest.raises(ValueError):
        topk_pack(S, torch.tensor([1, 2, 3], device="cuda"))          # one k per row
    with pytest.raises(ValueError):
        topk_pack(S, torch.tensor([1.0, 2.0, 3.0, 4.0], device="cuda"))
    with pytest.raises(SdrmError):
        topk_pack(S.cpu(), [1, 2, 3, 4])
    with pytest.raises(ValueError):
        topk_pack(S.double(), [1, 2, 3, 4])
    with pytest.raises(ValueError):
        topk_pack(S[0], [1])
    with pytest.raises(ValueError):
        topk_pack(S.t(), [1] * 50)
    with pytest.raises(ValueError):
        topk_pack(torch.zeros(2, (1 << 20) + 1, device="cuda"), [1, 1])
    pm = topk_pack(S, torch.tensor([1, 2, 3, 50], device="cuda"))   # a good call after the bad ones
    assert pm.numpy().sum(axis=1).tolist() == [1, 2, 3, 50]


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("m,n,n_cols", [(500, 500, 729), (843, 400, 1008), (300, 900, 3125), (1, 5, 40)])
def test_activity_matched_against_oracle(dtype, m, n, n_cols):
    from sdrm_b200.fidelity import compare
    from sdrm_b200.sparsify import activity_matched_device, row_activity
    rng = np.random.default_rng(m + n + n_cols)
    real = sp.csr_matrix((rng.random((n, n_cols)) < rng.random((n, 1)) * 0.12).astype(np.float32))
    a = row_activity(real)
    S = torch.from_numpy(_scores(rng, m, n_cols, "continuous")).cuda().to(dtype)
    for q in (0.95, 0.5):
        pm = activity_matched_device(S, q, a)
        want, k = oracle.activity_matched(S, q, a)
        _check_packed(pm, want, k)
        assert pm.to_sparse().threshold is None
        if m == n:
            assert np.array_equal(np.sort(pm.numpy().sum(axis=1)), np.sort(a))
            assert compare(real, pm, k=None).summary()["activity_ks"] == 0.0


@pytest.mark.parametrize("mode", ["full", "random"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_from_sampler(mode, dtype):
    from helpers import random_modules
    from sdrm_b200.sparsify import activity_matched_device
    from sdrm_b200.train_SDRM import sample_ddpm
    n, I, H, L, T, nh = 777, 1008, 64, 48, 7, 1
    dn, vae = random_modules(I, H, L, T, nh, seed=11, device="cuda")
    t_rows = np.random.RandomState(5).randint(1, T, size=n) if mode == "random" else None
    S = sample_ddpm(n, dn, vae, L, 1.0, timesteps="random" if mode == "random" else None, n_timesteps=T, seed=9, t_rows=t_rows,
                    out_dtype=dtype)
    a = np.random.default_rng(3).zipf(1.7, size=n).clip(0, I)
    pm = activity_matched_device(S, 0.9425, a)
    want, k = oracle.activity_matched(S, 0.9425, a)
    _check_packed(pm, want, k)
    assert np.array_equal(np.sort(k), np.sort(a))


@pytest.mark.parametrize("gather", ["bits", "csr"])
@pytest.mark.parametrize("mode", [None, "random"])
def test_sharded_one_process_equals_direct(gather, mode):
    from helpers import random_modules
    from sdrm_b200.distributed import sample_ddpm_sharded
    from sdrm_b200.sparsify import activity_matched_device
    from sdrm_b200.train_SDRM import sample_ddpm
    n, I, H, L, T, nh = 513, 300, 64, 40, 8, 1
    dn, vae = random_modules(I, H, L, T, nh, seed=21, device="cuda")
    a = np.random.default_rng(1).integers(0, 60, size=400)
    got, span = sample_ddpm_sharded(n, dn, vae, L, 1.0, timesteps=mode, n_timesteps=T, seed=77, gather=gather, sparsity=0.95,
                                    activity=a)
    t_rows = np.random.RandomState(77).randint(1, T, size=n).astype(np.int32) if mode == "random" else None
    S = sample_ddpm(n, dn, vae, L, 1.0, timesteps=mode, n_timesteps=T, seed=77, t_rows=t_rows)
    want = activity_matched_device(S, 0.95, a)
    assert span == (0, n)
    if gather == "bits":
        assert torch.equal(got.bits, want.bits) and got.threshold is None and int(got.ones) == int(want.ones)
    else:
        w = want.to_sparse()
        assert torch.equal(got.indptr, w.indptr) and torch.equal(got.indices, w.indices) and got.threshold is None


def test_sharded_activity_needs_a_binarising_gather():
    from helpers import random_modules
    from sdrm_b200.distributed import sample_ddpm_sharded
    dn, vae = random_modules(40, 16, 8, 5, 0, seed=1, device="cuda")
    for gather in (False, True):
        with pytest.raises(ValueError):
            sample_ddpm_sharded(10, dn, vae, 8, 1.0, n_timesteps=5, seed=0, gather=gather, sparsity=0.9, activity=[1, 2])


def _tiny_dataset(tmp_path, U=150, I=60):
    import pickle

    from privacy_oracle import random_rows
    rng = np.random.default_rng(2)
    train = sp.csr_matrix(random_rows(rng, U, I, 0.1).astype(np.float64))
    train[0, 59] = 0.0            # an explicit stored zero: counted by SPARSITY, not by the activity
    train[1, 3] = 1.0
    valid = sp.csr_matrix(random_rows(rng, 120, I, 0.15).astype(np.float64))
    os.makedirs(tmp_path / "ml-100k")
    for kind, mat in (("train_test", train), ("valid", valid)):
        with open(tmp_path / "ml-100k" / f"ml-100k_{kind}.pkl", "wb") as fh:
            pickle.dump(mat, fh)
    return train


def test_main_binarise_activity(tmp_path, monkeypatch, capsys):
    """main.py --binarise activity: every column's rows have TRAIN_DATA's activity histogram exactly; --binarise equal-sparsity
    returns and prints exactly what no flag does."""
    import main as cli
    import sdrm_b200.train_SDRM as ts
    from helpers import random_modules
    from sdrm_b200.sparsify import row_activity
    train = _tiny_dataset(tmp_path)
    monkeypatch.setattr(ts, "train_SDRM", lambda **kw: random_modules(kw["N_ITEMS"], kw["VAE_HIDDEN"], kw["DIFF_LATENT"],
                                                                      kw["TIMESTEPS"], kw["N_HIDDEN_MLP_LAYERS"], seed=4,
                                                                      device="cuda"))
    monkeypatch.chdir(tmp_path)
    argv = ["--dataset", "ml-100k", "--data-dir", str(tmp_path), "--runs", "1", "--seed", "5", "--SDRM-timesteps", "6",
            "--MLP-latent-neurons", "16", "--VAE-hidden-layer-neurons", "24", "--MLP-hidden-layers", "1"]
    plain = cli.main(argv)
    out0 = capsys.readouterr().out
    same = cli.main(argv + ["--binarise", "equal-sparsity"])
    out1 = capsys.readouterr().out
    for c in cli.COLS:
        assert np.array_equal(plain[c], same[c], equal_nan=True), c
    assert [ln for ln in out1.splitlines() if "took" not in ln] == [ln for ln in out0.splitlines() if "took" not in ln]

    want = np.sort(row_activity(train))
    recorded = []
    real = cli.binarise_activity

    def recording(scores, sparsity, activity):
        res = real(scores, sparsity, activity)
        recorded.append(res)
        return res
    monkeypatch.setattr(cli, "binarise_activity", recording)
    cli.main(argv + ["--binarise", "activity", "--save-synthetic", str(tmp_path / "synth")])
    assert len(recorded) == 3
    for dense, pm in recorded:
        assert pm.threshold is None
        assert np.array_equal(np.sort(dense.sum(axis=1)), want)
    for name in cli.COLS:
        mat = sp.load_npz(tmp_path / "synth" / f"run1_{name}.npz")
        assert np.array_equal(np.sort(np.diff(mat.indptr)), want), name


@pytest.mark.timeout(600)
def test_cli_activity_from(tmp_path):
    from helpers import random_modules
    from sdrm_b200.distributed import sample_ddpm_sharded
    from sdrm_b200.synthesize import load_generator, save_generator
    from sdrm_b200.sparsify import row_activity
    I, H, L, T, nh, nd = 500, 64, 32, 9, 1, 1.0
    dn, vae = random_modules(I, H, L, T, nh, seed=8, device="cuda")
    gen = save_generator(str(tmp_path / "g.pt"), dn, vae, noise_divider=nd, sparsity=0.97)
    rng = np.random.default_rng(4)
    real = sp.csr_matrix((rng.random((700, I)) < rng.random((700, 1)) * 0.1).astype(np.float32))
    real_path = str(tmp_path / "real.npz")
    sp.save_npz(real_path, real)
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    out = str(tmp_path / "x.npz")
    r = subprocess.run([sys.executable, "-m", "sdrm_b200.synthesize", "--generator", gen, "--users", "1234", "--out", out,
                        "--activity-from", real_path, "--seed", "3"], cwd=ROOT, env=env, capture_output=True, text=True, timeout=500)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "1234 users" in r.stdout and "threshold none" in r.stdout
    got = sp.load_npz(out)
    d2, v2, meta = load_generator(gen, torch.device("cuda"))
    S, _ = sample_ddpm_sharded(1234, d2, v2, L, nd, n_timesteps=T, seed=3)
    a = row_activity(real)
    want, k = oracle.activity_matched(S, 0.97, a)
    assert np.array_equal(np.diff(got.indptr), k)
    assert np.array_equal(got.toarray().astype(bool), want)
    bad = sp.csr_matrix(np.ones((3, I + 1), dtype=np.float32))
    sp.save_npz(real_path, bad)
    r = subprocess.run([sys.executable, "-m", "sdrm_b200.synthesize", "--generator", gen, "--users", "10", "--out", out,
                        "--activity-from", real_path], cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "items" in r.stderr


@pytest.mark.timeout(900)
def test_cfg5_shard_real_size():
    """125 000 x 20 000 fp32 (a cfg-5 shard, 10 GB, every row staged): exact popcounts for every row, and the oracle's per-row
    select on a few hundred rows spread over the matrix (the targets checked against the oracle from K4's counts)."""
    from sdrm_b200.sparsify import _packed_indptr, activity_matched_device, equal_sparsity_device
    rows, n_cols, q = 125_000, 20_000, 0.99
    g = torch.Generator(device="cuda").manual_seed(17)
    S = torch.randn((rows, n_cols), generator=g, device="cuda")
    S[::97] = torch.round(S[::97] * 2) / 2      # heavily tied rows among them
    a = np.random.default_rng(5).zipf(1.5, size=100_000).clip(0, n_cols)
    pm = activity_matched_device(S, q, a)
    c = torch.diff(_packed_indptr(equal_sparsity_device(S, q).bits, n_cols)).cpu().numpy()
    k = oracle.targets(c, a)
    got_counts = torch.diff(_packed_indptr(pm.bits, n_cols)).cpu().numpy()
    assert np.array_equal(got_counts, k)
    assert int(pm.ones.item()) == int(k.sum())
    pick = np.unique(np.concatenate([np.linspace(0, rows - 1, 300).astype(np.int64), np.arange(0, rows, 97)[:40]]))
    idx = torch.from_numpy(pick).cuda()
    sub = S.index_select(0, idx)
    want = oracle.topk_dense(sub, k[pick])
    from sdrm_b200.sparsify import PackedMatrix
    got = PackedMatrix(pm.bits.index_select(0, idx), n_cols, None, None).numpy(np.int64).astype(bool)
    assert np.array_equal(got, want)
    del S, pm, sub
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------------------------------------
# two GPUs
# ------------------------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


CASES = [   # (n, timesteps, seed, sparsity, gather): full- and multi-resolution rows, and n = 1 (rank 1's block is empty)
    (301, None, 55, 0.9, "bits"),
    (257, "random", 56, 0.95, "csr"),
    (1, None, 57, 0.5, "bits"),
    (1, None, 58, 0.5, "csr"),
]
SHAPE = (190, 48, 72, 6, 1, 1.0)   # I, H, L, T, nh, nd
ACTIVITY = np.random.default_rng(9).integers(0, 40, size=211)


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
        from helpers import random_modules
        from sdrm_b200 import distributed as sdd
        I, H, L, T, nh, nd = SHAPE
        dn, vae = random_modules(I, H, L, T, nh, seed=3, device=dev)
        res = []
        for n, ts_, seed, q, gather in CASES:
            out, span = sdd.sample_ddpm_sharded(n, dn, vae, L, nd, timesteps=ts_, n_timesteps=T, seed=seed, gather=gather,
                                                sparsity=q, activity=ACTIVITY)
            if gather == "bits":
                res.append((span, out.bits.cpu(), int(out.ones.item()), out.threshold))
            else:
                res.append((span, out.indptr.cpu(), out.indices.cpu(), out.threshold))
        torch.save(res, os.path.join(out_dir, f"rank{rank}.pt"))
    except Exception:
        import traceback
        with open(os.path.join(out_dir, f"rank{rank}.err"), "w") as fh:
            fh.write(traceback.format_exc())
        raise
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_rank_activity_gather():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from helpers import random_modules
    from sdrm_b200.sparsify import activity_matched_device
    from sdrm_b200.train_SDRM import sample_ddpm
    world = 2
    ctx = mp.get_context("spawn")
    port = _free_port()
    out_dir = tempfile.mkdtemp(prefix="sdrm_activity_gpu_")
    procs = [ctx.Process(target=_worker, args=(r, world, port, out_dir)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        for p in procs:
            p.join(280)
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
                p.join()
    for r, p in enumerate(procs):
        err = os.path.join(out_dir, f"rank{r}.err")
        assert p.exitcode == 0, open(err).read() if os.path.exists(err) else f"rank {r} exit code {p.exitcode}"
    res = [torch.load(os.path.join(out_dir, f"rank{r}.pt"), weights_only=False) for r in range(world)]
    I, H, L, T, nh, nd = SHAPE
    dn, vae = random_modules(I, H, L, T, nh, seed=3, device="cuda")
    for c, (n, ts_, seed, q, gather) in enumerate(CASES):
        t_rows = np.random.RandomState(seed).randint(1, T, size=n).astype(np.int32) if ts_ == "random" else None
        whole = sample_ddpm(n, dn, vae, L, nd, timesteps=ts_, n_timesteps=T, seed=seed, t_rows=t_rows)
        pm = activity_matched_device(whole, q, ACTIVITY)
        for rank in range(world):
            span, x, y, thr = res[rank][c]
            assert span == (0, n) and thr is None
            if gather == "bits":
                assert torch.equal(x, pm.bits.cpu()) and y == int(pm.ones.item()), (c, rank)
            else:
                want = pm.to_sparse()
                assert torch.equal(x, want.indptr.cpu()) and torch.equal(y, want.indices.cpu()), (c, rank)
