"""GPU tests of synthetic rows as CSR: K10 (bits -> CSR) bit-exact against a NumPy oracle on every shape edge, past 2^31 ones,
from the sampler's binarised rows, the generator checkpoint, the synthesize CLI, main.py --save-synthetic / --save-generator,
and (on two GPUs) the sharded gather="csr"."""
import os
import socket
import subprocess
import sys
import tempfile

import numpy as np
import pytest
import scipy.sparse as sp
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _oracle(dense):
    """indptr / indices of a dense 0/1 matrix (row-major nonzero order: ascending columns within a row)."""
    counts = dense.sum(axis=1, dtype=np.int64)
    indptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    return indptr, np.nonzero(dense)[1].astype(np.int32)


def _packed(rng, rows, n_cols, density, extra_words, lead=2, trail=3):
    """Bits of `rows` random rows at `density` inside a larger matrix: `lead` rows before and `trail` after, `extra_words` words
    of garbage past ceil(n_cols / 32) per row, and garbage in the last word's bits at or past n_cols.  Returns (dense, the
    [rows, need] view with row stride need + extra_words, the full matrix)."""
    need = (n_cols + 31) // 32
    ld = need + extra_words
    dense = rng.random((rows, n_cols), dtype=np.float32) < density if 0 < density < 1 else np.full((rows, n_cols), density == 1)
    padded = np.zeros((rows, need * 32), dtype=bool)
    padded[:, :n_cols] = dense
    words = np.packbits(padded, axis=1, bitorder="little").view(np.uint32).reshape(rows, need)
    full = rng.integers(0, 2 ** 32, size=(lead + rows + trail, ld), dtype=np.uint32)   # garbage everywhere ...
    tail = n_cols % 32
    block = full[lead:lead + rows]
    block[:, :need] = words
    if tail:   # ... including the last word's unused high bits
        block[:, need - 1] |= rng.integers(0, 2 ** 32, size=rows, dtype=np.uint32) & np.uint32(~((1 << tail) - 1) & 0xFFFFFFFF)
    full_t = torch.from_numpy(full.view(np.int32)).cuda()
    return dense, full_t[lead:lead + rows, :need], full_t


@pytest.mark.parametrize("rows", [0, 1, 7, 4099])
@pytest.mark.parametrize("n_cols", [1, 31, 32, 33, 729, 1008, 3125, 8582, 20000])
def test_k10_against_numpy_oracle(rows, n_cols):
    from sdrm_b200.sparsify import packed_to_csr
    rng = np.random.default_rng(rows * 100003 + n_cols)
    for density in (0.0, 0.001, 0.01, 0.5, 1.0):
        for extra in (0, 3):
            dense, view, _ = _packed(rng, rows, n_cols, density, extra)
            assert view.stride(0) == view.shape[1] + extra
            want_ptr, want_idx = _oracle(dense)
            sr = packed_to_csr(view, n_cols)
            assert sr.shape == (rows, n_cols) and sr.nnz == len(want_idx)
            assert sr.indptr.dtype == torch.int64 and sr.indices.dtype == torch.int32
            assert np.array_equal(sr.indptr.cpu().numpy(), want_ptr), (density, extra)
            assert np.array_equal(sr.indices.cpu().numpy(), want_idx), (density, extra)
            again = packed_to_csr(view, n_cols)
            assert torch.equal(again.indptr, sr.indptr) and torch.equal(again.indices, sr.indices)


def test_k10_row_slice_of_packed_matrix():
    """PackedMatrix.to_sparse on a row slice (pointer offset, parent's row stride) of threshold_pack's output."""
    from sdrm_b200.sparsify import PackedMatrix, threshold_pack
    g = torch.Generator(device="cuda").manual_seed(3)
    S = torch.rand((1000, 3125), generator=g, device="cuda")
    pm = threshold_pack(S, 0.97)
    dense = pm.numpy(np.int64)
    part = PackedMatrix(pm.bits[123:777], pm.n_cols, pm.threshold, None).to_sparse()
    want = sp.csr_matrix(dense[123:777])
    got = part.to_scipy()
    assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)


def test_k10_nnz_past_int32():
    """110 000 x 20 000 ones: nnz = 2.2e9 > 2^31; indptr and the row placement must use 64-bit arithmetic (8.8 GB of indices)."""
    from sdrm_b200.sparsify import packed_to_csr
    rows, n_cols = 110_000, 20_000
    bits = torch.full((rows, n_cols // 32), -1, dtype=torch.int32, device="cuda")
    sr = packed_to_csr(bits, n_cols)
    assert sr.nnz == rows * n_cols and sr.nnz > 2 ** 31
    assert torch.equal(sr.indptr, torch.arange(rows + 1, dtype=torch.int64, device="cuda") * n_cols)
    cols = torch.arange(n_cols, dtype=torch.int32, device="cuda")
    for r in (0, 1, rows // 2, 107_374, 107_375, rows - 2, rows - 1):    # (row 107 374 straddles the 2^31-th entry)
        assert torch.equal(sr.indices[r * n_cols:(r + 1) * n_cols], cols), r
    del sr, bits
    torch.cuda.empty_cache()


def _check_same_csr(got, dense):
    want = sp.csr_matrix(dense)
    assert got.shape == want.shape and got.dtype == want.dtype == np.int64
    assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)
    assert np.array_equal(got.data, want.data) and got.has_canonical_format


@pytest.mark.parametrize("mode", ["full", "random"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("steps", [None, 3])
def test_from_sampler(mode, dtype, steps):
    from helpers import random_modules
    from sdrm_b200.sparsify import equal_sparsity_device
    from sdrm_b200.train_SDRM import sample_ddpm
    n, I, H, L, T, nh = 777, 1008, 64, 48, 7, 1
    dn, vae = random_modules(I, H, L, T, nh, seed=11, device="cuda")
    t_rows = np.random.RandomState(5).randint(1, T, size=n) if mode == "random" else None
    S = sample_ddpm(n, dn, vae, L, 1.0, timesteps="random" if mode == "random" else None, n_timesteps=T, seed=9, t_rows=t_rows,
                    out_dtype=dtype, sampling_steps=steps)
    for q in (0.9425, 0.0):
        pm = equal_sparsity_device(S, q)
        sr = pm.to_sparse()
        assert sr.threshold == pm.threshold and sr.nnz == int(pm.ones.item())
        got = sr.to_scipy()
        dense = pm.numpy(np.int64)
        _check_same_csr(got, dense)
        if q == 0.0:
            assert got.nnz == n * I


def test_from_sampler_all_zero_nan_threshold():
    from helpers import random_modules
    from sdrm_b200.sparsify import equal_sparsity_device
    from sdrm_b200.train_SDRM import sample_ddpm
    n, I, H, L, T, nh = 300, 200, 32, 24, 6, 0
    dn, vae = random_modules(I, H, L, T, nh, seed=2, device="cuda")
    with torch.no_grad():
        vae.decoder[2].bias[17] = float("nan")     # one NaN column: np.quantile is NaN, no score is >= NaN
    S = sample_ddpm(n, dn, vae, L, 1.0, n_timesteps=T, seed=1)
    pm = equal_sparsity_device(S, 0.9)
    assert np.isnan(pm.threshold)
    sr = pm.to_sparse()
    assert sr.nnz == 0 and torch.equal(sr.indptr, torch.zeros(n + 1, dtype=torch.int64, device="cuda"))
    got = sr.to_scipy()
    _check_same_csr(got, pm.numpy(np.int64))
    assert got.nnz == 0


@pytest.mark.parametrize("multi_resolution", [False, True])
def test_generator_checkpoint_same_rows(tmp_path, multi_resolution):
    from helpers import random_modules
    from sdrm_b200.distributed import sample_ddpm_sharded
    from sdrm_b200.synthesize import load_generator, save_generator
    I, H, L, T, nh, nd = 300, 64, 40, 8, 2, 0.7
    dn, vae = random_modules(I, H, L, T, nh, seed=21, device="cuda")
    path = save_generator(str(tmp_path / "g.pt"), dn, vae, noise_divider=nd, sparsity=0.95)
    d2, v2, meta = load_generator(path, torch.device("cuda"))
    kw = dict(timesteps="random" if multi_resolution else None, n_timesteps=T, seed=77)
    a, _ = sample_ddpm_sharded(513, dn, vae, L, nd, **kw)
    b, _ = sample_ddpm_sharded(513, d2, v2, L, meta["noise_divider"], **kw)
    assert torch.equal(a, b)
    ca, _ = sample_ddpm_sharded(513, dn, vae, L, nd, gather="csr", sparsity=0.95, **kw)
    cb, _ = sample_ddpm_sharded(513, d2, v2, L, nd, gather="csr", sparsity=meta["sparsity"], **kw)
    assert torch.equal(ca.indptr, cb.indptr) and torch.equal(ca.indices, cb.indices)


@pytest.mark.timeout(600)
def test_cli_writes_the_sharded_result(tmp_path):
    from helpers import random_modules
    from sdrm_b200.distributed import sample_ddpm_sharded
    from sdrm_b200.synthesize import load_generator, save_generator
    I, H, L, T, nh, nd = 500, 64, 32, 9, 1, 1.0
    dn, vae = random_modules(I, H, L, T, nh, seed=8, device="cuda")
    gen = save_generator(str(tmp_path / "g.pt"), dn, vae, noise_divider=nd, sparsity=0.97)
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    for flags, kw in (([], dict(sparsity=0.97)),
                      (["--multi-resolution", "--bf16", "--sampling-steps", "4", "--sparsity", "0.9", "--seed", "12"],
                       dict(timesteps="random", out_dtype=torch.bfloat16, sampling_steps=4, sparsity=0.9, seed=12))):
        out = str(tmp_path / "x.npz")
        r = subprocess.run([sys.executable, "-m", "sdrm_b200.synthesize", "--generator", gen, "--users", "1234", "--out", out] + flags,
                           cwd=ROOT, env=env, capture_output=True, text=True, timeout=500)
        assert r.returncode == 0, r.stdout + r.stderr
        assert "1234 users" in r.stdout and "nnz" in r.stdout and "threshold" in r.stdout
        got = sp.load_npz(out)
        d2, v2, meta = load_generator(gen, torch.device("cuda"))
        kw = dict(kw)
        kw.setdefault("seed", 0)
        want, _ = sample_ddpm_sharded(1234, d2, v2, L, nd, n_timesteps=T, gather="csr", **kw)
        want = want.to_scipy()
        assert got.shape == want.shape and got.dtype == want.dtype
        assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)
        assert np.array_equal(got.data, want.data)
        os.remove(out)


def test_main_save_synthetic_and_generator(tmp_path, monkeypatch, capsys):
    """main.py --save-synthetic / --save-generator write the run's binarised rows and generators, and change nothing it returns."""
    import pickle

    import main as cli
    import sdrm_b200.train_SDRM as ts
    from helpers import random_modules
    from privacy_oracle import random_rows
    from sdrm_b200.synthesize import load_generator
    rng = np.random.default_rng(2)
    U, I = 150, 60
    train = sp.csr_matrix(random_rows(rng, U, I, 0.1).astype(np.float64))
    train[0, 59] = 0.0
    valid = sp.csr_matrix(random_rows(rng, 120, I, 0.15).astype(np.float64))
    os.makedirs(tmp_path / "ml-100k")
    for kind, mat in (("train_test", train), ("valid", valid)):
        with open(tmp_path / "ml-100k" / f"ml-100k_{kind}.pkl", "wb") as fh:
            pickle.dump(mat, fh)
    trained = []

    def fake_train(**kw):   # untrained modules: the test is about the files, not the model
        mods = random_modules(kw["N_ITEMS"], kw["VAE_HIDDEN"], kw["DIFF_LATENT"], kw["TIMESTEPS"], kw["N_HIDDEN_MLP_LAYERS"],
                              seed=4 + len(trained), device="cuda")
        trained.append(mods)
        return mods
    monkeypatch.setattr(ts, "train_SDRM", fake_train)
    monkeypatch.chdir(tmp_path)
    argv = ["--dataset", "ml-100k", "--data-dir", str(tmp_path), "--runs", "2", "--seed", "5", "--SDRM-timesteps", "6",
            "--MLP-latent-neurons", "16", "--VAE-hidden-layer-neurons", "24", "--MLP-hidden-layers", "1"]
    plain = cli.main(argv)
    out0 = capsys.readouterr().out
    trained.clear()
    recorded = []
    real_binarise = cli.binarise

    def recording_binarise(scores, sparsity):
        res = real_binarise(scores, sparsity)
        recorded.append(res[0])
        return res
    monkeypatch.setattr(cli, "binarise", recording_binarise)
    saved = cli.main(argv + ["--save-synthetic", str(tmp_path / "synth"), "--save-generator", str(tmp_path / "gen")])
    out1 = capsys.readouterr().out
    for c in cli.COLS:
        assert np.array_equal(plain[c], saved[c], equal_nan=True), c
    assert [ln for ln in out1.splitlines() if "took" not in ln] == [ln for ln in out0.splitlines() if "took" not in ln]
    sparsity = 1 - train.nnz / (U * I)
    assert len(recorded) == 6 and len(trained) == 2
    for run in (1, 2):
        dense = dict(zip(["M-SDRM", "F-SDRM", "MultiVAE++"], recorded[3 * (run - 1): 3 * run]))
        for name in cli.COLS:
            mat = sp.load_npz(tmp_path / "synth" / f"run{run}_{name}.npz")
            assert mat.format == "csr" and mat.shape == (U, I) and mat.has_canonical_format
            assert np.array_equal(mat.toarray(), dense[name]), (run, name)
        d2, v2, meta = load_generator(str(tmp_path / "gen" / f"run{run}_generator.pt"), torch.device("cuda"))
        assert meta["sparsity"] == sparsity and meta["T"] == 6 and meta["noise_divider"] == 0.5
        for a, b in zip(trained[run - 1], (d2, v2)):
            sa, sb = a.state_dict(), b.state_dict()
            assert sa.keys() == sb.keys() and all(torch.equal(sa[k], sb[k]) for k in sa)


# ------------------------------------------------------------------------------------------------------------------------------
# two GPUs
# ------------------------------------------------------------------------------------------------------------------------------
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


CASES = [   # (n, timesteps, seed, sparsity): full- and multi-resolution rows, and n = 1 (rank 1's block is empty)
    (301, None, 55, 0.9),
    (257, "random", 56, 0.95),
    (1, None, 57, 0.5),
]
SHAPE = (190, 48, 72, 6, 1, 1.0)   # I, H, L, T, nh, nd


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
        for n, ts_, seed, q in CASES:
            sr, span = sdd.sample_ddpm_sharded(n, dn, vae, L, nd, timesteps=ts_, n_timesteps=T, seed=seed, gather="csr", sparsity=q)
            res.append((span, sr.indptr.cpu(), sr.indices.cpu(), float(sr.threshold), sr.shape))
        torch.save(res, os.path.join(out_dir, f"rank{rank}.pt"))
    except Exception:
        import traceback
        with open(os.path.join(out_dir, f"rank{rank}.err"), "w") as fh:
            fh.write(traceback.format_exc())
        raise
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_rank_csr_gather():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from helpers import random_modules
    from sdrm_b200.sparsify import equal_sparsity_device
    from sdrm_b200.train_SDRM import sample_ddpm
    world = 2
    ctx = mp.get_context("spawn")
    port = _free_port()
    out_dir = tempfile.mkdtemp(prefix="sdrm_csr_gpu_")
    procs = [ctx.Process(target=_worker, args=(r, world, port, out_dir)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(280)
    for r, p in enumerate(procs):
        err = os.path.join(out_dir, f"rank{r}.err")
        assert p.exitcode == 0, open(err).read() if os.path.exists(err) else f"rank {r} exit code {p.exitcode}"
    res = [torch.load(os.path.join(out_dir, f"rank{r}.pt"), weights_only=False) for r in range(world)]
    I, H, L, T, nh, nd = SHAPE
    dn, vae = random_modules(I, H, L, T, nh, seed=3, device="cuda")
    for c, (n, ts_, seed, q) in enumerate(CASES):
        t_rows = np.random.RandomState(seed).randint(1, T, size=n).astype(np.int32) if ts_ == "random" else None
        whole = sample_ddpm(n, dn, vae, L, nd, timesteps=ts_, n_timesteps=T, seed=seed, t_rows=t_rows)
        pm = equal_sparsity_device(whole, q)
        want = pm.to_sparse()
        for rank in range(world):
            span, indptr, indices, thr, shape = res[rank][c]
            assert span == (0, n) and shape == (n, I)
            assert thr == float(pm.threshold), (c, rank)
            assert torch.equal(indptr, want.indptr.cpu()) and torch.equal(indices, want.indices.cpu()), (c, rank)
