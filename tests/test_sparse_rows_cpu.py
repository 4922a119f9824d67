"""CPU tests of the bits -> CSR path (K10, sparsify.packed_to_csr / PackedMatrix.to_sparse), the generator checkpoint and the
synthesize CLI: every check that needs no device."""
import ctypes

import numpy as np
import pytest
import torch

from sdrm_b200 import sparsify
from sdrm_b200.sparsify import PackedMatrix, packed_to_csr


@pytest.fixture(scope="module")
def lib():
    from sdrm_b200 import _lib
    from sdrm_b200.csrc import build
    build.build()
    return _lib.load()


def test_c_abi_host_checks(lib):
    """Bad arguments return SDRM_ERR_BAD_ARG (-1) before anything touches a device."""
    assert lib.sdrm_packed_csr_workspace_bytes(0) == 0 and lib.sdrm_packed_csr_workspace_bytes(-5) == 0
    assert lib.sdrm_packed_csr_workspace_bytes(1) == 8 and lib.sdrm_packed_csr_workspace_bytes(128) == 8
    assert lib.sdrm_packed_csr_workspace_bytes(129) == 16
    buf = ctypes.create_string_buffer(4096)
    p = ctypes.c_void_p((ctypes.addressof(buf) + 15) // 16 * 16)
    ind, ix = lib.sdrm_packed_csr_indptr, lib.sdrm_packed_csr_indices
    assert ind(None, 2, 4, 40, p, p, 4096, None) == -1 and b"d_words" in lib.sdrm_last_error()
    assert ind(p, 2, 4, 40, None, p, 4096, None) == -1 and b"d_indptr" in lib.sdrm_last_error()
    assert ind(p, 2, 4, 40, p, None, 4096, None) == -1 and b"d_workspace" in lib.sdrm_last_error()
    assert ind(p, 2, 4, 0, p, p, 4096, None) == -1                  # n_cols < 1
    assert ind(p, 2, 4, -3, p, p, 4096, None) == -1
    assert ind(p, 1, 4, 33, p, p, 4096, None) == -1                 # words_ld < ceil(33 / 32)
    assert b"words_ld" in lib.sdrm_last_error()
    assert ind(p, 2, -1, 40, p, p, 4096, None) == -1                # rows < 0
    assert ind(p, 2, 200, 40, p, p, 8, None) == -5                  # workspace below sdrm_packed_csr_workspace_bytes(200)
    assert ix(None, 2, 4, 40, p, p, None) == -1
    assert ix(p, 2, 4, 40, None, p, None) == -1
    assert ix(p, 2, 4, 40, p, None, None) == -1
    assert ix(p, 2, 4, 0, p, p, None) == -1
    assert ix(p, 1, 4, 33, p, p, None) == -1
    assert ix(p, 2, -2, 40, p, p, None) == -1
    assert ix(None, 1, 0, 1, None, None, None) == 0                 # zero rows: nothing to do, no pointer needed


def test_python_argument_errors_before_any_launch():
    ok = torch.zeros((3, 2), dtype=torch.int32)
    with pytest.raises(TypeError):
        packed_to_csr(np.zeros((3, 2), dtype=np.int32), 40)
    with pytest.raises(ValueError):
        packed_to_csr(ok.to(torch.int64), 40)
    with pytest.raises(ValueError):
        packed_to_csr(torch.zeros((3, 2, 1), dtype=torch.int32), 40)
    with pytest.raises(ValueError):
        packed_to_csr(torch.zeros((2, 3), dtype=torch.int32).t(), 40)   # word stride != 1
    with pytest.raises(ValueError, match="words per row"):
        packed_to_csr(ok, 65)
    for bad in (0, -1, 2 ** 31):
        with pytest.raises(ValueError):
            packed_to_csr(ok, bad)
    for bad in (40.0, True, "40"):
        with pytest.raises(TypeError):
            packed_to_csr(ok, bad)


def test_no_cpu_fallback():
    from sdrm_b200 import _lib
    with pytest.raises(_lib.SdrmError):
        packed_to_csr(torch.zeros((3, 2), dtype=torch.int32), 40)
    with pytest.raises(_lib.SdrmError):
        PackedMatrix(torch.zeros((3, 2), dtype=torch.int32), 40, 0.5, None).to_sparse()


def test_sparse_rows_shape_and_nnz():
    sr = sparsify.SparseRows(torch.tensor([0, 2, 2, 5]), torch.tensor([1, 4, 0, 3, 9], dtype=torch.int32), 10, threshold=0.25)
    assert sr.shape == (3, 10) and sr.nnz == 5 and sr.threshold == 0.25


def _modules(nh=2, L=12, H=20, I=30, T=7, D=None, seed=0):
    from sdrm_b200.models import SDRM, VAE
    torch.manual_seed(seed)
    return SDRM(N_ITEMS=L, EMB_DIM=T, LATENT_DIM=D or L, n_hidden_layers=nh), VAE(I, H, L, p_drop=0.3)


@pytest.mark.parametrize("nh,D", [(0, None), (2, None), (1, 17)])
def test_generator_round_trip_cpu(tmp_path, nh, D):
    from sdrm_b200.models import make_schedule
    from sdrm_b200.synthesize import load_generator, save_generator
    diff, vae = _modules(nh=nh, D=D)
    path = save_generator(str(tmp_path / "g.pt"), diff, vae, noise_divider=0.5, sparsity=0.9425)
    d2, v2, meta = load_generator(path, "cpu")
    assert meta["T"] == 7 and meta["noise_divider"] == 0.5 and meta["sparsity"] == 0.9425
    assert meta["sdrm_args"] == dict(N_ITEMS=12, EMB_DIM=7, LATENT_DIM=D or 12, n_hidden_layers=nh)
    assert meta["vae_args"] == dict(input_dim=30, hidden_dim=20, latent_dim=12, p_drop=0.3)
    assert (d2.N_ITEMS, d2.EMB_DIM, d2.LATENT_DIM, d2.n_hidden_layers) == (12, 7, D or 12, nh)
    assert (v2.input_dim, v2.hidden_dim, v2.latent_dim, v2.dropout.p) == (30, 20, 12, 0.3)
    for a, b in ((diff, d2), (vae, v2)):
        sa, sb = a.state_dict(), b.state_dict()
        assert sa.keys() == sb.keys()
        assert all(torch.equal(sa[k], sb[k]) for k in sa)
    if nh > 1:   # the shared hidden layer stays one module pair
        assert d2.dnn[2] is d2.dnn[4]
    assert not d2.training and not v2.training
    for x, y in zip(d2.sdrm_schedule, make_schedule(7, device="cpu")):
        assert torch.equal(x, y)


def test_load_generator_rejects_other_files(tmp_path):
    from sdrm_b200.synthesize import load_generator
    torch.save({"weights": torch.zeros(3)}, tmp_path / "x.pt")
    with pytest.raises(ValueError, match="not an SDRM generator"):
        load_generator(str(tmp_path / "x.pt"), "cpu")
    torch.save({"format": "sdrm_b200.generator", "version": 99}, tmp_path / "y.pt")
    with pytest.raises(ValueError, match="version"):
        load_generator(str(tmp_path / "y.pt"), "cpu")


def test_cli_parses_and_rejects_bad_flags():
    from sdrm_b200.synthesize import parse_args
    a = parse_args(["--generator", "g.pt", "--users", "100", "--out", "x.npz"])
    assert (a.seed, a.multi_resolution, a.sampling_steps, a.eta, a.bf16, a.sparsity) == (0, False, None, None, False, None)
    a = parse_args(["--generator", "g.pt", "--users", "7", "--out", "x.npz", "--seed", "3", "--multi-resolution",
                    "--sampling-steps", "5", "--eta", "0.5", "--bf16", "--sparsity", "0.99"])
    assert (a.users, a.seed, a.multi_resolution, a.sampling_steps, a.eta, a.bf16, a.sparsity) == (7, 3, True, 5, 0.5, True, 0.99)
    base = ["--generator", "g.pt", "--users", "10", "--out", "x.npz"]
    for bad in ([], ["--users", "10", "--out", "x.npz"], base[:4], base[2:],
                base[:3] + ["0"] + base[4:], base[:3] + ["ten"] + base[4:], base[:5] + ["x.csv"],
                base + ["--sparsity", "1.5"], base + ["--sparsity", "-0.1"], base + ["--eta", "2"],
                base + ["--sampling-steps", "0"], base + ["--seed", "1.5"], base + ["--unknown"]):
        with pytest.raises(SystemExit):
            parse_args(bad)


def test_cli_no_cpu_fallback(tmp_path):
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from sdrm_b200 import _lib
    from sdrm_b200.synthesize import main
    with pytest.raises(_lib.SdrmError):
        main(["--generator", str(tmp_path / "g.pt"), "--users", "3", "--out", str(tmp_path / "x.npz")])
    assert not (tmp_path / "x.npz").exists()


def test_sharded_csr_needs_sparsity_before_sampling():
    from sdrm_b200.distributed import sample_ddpm_sharded

    def sampler(*a, **k):
        raise AssertionError("sampled before the argument check")
    with pytest.raises(ValueError, match="sparsity"):
        sample_ddpm_sharded(10, None, None, 8, seed=1, gather="csr", sampler=sampler)


def test_main_flags_default_off():
    import main as cli
    a = cli.build_parser().parse_args([])
    assert a.save_generator is None and a.save_synthetic is None
    a = cli.build_parser().parse_args(["--save-generator", "g", "--save-synthetic", "s"])
    assert (a.save_generator, a.save_synthetic) == ("g", "s")
