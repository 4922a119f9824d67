"""GPU tests of the fidelity audit (sdrm_b200/fidelity.py): the item-major prep is bit-exact, K9's six sums match the float64
oracle on every shape, exact cases hold exactly, the item neighbours equal the K8 oracle, every input format gives the same
report, and main.py --fidelity-audit changes nothing else a run prints or returns."""
import math
import os

import numpy as np
import pytest
import torch

from fidelity_oracle import pair_sums, report
from privacy_oracle import nearest_oracle, random_rows
from test_privacy_gpu import _formats

pytestmark = pytest.mark.gpu


def _image(X, kind="dense"):
    from sdrm_b200.fidelity import _item_image
    U, I = X.shape
    return _item_image(X, kind, U, I, torch.device("cuda"))


def _expected_image(D):
    """Item-major 0/1 image of dense rows D [users, items] with K8's pitch over the users."""
    U, I = D.shape
    pitch = (U + 127) // 128 * 128
    img = torch.zeros((I, pitch), dtype=torch.uint8)
    img[:, :U] = torch.from_numpy((np.asarray(D) != 0).T.astype(np.uint8))
    return img


@pytest.mark.parametrize("users", [1, 127, 128, 129, 5000])
@pytest.mark.parametrize("items", [1, 45, 300])
def test_prep_bit_exact(users, items):
    rng = np.random.default_rng(users * 7 + items)
    D = random_rows(rng, users, items, 0.2)
    fmts = _formats(D, rng)   # packed rows with garbage past n_cols, CSR with explicit zeros, duplicates and unsorted indices
    want = _expected_image(D)
    item_ones = torch.from_numpy(D.sum(0).astype(np.int32))
    user_ones = torch.from_numpy(D.sum(1).astype(np.int32))
    kinds = {"packed": "bits", "scipy": "scipy", "torch_csr": "torch_csr", "device_csr": "device_csr", "dense_torch": "dense",
             "dense_numpy": "dense"}
    for name, x in fmts.items():
        img, io, uo = _image(x, kinds[name])
        assert torch.equal(img.cpu(), want), name
        assert torch.equal(io.cpu(), item_ones), name
        assert torch.equal(uo.cpu(), user_ones), name


def test_bad_csr_raises():
    from sdrm_b200.fidelity import compare
    ok = torch.zeros((4, 10)).cuda()
    bad_index = torch.sparse_csr_tensor(torch.tensor([0, 1, 2, 2, 3]), torch.tensor([0, 10, 3]), torch.ones(3), size=(4, 10))
    with pytest.raises(ValueError, match="outside"):
        compare(bad_index, ok, k=None)
    neg = torch.sparse_csr_tensor(torch.tensor([0, 1]), torch.tensor([-1]), torch.ones(1), size=(1, 10), check_invariants=False)
    with pytest.raises(ValueError, match="outside"):
        compare(ok, neg, k=None)
    for indptr in ([0, 2, 1], [0, 1, 5]):
        bad = torch.sparse_csr_tensor(torch.tensor(indptr), torch.tensor([1, 2]), torch.ones(2), size=(2, 10),
                                      check_invariants=False)
        with pytest.raises(ValueError, match="indptr"):
            compare(bad, ok, k=None)


def _check_sums(rep, R, S):
    P = R.shape[1] * (R.shape[1] - 1) / 2
    ref = pair_sums(R, S, device="cuda")
    assert torch.allclose(rep.sums.cpu(), ref, rtol=0, atol=1e-9 * max(1.0, P)), (rep.sums.cpu(), ref)


@pytest.mark.parametrize("items", [1, 2, 127, 128, 129, 300, 1000])
def test_sums_against_oracle(items):
    from sdrm_b200.fidelity import compare
    rng = np.random.default_rng(items)
    R, S = random_rows(rng, 700, items, 0.08), random_rows(rng, 333, items, 0.12)
    if items > 4:
        R[:, 1] = 0            # constant items in one set only
        S[:, 2] = 1
        R[:, items - 1] = 1
    rep = compare(R, S, k=None if items == 1 else min(10, items - 1))
    _check_sums(rep, R, S)
    assert torch.equal(rep.item_ones_real.cpu(), torch.from_numpy(R.sum(0).astype(np.int32)))
    assert torch.equal(rep.user_ones_synth.cpu(), torch.from_numpy(S.sum(1).astype(np.int32)))


def test_exact_cases():
    from sdrm_b200.fidelity import compare
    rng = np.random.default_rng(5)
    X, Y = random_rows(rng, 500, 400, 0.05), random_rows(rng, 650, 400, 0.07)
    X[:, 7] = 0
    same = compare(X, X, k=5)
    assert float(same.sums[0]) == 0.0
    s = same.summary()
    assert s["phi_pcd"] == 0.0 and abs(s["phi_corr"] - 1.0) < 1e-12 and s["neighbour_recall_at_k"] == 1.0
    a, b = compare(X, Y, k=None), compare(X, Y, k=None)
    assert torch.equal(a.sums, b.sums)            # bit-identical from call to call
    sw = compare(Y, X, k=None).sums.cpu()
    ab = a.sums.cpu()
    assert sw[0] == ab[0] and sw[5] == ab[5]      # S_dd and S_rs
    assert sw[1] == ab[2] and sw[2] == ab[1] and sw[3] == ab[4] and sw[4] == ab[3]


def test_neighbours_against_oracle():
    from sdrm_b200.fidelity import compare
    rng = np.random.default_rng(9)
    R, S = random_rows(rng, 400, 260, 0.05), random_rows(rng, 300, 260, 0.06)
    R[:, 10] = 0
    R[:, 11] = R[:, 12]
    for k in (1, 8, 16):
        rep = compare(R, S, k=k)
        for nb, X in ((rep.neighbours_real, R), (rep.neighbours_synth, S)):
            idx, c, u = nearest_oracle(X.T, X.T, k, exclude_same_index=True, device="cuda")
            assert torch.equal(nb.index.cpu(), idx) and torch.equal(nb.intersection.cpu(), c) and torch.equal(nb.union.cpu(), u)
        want = report(R, S, k=k, device="cuda").summary()["neighbour_recall_at_k"]
        assert rep.summary()["neighbour_recall_at_k"] == pytest.approx(want, abs=1e-15)


def test_input_formats_agree():
    from sdrm_b200.fidelity import compare
    rng = np.random.default_rng(3)
    R, S = random_rows(rng, 260, 333, 0.06), random_rows(rng, 150, 333, 0.06)
    fr, fs = _formats(R, rng), _formats(S, rng)
    first = None
    for a in fr:
        for b in (a, "dense_numpy"):
            rep = compare(fr[a], fs[b], k=4)
            if first is None:
                _check_sums(rep, R, S)
                first = rep
            assert torch.equal(rep.sums, first.sums), (a, b)
            for f in ("item_ones_real", "item_ones_synth", "user_ones_real", "user_ones_synth"):
                assert torch.equal(getattr(rep, f), getattr(first, f)), (a, b, f)
            for f in ("index", "intersection", "union"):
                assert torch.equal(getattr(rep.neighbours_real, f), getattr(first.neighbours_real, f)), (a, b, f)
                assert torch.equal(getattr(rep.neighbours_synth, f), getattr(first.neighbours_synth, f)), (a, b, f)


@pytest.mark.parametrize("ur,us,items,density", [(938, 843, 1008, 0.0575), (10621, 9558, 8582, 0.00115)])
def test_dataset_shapes(ur, us, items, density):
    from sdrm_b200.fidelity import compare
    rng = np.random.default_rng(ur)
    R, S = random_rows(rng, ur, items, density), random_rows(rng, us, items, density)
    got = compare(R, S, k=10).summary()
    want = report(R, S, k=10, device="cuda").summary()
    P = items * (items - 1) / 2
    assert got.keys() == want.keys()
    for key in got:
        if isinstance(want[key], float) and math.isnan(want[key]):
            assert math.isnan(got[key]), key
        elif key.startswith("phi"):
            assert got[key] == pytest.approx(want[key], rel=1e-9, abs=1e-9 * P), key
        else:
            assert got[key] == pytest.approx(want[key], rel=1e-12, abs=1e-15), key


def test_main_fidelity_audit(tmp_path, monkeypatch, capsys):
    """main.py --fidelity-audit prints the audit table; without the flag the run prints and returns what it did before."""
    import pickle

    import scipy.sparse as sp

    import main as cli
    import sdrm_b200.train_SDRM as ts
    from helpers import random_modules
    rng = np.random.default_rng(2)
    U, I = 150, 60
    train = sp.csr_matrix(random_rows(rng, U, I, 0.1).astype(np.float64))
    train[0, 59] = 0.0
    valid = sp.csr_matrix(random_rows(rng, 120, I, 0.15).astype(np.float64))
    os.makedirs(tmp_path / "ml-100k")
    for kind, mat in (("train_test", train), ("valid", valid)):
        with open(tmp_path / "ml-100k" / f"ml-100k_{kind}.pkl", "wb") as fh:
            pickle.dump(mat, fh)

    def fake_train(**kw):   # untrained modules: the test is about the audit, not the model
        return random_modules(kw["N_ITEMS"], kw["VAE_HIDDEN"], kw["DIFF_LATENT"], kw["TIMESTEPS"], kw["N_HIDDEN_MLP_LAYERS"],
                              seed=4, device="cuda")
    monkeypatch.setattr(ts, "train_SDRM", fake_train)
    monkeypatch.chdir(tmp_path)
    argv = ["--dataset", "ml-100k", "--data-dir", str(tmp_path), "--runs", "2", "--seed", "5", "--SDRM-timesteps", "6",
            "--MLP-latent-neurons", "16", "--VAE-hidden-layer-neurons", "24", "--MLP-hidden-layers", "1"]
    plain = cli.main(argv)
    out0 = capsys.readouterr().out
    audited = cli.main(argv + ["--fidelity-audit"])
    out1 = capsys.readouterr().out
    for c in cli.COLS:
        assert np.array_equal(plain[c], audited[c], equal_nan=True), c
    assert "Fidelity audit" not in out0
    lines = out1.splitlines()
    rest = lines
    for run in (1, 2):
        start = rest.index(f"Fidelity audit (run {run}): synthetic rows against the training rows")
        block = rest[start:start + 7]
        assert all(name in block[i + 3] for i, name in enumerate(cli.COLS + ["real split-half (baseline)"])), block
        assert all(col in block[1] for col in cli.FIDELITY_COLS)
        rest = rest[:start - 1] + rest[start + 7:]
    assert [ln for ln in rest if "took" not in ln] == [ln for ln in out0.splitlines() if "took" not in ln]
