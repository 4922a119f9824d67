"""GPU tests of the K8 nearest-rows search (sdrm_b200/privacy.py): index, intersection and union equal the test oracle bit for
bit on every shape, edge case and input format; the split + merge path and query shards give the same result as one launch."""
import os
import socket
import tempfile

import numpy as np
import pytest
import torch

from privacy_oracle import nearest_oracle, random_rows

pytestmark = pytest.mark.gpu


def _check(res, Q, R, k, exclude=False, offset=0):
    idx, c, u = nearest_oracle(Q, R, k, exclude_same_index=exclude, q_index_offset=offset, device="cuda")
    assert torch.equal(res.index.cpu(), idx)
    assert torch.equal(res.intersection.cpu(), c)
    assert torch.equal(res.union.cpu(), u)
    assert torch.equal(res.query_ones.cpu(), torch.as_tensor((np.asarray(Q) != 0).sum(1), dtype=torch.int32))


def _run(Q, R, k, **kw):
    from sdrm_b200.privacy import nearest_rows
    res = nearest_rows(Q, R, k=k, **kw)
    _check(res, Q, R, k, kw.get("exclude_same_index", False))
    return res


@pytest.mark.parametrize("k", [1, 2, 8, 16])
@pytest.mark.parametrize("items", [1, 31, 33, 127, 129, 729, 1008, 3125, 8582, 20000])
def test_items_and_k(items, k):
    rng = np.random.default_rng(items * 31 + k)
    density = min(0.5, max(0.02, 8.0 / items))
    Q, R = random_rows(rng, 129, items, density), random_rows(rng, 300, items, density)
    _run(Q, R, k)


@pytest.mark.parametrize("n,m,k", [(1, 1, 1), (1, 938, 16), (127, 128, 8), (128, 127, 2), (129, 129, 16), (843, 938, 8),
                                   (938, 843, 1), (5, 16, 16), (128, 1, 1)])
def test_row_counts(n, m, k):
    rng = np.random.default_rng(n * 1000 + m)
    _run(random_rows(rng, n, 200, 0.06), random_rows(rng, m, 200, 0.06), k)


@pytest.mark.parametrize("k", [1, 8])
def test_empty_rows_duplicates_and_ties(k):
    rng = np.random.default_rng(7)
    I = 300
    Q, R = random_rows(rng, 200, I, 0.05), random_rows(rng, 600, I, 0.05)
    Q[:5] = 0                     # empty queries: J = 1 to empty references, 0 to the rest (all tied)
    R[[3, 250, 257, 599]] = 0     # empty references, one per tile and at the end
    Q[10:20] = R[100:110]         # exact copies
    R[300:340] = R[120]           # 40 identical references: heavy ties across tile borders
    Q[20] = R[120]
    # many references at the same J against query 30: each holds one distinct item of the query's 4 and nothing else
    Q[30] = 0
    Q[30, :4] = 1
    R[400:480] = 0
    R[np.arange(400, 480), np.arange(80) % 4] = 1
    _run(Q, R, k)
    _run(R, Q, k)                 # empty rows on the other side
    z = np.zeros((3, I), dtype=np.uint8)
    _run(z, z, min(k, 3))         # only empty rows: u = 0 everywhere


@pytest.mark.parametrize("k", [1, 2, 8, 16])
def test_exclude_same_index(k):
    rng = np.random.default_rng(11)
    R = random_rows(rng, 700, 500, 0.05)
    R[50] = R[60]                 # a duplicate: row 50's best is 60 (and vice versa) once itself is excluded
    R[5] = 0
    R[6] = 0
    _run(R, R, k, exclude_same_index=True)
    _run(R[:300], R, k, exclude_same_index=True)     # fewer queries than references


@pytest.mark.parametrize("n,m,items,density", [(843, 938, 1008, 0.0575), (5429, 6034, 3125, 0.0447), (9558, 10621, 8582, 0.00115)])
@pytest.mark.parametrize("k", [1, 8])
def test_dataset_shapes(n, m, items, density, k):
    rng = np.random.default_rng(n + k)
    _run(random_rows(rng, n, items, density), random_rows(rng, m, items, density), k)


def _formats(D, rng):
    """The same 0/1 rows as every accepted input type, with the traps each format can carry."""
    import scipy.sparse as sp

    from sdrm_b200.sparsify import PackedMatrix
    from sdrm_b200.training import DeviceCSR
    rows, I = D.shape
    wpr = (I + 31) // 32
    packed = np.packbits(np.pad(D, ((0, 0), (0, 32 * wpr - I))), axis=1, bitorder="little").view(np.uint32)
    garbage = packed.copy()
    if I % 32:
        garbage[:, -1] |= np.uint32(0xFFFFFFFF) << np.uint32(I % 32)   # caller garbage past n_cols
    words = np.concatenate([garbage, np.full((rows, 1), 0xFFFFFFFF, dtype=np.uint32)], axis=1).view(np.int32)
    bits = torch.from_numpy(words).cuda()[:, :wpr]                     # a row-strided view
    pm = PackedMatrix(bits, I, 0.0, None)
    # CSR with unsorted indices, duplicated columns and explicit zeros (also on columns that hold no interaction)
    indptr, indices, data = [0], [], []
    for r in range(rows):
        cols = list(np.flatnonzero(D[r]))
        dup = cols[: len(cols) // 3]
        zeros = list(rng.choice(np.flatnonzero(D[r] == 0), size=min(3, int((D[r] == 0).sum())), replace=False))
        ent = [(c, 1.0) for c in cols + dup] + [(c, 0.0) for c in zeros]
        rng.shuffle(ent)
        indices += [e[0] for e in ent]
        data += [e[1] for e in ent]
        indptr.append(len(indices))
    csr = sp.csr_matrix((np.array(data, dtype=np.float64), np.array(indices, dtype=np.int32), np.array(indptr)), shape=D.shape)
    tcsr = torch.sparse_csr_tensor(torch.tensor(indptr), torch.tensor(indices), torch.tensor(data, dtype=torch.float32),
                                   size=D.shape).cuda()
    return {"packed": pm, "scipy": csr, "torch_csr": tcsr, "device_csr": DeviceCSR(csr, "cuda"),
            "dense_torch": torch.from_numpy(D.astype(np.float32) * 3).cuda(), "dense_numpy": D.astype(np.int64)}


def test_input_formats_agree():
    from sdrm_b200.privacy import nearest_rows
    rng = np.random.default_rng(3)
    I = 333
    Q, R = random_rows(rng, 150, I, 0.06), random_rows(rng, 420, I, 0.06)
    Q[0] = 0
    Q[1] = R[7]
    fq, fr = _formats(Q, rng), _formats(R, rng)
    first = None
    for a in fq:
        for b in (a, "dense_numpy"):
            res = nearest_rows(fq[a], fr[b], k=4)
            if first is None:
                _check(res, Q, R, 4)
                first = res
            for f in ("index", "intersection", "union", "query_ones"):
                assert torch.equal(getattr(res, f), getattr(first, f)), (a, b, f)


def test_split_merge_and_query_shards():
    from sdrm_b200.privacy import _image, _search
    rng = np.random.default_rng(17)
    I = 700
    Q, R = random_rows(rng, 300, I, 0.04), random_rows(rng, 2000, I, 0.04)
    Q[100:110] = R[50:60]
    qi, qo = _image(Q, "dense", 300, I, torch.device("cuda"))
    ri, ro = _image(R, "dense", 2000, I, torch.device("cuda"))
    for k in (1, 8, 16):
        one = _search(qi, qo, ri, ro, I, k, splits=1)
        for s in (0, 2, 3, 8):     # 8 reference tiles: up to one tile per CTA
            assert all(torch.equal(x, y) for x, y in zip(one, _search(qi, qo, ri, ro, I, k, splits=s))), (k, s)
        exc = _search(ri, ro, ri, ro, I, k, exclude_same_index=True, splits=1)
        a = _search(ri[:1111], ro[:1111], ri, ro, I, k, exclude_same_index=True, splits=3)
        b = _search(ri[1111:], ro[1111:], ri, ro, I, k, exclude_same_index=True, q_index_offset=1111)
        assert all(torch.equal(x, torch.cat([y, z])) for x, y, z in zip(exc, a, b)), k
        idx, c, u = nearest_oracle(R, R, k, exclude_same_index=True, device="cuda")
        assert torch.equal(exc[0].cpu(), idx) and torch.equal(exc[1].cpu(), c) and torch.equal(exc[2].cpu(), u)


def test_bad_csr_raises():
    from sdrm_b200.privacy import _csr_image, nearest_rows
    dev = torch.device("cuda")
    ok = torch.zeros((4, 10)).cuda()
    bad_index = torch.sparse_csr_tensor(torch.tensor([0, 1, 2, 2, 3]), torch.tensor([0, 10, 3]), torch.ones(3), size=(4, 10))
    with pytest.raises(ValueError, match="outside"):
        nearest_rows(bad_index, ok, k=1)
    with pytest.raises(ValueError, match="outside"):
        _csr_image(torch.tensor([0, 1]), torch.tensor([-1]), None, 1, 10, dev)
    with pytest.raises(ValueError, match="indptr"):
        _csr_image(torch.tensor([0, 2, 1]), torch.tensor([1, 2]), None, 2, 10, dev)
    with pytest.raises(ValueError, match="indptr"):
        _csr_image(torch.tensor([0, 1, 5]), torch.tensor([1, 2]), None, 2, 10, dev)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from sdrm_b200.privacy import nearest_rows
        rng = np.random.default_rng(23)
        R = random_rows(rng, 301, 257, 0.05)
        res = nearest_rows(R, R, k=3, exclude_same_index=True, group=dist.group.WORLD)
        torch.save((res.index.cpu(), res.intersection.cpu(), res.union.cpu()), os.path.join(out_dir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_rank_group():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    port, out_dir = _free_port(), tempfile.mkdtemp(prefix="sdrm_privacy_")
    procs = [ctx.Process(target=_worker, args=(r, 2, port, out_dir)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(280)
    assert all(p.exitcode == 0 for p in procs)
    R = random_rows(np.random.default_rng(23), 301, 257, 0.05)
    ref = nearest_oracle(R, R, 3, exclude_same_index=True, device="cuda")
    for r in range(2):
        got = torch.load(os.path.join(out_dir, f"rank{r}.pt"))
        assert all(torch.equal(x, y) for x, y in zip(got, ref))


def test_main_privacy_audit(tmp_path, monkeypatch, capsys):
    """main.py --privacy-audit prints the audit table; without the flag the run prints and returns what it did before."""
    import pickle

    import scipy.sparse as sp

    import main as cli
    import sdrm_b200.train_SDRM as ts
    from helpers import random_modules
    rng = np.random.default_rng(2)
    U, I = 150, 60
    train = sp.csr_matrix(random_rows(rng, U, I, 0.1).astype(np.float64))
    train[0, 59] = 0.0     # an explicit stored zero: it counts in SPARSITY like in the reference
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
    argv = ["--dataset", "ml-100k", "--data-dir", str(tmp_path), "--runs", "1", "--seed", "5", "--SDRM-timesteps", "6",
            "--MLP-latent-neurons", "16", "--VAE-hidden-layer-neurons", "24", "--MLP-hidden-layers", "1"]
    plain = cli.main(argv)
    out0 = capsys.readouterr().out
    audited = cli.main(argv + ["--privacy-audit"])
    out1 = capsys.readouterr().out
    for c in cli.COLS:
        assert np.array_equal(plain[c], audited[c], equal_nan=True), c
    assert "Privacy audit" not in out0
    lines = out1.splitlines()
    start = lines.index("Privacy audit (run 1): distance to the closest training row")
    block = lines[start:start + 7]
    assert all(name in block[i + 3] for i, name in enumerate(cli.COLS + ["real vs real (baseline)"])), block
    assert all(col in block[1] for col in cli.AUDIT_COLS)
    rest = lines[:start - 1] + lines[start + 7:]
    assert [ln for ln in rest if "took" not in ln] == [ln for ln in out0.splitlines() if "took" not in ln]
