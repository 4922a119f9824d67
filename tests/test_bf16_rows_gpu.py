"""bfloat16 synthetic rows: sdrm_sample_bf16 on every data flow of the sampler kernels (K6, and K1's single CTAs, pairs, pairs with
several tiles per CTA, column split of 8 / 4, resident and interleaved sub-tiles), in every placement the fp32 path accepts, through
sample_ddpm / sample_ddpm_host / sample_ddpm_sharded, and K4 equal-sparsity thresholding of bfloat16 score matrices.

The contract: every bfloat16 logit is the round-to-nearest-even bfloat16 of the fp32 logit of the same rows, seed and start steps,
bit for bit (out_bf16.view(int16) == out_fp32.to(torch.bfloat16).view(int16)); the latent output stays fp32 and unchanged.  K4 on
bfloat16 scores: threshold bit-identical to np.quantile(S.astype(np.float32).flatten(), q), bits equal to S >= thr (<= thr)."""
import os
import re

import numpy as np
import pytest
import torch

from helpers import random_modules
from sdrm_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BF16_ENTRIES = ("sdrm_sample_bf16", "sdrm_key_histogram_bf16", "sdrm_threshold_pack_bf16", "sdrm_select_histogram_bf16",
                "sdrm_select_walk_bf16", "sdrm_select_threshold_pack_bf16")


def _bits16(t):
    return t.cpu().view(torch.int16)


def _rounded(fp32):
    return _bits16(fp32.to(torch.bfloat16))


# ------------------------------------------------------------------------------------------------------------------------------
# CPU: header / binding table, the bfloat16 radix-select digits, argument checks that need no device
# ------------------------------------------------------------------------------------------------------------------------------
def test_header_declares_the_bf16_entries():
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "sdrm_b200.h")).read(), flags=re.S)
    for name in BF16_ENTRIES:
        assert re.search(r"\b%s\s*\(" % name, text), name
        assert name in _lib.SIGNATURES, name
    # the same arguments as the fp32 entries (only the pointer type of the scores / logits differs)
    assert _lib.SIGNATURES["sdrm_sample_bf16"] == _lib.SIGNATURES["sdrm_sample"]
    for base in ("sdrm_key_histogram", "sdrm_threshold_pack", "sdrm_select_histogram", "sdrm_select_walk", "sdrm_select_threshold_pack"):
        assert _lib.SIGNATURES[base + "_bf16"] == _lib.SIGNATURES[base], base
    assert re.search(r"sdrm_sample_bf16\([^;]*uint16_t\* d_logits", text)


def _np_keys(f32):
    u = f32.view(np.uint32).astype(np.uint64)
    return np.where(u & 0x80000000, ~u & 0xFFFFFFFF, u | 0x80000000).astype(np.uint64)


def test_select_ranks_with_the_bf16_digits():
    """Host radix select over two digits (11 + 5 bits) of float32 keys of bfloat16 values: every order statistic exact."""
    from sdrm_b200.sparsify import _DIGITS_BF16, select_ranks
    rng = np.random.RandomState(3)
    vals = torch.from_numpy(np.concatenate([rng.randn(3000) * 5, rng.randint(-3, 4, size=2000), [0.0, -0.0, np.inf, -np.inf, 1e-40, -1e-40]])
                            .astype(np.float32)).to(torch.bfloat16).float().numpy()
    keys = _np_keys(vals)

    def hist_fn(prefix, prefix_bits, shift, bits):
        sel = keys if prefix_bits == 0 else keys[(keys >> np.uint64(32 - prefix_bits)) == prefix]
        return np.bincount(((sel >> np.uint64(shift)) & np.uint64((1 << bits) - 1)).astype(np.int64), minlength=2048)
    srt = np.sort(vals)
    ranks = [0, 1, 17, 2500, 4999, len(vals) - 2, len(vals) - 1]
    got = select_ranks(hist_fn, ranks, _DIGITS_BF16)
    for r, g in zip(ranks, got):
        assert np.float32(g).view(np.uint32) == srt[r].view(np.uint32) or (g == 0 and srt[r] == 0), (r, g, srt[r])


def test_argument_checks_without_a_device():
    from sdrm_b200.sparsify import equal_sparsity_device, threshold_pack
    from sdrm_b200.train_SDRM import sample_ddpm, sample_ddpm_host
    with pytest.raises(ValueError):
        sample_ddpm(4, None, None, 8, out_dtype=torch.float16)
    with pytest.raises(ValueError):
        sample_ddpm(4, None, None, 8, out=torch.empty(4, 8), out_dtype=torch.bfloat16)
    with pytest.raises(ValueError):
        sample_ddpm_host(4, None, None, 8, host_out=torch.empty(4, 8), out_dtype=torch.bfloat16)
    for f in (lambda s: equal_sparsity_device(s, 0.9), lambda s: threshold_pack(s, 0.0)):
        with pytest.raises(_lib.SdrmError):
            f(torch.zeros(4, 8, dtype=torch.bfloat16))


# ------------------------------------------------------------------------------------------------------------------------------
# GPU A. every data flow, full and multi resolution, item counts of every residue class that matters to the store paths
# ------------------------------------------------------------------------------------------------------------------------------
# I, H, L, T, nh, nd: "k1" is wider than 64 (K1 and the column split), "k6" has every width <= 64
KINDS = {"k1": (150, 200, 7, 2, 1.0), "k6": (48, 40, 7, 2, 1.0)}
ITEMS = (336, 729, 730, 1004, 333, 8582)   # I % 8 = 0, 1, 2, 4, 5, 6


def _model(kind, I, seed):
    from test_sampler_gpu import _engine
    H, L, T, nh, nd = KINDS[kind]
    diff, vae = random_modules(I, H, L, T, nh, seed=seed, device="cuda")
    return diff, vae, _engine(diff, vae, T, nd)


def _flows(kind, multires):
    from test_sampler_edges_gpu import FULLRES_K1, MULTIRES_K1, NARROW_FLOWS
    if kind == "k6":
        return NARROW_FLOWS
    return MULTIRES_K1 if multires else FULLRES_K1


def _multires_inputs(n, T, seed=7):
    """the public call's layout: sorted start steps (longest first) with whole tiles of zero start steps, and row_ids"""
    rng = np.random.RandomState(seed)
    t = rng.randint(1, T + 1, size=n)
    t[rng.rand(n) < 0.45] = 0
    order = np.argsort(-t, kind="stable")
    return torch.from_numpy(t[order].astype(np.int32)).cuda(), torch.from_numpy(order.astype(np.int32)).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("I", ITEMS)
@pytest.mark.parametrize("kind", ["k1", "k6"])
def test_every_flow_bf16_rows_are_the_rounded_fp32_rows(kind, I):
    from test_sampler_edges_gpu import _run
    H, L, T, nh, nd = KINDS[kind]
    n = 300                                                   # 3 row tiles, the last one ragged (44 rows)
    diff, vae, eng = _model(kind, I, seed=40 + I % 8)
    ts, rid = _multires_inputs(n, T)
    for mode, kw in (("full", {}), ("multires", {"t_start": ts, "row_ids": rid})):
        for flow in _flows(kind, mode == "multires"):
            lat32, lat16 = torch.empty(n, L, device="cuda"), torch.empty(n, L, device="cuda")
            ref = _run(eng, flow, n, seed=91, row_offset=1000, latent_out=lat32, **kw)
            out = torch.empty(n, I, dtype=torch.bfloat16, device="cuda")
            got = _run(eng, flow, n, seed=91, row_offset=1000, latent_out=lat16, out=out, **kw)
            assert got.data_ptr() == out.data_ptr() and got.dtype == torch.bfloat16
            assert torch.isfinite(ref).all(), (mode, flow)
            assert torch.equal(_bits16(got), _rounded(ref)), (mode, flow, int((_bits16(got) != _rounded(ref)).sum()))
            assert torch.equal(lat16.cpu().view(torch.int32), lat32.cpu().view(torch.int32)), (mode, flow)


# ------------------------------------------------------------------------------------------------------------------------------
# GPU B. placement: bf16 logits into views of a larger buffer; values equal a contiguous launch, nothing outside the view written
# ------------------------------------------------------------------------------------------------------------------------------
PLACEMENTS = {   # name: (first column of the view, leading dimension - I)  for I = 333
    "misaligned": (1, 3),      # ld = 336 (a multiple of 8), base 2 bytes past a 16-byte boundary
    "odd_ld": (0, 4),          # ld = 337
    "aligned_wide": (8, 27),   # ld = 360, base 16-byte aligned: the vector store path (up to the ragged last group)
}
SENTINEL16 = 0x7FAB            # a bfloat16 NaN payload no kernel produces: compared as bits


@pytest.mark.gpu
@pytest.mark.parametrize("placement", sorted(PLACEMENTS))
@pytest.mark.parametrize("kind", ["k1", "k6"])
def test_bf16_output_placement_and_guards(kind, placement):
    from test_sampler_edges_gpu import _run
    I = 333
    H, L, T, nh, nd = KINDS[kind]
    n = 300
    diff, vae, eng = _model(kind, I, seed=32)
    c0, extra = PLACEMENTS[placement]
    ld = I + extra
    rng = np.random.RandomState(5)
    ts = torch.from_numpy(rng.randint(1, T + 1, size=n).astype(np.int32)).cuda()
    perm = torch.from_numpy(rng.permutation(n).astype(np.int32)).cuda()
    for vname, (kw, multires) in {"full": ({}, False), "multires_row_ids": ({"t_start": ts, "row_ids": perm}, True)}.items():
        for flow in _flows(kind, multires):
            ref = _run(eng, flow, n, seed=44, out=torch.empty(n, I, dtype=torch.bfloat16, device="cuda"), **kw).clone()
            buf = torch.full((n + 2, ld), SENTINEL16, dtype=torch.int16, device="cuda").view(torch.bfloat16)
            view = buf[1:n + 1, c0:c0 + I]
            assert view.stride(0) == ld
            got = _run(eng, flow, n, seed=44, out=view, **kw)
            assert got.data_ptr() == view.data_ptr()
            assert torch.equal(_bits16(view), _bits16(ref)), (vname, flow)
            b = _bits16(buf)
            inside = torch.zeros_like(b, dtype=torch.bool)
            inside[1:n + 1, c0:c0 + I] = True
            assert (b[~inside] == SENTINEL16).all(), (vname, flow, int((b[~inside] != SENTINEL16).sum()))


# ------------------------------------------------------------------------------------------------------------------------------
# GPU C. the public calls: sample_ddpm, sample_ddpm_host (one and several chunks), sample_ddpm_sharded (three gather modes)
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("chunk_rows", [None, 300])
def test_host_and_sharded_paths_in_bf16(chunk_rows):
    from sdrm_b200.distributed import sample_ddpm_sharded
    from sdrm_b200.sparsify import equal_sparsity_device
    from sdrm_b200.train_SDRM import sample_ddpm, sample_ddpm_host
    I, (H, L, T, nh, nd) = 729, KINDS["k1"]
    n, seed, off = 1000, 0x5EED6, 321
    diff, vae = random_modules(I, H, L, T, nh, seed=35, device="cuda")
    ref32 = sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, row_offset=off)
    ref = sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, row_offset=off, out_dtype=torch.bfloat16)
    assert ref.dtype == torch.bfloat16 and torch.equal(_bits16(ref), _rounded(ref32))
    got = sample_ddpm_host(n, diff, vae, L, nd, n_timesteps=T, seed=seed, row_offset=off, chunk_rows=chunk_rows, out_dtype=torch.bfloat16)
    assert got.device.type == "cpu" and got.dtype == torch.bfloat16 and torch.equal(_bits16(got), _bits16(ref))
    host = torch.full((n, I), float("nan"), dtype=torch.bfloat16)
    assert sample_ddpm_host(n, diff, vae, L, nd, n_timesteps=T, seed=seed, row_offset=off, host_out=host, chunk_rows=chunk_rows) is host
    assert torch.equal(_bits16(host), _bits16(ref))
    # the fp32 host path behind the same engine still gives fp32 rows (the chunk buffers follow the dtype)
    assert torch.equal(sample_ddpm_host(n, diff, vae, L, nd, n_timesteps=T, seed=seed, row_offset=off, chunk_rows=chunk_rows), ref32.cpu())
    if chunk_rows is not None:
        return
    ref0 = sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, out_dtype=torch.bfloat16)
    rows, span = sample_ddpm_sharded(n, diff, vae, L, nd, n_timesteps=T, seed=seed, out_dtype=torch.bfloat16)
    assert span == (0, n) and torch.equal(_bits16(rows), _bits16(ref0))
    rows, span = sample_ddpm_sharded(n, diff, vae, L, nd, n_timesteps=T, seed=seed, out_dtype=torch.bfloat16, gather=True)
    assert span == (0, n) and torch.equal(_bits16(rows), _bits16(ref0))
    pm, span = sample_ddpm_sharded(n, diff, vae, L, nd, n_timesteps=T, seed=seed, out_dtype=torch.bfloat16, gather="bits", sparsity=0.95)
    pm1 = equal_sparsity_device(ref0, 0.95)
    assert float(pm.threshold) == float(pm1.threshold) and torch.equal(pm.bits, pm1.bits)
    assert int(pm.ones.item()) == int(pm1.ones.item())
    thr = np.quantile(ref0.float().cpu().numpy().flatten(), 0.95)
    assert np.float32(pm.threshold).view(np.uint32) == np.float32(thr).view(np.uint32)


def _two_rank_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from sdrm_b200 import distributed as sdd
        I, (H, L, T, nh, nd) = 729, KINDS["k1"]
        dn, vae = random_modules(I, H, L, T, nh, seed=3, device=dev)
        pm, _ = sdd.sample_ddpm_sharded(301, dn, vae, L, nd, n_timesteps=T, seed=55, gather="bits", sparsity=0.9,
                                        out_dtype=torch.bfloat16)
        rows, _ = sdd.sample_ddpm_sharded(301, dn, vae, L, nd, n_timesteps=T, seed=55, gather=True, out_dtype=torch.bfloat16)
        torch.save((pm.bits.cpu(), float(pm.threshold), int(pm.ones.item()), rows.cpu()), os.path.join(out_dir, f"rank{rank}.pt"))
    except Exception:
        import traceback
        with open(os.path.join(out_dir, f"rank{rank}.err"), "w") as fh:
            fh.write(traceback.format_exc())
        raise
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.timeout(300)
def test_two_rank_bf16_bits_use_the_global_threshold():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import tempfile
    import torch.multiprocessing as mp
    from test_distributed_gpu import _free_port
    from sdrm_b200.sparsify import equal_sparsity_device
    from sdrm_b200.train_SDRM import sample_ddpm
    ctx = mp.get_context("spawn")
    out_dir = tempfile.mkdtemp(prefix="sdrm_bf16_2gpu_")
    port = _free_port()
    procs = [ctx.Process(target=_two_rank_worker, args=(r, 2, port, out_dir)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(280)
    for r, p in enumerate(procs):
        err = os.path.join(out_dir, f"rank{r}.err")
        assert p.exitcode == 0, open(err).read() if os.path.exists(err) else f"rank {r} exit code {p.exitcode}"
    I, (H, L, T, nh, nd) = 729, KINDS["k1"]
    dn, vae = random_modules(I, H, L, T, nh, seed=3, device="cuda")
    whole = sample_ddpm(301, dn, vae, L, nd, n_timesteps=T, seed=55, out_dtype=torch.bfloat16)
    pm1 = equal_sparsity_device(whole, 0.9)
    for r in range(2):
        bits, thr, ones, rows = torch.load(os.path.join(out_dir, f"rank{r}.pt"), weights_only=False)
        assert torch.equal(_bits16(rows), _bits16(whole))
        assert thr == float(pm1.threshold) and ones == int(pm1.ones.item()) and torch.equal(bits, pm1.bits.cpu())


# ------------------------------------------------------------------------------------------------------------------------------
# GPU D. K4 on bfloat16 scores
# ------------------------------------------------------------------------------------------------------------------------------
QS = (0.0, 1.0, 0.5, 0.99, 0.937, 0.955, 0.9, 0.123)


def _scores(name, rng):
    if name == "normal":
        a = rng.randn(300, 333) * 3
    elif name == "ties":          # a handful of distinct values: bfloat16 makes ties common, here every score is one
        a = rng.randint(-4, 5, size=(257, 130)) * 0.25
    elif name == "specials":      # +-0, negatives, +-inf, subnormals
        a = rng.randn(129, 77)
        flat = a.reshape(-1)
        idx = rng.permutation(flat.size)
        flat[idx[:40]] = 0.0
        flat[idx[40:80]] = -0.0
        flat[idx[80:90]] = np.inf
        flat[idx[90:100]] = -np.inf
        flat[idx[100:110]] = 1e-39
        flat[idx[110:120]] = -1e-39
        flat[idx[120:600]] = -np.abs(flat[idx[120:600]])
    else:
        raise ValueError(name)
    return torch.from_numpy(a.astype(np.float32)).to(torch.bfloat16).cuda()


def _check_k4(S, q, lower=False, host_walk=False):
    from sdrm_b200.sparsify import equal_sparsity_device
    Sf = S.float().cpu().numpy()
    qq = (1 - q) if lower else q
    thr = np.quantile(Sf.flatten(), qq)
    pm = equal_sparsity_device(S, q, lower=lower, host_walk=host_walk)
    same = np.float32(pm.threshold).view(np.uint32) == np.float32(thr).view(np.uint32)
    assert same or (np.isnan(pm.threshold) and np.isnan(thr)), (q, lower, pm.threshold, thr)   # (inf - inf in NumPy's _lerp: NaN)
    want = (Sf <= thr) if lower else (Sf >= thr)
    got = pm.numpy(np.int64).astype(bool)
    assert np.array_equal(got, want), (q, lower, int((got != want).sum()))
    assert int(pm.ones.item()) == int(want.sum())
    return pm


class _CountHist:
    """Counts the histogram passes K4 launches (every histogram entry of the C ABI launches one kernel)."""

    def __init__(self, monkeypatch):
        self.calls = {}
        lib = _lib.load()
        for name in ("sdrm_select_histogram", "sdrm_select_histogram_bf16", "sdrm_key_histogram", "sdrm_key_histogram_bf16"):
            fn = getattr(lib, name)

            def wrapped(*a, _fn=fn, _name=name):
                self.calls[_name] = self.calls.get(_name, 0) + 1
                return _fn(*a)
            monkeypatch.setattr(lib, name, wrapped)


@pytest.mark.gpu
@pytest.mark.parametrize("data", ["normal", "ties", "specials"])
def test_k4_bf16_threshold_and_bits_match_numpy(data, monkeypatch):
    from sdrm_b200.sparsify import _select_pack_device, quantile_device
    S = _scores(data, np.random.RandomState(11))
    counter = _CountHist(monkeypatch)

    def delta(before, name):
        return counter.calls.get(name, 0) - before.get(name, 0)
    for q in QS:
        for lower in (False, True):
            before = dict(counter.calls)
            _check_k4(S, q, lower)
            # every device selection is two histogram passes; when its walk flags the rare case it does not handle, the
            # host walk takes over (one pass per digit and distinct prefix); only the bfloat16 entries run
            d_sel, d_key = delta(before, "sdrm_select_histogram_bf16"), delta(before, "sdrm_key_histogram_bf16")
            assert d_sel in (2, 4) and d_key in (0, 2, 3) and (d_key > 0) == (d_sel == 4), (q, lower, d_sel, d_key)
            assert d_sel + d_key == sum(counter.calls.values()) - sum(before.values())
    if data == "normal":   # the common case: no fallback, the whole binarisation reads the matrix three times
        for q in (0.9, 0.99):
            before = dict(counter.calls)
            assert _select_pack_device(S, q, None, False) is not None
            assert delta(before, "sdrm_select_histogram_bf16") == 2 and sum(counter.calls.values()) - sum(before.values()) == 2
    for q in QS:
        thr, ref = quantile_device(S, q), np.quantile(S.float().cpu().numpy().flatten(), q)
        assert np.float32(thr).view(np.uint32) == np.float32(ref).view(np.uint32) or (np.isnan(thr) and np.isnan(ref)), (q, thr, ref)
    # the host walk (histograms copied to the host between the passes): same answers
    for q in (0.5, 0.99):
        _check_k4(S, q, host_walk=True)
    # a row stride larger than the width: the same scores in a view of a wider buffer
    wide = torch.zeros(S.shape[0], S.shape[1] + 13, dtype=torch.bfloat16, device="cuda")
    wide[:, 5:5 + S.shape[1]] = S
    V = wide[:, 5:5 + S.shape[1]]
    assert V.stride(0) > V.shape[1]
    for q in (0.5, 0.99):
        pm_v, pm_s = _check_k4(V, q), _check_k4(S, q)
        assert torch.equal(pm_v.bits, pm_s.bits)


@pytest.mark.gpu
def test_k4_bf16_nan_and_host_walk_fallback(monkeypatch):
    from sdrm_b200.sparsify import _select_pack_device, equal_sparsity_device, quantile_device
    S = _scores("normal", np.random.RandomState(12))
    S[17, 5] = float("nan")
    assert np.isnan(quantile_device(S, 0.9))
    pm = equal_sparsity_device(S, 0.9)
    assert np.isnan(pm.threshold) and int(pm.ones.item()) == 0 and not pm.numpy().any()
    # two order statistics in different top-digit bins (-1 and +1: different sign bits): the device walk flags the fallback
    F = torch.cat([torch.full((50, 64), -1.0), torch.full((50, 64), 1.0)]).to(torch.bfloat16).cuda()
    assert _select_pack_device(F, 0.5, None, False) is None
    counter = _CountHist(monkeypatch)
    for q in (0.3, 0.5, 0.7):
        _check_k4(F, q)
        _check_k4(F, q, lower=True)
        _check_k4(F, q, host_walk=True)
    assert set(counter.calls) <= {"sdrm_select_histogram_bf16", "sdrm_key_histogram_bf16"}
    # a negative and a positive order statistic straddling zero in a random matrix: q picks the ranks around the sign change
    R = _scores("normal", np.random.RandomState(13))
    n_neg = int((R.float() < 0).sum())
    q = (n_neg - 0.5) / (R.numel() - 1)
    _check_k4(R, q)
    _check_k4(R, q, host_walk=True)


@pytest.mark.gpu
def test_bf16_argument_checks():
    from sdrm_b200.sparsify import equal_sparsity_device, threshold_pack
    I = 333
    diff, vae, eng = _model("k1", I, seed=50)
    bad = {
        "short": torch.empty(10, I, dtype=torch.bfloat16, device="cuda"),
        "narrow": torch.empty(300, I - 1, dtype=torch.bfloat16, device="cuda"),
        "col_stride": torch.empty(I, 300, dtype=torch.bfloat16, device="cuda").t(),
        "fp16": torch.empty(300, I, dtype=torch.float16, device="cuda"),
        "1d": torch.empty(300 * I, dtype=torch.bfloat16, device="cuda"),
    }
    for name, out in bad.items():
        with pytest.raises(ValueError):
            eng.sample(300, seed=1, out=out)
    with pytest.raises(_lib.SdrmError):
        eng.sample(300, seed=1, out=torch.empty(300, I, dtype=torch.bfloat16))
    # the C entry checks its own arguments: ld below I, null logits
    ws, need = eng.workspace(300)
    lib = eng.lib
    out = torch.empty(300, I, dtype=torch.bfloat16, device="cuda")
    assert lib.sdrm_sample_bf16(eng.handle, 300, 0, None, None, 1, None, _lib.ptr(out), I - 1, None, None, None, _lib.ptr(ws), need,
                                _lib.stream_ptr()) == -1
    assert lib.sdrm_sample_bf16(eng.handle, 300, 0, None, None, 1, None, None, I, None, None, None, _lib.ptr(ws), need,
                                _lib.stream_ptr()) == -1
    S = torch.randn(64, 100, device="cuda").to(torch.bfloat16)
    for f in (lambda s: equal_sparsity_device(s, 0.9), lambda s: threshold_pack(s, 0.0)):
        with pytest.raises(ValueError):
            f(S.half())
        with pytest.raises(ValueError):
            f(S.t())
        with pytest.raises(ValueError):
            f(S[0])
        with pytest.raises(_lib.SdrmError):
            f(S.cpu())
    st = torch.zeros(lib.sdrm_select_state_bytes(), dtype=torch.uint8, device="cuda")
    h = torch.zeros(2048, dtype=torch.int64, device="cuda")
    assert lib.sdrm_select_histogram_bf16(_lib.ptr(S), 64, 100, 100, _lib.ptr(st), 2, _lib.ptr(h), _lib.stream_ptr()) == -1   # two digits
    assert lib.sdrm_select_walk_bf16(_lib.ptr(h), _lib.ptr(st), 2, 0.5, 1, _lib.stream_ptr()) == -1
    assert lib.sdrm_threshold_pack_bf16(_lib.ptr(S), 64, 100, 99, 0.0, 0, _lib.ptr(h), 4, None, _lib.stream_ptr()) == -1       # ld < n_cols
    assert lib.sdrm_key_histogram_bf16(_lib.ptr(S), 64, 100, 100, 0, 0, 16, 5, _lib.ptr(h), _lib.stream_ptr()) == -1          # digit layout
