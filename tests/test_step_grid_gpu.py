"""Fewer-step sampling (sdrm_set_step_grid; sample_ddpm's sampling_steps / eta) on every data flow of the sampler kernels (K6, and
K1's single CTAs, pairs, pairs with several tiles per CTA, column split of 8 / 4, resident and interleaved sub-tiles): the explicit
full grid reproduces the default chain bit for bit, strided DDPM and DDIM grids match the CPU oracle, eta = 0 never reads the
noise, the flows agree bit for bit, the host-delivery and sharded entry points follow the grid, and the handle's grid state
survives re-packs and rejected grids as documented."""
import ctypes as C
import os
import socket
import tempfile

import numpy as np
import pytest
import torch

from helpers import max_scaled_err, random_modules, rel_fro, state_dicts
from sdrm_b200 import _lib
from sdrm_b200.train_SDRM import grid_start_steps, step_grid
from test_sampler_edges_gpu import MODELS, _flows_of, _model, _run, _slices
from test_sampler_gpu import TOL, TOL_MAX

pytestmark = pytest.mark.gpu


def _grid_size(eng):
    return int(eng.lib.sdrm_step_grid_size(eng.handle))


def _multires(n, T, tau, seed=7):
    """(physical grid start steps on the device, row_ids): t_j ~ U{1..T-1} mapped onto the grid and sorted as sample_ddpm does"""
    t = np.random.RandomState(seed).randint(1, T, size=n)
    s = grid_start_steps(t, tau)
    order = np.argsort(-s, kind="stable").astype(np.int32)
    return s, torch.from_numpy(s[order].astype(np.int32)).cuda(), torch.from_numpy(order).cuda()


# ------------------------------------------------------------------------------------------------------------------------------
# A. the explicit full grid [1 .. T] in DDPM mode runs the grid tables and reproduces the default chain bit for bit
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bf16", [False, True])
@pytest.mark.parametrize("multires", [False, True])
@pytest.mark.parametrize("kind", ["k1", "k6"])
def test_full_grid_is_bit_identical_to_the_default_chain(kind, multires, bf16):
    I, H, L, T, nh, nd = MODELS[kind]
    n = 1000
    diff, vae, eng = _model(kind, seed=41)
    kw = {}
    if multires:
        _, kw["t_start"], kw["row_ids"] = _multires(n, T, list(range(1, T + 1)))
    dt = torch.bfloat16 if bf16 else torch.float32
    for flow in _flows_of(kind, multires):
        outs = []
        for grid in (None, range(1, T + 1)):
            eng.set_step_grid(grid)
            assert _grid_size(eng) == (0 if grid is None else T)
            lat = torch.empty(n, L, device="cuda")
            out = _run(eng, flow, n, seed=0xF00D, row_offset=123, latent_out=lat, out=torch.empty(n, I, dtype=dt, device="cuda"))
            outs.append((out.cpu(), lat.cpu()))
        eng.set_step_grid(None)
        (a, la), (b, lb) = outs
        assert torch.equal(a.view(torch.int16 if bf16 else torch.int32), b.view(torch.int16 if bf16 else torch.int32)), flow
        assert torch.equal(la.view(torch.int32), lb.view(torch.int32)), flow


# ------------------------------------------------------------------------------------------------------------------------------
# B. strided DDPM and DDIM grids against the CPU oracle, with injected noise slabs [S+1, n, L] and with in-kernel Philox
#    (whose streams of step j are those of step index j: philox_ref.sampler_noise with S steps)
# ------------------------------------------------------------------------------------------------------------------------------
def _grids(T):
    return {
        "S1": (step_grid(T, 1).tolist(), None),
        "S2": (step_grid(T, 2).tolist(), None),
        "S3": (step_grid(T, 3).tolist(), None),
        "half": (step_grid(T, T // 2).tolist(), None),
        "irregular": ([1, 2, 5, T], None),
        "ddim0": (step_grid(T, 3).tolist(), 0.0),
        "ddim05": ([2, 3, 6, T], 0.5),
        "ddim1": (list(range(1, T + 1)), 1.0),
    }


@pytest.mark.parametrize("grid", ["S1", "S2", "S3", "half", "irregular", "ddim0", "ddim05", "ddim1"])
@pytest.mark.parametrize("kind", ["k1", "k6"])
def test_grid_chain_matches_the_oracle(kind, grid):
    from oracle import philox_ref
    import grid_oracle as go
    I, H, L, T, nh, nd = MODELS[kind]
    tau, eta = _grids(T)[grid]
    S = len(tau)
    n = 300                                                   # 3 row tiles, the last one 44 rows
    diff, vae, eng = _model(kind, seed=42)
    dsd, vsd = state_dicts(diff, vae)
    eng.set_step_grid(tau, eta)
    assert _grid_size(eng) == S
    seed, off = 0x6121D, 64
    xT, z, keep = (torch.from_numpy(a) for a in philox_ref.sampler_noise(seed, off, n, L, S))
    inj = dict(inj_xT=xT.cuda(), inj_z=z.cuda(), inj_keep=keep.cuda())
    refs = {s: go.sample_grid(dsd, vsd, T, nd, xT[s:s + 12], z[:, s:s + 12], keep[:, s:s + 12], tau, eta) for s in _slices(n)}
    emus = {s: go.sample_bf16_emulated_grid(dsd, vsd, T, nd, xT[s:s + 12], z[:, s:s + 12], keep[:, s:s + 12], tau, eta)
            for s in _slices(n)}
    res = {}
    for flow in _flows_of(kind, False):
        out_i = _run(eng, flow, n, row_offset=off, **inj).cpu()
        out_p = _run(eng, flow, n, row_offset=off, seed=seed).cpu()
        for o in (out_i, out_p):
            assert torch.isfinite(o).all(), flow
            for s, ref in refs.items():
                got = o[s:s + 12]
                assert rel_fro(got, ref) < TOL and max_scaled_err(got, ref) < TOL_MAX, (flow, s, rel_fro(got, ref))
                assert rel_fro(got, emus[s]) < 2e-4, (flow, s, rel_fro(got, emus[s]))
        res[flow] = (out_i, out_p)
    k1 = [f for f in res if f != "k6"]
    for f in k1[1:]:                                          # in-kernel Philox and injected noise: every K1 flow alike
        assert torch.equal(res[k1[0]][0], res[f][0]) and torch.equal(res[k1[0]][1], res[f][1]), (k1[0], f)


@pytest.mark.parametrize("eta", [None, 0.5])
@pytest.mark.parametrize("kind", ["k1", "k6"])
def test_multiresolution_grid_matches_the_oracle(kind, eta):
    """Rows enter the grid at s_j = #{k : tau_k <= t_j}; t_j below tau_1 gives s_j = 0 (the row decodes x_T)."""
    from oracle import philox_ref
    import grid_oracle as go
    I, H, L, T, nh, nd = MODELS[kind]
    tau = [3, 5, T]
    n = 1000
    diff, vae, eng = _model(kind, seed=43)
    dsd, vsd = state_dicts(diff, vae)
    eng.set_step_grid(tau, eta)
    s_log, t_dev, row_ids = _multires(n, T, tau, seed=8)
    assert (s_log == 0).any() and (s_log == 1).any() and (s_log == 2).any()
    seed = 0xD1CE
    xT, z, keep = (torch.from_numpy(a) for a in philox_ref.sampler_noise(seed, 0, n, L, len(tau)))
    inj = dict(inj_xT=xT.cuda(), inj_z=z.cuda(), inj_keep=keep.cuda())
    zero = torch.from_numpy(s_log == 0)
    refs = {s: go.sample_grid(dsd, vsd, T, nd, xT[s:s + 12], z[:, s:s + 12], keep[:, s:s + 12], tau, eta, t_start=s_log[s:s + 12])
            for s in _slices(n)}
    emus = {s: go.sample_bf16_emulated_grid(dsd, vsd, T, nd, xT[s:s + 12], z[:, s:s + 12], keep[:, s:s + 12], tau, eta,
                                            t_start=s_log[s:s + 12]) for s in _slices(n)}
    res = {}
    for flow in _flows_of(kind, True):
        lat = torch.empty(n, L, device="cuda")
        out_i = _run(eng, flow, n, t_start=t_dev, row_ids=row_ids, latent_out=lat, **inj).cpu()
        out_p = _run(eng, flow, n, t_start=t_dev, row_ids=row_ids, seed=seed).cpu()
        assert torch.equal(lat.cpu()[zero], xT[zero]), flow      # s_j = 0: x_0 = x_T, bit for bit
        for o in (out_i, out_p):
            for s, ref in refs.items():
                got = o[s:s + 12]
                assert rel_fro(got, ref) < TOL and max_scaled_err(got, ref) < TOL_MAX, (flow, s, rel_fro(got, ref))
                assert rel_fro(got, emus[s]) < 2e-4, (flow, s)
        res[flow] = (out_i, out_p)
    k1 = [f for f in res if f != "k6"]
    for f in k1[1:]:
        assert torch.equal(res[k1[0]][0], res[f][0]) and torch.equal(res[k1[0]][1], res[f][1]), (k1[0], f)


# ------------------------------------------------------------------------------------------------------------------------------
# C. eta = 0 adds no noise: the injected z is never read (garbage in it changes nothing)
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["k1", "k6"])
def test_ddim_eta0_reads_no_noise(kind):
    from oracle import philox_ref
    I, H, L, T, nh, nd = MODELS[kind]
    n, tau = 300, step_grid(MODELS[kind][3], 4).tolist()
    diff, vae, eng = _model(kind, seed=44)
    eng.set_step_grid(tau, 0.0)
    xT, z, keep = (torch.from_numpy(a).cuda() for a in philox_ref.sampler_noise(5, 0, n, L, len(tau)))
    garbage = torch.full_like(z, float("nan"))
    for flow in _flows_of(kind, False):
        a = _run(eng, flow, n, inj_xT=xT, inj_z=z, inj_keep=keep).cpu()
        b = _run(eng, flow, n, inj_xT=xT, inj_z=garbage, inj_keep=keep).cpu()
        assert torch.isfinite(b).all() and torch.equal(a, b), flow


# ------------------------------------------------------------------------------------------------------------------------------
# D. the public entry points: sample_ddpm, sample_ddpm_host (one chunk, several) and sample_ddpm_sharded (every gather mode)
# ------------------------------------------------------------------------------------------------------------------------------
def test_sample_ddpm_follows_the_grid():
    from sdrm_b200.train_SDRM import engine_for, sample_ddpm
    I, H, L, T, nh, nd = MODELS["k1"]
    n, seed = 700, 0xAB
    diff, vae = random_modules(I, H, L, T, nh, seed=45, device="cuda")
    default = sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed).cpu()
    eng = engine_for(diff)
    # the explicit full grid equals the default; S = 3 equals the engine's grid launch
    assert torch.equal(sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, sampling_steps=list(range(1, T + 1))).cpu(), default)
    s3 = sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, sampling_steps=3).cpu()
    assert _grid_size(eng) == 3 and not torch.equal(s3, default)
    eng.set_step_grid(step_grid(T, 3))
    assert torch.equal(eng.sample(n, seed=seed).cpu(), s3)
    # bfloat16 rows are the rounded float32 rows of the same grid
    b16 = sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, sampling_steps=3, out_dtype=torch.bfloat16).cpu()
    assert torch.equal(b16.view(torch.int16), s3.to(torch.bfloat16).view(torch.int16))
    # reuse_packed keeps the handle's grid in step with each call's arguments
    d2 = sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, reuse_packed=True).cpu()
    assert _grid_size(eng) == 0 and torch.equal(d2, default)
    assert torch.equal(sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, reuse_packed=True, sampling_steps=3).cpu(), s3)
    # DDIM: eta alone runs the full grid
    dd = sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, eta=0.0).cpu()
    assert _grid_size(eng) == T and torch.isfinite(dd).all()
    # multi-resolution: the drawn t_j are mapped onto the grid and sorted
    t_rows = np.random.RandomState(3).randint(1, T, size=n)
    m = sample_ddpm(n, diff, vae, L, nd, timesteps="random", n_timesteps=T, seed=seed, t_rows=t_rows, sampling_steps=[3, 5, T]).cpu()
    s = grid_start_steps(t_rows, [3, 5, T])
    order = np.argsort(-s, kind="stable").astype(np.int32)
    eng.set_step_grid([3, 5, T])
    ref = eng.sample(n, seed=seed, t_start=torch.from_numpy(s[order].astype(np.int32)), row_ids=torch.from_numpy(order)).cpu()
    assert torch.equal(m, ref)
    # bad values raise before any launch and leave the handle's grid alone
    for bad in (dict(sampling_steps=0), dict(sampling_steps=T + 1), dict(sampling_steps=[2, 2]), dict(eta=1.5), dict(eta=-1.0)):
        with pytest.raises(ValueError):
            sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, **bad)
        assert _grid_size(eng) == 3


@pytest.mark.parametrize("chunk_rows", [None, 300])
def test_sample_ddpm_host_follows_the_grid(chunk_rows):
    from sdrm_b200.train_SDRM import sample_ddpm, sample_ddpm_host
    I, H, L, T, nh, nd = MODELS["k1"]
    n, seed, off = 1000, 0x5EED6, 99
    diff, vae = random_modules(I, H, L, T, nh, seed=46, device="cuda")
    for kw in (dict(sampling_steps=3), dict(sampling_steps=[1, 4, T], eta=0.5)):
        ref = sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, row_offset=off, **kw).cpu()
        got = sample_ddpm_host(n, diff, vae, L, nd, n_timesteps=T, seed=seed, row_offset=off, chunk_rows=chunk_rows, **kw)
        assert torch.equal(got, ref), kw
    with pytest.raises(ValueError):
        sample_ddpm_host(n, diff, vae, L, nd, n_timesteps=T, seed=seed, sampling_steps=T + 1)


def test_sample_ddpm_sharded_follows_the_grid():
    from sdrm_b200 import distributed as sdd
    from sdrm_b200.sparsify import equal_sparsity_device
    from sdrm_b200.train_SDRM import sample_ddpm
    I, H, L, T, nh, nd = MODELS["k1"]
    n, seed = 600, 57
    diff, vae = random_modules(I, H, L, T, nh, seed=47, device="cuda")
    kw = dict(sampling_steps=4, eta=0.5)
    ref = sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, **kw)
    rows, span = sdd.sample_ddpm_sharded(n, diff, vae, L, nd, n_timesteps=T, seed=seed, **kw)
    assert span == (0, n) and torch.equal(rows.cpu(), ref.cpu())
    rows, _ = sdd.sample_ddpm_sharded(n, diff, vae, L, nd, n_timesteps=T, seed=seed, gather=True, **kw)
    assert torch.equal(rows.cpu(), ref.cpu())
    pm, _ = sdd.sample_ddpm_sharded(n, diff, vae, L, nd, n_timesteps=T, seed=seed, gather="bits", sparsity=0.9, **kw)
    pm1 = equal_sparsity_device(ref, 0.9)
    assert torch.equal(pm.bits.cpu(), pm1.bits.cpu()) and float(pm.threshold) == float(pm1.threshold)
    b16, _ = sdd.sample_ddpm_sharded(n, diff, vae, L, nd, n_timesteps=T, seed=seed, out_dtype=torch.bfloat16, **kw)
    assert torch.equal(b16.cpu().view(torch.int16), ref.cpu().to(torch.bfloat16).view(torch.int16))
    t_all = np.random.RandomState(seed & 0x7FFFFFFF).randint(1, T, size=n).astype(np.int32)
    rnd, _ = sdd.sample_ddpm_sharded(n, diff, vae, L, nd, timesteps="random", n_timesteps=T, seed=seed, **kw)
    assert torch.equal(rnd.cpu(), sample_ddpm(n, diff, vae, L, nd, timesteps="random", n_timesteps=T, seed=seed, t_rows=t_all,
                                               **kw).cpu())


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _sharded_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        import sys
        sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
        from helpers import random_modules as rm
        from sdrm_b200 import distributed as sdd
        I, H, L, T, nh, nd = 333, 150, 200, 7, 2, 1.0
        diff, vae = rm(I, H, L, T, nh, seed=48, device=dev)
        rows, _ = sdd.sample_ddpm_sharded(601, diff, vae, L, nd, n_timesteps=T, seed=58, gather=True, sampling_steps=3)
        pm, _ = sdd.sample_ddpm_sharded(601, diff, vae, L, nd, n_timesteps=T, seed=58, gather="bits", sparsity=0.9, sampling_steps=3)
        torch.save((rows.cpu(), pm.bits.cpu()), os.path.join(out_dir, f"rank{rank}.pt"))
    except Exception:
        import traceback
        with open(os.path.join(out_dir, f"rank{rank}.err"), "w") as fh:
            fh.write(traceback.format_exc())
        raise
    finally:
        dist.destroy_process_group()


def test_two_rank_sharded_grid_equals_one_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from sdrm_b200.sparsify import equal_sparsity_device
    from sdrm_b200.train_SDRM import sample_ddpm
    world, port, out_dir = 2, _free_port(), tempfile.mkdtemp(prefix="sdrm_grid_gpu_")
    ctx = mp.get_context("spawn")
    procs = [ctx.Process(target=_sharded_worker, args=(r, world, port, out_dir)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(280)
    for r, p in enumerate(procs):
        err = os.path.join(out_dir, f"rank{r}.err")
        assert p.exitcode == 0, open(err).read() if os.path.exists(err) else f"rank {r} exit code {p.exitcode}"
    I, H, L, T, nh, nd = MODELS["k1"]
    diff, vae = random_modules(I, H, L, T, nh, seed=48, device="cuda")
    whole = sample_ddpm(601, diff, vae, L, nd, n_timesteps=T, seed=58, sampling_steps=3)
    bits = equal_sparsity_device(whole, 0.9).bits.cpu()
    for r in range(world):
        rows, b = torch.load(os.path.join(out_dir, f"rank{r}.pt"))
        assert torch.equal(rows, whole.cpu()) and torch.equal(b, bits)


# ------------------------------------------------------------------------------------------------------------------------------
# E. the handle's grid state: a re-pack resets it, S = 0 resets it, rejected grids change nothing, t_start above S is refused
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["k1", "k6"])
def test_handle_grid_state(kind):
    from sdrm_b200.models import make_schedule
    I, H, L, T, nh, nd = MODELS[kind]
    n = 300
    diff, vae, eng = _model(kind, seed=49)
    default = eng.sample(n, seed=9, check=True).cpu()
    tau = [2, 4, T]
    eng.set_step_grid(tau, 0.5)
    on_grid = eng.sample(n, seed=9, check=True).cpu()
    assert _grid_size(eng) == 3 and not torch.equal(on_grid, default)
    # rejected grids (host-side checks of sdrm_set_step_grid) leave the grid set and the handle sampling as before
    lib = eng.lib
    st = _lib.stream_ptr()
    bad = [([2, 2, T], 0, 0.0), ([0, 3], 0, 0.0), ([1, T + 1], 0, 0.0), ([3, 1], 1, 0.5), (list(range(1, T + 2)), 0, 0.0),
           ([1, 2], 2, 0.0), ([1, 2], 1, 1.5), ([1, 2], 1, -0.25), ([1, 2], 1, float("nan"))]
    for ts, mode, eta in bad:
        arr = (C.c_int32 * len(ts))(*ts)
        assert lib.sdrm_set_step_grid(eng.handle, arr, len(ts), mode, eta, st) == -1, (ts, mode, eta)
        assert _grid_size(eng) == 3
    assert lib.sdrm_set_step_grid(eng.handle, None, 2, 0, 0.0, st) == -1
    with pytest.raises(_lib.SdrmError):
        eng.set_step_grid([5, 3])
    assert torch.equal(eng.sample(n, seed=9, check=True).cpu(), on_grid)
    # t_start above S is refused on the host path; S itself is fine
    with pytest.raises(ValueError):
        eng.sample(n, seed=9, t_start=torch.full((n,), 4, dtype=torch.int32))
    eng.sample(n, seed=9, t_start=torch.full((n,), 3, dtype=torch.int32), check=True)
    # S = 0 restores the full chain
    eng.set_step_grid(None)
    assert _grid_size(eng) == 0 and torch.equal(eng.sample(n, seed=9, check=True).cpu(), default)
    assert lib.sdrm_set_step_grid(eng.handle, (C.c_int32 * 3)(*tau), 3, 0, 0.0, st) == 0 and _grid_size(eng) == 3
    assert lib.sdrm_set_step_grid(eng.handle, None, 0, 0, 0.0, st) == 0 and _grid_size(eng) == 0
    assert torch.equal(eng.sample(n, seed=9, check=True).cpu(), default)
    # a re-pack of the denoiser resets the handle (and the engine's record of it) to the full chain
    eng.set_step_grid(tau, 0.5)
    eng.pack_denoiser(diff, make_schedule(T, device="cuda"), nd)
    assert _grid_size(eng) == 0 and eng.steps == T
    assert torch.equal(eng.sample(n, seed=9, check=True).cpu(), default)
    eng.set_step_grid(tau, 0.5)                              # (not skipped as already set: the pack cleared the record)
    assert _grid_size(eng) == 3 and torch.equal(eng.sample(n, seed=9, check=True).cpu(), on_grid)
