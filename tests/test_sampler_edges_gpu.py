"""Edge contracts of sdrm_sample on every data flow of the sampler kernels (K6, and K1's single CTAs, pairs, pairs with several
tiles per CTA, column split of 8 / 4, resident and interleaved sub-tiles): rows with a start step of 0 or below (no reverse step:
the row decodes x_T), where the outputs land (strided, misaligned and odd-pitched views; nothing written outside them), PReLU
slopes outside [0, 1], the packing limits, and the chunked host-delivery path sample_ddpm_host.  Reference: the CPU oracle on
row slices (first tile, a middle tile, the ragged last tile), and the flows bit for bit against each other."""
import numpy as np
import pytest
import torch

from helpers import max_scaled_err, random_modules, rel_fro, state_dicts
from sdrm_b200 import _lib
from test_sampler_gpu import TOL, TOL_MAX, _engine

pytestmark = pytest.mark.gpu

# flow -> (options that force it, (sdrm_last_cluster_size, sdrm_last_split_size, sdrm_last_resident_mode) that prove it ran).
FLOWS = {
    "k6": ({_lib.OPT_ENGINE: 2}, (0, 0, 0)),
    "single": ({_lib.OPT_ENGINE: 1, _lib.OPT_CLUSTER: 1, _lib.OPT_NO_SPLIT: 1}, (1, 0, 0)),
    "pair": ({_lib.OPT_ENGINE: 1, _lib.OPT_CLUSTER: 2, _lib.OPT_NO_SPLIT: 1, _lib.OPT_RESIDENT: 1}, (2, 0, 0)),
    # one CTA pair for the whole launch: every CTA runs several row tiles one after the other
    "pair_grid": ({_lib.OPT_ENGINE: 1, _lib.OPT_CLUSTER: 2, _lib.OPT_NO_SPLIT: 1, _lib.OPT_RESIDENT: 1, _lib.OPT_SUBTILES: 1,
                   _lib.OPT_GRID_LIMIT: 2}, (2, 0, 0)),
    "split8": ({_lib.OPT_ENGINE: 1, _lib.OPT_CLUSTER: 8}, (1, 8, 0)),
    "split4": ({_lib.OPT_ENGINE: 1, _lib.OPT_CLUSTER: 4}, (1, 4, 0)),
    # full resolution only (a multi-resolution pair runs one streaming tile at a time)
    "resident": ({_lib.OPT_ENGINE: 1, _lib.OPT_CLUSTER: 2, _lib.OPT_NO_SPLIT: 1}, (2, 0, 1)),
    "subtiles": ({_lib.OPT_ENGINE: 1, _lib.OPT_CLUSTER: 2, _lib.OPT_NO_SPLIT: 1, _lib.OPT_SUBTILES: 2, _lib.OPT_GRID_LIMIT: 2},
                 (2, 0, 0)),
}
MULTIRES_K1 = ("single", "pair", "pair_grid", "split8", "split4")
FULLRES_K1 = MULTIRES_K1 + ("resident", "subtiles")
# I, H, L, T, nh, nd   ("k1": wider than 64, so the engine takes K1 and the column split; "k6": every width <= 64)
MODELS = {
    "k1": (333, 150, 200, 7, 2, 1.0),
    "k6": (333, 48, 40, 7, 2, 1.0),
}
NARROW_FLOWS = ("k6", "single", "pair")   # (the column split needs a denoiser wider than 64)

SENTINEL = 0x7FC0DEAD   # a NaN payload no kernel produces: compared as bits


def _run(eng, flow, n, **kw):
    """One sdrm_sample on `flow`; asserts that the launch took it and restores the automatic choice."""
    opts, (cluster, split, resident) = FLOWS[flow]
    lib = eng.lib
    try:
        for k, v in opts.items():
            eng.set_option(k, v)
        out = eng.sample(n, check=True, **kw)
        got = (lib.sdrm_last_cluster_size(eng.handle), lib.sdrm_last_split_size(eng.handle), lib.sdrm_last_resident_mode(eng.handle))
        assert got[0] == cluster and split in (None, got[1]) and resident in (None, got[2]), (flow, got)
    finally:
        for k in opts:
            eng.set_option(k, 0)
    return out


def _model(kind, seed, slopes=None):
    I, H, L, T, nh, nd = MODELS[kind]
    diff, vae = random_modules(I, H, L, T, nh, seed=seed, device="cuda")
    if slopes is not None:
        with torch.no_grad():
            diff.dnn[1].weight.fill_(slopes[0])
            diff.dnn[3].weight.fill_(slopes[1])   # (the ONE shared hidden PReLU)
    return diff, vae, _engine(diff, vae, T, nd)


def _flows_of(kind, multires):
    if kind == "k6":
        return NARROW_FLOWS
    return MULTIRES_K1 if multires else FULLRES_K1


def _slices(n):
    return sorted({0, (n // 2) // 128 * 128 - 6, n - 12})   # first tile, straddling a tile boundary mid-launch, ragged last tile


def _sentinel(shape):
    return torch.full(shape, SENTINEL, dtype=torch.int32, device="cuda").view(torch.float32)


# ------------------------------------------------------------------------------------------------------------------------------
# A. start steps of 0 and below: the row runs no reverse step and decodes x_T (K6, the oracle and the host check of engine.py
#    agree); K1 must do so for whole tiles (pairs: both tiles) of such rows too, where the chain runs no layer at all
# ------------------------------------------------------------------------------------------------------------------------------
def _t_layout(name, n, T):
    """(logical start steps as given, physical t_start of the launch, row_ids or None)"""
    rng = np.random.RandomState(7)
    t = rng.randint(1, T + 1, size=n).astype(np.int64)
    if name == "sorted_tail":          # the public call's order: longest chains first, whole tiles of zeros at the end
        t[rng.rand(n) < 0.45] = 0
        order = np.argsort(-t, kind="stable")
        return t, t[order], order
    if name == "zero_tiles_between":   # tiles 4 and 5 (one CTA pair's second tile pair under the grid cap) after real tiles
        t[4 * 128:6 * 128] = 0
    elif name == "mixed":              # zeros inside tiles that run the chain
        t[rng.rand(n) < 0.3] = 0
    elif name == "negative":           # device entries below 0 are clamped to 0; tiles 6 and 7 have no other entry
        t[rng.rand(n) < 0.3] = -1
        t[:40:3] = -(2 ** 31)
        t[6 * 128:] = rng.choice([-1, -5, -(2 ** 31)], size=n - 6 * 128)
    elif name == "all_zero":
        t[:] = 0
    return t, t, None


@pytest.mark.parametrize("layout", ["sorted_tail", "zero_tiles_between", "mixed", "negative", "all_zero"])
@pytest.mark.parametrize("kind", ["k1", "k6"])
def test_zero_and_negative_start_steps(kind, layout):
    from oracle import philox_ref
    from oracle import sdrm_oracle as orc
    I, H, L, T, nh, nd = MODELS[kind]
    n = 1000                                                  # 8 row tiles, the last one ragged (104 rows)
    diff, vae, eng = _model(kind, seed=31)
    t_log, t_phys, order = _t_layout(layout, n, T)
    t_dev = torch.from_numpy(t_phys.astype(np.int32)).cuda()
    row_ids = torch.from_numpy(order.astype(np.int32)).cuda() if order is not None else None
    seed = 0xA11CE
    xT, z, keep = (torch.from_numpy(a) for a in philox_ref.sampler_noise(seed, 0, n, L, T))
    inj = dict(inj_xT=xT.cuda(), inj_z=z.cuda(), inj_keep=keep.cuda())
    t_clamped = torch.from_numpy(np.clip(t_log, 0, T))
    zero = t_clamped == 0
    dsd, vsd = state_dicts(diff, vae)
    ref_zero = orc.vae_decode(vsd, xT[zero])                  # rows without a reverse step: decode(x_T)
    refs = {s: orc.sample_random(dsd, vsd, T, nd, xT[s:s + 12], z[:, s:s + 12], keep[:, s:s + 12], t_clamped[s:s + 12])
            for s in _slices(n)}
    res = {}
    for flow in _flows_of(kind, True):
        lat, lat_i = _sentinel((n, L)), _sentinel((n, L))
        out = _run(eng, flow, n, t_start=t_dev, row_ids=row_ids, seed=seed, latent_out=lat).cpu()
        out_i = _run(eng, flow, n, t_start=t_dev, row_ids=row_ids, latent_out=lat_i, **inj).cpu()
        lat, lat_i = lat.cpu(), lat_i.cpu()
        for o in (out, out_i):
            assert torch.isfinite(o).all(), flow
            if zero.any():
                e_fro, e_max = rel_fro(o[zero], ref_zero), max_scaled_err(o[zero], ref_zero)
                assert e_fro < TOL and e_max < TOL_MAX, (flow, e_fro, e_max)
            for s, ref in refs.items():
                assert rel_fro(o[s:s + 12], ref) < TOL and max_scaled_err(o[s:s + 12], ref) < TOL_MAX, (flow, s, rel_fro(o[s:s + 12], ref))
        assert torch.isfinite(lat).all() and torch.isfinite(lat_i).all(), flow   # (a sentinel NaN: a latent row never written)
        assert torch.equal(lat_i[zero], xT[zero]), flow      # x_0 = x_T, bit for bit
        res[flow] = (out, lat, out_i, lat_i)
    k1 = [f for f in res if f != "k6"]
    for f in k1[1:]:
        assert all(torch.equal(a, b) for a, b in zip(res[k1[0]], res[f])), (k1[0], f)


# ------------------------------------------------------------------------------------------------------------------------------
# B. output placement: logits into a view of a larger buffer (misaligned base, odd pitch, wide aligned pitch), latent into a
#    row slice; the values equal a contiguous launch and nothing outside the views is touched
# ------------------------------------------------------------------------------------------------------------------------------
PLACEMENTS = {   # name: (first column of the view, leading dimension - I)  for I = 333
    "misaligned": (1, 3),      # ld = 336 (a multiple of 4), base 4 bytes past a 16-byte boundary
    "odd_ld": (0, 4),          # ld = 337
    "aligned_wide": (4, 19),   # ld = 352, base 16-byte aligned: the vector store path (up to the ragged last group)
}


@pytest.mark.parametrize("placement", sorted(PLACEMENTS))
@pytest.mark.parametrize("kind", ["k1", "k6"])
def test_output_placement_and_guards(kind, placement):
    I, H, L, T, nh, nd = MODELS[kind]
    n = 300                                                   # 3 row tiles, the last one 44 rows
    diff, vae, eng = _model(kind, seed=32)
    c0, extra = PLACEMENTS[placement]
    ld = I + extra
    rng = np.random.RandomState(5)
    ts = torch.from_numpy(rng.randint(1, T + 1, size=n).astype(np.int32)).cuda()
    perm = torch.from_numpy(rng.permutation(n).astype(np.int32)).cuda()
    variants = {"full": ({}, False), "multires_row_ids": ({"t_start": ts, "row_ids": perm}, True)}
    for vname, (kw, multires) in variants.items():
        for flow in _flows_of(kind, multires):
            lat_ref = torch.empty(n, L, device="cuda")
            ref = _run(eng, flow, n, seed=44, latent_out=lat_ref, **kw).clone()
            buf, lbuf = _sentinel((n + 2, ld)), _sentinel((n + 2, L))
            view = buf[1:n + 1, c0:c0 + I]
            assert view.stride(0) == ld
            got = _run(eng, flow, n, seed=44, out=view, latent_out=lbuf[1:n + 1], **kw)
            assert got.data_ptr() == view.data_ptr()
            what = (vname, flow)
            assert torch.equal(view.cpu().view(torch.int32), ref.cpu().view(torch.int32)), what
            assert torch.equal(lbuf[1:n + 1].cpu().view(torch.int32), lat_ref.cpu().view(torch.int32)), what
            b = buf.cpu().view(torch.int32)
            inside = torch.zeros_like(b, dtype=torch.bool)
            inside[1:n + 1, c0:c0 + I] = True
            assert (b[~inside] == SENTINEL).all(), (what, int((b[~inside] != SENTINEL).sum()))
            lb = lbuf.cpu().view(torch.int32)
            assert (lb[0] == SENTINEL).all() and (lb[n + 1] == SENTINEL).all(), what


# ------------------------------------------------------------------------------------------------------------------------------
# C. PReLU slopes outside [0, 1] (trained slopes can leave it) and at its ends; two different slopes also catch a swapped slope
#    pointer of the chain's first and hidden layers
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("slopes", [(-0.5, 1.5), (1.5, -0.5), (0.0, 1.0)])
@pytest.mark.parametrize("kind", ["k1", "k6"])
def test_prelu_slopes_on_every_flow(kind, slopes):
    from oracle import philox_ref
    from oracle import sdrm_oracle as orc
    I, H, L, T, nh, nd = MODELS[kind]
    n = 600                                                   # 5 row tiles
    diff, vae, eng = _model(kind, seed=33, slopes=slopes)
    seed, off = 0x51095, 4096
    outs = {flow: _run(eng, flow, n, row_offset=off, seed=seed).cpu() for flow in _flows_of(kind, False)}
    dsd, vsd = state_dicts(diff, vae)
    for s in _slices(n):
        xT, z, keep = (torch.from_numpy(a) for a in philox_ref.sampler_noise(seed, off + s, 12, L, T))
        ref = orc.sample_full(dsd, vsd, T, nd, xT, z, keep)
        emu = orc.sample_bf16_emulated(dsd, vsd, T, nd, xT, z, keep)
        for flow, out in outs.items():
            got = out[s:s + 12]
            assert rel_fro(got, ref) < TOL and max_scaled_err(got, ref) < TOL_MAX, (flow, s, rel_fro(got, ref))
            assert rel_fro(got, emu) < 2e-4, (flow, s, rel_fro(got, emu))
    k1 = [f for f in outs if f != "k6"]
    for f in k1[1:]:
        assert torch.equal(outs[k1[0]], outs[f]), (k1[0], f)


# ------------------------------------------------------------------------------------------------------------------------------
# D. widths and depths above the compiled limits (L, D, H <= 2048, nh <= 6) are rejected, and the handle stays usable
# ------------------------------------------------------------------------------------------------------------------------------
def test_pack_rejects_shapes_above_the_limits():
    from oracle import philox_ref
    from oracle import sdrm_oracle as orc
    from sdrm_b200.models import SDRM, VAE, make_schedule
    I, H, L, T, nh, nd = MODELS["k1"]
    n = 300
    diff, vae, eng = _model("k1", seed=34)
    before = eng.sample(n, seed=3, check=True).clone()
    for bad_L, bad_nh in ((2049, nh), (L, 7)):
        bad = SDRM(N_ITEMS=bad_L, EMB_DIM=T, LATENT_DIM=bad_L, n_hidden_layers=bad_nh).cuda()
        with pytest.raises(_lib.SdrmError):
            eng.pack_denoiser(bad, make_schedule(T, device="cuda"), nd)
    with pytest.raises(_lib.SdrmError):
        eng.pack_decoder(VAE(I, 2049, L).cuda())
    eng.pack_denoiser(diff, make_schedule(T, device="cuda"), nd)
    eng.pack_decoder(vae)
    out = eng.sample(n, seed=3, check=True).cpu()
    assert torch.equal(out, before.cpu())
    dsd, vsd = state_dicts(diff, vae)
    for s in _slices(n):
        xT, z, keep = (torch.from_numpy(a) for a in philox_ref.sampler_noise(3, s, 12, L, T))
        ref = orc.sample_full(dsd, vsd, T, nd, xT, z, keep)
        assert rel_fro(out[s:s + 12], ref) < TOL and max_scaled_err(out[s:s + 12], ref) < TOL_MAX, s


# ------------------------------------------------------------------------------------------------------------------------------
# E. sample_ddpm_host: chunks of rows on two device buffers, copied to the host on a side stream; rows identical to sample_ddpm
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("chunk_rows", [None, 300, 384])   # one chunk; chunks straddling row tiles; tile-aligned chunks; ragged last
def test_sample_ddpm_host_rows_equal_sample_ddpm(chunk_rows):
    from sdrm_b200.models import VAE
    from sdrm_b200.train_SDRM import sample_ddpm, sample_ddpm_host
    I, H, L, T, nh, nd = MODELS["k1"]
    n, seed, off = 1000, 0x5EED5, 777
    diff, vae = random_modules(I, H, L, T, nh, seed=35, device="cuda")
    ref = sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, row_offset=off).cpu()
    got = sample_ddpm_host(n, diff, vae, L, nd, n_timesteps=T, seed=seed, row_offset=off, chunk_rows=chunk_rows)
    assert got.device.type == "cpu" and got.shape == (n, I) and torch.equal(got, ref)
    host = torch.full((n, I), float("nan"))
    assert sample_ddpm_host(n, diff, vae, L, nd, n_timesteps=T, seed=seed, row_offset=off, host_out=host, chunk_rows=chunk_rows) is host
    assert torch.equal(host, ref)
    # another item count behind the same denoiser (the same engine): the chunk buffers are reallocated
    torch.manual_seed(36)
    vae2 = VAE(input_dim=I + 61, hidden_dim=H, latent_dim=L).cuda().eval()
    ref2 = sample_ddpm(n, diff, vae2, L, nd, n_timesteps=T, seed=seed, row_offset=off).cpu()
    got2 = sample_ddpm_host(n, diff, vae2, L, nd, n_timesteps=T, seed=seed, row_offset=off, chunk_rows=chunk_rows)
    assert got2.shape == (n, I + 61) and torch.equal(got2, ref2)
    with pytest.raises(NotImplementedError):
        sample_ddpm_host(n, diff, vae, L, nd, timesteps="random", n_timesteps=T, seed=seed)
