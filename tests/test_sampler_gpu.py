"""GPU parity of K1 (sdrm_sample through the C ABI) against the oracle and the reference goldens."""
import numpy as np
import pytest
import torch

from conftest import SAMPLER_GOLDENS, load_golden
from helpers import max_scaled_err, modules_from_golden, random_modules, rel_fro, state_dicts

pytestmark = pytest.mark.gpu

TOL = 1e-3      # north_star: synthetic rows within 1e-3 relative (bf16 operands, fp32 accumulate) -> rel-Frobenius
TOL_MAX = 3e-3  # worst single element, |d| / max(1, |ref|): measured 4.9e-5 ... 1.0e-3 at the full chain lengths of cfg 1-3 / cfg 5 and 2.3e-3 at cfg 4 (nd = 0.2) (r02)


def _engine(diff, vae, T, nd):
    from sdrm_b200.engine import SamplerEngine
    from sdrm_b200.models import make_schedule
    eng = SamplerEngine()
    eng.pack_denoiser(diff, make_schedule(T, device="cuda"), nd)
    eng.pack_decoder(vae)
    return eng


@pytest.mark.parametrize("name", SAMPLER_GOLDENS)
@pytest.mark.parametrize("mode", ["full", "random"])
@pytest.mark.parametrize("engine", ["auto", "tcgen05"])
def test_golden_injected_noise(name, mode, engine):
    """Same weights + same noise tensors the REFERENCE consumed -> rows match the reference output.  `auto` takes the
    small-chain kernel (K6) for the fixtures whose widths are all <= 64 and the tcgen05 layer engine (K1) for the others;
    `tcgen05` forces K1 for every fixture."""
    from sdrm_b200 import _lib
    g = load_golden(name)
    diff, vae = modules_from_golden(g, "cuda")
    eng = _engine(diff, vae, g["T"], g["nd"])
    eng.set_option(_lib.OPT_ENGINE, 1 if engine == "tcgen05" else 0)
    c = g[mode]
    n = g["n"]
    lat = torch.empty(n, g["L"], device="cuda")
    t_start = c.get("t_start")
    out = eng.sample(n, t_start=t_start.cuda() if t_start is not None else None, latent_out=lat,
                     inj_xT=c["xT"].cuda().contiguous(), inj_z=c["z"].cuda().contiguous(),
                     inj_keep=c["keep"].cuda().contiguous(), check=True)
    ref = c["logits_ref"]
    assert torch.isfinite(out).all()
    assert rel_fro(out.cpu(), ref) < TOL, (rel_fro(out.cpu(), ref))
    assert max_scaled_err(out.cpu(), ref) < TOL_MAX


@pytest.mark.parametrize("shape", [
    # n, I, H, L, T, nh, nd   (dataset-shaped, shortened chains so the CPU oracle stays fast)
    (843, 1008, 930, 830, 12, 2, 1.0),    # cfg 1 ml-100k
    (700, 3125, 490, 340, 10, 1, 1.0),    # cfg 2 ml-1m
    (1200, 8582, 40, 40, 16, 5, 1.0),     # cfg 3 adm
    (1208, 729, 550, 400, 43, 0, 0.2),    # cfg 4 alb, full T
    (300, 2000, 1000, 950, 6, 4, 1.0),    # cfg 5 layer shapes (I shortened)
    (130, 500, 2048, 2048, 3, 1, 1.0),    # the widest latent, hidden and VAE hidden the library takes (8 x 256 columns)
    (200, 1, 40, 65, 6, 1, 1.0),          # one column wider than the small-chain kernel takes; a single item
    (300, 400, 100, 120, 1, 6, 0.0),      # K1: one step (no dropout mask or noise from the noise warps, no discard), nh = 6
    (400, 150, 48, 40, 2, 6, 0.5),        # K6 (every width <= 64): two steps, nh = 6
])
def test_vs_oracle_philox_noise(shape):
    """In-kernel Philox noise: the oracle is fed the numpy restatement of the same streams."""
    from oracle import philox_ref
    from oracle import sdrm_oracle as orc
    n, I, H, L, T, nh, nd = shape
    diff, vae = random_modules(I, H, L, T, nh, seed=3, device="cuda")
    eng = _engine(diff, vae, T, nd)
    seed, row_offset = 0x1234ABCD5678, 1000
    lat = torch.empty(n, L, device="cuda")
    out = eng.sample(n, row_offset=row_offset, seed=seed, latent_out=lat, check=True).cpu()
    xT, z, keep = philox_ref.sampler_noise(seed, row_offset, n, L, T)
    dsd, vsd = state_dicts(diff, vae)
    ref, ref_lat = orc.sample_full(dsd, vsd, T, nd, torch.from_numpy(xT), torch.from_numpy(z), torch.from_numpy(keep),
                                   return_latent=True)
    emu = orc.sample_bf16_emulated(dsd, vsd, T, nd, torch.from_numpy(xT), torch.from_numpy(z), torch.from_numpy(keep))
    e_lat, e_out, e_emu = rel_fro(lat.cpu(), ref_lat), rel_fro(out, ref), rel_fro(out, emu)
    print(f"shape={shape} latent rel {e_lat:.2e} logits rel {e_out:.2e} vs bf16-emulation {e_emu:.2e} "
          f"max scaled {max_scaled_err(out, ref):.2e}")
    assert e_out < TOL and e_lat < TOL
    assert max_scaled_err(out, ref) < TOL_MAX
    assert e_emu < 2e-4  # same rounding points -> much tighter: isolates kernel bugs from bf16 effects


def test_partition_invariance():
    """Rows depend only on (seed, global row id): any sharding / tile placement gives identical bits."""
    n, I, H, L, T, nh, nd = 700, 300, 64, 72, 9, 1, 1.0
    diff, vae = random_modules(I, H, L, T, nh, seed=5, device="cuda")
    eng = _engine(diff, vae, T, nd)
    whole = eng.sample(n, row_offset=0, seed=99, check=True).clone()
    a = eng.sample(389, row_offset=0, seed=99, check=True).clone()
    b = eng.sample(n - 389, row_offset=389, seed=99, check=True).clone()
    assert torch.equal(whole, torch.cat([a, b]))


def test_single_and_pair_mode_are_bit_identical():
    """The chain runs on single CTAs (cta_group::1) or CTA pairs (cta_group::2, UMMA M=256); rows do not change."""
    from sdrm_b200 import _lib
    lib = _lib.load()
    n, I, H, L, T, nh, nd = 1400, 700, 200, 264, 7, 2, 1.0     # 11 row tiles; ragged last tile; a ghost tile for the last pair
    diff, vae = random_modules(I, H, L, T, nh, seed=6, device="cuda")
    eng = _engine(diff, vae, T, nd)
    outs, rnd, srt = {}, {}, {}
    rng = np.random.RandomState(9)
    t_any = torch.from_numpy(rng.randint(1, T, size=n).astype(np.int32)).cuda()      # multi-resolution chains, rows in any order
    order = np.argsort(-t_any.cpu().numpy(), kind="stable").astype(np.int32)          # ... and sorted by chain length (the public call)
    t_sorted, row_ids = t_any[torch.from_numpy(order).cuda().long()].contiguous(), torch.from_numpy(order).cuda()
    try:
        for c in (1, 2):
            eng.set_option(_lib.OPT_CLUSTER, c)
            outs[c] = eng.sample(n, seed=77, check=True).clone()
            assert lib.sdrm_last_cluster_size(eng.handle) == c
            # a pair runs the longer of its two tiles' chains; rows with shorter chains wait for their start step
            rnd[c] = eng.sample(n, t_start=t_any, seed=77, check=True).clone()
            assert lib.sdrm_last_cluster_size(eng.handle) == c
            srt[c] = eng.sample(n, t_start=t_sorted, row_ids=row_ids, seed=77, check=True).clone()
            eng.set_option(_lib.OPT_GRID_LIMIT, 4)                                    # several tiles per CTA
            assert torch.equal(eng.sample(n, t_start=t_sorted, row_ids=row_ids, seed=77, check=True), srt[c])
            eng.set_option(_lib.OPT_GRID_LIMIT, 0)
    finally:
        eng.set_option(_lib.OPT_CLUSTER, 0)
        eng.set_option(_lib.OPT_GRID_LIMIT, 0)
    assert lib.sdrm_resident_ctas(eng.handle, 2) >= 2 and lib.sdrm_resident_ctas(eng.handle, 4) == 0
    for c in outs:
        assert torch.equal(outs[1], outs[c]), c
        assert torch.equal(rnd[1], rnd[c]) and torch.equal(srt[1], srt[c]), c
    assert torch.equal(rnd[1], srt[1])      # a row's chain does not depend on where the row sits in the launch
    assert not torch.equal(outs[1], rnd[1])


@pytest.mark.parametrize("shape", [
    # n, I, H, L, T, nh       resident geometry
    (1500, 700, 200, 264, 7, 2),     # KB = 5 (odd: a lone last weight k-block), 2 chunks, 3 stages left
    (900, 300, 128, 120, 9, 1),      # one chunk, KB = 2
    (2000, 729, 550, 400, 6, 0),     # cfg-4 widths: KB = 7 -> 2 stages left, no hidden layer
    (1000, 500, 300, 512, 5, 1),     # the widest denoiser the mode takes (2 x 256 columns, KB = 8)
    (700, 400, 200, 520, 4, 1),      # too wide (3 chunks): stays in streaming mode
    (1000, 300, 200, 128, 5, 1),     # 128 columns: one tile per CTA streams; several tiles per CTA interleave (w = 128)
    (1000, 300, 200, 129, 5, 1),     # one column more: KB = 3 (w = 192) -> resident with one tile per CTA
    (1000, 300, 200, 256, 5, 1),     # one chunk of 256 columns (w = 256)
    (1000, 300, 200, 257, 5, 1),     # two chunks of 144 columns, KB = 5 (w = 320: the widest that interleaves sub-tiles)
    (700, 300, 200, 513, 4, 1),      # 3 chunks: streaming
])
def test_resident_mode_is_bit_identical_to_streaming(shape):
    """Pair-mode launches of denoisers up to 512 wide keep the chain's activation tile in shared memory (resident mode), with
    one row tile per CTA or several in sequence (grid cap); SDRM_OPT_RESIDENT = 1 forces the L2-streaming path.  Same
    arithmetic, same rows.  (Automatic choice, engine_host.cu: one tile per CTA -> resident above 128 columns; several tiles per
    CTA -> two interleaved streaming sub-tiles up to 320 columns, resident above.)"""
    from sdrm_b200 import _lib
    lib = _lib.load()
    n, I, H, L, T, nh = shape
    w = max((L + 63) // 64 * 64, (L + 15) // 16 * 16 if L <= 256 else 2 * (((L + 1) // 2 + 15) // 16 * 16))
    fits = L <= 512
    diff, vae = random_modules(I, H, L, T, nh, seed=11, device="cuda")
    eng = _engine(diff, vae, T, 1.0)
    lat = [torch.empty(n, L, device="cuda") for _ in range(4)]
    eng.set_option(_lib.OPT_NO_SPLIT, 1)    # (launches of a few row tiles would take the column-split flow: its own test below)
    try:
        a = eng.sample(n, seed=5, latent_out=lat[0], check=True).clone()
        assert lib.sdrm_last_resident_mode(eng.handle) == (1 if fits and w > 128 else 0)
        eng.set_option(_lib.OPT_RESIDENT, 1)
        b = eng.sample(n, seed=5, latent_out=lat[1], check=True).clone()
        assert lib.sdrm_last_resident_mode(eng.handle) == 0
        eng.set_option(_lib.OPT_RESIDENT, 0)
        eng.set_option(_lib.OPT_GRID_LIMIT, 4)          # two pairs: every CTA runs several row tiles
        c = eng.sample(n, seed=5, latent_out=lat[2], check=True).clone()   # automatic: sub-tiles or resident by width
        assert lib.sdrm_last_resident_mode(eng.handle) == (1 if fits and w > 320 else 0)
        eng.set_option(_lib.OPT_SUBTILES, 1)            # one tile at a time: resident whenever it fits
        d = eng.sample(n, seed=5, latent_out=lat[3], check=True)
        assert lib.sdrm_last_resident_mode(eng.handle) == (1 if fits else 0)
    finally:
        eng.set_option(_lib.OPT_RESIDENT, 0)
        eng.set_option(_lib.OPT_GRID_LIMIT, 0)
        eng.set_option(_lib.OPT_SUBTILES, 0)
        eng.set_option(_lib.OPT_NO_SPLIT, 0)
    for o, l_ in ((b, lat[1]), (c, lat[2]), (d, lat[3])):
        assert torch.equal(a, o) and torch.equal(lat[0], l_)


@pytest.mark.parametrize("shape", [
    # n, I, H, L, T, nh      normal geometry -> 8-chunk geometry (clusters of 8); clusters of 4 keep the normal geometry
    (843, 1008, 930, 830, 9, 2),     # cfg-1 widths: 4 chunks of 208 -> 8 of 112 (7 tiles = 56 CTAs)
    (700, 400, 200, 520, 5, 1),      # 3 chunks of 176 (on 4 CTAs one idles in the chain) -> 8 of 80; decoder layers of 1 and 2 chunks
    (300, 2000, 1000, 950, 6, 4),    # cfg-5 widths, ragged last tile; 8 logits chunks in either geometry (two per CTA on 4 CTAs)
    (260, 600, 300, 1300, 4, 1),     # 6 chunks of 224 -> 8 of 176 (on 4 CTAs: two chunks for CTAs 0 and 1)
    (128, 300, 96, 600, 3, 0),       # a single row tile, no hidden layer
    (1208, 729, 550, 400, 8, 0),     # cfg-4 widths: 2 chunks of 208 -> 8 of 64 (the resident flow's territory: the split is faster)
    (900, 500, 300, 264, 6, 2),      # 2 chunks of 144 -> 8 of 48
    (6000, 300, 200, 600, 3, 1),     # 47 row tiles: only clusters of 2 fit (normal geometry, CTA j takes the chunks j and j + 2 of 3)
    (1500, 400, 128, 200, 7, 3),     # a single-chunk denoiser: 8 chunks of 32 columns
    (500, 300, 100, 72, 9, 1),       # 8 chunks of 16 columns (the narrowest UMMA)
    (300, 700, 300, 2048, 3, 1),     # the widest denoiser: 8 chunks of 256 in either geometry (two per CTA on 4 CTAs)
    (500, 10, 100, 65, 5, 1),        # one chunk of 80 -> 8 of 16; fewer items than one 16-column logits chunk
])
def test_column_split_mode_is_bit_identical_to_streaming(shape):
    """Full-resolution launches of a few row tiles of a wide denoiser (>= 3 N chunks per chain layer) split every tile's chunks over
    a cluster of 8 CTAs in an 8-chunk geometry of the layers (a second set of weight images), or of 4 CTAs in the normal geometry
    (engine_host.cu, SDRM_OPT_NO_SPLIT / SDRM_OPT_CLUSTER); the chunk barriers span the cluster.  Same arithmetic, same rows, same
    latent as the one-CTA-per-tile flows, with in-kernel Philox noise and with injected noise tensors."""
    from oracle import philox_ref
    from sdrm_b200 import _lib
    lib = _lib.load()
    n, I, H, L, T, nh = shape
    want = 8 if n <= 2000 else 2
    diff, vae = random_modules(I, H, L, T, nh, seed=13, device="cuda")
    eng = _engine(diff, vae, T, 1.0)
    lat = [torch.empty(n, L, device="cuda") for _ in range(4)]
    try:
        a = eng.sample(n, seed=21, latent_out=lat[0], check=True).clone()
        assert lib.sdrm_last_split_size(eng.handle) == want
        a2 = eng.sample(n, seed=21, check=True).clone()          # (a second launch on the same scratch)
        eng.set_option(_lib.OPT_CLUSTER, 4)
        a4 = eng.sample(n, seed=21, check=True).clone()
        assert lib.sdrm_last_split_size(eng.handle) == (4 if want == 8 else 0)   # (47 tiles x 4 CTAs do not fit: pair flow)
        eng.set_option(_lib.OPT_CLUSTER, 0)
        ts = torch.from_numpy(np.random.RandomState(3).randint(1, T, size=n).astype(np.int32)).cuda()
        e = eng.sample(n, t_start=ts, seed=21, check=True).clone()      # multi-resolution chains (per-row start steps) split too
        assert lib.sdrm_last_split_size(eng.handle) == want
        eng.set_option(_lib.OPT_NO_SPLIT, 1)
        b = eng.sample(n, seed=21, latent_out=lat[1], check=True).clone()
        assert lib.sdrm_last_split_size(eng.handle) == 0
        f = eng.sample(n, t_start=ts, seed=21, check=True).clone()      # multi-resolution chains, one CTA per tile
        assert lib.sdrm_last_split_size(eng.handle) == 0
        inj = dict(zip(("inj_xT", "inj_z", "inj_keep"), (torch.from_numpy(t).cuda().contiguous() for t in philox_ref.sampler_noise(21, 0, n, L, T))))
        d = eng.sample(n, seed=0, latent_out=lat[3], check=True, **inj).clone()
        eng.set_option(_lib.OPT_NO_SPLIT, 0)
        c = eng.sample(n, seed=0, latent_out=lat[2], check=True, **inj)
        assert lib.sdrm_last_split_size(eng.handle) == want
    finally:
        eng.set_option(_lib.OPT_NO_SPLIT, 0)
        eng.set_option(_lib.OPT_CLUSTER, 0)
    assert torch.isfinite(a).all()
    assert torch.equal(a, a2) and torch.equal(a, a4)
    assert torch.equal(a, b) and torch.equal(lat[0], lat[1])
    assert torch.equal(c, d) and torch.equal(lat[2], lat[3])
    assert torch.equal(e, f)
    assert rel_fro(c.cpu(), a.cpu()) < 1e-4   # (the numpy restatement of the noise differs from MUFU Box-Muller in the last bits)


def test_interleaved_sub_tiles_are_bit_identical():
    """A CTA pair that owns several row tiles interleaves two of them layer by layer (ChainParams::n_sub = 2, an odd last
    tile runs alone); the grid cap makes a small launch take that path (12 row tiles on 2 pairs = 3 tiles per CTA)."""
    from sdrm_b200 import _lib
    lib = _lib.load()
    n, I, H, L, T, nh, nd = 1500, 700, 200, 264, 7, 2, 1.0
    diff, vae = random_modules(I, H, L, T, nh, seed=6, device="cuda")
    eng = _engine(diff, vae, T, nd)
    ref = eng.sample(n, seed=77, check=True).clone()
    lat_ref = torch.empty(n, L, device="cuda")
    eng.sample(n, seed=77, latent_out=lat_ref, check=True)
    try:
        for cluster, limit in ((2, 4), (2, 8)):
            eng.set_option(_lib.OPT_CLUSTER, cluster)
            eng.set_option(_lib.OPT_GRID_LIMIT, limit)
            for sub in (1, 2):
                eng.set_option(_lib.OPT_SUBTILES, sub)
                lat = torch.empty(n, L, device="cuda")
                out = eng.sample(n, seed=77, latent_out=lat, check=True)
                assert torch.equal(out, ref), (cluster, limit, sub)
                assert torch.equal(lat, lat_ref), (cluster, limit, sub)
    finally:
        eng.set_option(_lib.OPT_CLUSTER, 0)
        eng.set_option(_lib.OPT_GRID_LIMIT, 0)
        eng.set_option(_lib.OPT_SUBTILES, 0)


def test_random_mode_matches_oracle():
    from oracle import philox_ref
    from oracle import sdrm_oracle as orc
    n, I, H, L, T, nh, nd = 500, 256, 96, 88, 21, 2, 0.7
    diff, vae = random_modules(I, H, L, T, nh, seed=8, device="cuda")
    eng = _engine(diff, vae, T, nd)
    rng = np.random.RandomState(4)
    t_start = torch.from_numpy(rng.randint(1, T, size=n).astype(np.int32))
    out = eng.sample(n, t_start=t_start.cuda(), seed=321, check=True).cpu()
    xT, z, keep = philox_ref.sampler_noise(321, 0, n, L, T)
    dsd, vsd = state_dicts(diff, vae)
    ref = orc.sample_random(dsd, vsd, T, nd, torch.from_numpy(xT), torch.from_numpy(z), torch.from_numpy(keep), t_start)
    assert rel_fro(out, ref) < TOL


def test_empty_and_ragged():
    n, I, H, L, T, nh, nd = 1, 17, 8, 5, 3, 0, 1.0   # one row, ragged dims far from multiples of 16
    diff, vae = random_modules(I, H, L, T, nh, seed=1, device="cuda")
    eng = _engine(diff, vae, T, nd)
    out = eng.sample(n, seed=1, check=True)
    assert out.shape == (1, I) and torch.isfinite(out).all()
    assert eng.sample(0).shape == (0, I)


def test_headline_config_rows_match_oracle_at_full_scale():
    """BASELINE.json's scale-up configuration itself (T=178, L=950, H=1000, nh=4, I=20 000) on two full waves of CTA pairs:
    rows taken from the first, a middle and the ragged last tile of a 37 900-row launch are compared with the oracle over
    the WHOLE 178-step chain, and the launch is checked for determinism and sharding invariance."""
    from oracle import philox_ref
    from oracle import sdrm_oracle as orc
    n, I, H, L, T, nh, nd = 37900, 20000, 1000, 950, 178, 4, 1.0
    diff, vae = random_modules(I, H, L, T, nh, seed=11, device="cuda")
    eng = _engine(diff, vae, T, nd)
    seed, row_offset = 0xC0FFEE1234, 5_000_000_000          # row ids beyond 2^32 exercise the high counter word
    out = eng.sample(n, row_offset=row_offset, seed=seed, check=True)
    assert torch.isfinite(out).all()
    again = eng.sample(n, row_offset=row_offset, seed=seed, check=True)
    assert torch.equal(out, again)                            # deterministic
    lo = 19000
    shard = eng.sample(700, row_offset=row_offset + lo, seed=seed, check=True)
    assert torch.equal(shard, out[lo:lo + 700])               # rows depend only on (seed, global row id)
    dsd, vsd = state_dicts(diff, vae)
    for start in (0, 18944 + 37, n - 12):                     # first tile, second wave, ragged last tile
        rows = 12
        xT, z, keep = philox_ref.sampler_noise(seed, row_offset + start, rows, L, T)
        ref = orc.sample_full(dsd, vsd, T, nd, torch.from_numpy(xT), torch.from_numpy(z), torch.from_numpy(keep))
        got = out[start:start + rows].cpu()
        assert rel_fro(got, ref) < TOL, (start, rel_fro(got, ref))
        assert max_scaled_err(got, ref) < TOL_MAX


# BASELINE.json configs 1-3 at their REAL sizes and FULL chain lengths (T = 83 / 78 / 93); the CPU oracle runs the whole chain on
# 12-row slices (rows depend only on (seed, global row id), so a slice of the launch equals a launch of the slice).
FULL_T_CONFIGS = {
    "cfg1": (843, 1008, 930, 830, 83, 2, 1.0),
    "cfg2": (5429, 3125, 490, 340, 78, 1, 1.0),
    "cfg3": (9558, 8582, 40, 40, 93, 5, 1.0),
}


@pytest.mark.parametrize("cfg", sorted(FULL_T_CONFIGS))
def test_dataset_configs_full_chain_length(cfg):
    from oracle import philox_ref
    from oracle import sdrm_oracle as orc
    n, I, H, L, T, nh, nd = FULL_T_CONFIGS[cfg]
    diff, vae = random_modules(I, H, L, T, nh, seed=21, device="cuda")
    eng = _engine(diff, vae, T, nd)
    seed, row_offset = 0xABCDEF0123, 77
    out = eng.sample(n, row_offset=row_offset, seed=seed, check=True)
    assert torch.isfinite(out).all()
    dsd, vsd = state_dicts(diff, vae)
    worst_fro, worst_el = 0.0, 0.0
    for start in (0, (n // 2) // 128 * 128 + 19, n - 12):     # first tile, a middle tile, the ragged last tile
        xT, z, keep = philox_ref.sampler_noise(seed, row_offset + start, 12, L, T)
        ref = orc.sample_full(dsd, vsd, T, nd, torch.from_numpy(xT), torch.from_numpy(z), torch.from_numpy(keep))
        got = out[start:start + 12].cpu()
        worst_fro = max(worst_fro, rel_fro(got, ref))
        worst_el = max(worst_el, max_scaled_err(got, ref))
    print(f"{cfg} full T={T}: logits rel-Frobenius {worst_fro:.2e}, worst element |d|/max(1,|ref|) {worst_el:.2e}")
    assert worst_fro < TOL and worst_el < TOL_MAX


def test_random_mode_at_cfg1_shape_through_the_public_call():
    """sample_ddpm(timesteps='random') at the ml-100k shape (843 users, T = 83): t_j ~ np.random.randint(1, T) like the reference
    (train_SDRM.py:42); the call sorts the rows by chain length internally and must return them in logical order."""
    from oracle import philox_ref
    from oracle import sdrm_oracle as orc
    from sdrm_b200.train_SDRM import sample_ddpm
    n, I, H, L, T, nh, nd = FULL_T_CONFIGS["cfg1"]
    diff, vae = random_modules(I, H, L, T, nh, seed=22, device="cuda")
    np.random.seed(31)
    t_np = np.random.randint(1, T, size=n)             # the draw the call makes itself ...
    np.random.seed(31)                                  # ... replayed
    out = sample_ddpm(n, diff, vae, L, nd, timesteps="random", n_timesteps=T, seed=4242)
    assert out.shape == (n, I) and torch.isfinite(out).all()
    dsd, vsd = state_dicts(diff, vae)
    for start in (0, 400, n - 16):
        xT, z, keep = philox_ref.sampler_noise(4242, start, 16, L, T)
        ref = orc.sample_random(dsd, vsd, T, nd, torch.from_numpy(xT), torch.from_numpy(z), torch.from_numpy(keep), t_np[start:start + 16])
        got = out[start:start + 16].cpu()
        assert rel_fro(got, ref) < TOL, (start, rel_fro(got, ref))
        assert max_scaled_err(got, ref) < TOL_MAX


def test_packed_weights_follow_in_place_data_edits():
    """ADVICE r1: an edit through `.data` bumps no version counter; the default call re-packs, so it must see the new weights,
    and `reuse_packed=True` must be the only way to keep the old images."""
    from sdrm_b200.train_SDRM import sample_ddpm
    n, I, H, L, T, nh, nd = 200, 150, 64, 48, 5, 1, 1.0
    diff, vae = random_modules(I, H, L, T, nh, seed=2, device="cuda")
    a = sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=9).clone()
    diff.dnn[0].weight.data.mul_(0.5)                       # no _version bump
    vae.decoder[2].bias.data.add_(1.0)
    stale = sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=9, reuse_packed=True).clone()
    fresh = sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=9).clone()
    assert torch.equal(stale, a)                            # opted-in reuse keeps the old images (documented)
    assert not torch.equal(fresh, a)
    diff2, vae2 = random_modules(I, H, L, T, nh, seed=2, device="cuda")
    diff2.dnn[0].weight.data.mul_(0.5)
    vae2.decoder[2].bias.data.add_(1.0)
    assert torch.equal(fresh, sample_ddpm(n, diff2, vae2, L, nd, n_timesteps=T, seed=9))


def test_t_start_out_of_range_is_clamped():
    n, I, H, L, T, nh, nd = 130, 60, 32, 24, 6, 1, 1.0
    diff, vae = random_modules(I, H, L, T, nh, seed=4, device="cuda")
    eng = _engine(diff, vae, T, nd)
    t = torch.full((n,), T, dtype=torch.int32)
    ref = eng.sample(n, t_start=t.cuda(), seed=5, check=True).clone()
    bad = t.clone().cuda()
    bad[::3] = T + 1000                                     # device tensor: the host cannot validate it; the kernel clamps to T
    out = eng.sample(n, t_start=bad, seed=5, check=True)
    assert torch.equal(out, ref)
    with pytest.raises(ValueError):
        eng.sample(n, t_start=torch.full((n,), T + 1, dtype=torch.int32), seed=5)   # host tensor: validated


@pytest.mark.parametrize("shape", [
    # n, I, H, L, T, nh, nd
    (9558, 8582, 40, 40, 93, 5, 1.0),     # cfg 3 (ADM / NeuMF) at its real size and chain length
    (700, 333, 64, 64, 11, 2, 0.7),       # the widest shape the small-chain kernel takes
    (45, 50, 17, 9, 7, 0, 1.0),           # ragged, no hidden layer
    (300, 100, 24, 40, 5, 1, 1.0),        # VAE hidden narrower than the latent
])
def test_small_chain_kernel_vs_layer_engine_and_oracle(shape):
    """K6 and K1 draw the same Philox streams and round at the same points, so for the same (seed, row) they agree far inside
    the oracle tolerance; both are checked against the oracle on row slices (full chain length)."""
    from oracle import philox_ref
    from oracle import sdrm_oracle as orc
    from sdrm_b200 import _lib
    n, I, H, L, T, nh, nd = shape
    diff, vae = random_modules(I, H, L, T, nh, seed=17, device="cuda")
    eng = _engine(diff, vae, T, nd)
    seed, off = 0x5EED1234, 12345
    outs, lats = {}, {}
    for choice in (1, 2):
        eng.set_option(_lib.OPT_ENGINE, choice)
        lat = torch.empty(n, L, device="cuda")
        outs[choice] = eng.sample(n, row_offset=off, seed=seed, latent_out=lat, check=True).clone()
        lats[choice] = lat
        assert eng.lib.sdrm_last_cluster_size(eng.handle) == (0 if choice == 2 else eng.lib.sdrm_last_cluster_size(eng.handle))
    eng.set_option(_lib.OPT_ENGINE, 0)
    auto = eng.sample(n, row_offset=off, seed=seed, check=True)
    assert torch.equal(auto, outs[2])                       # automatic choice = the small-chain kernel at these widths
    assert rel_fro(outs[2].cpu(), outs[1].cpu()) < 3e-4 and rel_fro(lats[2].cpu(), lats[1].cpu()) < 3e-4
    dsd, vsd = state_dicts(diff, vae)
    for start in sorted({0, (n // 2) // 16 * 16 + 3, max(0, n - 12)}):
        rows = min(12, n - start)
        xT, z, keep = philox_ref.sampler_noise(seed, off + start, rows, L, T)
        ref = orc.sample_full(dsd, vsd, T, nd, torch.from_numpy(xT), torch.from_numpy(z), torch.from_numpy(keep))
        for choice in (1, 2):
            got = outs[choice][start:start + rows].cpu()
            assert rel_fro(got, ref) < TOL and max_scaled_err(got, ref) < TOL_MAX, (choice, start)


def test_small_chain_kernel_random_mode_and_row_ids():
    from oracle import philox_ref
    from oracle import sdrm_oracle as orc
    from sdrm_b200 import _lib
    n, I, H, L, T, nh, nd = 333, 120, 32, 40, 21, 2, 1.0
    diff, vae = random_modules(I, H, L, T, nh, seed=18, device="cuda")
    eng = _engine(diff, vae, T, nd)
    rng = np.random.RandomState(6)
    t_np = rng.randint(1, T, size=n).astype(np.int32)
    order = np.argsort(-t_np, kind="stable").astype(np.int32)
    outs = {}
    for choice in (1, 2):
        eng.set_option(_lib.OPT_ENGINE, choice)
        outs[choice] = eng.sample(n, t_start=torch.from_numpy(t_np[order]), row_ids=torch.from_numpy(order), seed=77, check=True).clone()
    xT, z, keep = philox_ref.sampler_noise(77, 0, n, L, T)
    dsd, vsd = state_dicts(diff, vae)
    ref = orc.sample_random(dsd, vsd, T, nd, torch.from_numpy(xT), torch.from_numpy(z), torch.from_numpy(keep), t_np)
    for choice in (1, 2):
        assert rel_fro(outs[choice].cpu(), ref) < TOL, choice
