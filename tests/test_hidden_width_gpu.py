"""Denoisers whose hidden width D differs from their latent width L: SDRM(N_ITEMS=L, LATENT_DIM=D), which train_SDRM builds
whenever DIFF_LATENT != VAE_LATENT.  The layers are Linear(L + T -> D), nh x the shared Linear(D -> D) and Linear(D -> L), so the
chain hands D-wide activations from layer to layer but L-wide state from step to step, and every chunk geometry, k-block count,
padded image and split-K factor of the kernels differs between the first, hidden and out layers.

  * a shape table whose premises (the chunk geometry each row is meant to exercise) are checked on the host without a GPU;
  * every sampler flow the row admits (K6, and K1's single CTAs, pairs, pairs with several tiles per CTA, interleaved sub-tiles,
    resident tiles, column split of 8 / 4 / 2) against the CPU oracle and its bf16-emulating twin, and bit for bit against the
    automatic launch; multi-resolution chains, injected noise, step grids, bfloat16 rows and the public call on chosen rows;
  * the training step's GEMMs (K5) against float64 autograd, and DiffusionTrainStep against the float64 oracle."""
import copy
import ctypes as C
from types import SimpleNamespace
from typing import Callable, NamedTuple

import numpy as np
import pytest
import torch

from helpers import max_scaled_err, rel_fro, state_dicts

TOL = 1e-3        # rel-Frobenius against the fp32 oracle (bf16 operands, fp32 accumulate)
TOL_MAX = 3e-3    # worst single element, |d| / max(1, |ref|)
TOL_EMU = 2e-4    # against the oracle that rounds where the kernels round: separates a kernel bug from bf16 effects
TOL_K6_K1 = 3e-4  # K6 and K1 round at the same points but sum in a different order
SMALL_MAX = 64    # widest latent / hidden / VAE-hidden width of the small-chain kernel (K6)
TILE_M = 128      # rows of a K1 row tile


class Row(NamedTuple):
    name: str
    n: int
    I: int
    H: int
    L: int
    D: int
    T: int
    nh: int
    nd: float
    flows: tuple          # the flows the row is meant to exercise (each one forced and proven through sdrm_last_*)
    premise: Callable     # (g, s) -> bool on the chain layers' (chunks, chunk columns, k-blocks), normal / column-split geometry
    why: str


# n, I, H, L, D, T, nh, nd.  T stays <= 9 so the CPU oracle stays fast.
ROWS = [
    Row("k6_L40_D64", 300, 150, 48, 40, 64, 7, 2, 1.0, ("k6", "single", "pair"),
        lambda g, s: g.first == (1, 64, 1) and g.out == (1, 48, 1),
        "K6: hidden images 64 wide, out image 48: padded images of different widths"),
    Row("k6_L64_D24", 333, 200, 64, 64, 24, 6, 1, 0.5, ("k6", "single", "pair"),
        lambda g, s: g.first == (1, 32, 1) and g.out == (1, 64, 1),
        "K6: latent 64, hidden 24 (the reverse)"),
    Row("k6_L9_D1_nh0", 45, 50, 17, 9, 1, 5, 0, 1.0, ("k6", "single", "pair"),
        lambda g, s: g.first == (1, 16, 1) and g.out == (1, 16, 1),
        "K6: a hidden width of 1, no hidden layer, one ragged tile"),
    Row("k1_L40_D65", 500, 300, 100, 40, 65, 6, 1, 1.0, ("single", "pair", "pair_grid", "split4", "resident_grid"),
        lambda g, s: g.first == (1, 80, 1) and g.hidden == (1, 80, 2) and g.out == (1, 48, 2),
        "hidden one column past SMALL_MAX (K1 with a latent <= 64): hidden reads 2 k-blocks, first 1"),
    Row("k1_L72_D16", 700, 300, 100, 72, 16, 5, 3, 1.0, ("single", "pair", "pair_grid", "split8", "split4", "subtiles"),
        lambda g, s: g.first == (1, 16, 2) and g.hidden == (1, 16, 1) and g.out == (1, 80, 1),
        "a single 16-column hidden chunk under an 80-column out chunk"),
    Row("pair_L264_D520", 1500, 700, 200, 264, 520, 7, 2, 1.0, ("single", "pair", "pair_grid", "split8", "split4"),
        lambda g, s: g.first == (3, 176, 5) and g.hidden == (3, 176, 9) and g.out == (2, 144, 9),
        "3 chunks of 176 feed 2 of 144 (streaming; too wide for the resident tile)"),
    Row("res_L128_D512", 1000, 500, 300, 128, 512, 5, 1, 1.0, ("resident", "resident_grid", "pair", "split8"),
        lambda g, s: g.first == (2, 256, 2) and g.out == (1, 128, 8),
        "resident: the out layer reads 8 k-blocks and writes 1 chunk"),
    Row("res_L512_D136", 1000, 400, 200, 512, 136, 5, 1, 1.0, ("resident", "resident_grid", "pair", "split8"),
        lambda g, s: g.first == (1, 144, 8) and g.out == (2, 256, 3),
        "resident, the reverse: the first layer reads 8 k-blocks and writes 1 chunk; out writes 2 of 256"),
    Row("res_L257_D256", 1000, 300, 200, 257, 256, 5, 2, 1.0, ("resident", "resident_grid", "subtiles", "pair"),
        lambda g, s: g.first == (1, 256, 5) and g.hidden == (1, 256, 4) and g.out == (2, 144, 4),
        "resident: a chunk boundary (2 x 144 out columns) over one 256-column hidden chunk"),
    Row("sub_L96_D320", 1500, 300, 128, 96, 320, 7, 2, 1.0, ("subtiles", "pair_grid", "resident"),
        lambda g, s: g.hidden == (2, 160, 5) and g.first == (2, 160, 2) and g.out == (1, 96, 5),
        "sub-tiles at w_max = 320, set by the hidden layer's k-blocks and the first layer's columns"),
    Row("sub_L320_D96", 1500, 300, 128, 320, 96, 7, 1, 1.0, ("subtiles", "pair_grid"),
        lambda g, s: g.first == (1, 96, 5) and g.out == (2, 160, 2),
        "sub-tiles at w_max = 320, set by the first layer's k-blocks and the out layer's columns"),
    Row("split_L200_D830", 843, 1008, 300, 200, 830, 6, 2, 1.0, ("split8", "split4", "pair"),
        lambda g, s: g.first == (4, 208, 4) and g.out == (1, 208, 13) and s.hidden == (8, 112, 13) and s.out == (8, 32, 13),
        "column split with nch_min = 1: posterior-owned state columns (8 x 32) narrower than the hidden chunks (8 x 112)"),
    Row("split_L830_D200", 843, 1008, 930, 830, 200, 6, 2, 1.0, ("split8", "split4", "pair"),
        lambda g, s: g.first == (1, 208, 13) and g.out == (4, 208, 4) and s.hidden == (8, 32, 4) and s.out == (8, 112, 4),
        "column split with nch_min = 1: posterior-owned state columns (8 x 112) wider than the hidden chunks (8 x 32)"),
    Row("split_L72_D1300", 500, 300, 100, 72, 1300, 4, 1, 1.0, ("split8", "split4", "pair"),
        lambda g, s: g.first == (6, 224, 2) and g.out == (1, 80, 21) and s.first == (8, 176, 2) and s.out == (8, 16, 21),
        "column split: 8 out chunks of 16 columns under 8 first-layer chunks of 176"),
    Row("split2_L600_D264", 6000, 300, 200, 600, 264, 3, 1, 1.0, ("auto_split2", "pair"),
        lambda g, s: g.first == (2, 144, 10) and g.hidden == (2, 144, 5) and g.out == (3, 208, 5),
        "47 row tiles with nch_min = 2: clusters of 2 in the normal geometry, 3 out chunks on 2 CTAs"),
    Row("nosplit_L600_D200", 6000, 300, 200, 600, 200, 3, 1, 1.0, ("auto_pair", "single"),
        lambda g, s: g.first == (1, 208, 10) and g.out == (3, 208, 4),
        "47 row tiles with nch_min = 1: must not take clusters of 2 / 4 (the single-chunk layers have no chunk to share)"),
    Row("wide_L2048_D64", 300, 700, 300, 2048, 64, 3, 1, 1.0, ("split8", "single", "pair"),
        lambda g, s: g.first == (1, 64, 32) and g.out == (8, 256, 1),
        "8 x 256 columns on the latent side only"),
    Row("wide_L64_D2048", 300, 700, 300, 64, 2048, 3, 1, 1.0, ("split8", "single", "pair"),
        lambda g, s: g.first == (8, 256, 1) and g.hidden == (8, 256, 32) and g.out == (1, 64, 32),
        "8 x 256 columns on the hidden side only (a latent <= 64: the split runs the normal geometry)"),
]
ROW = {r.name: r for r in ROWS}


def _lib_handle():
    from sdrm_b200 import _lib
    return _lib, _lib.load()


# flow -> (options that force it, (sdrm_last_cluster_size, sdrm_last_split_size, sdrm_last_resident_mode) that prove it ran;
# None = checked by the caller)
def _flows():
    from sdrm_b200 import _lib as L_
    K1 = {L_.OPT_ENGINE: 1}
    return {
        "auto": ({}, None),
        "k6": ({L_.OPT_ENGINE: 2}, (0, 0, 0)),
        "single": ({**K1, L_.OPT_CLUSTER: 1, L_.OPT_NO_SPLIT: 1}, (1, 0, 0)),
        # CTA pairs, one streaming tile per CTA; the same without the dead-buffer discard warp
        "pair": ({**K1, L_.OPT_CLUSTER: 2, L_.OPT_NO_SPLIT: 1, L_.OPT_RESIDENT: 1}, (2, 0, 0)),
        "pair_nodiscard": ({**K1, L_.OPT_CLUSTER: 2, L_.OPT_NO_SPLIT: 1, L_.OPT_RESIDENT: 1, L_.OPT_NO_DISCARD: 1}, (2, 0, 0)),
        # one CTA pair for the launch: every CTA runs its row tiles one after the other
        "pair_grid": ({**K1, L_.OPT_CLUSTER: 2, L_.OPT_NO_SPLIT: 1, L_.OPT_RESIDENT: 1, L_.OPT_SUBTILES: 1, L_.OPT_GRID_LIMIT: 2},
                      (2, 0, 0)),
        # one CTA pair, two interleaved sub-tiles per CTA
        "subtiles": ({**K1, L_.OPT_CLUSTER: 2, L_.OPT_NO_SPLIT: 1, L_.OPT_SUBTILES: 2, L_.OPT_GRID_LIMIT: 2}, (2, 0, 0)),
        # resident tile, one row tile per CTA / several in sequence on one pair
        "resident": ({**K1, L_.OPT_CLUSTER: 2, L_.OPT_NO_SPLIT: 1, L_.OPT_SUBTILES: 1}, (2, 0, 1)),
        "resident_grid": ({**K1, L_.OPT_CLUSTER: 2, L_.OPT_NO_SPLIT: 1, L_.OPT_SUBTILES: 1, L_.OPT_GRID_LIMIT: 2}, (2, 0, 1)),
        "split8": ({**K1, L_.OPT_CLUSTER: 8}, (1, 8, 0)),
        "split4": ({**K1, L_.OPT_CLUSTER: 4}, (1, 4, 0)),
        # automatic choices of many-tile launches
        "auto_split2": ({}, (1, 2, 0)),
        "auto_pair": ({}, (2, 0, 0)),
    }


def _geom(lib, N, K, split):
    a, b, c = C.c_int(), C.c_int(), C.c_int()
    assert lib.sdrm_layer_geometry(N, K, split, C.byref(a), C.byref(b), C.byref(c)) == 0
    return a.value, b.value, c.value


def _chain_geometry(lib, r):
    """(normal, column-split) geometry of the chain layers: first N = D, K = L; hidden N = K = D; out N = L, K = D"""
    return tuple(SimpleNamespace(first=_geom(lib, r.D, r.L, s), hidden=_geom(lib, r.D, r.D, s), out=_geom(lib, r.L, r.D, s))
                 for s in (0, 1))


def _admits(r, flow, g, s):
    """Whether the host plan (engine_host.cu plan_launch) can run `flow` for row r, from the chain geometry."""
    tiles = (r.n + TILE_M - 1) // TILE_M
    chain = [g.first] + ([g.hidden] if r.nh > 0 else []) + [g.out]
    nch = [c[0] for c in chain]
    kb_max = max(max(c[2], (c[0] * c[1] + 63) // 64) for c in chain)
    w_max = max(max(64 * c[2], c[0] * c[1]) for c in chain)
    wide = max(r.L, r.D) > SMALL_MAX
    # the 8-chunk images: a denoiser wider than 64 whose geometry they re-cut, and a decoder behind a latent wider than 64
    geom8 = wide and r.L > SMALL_MAX and any(getattr(g, k) != getattr(s, k) for k in ("first", "hidden", "out"))
    if flow == "k6":
        return max(r.L, r.D, r.H) <= SMALL_MAX
    if flow in ("single", "pair", "pair_nodiscard"):
        return True
    if flow == "pair_grid":
        return tiles >= 3
    if flow == "subtiles":
        return tiles >= 3 and w_max <= 320        # (the widths where the automatic plan interleaves sub-tiles)
    if flow == "resident":
        return max(nch) <= 2 and kb_max <= 8 and w_max > 128 and tiles <= 128
    if flow == "resident_grid":
        return max(nch) <= 2 and kb_max <= 8 and tiles >= 3
    if flow == "split8":
        return wide and tiles <= 16 and (geom8 or max(nch) > 4)
    if flow == "split4":
        return wide and tiles <= 16
    if flow == "auto_split2":
        return wide and tiles > 18 and min(nch) >= 2
    if flow == "auto_pair":
        return tiles > 18 and min(nch) == 1
    raise ValueError(flow)


# ------------------------------------------------------------------------------------------------------------------------------
# 1. the shape table's premises, on the host (no GPU)
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def built_lib():
    import __graft_entry__ as ge
    return C.CDLL(ge.build())


@pytest.mark.parametrize("r", ROWS, ids=lambda r: r.name)
def test_shape_table_premises(built_lib, r):
    """Each row's geometry is what the row claims, and each flow it names is one the launch plan can take for it.  If a change
    to the geometry quietly stops covering a case, this fails before any GPU run."""
    assert r.L != r.D, r.name
    g, s = _chain_geometry(built_lib, r)
    assert r.premise(g, s), (r.name, r.why, g, s)
    for f in r.flows:
        assert _admits(r, f, g, s), (r.name, f, g, s)
    small = max(r.L, r.D, r.H) <= SMALL_MAX
    assert ("k6" in r.flows) == small, r.name


def test_shape_table_covers_the_hidden_width_cases(built_lib):
    """Across the table: both orders of L and D on every flow family, nch_min = 1 under nch_max >= 3, a single 16-column chunk,
    and resident rows whose out layer reads 8 k-blocks and writes one chunk and the reverse."""
    geo = {r.name: _chain_geometry(built_lib, r) for r in ROWS}
    fams = {"k6": ("k6",), "resident": ("resident", "resident_grid"), "subtiles": ("subtiles",), "split": ("split8", "split4")}
    for fam, fl in fams.items():
        rows = [r for r in ROWS if any(f in r.flows for f in fl)]
        assert any(r.L < r.D for r in rows) and any(r.L > r.D for r in rows), fam
    nch = {k: [c[0] for c in (g.first, g.hidden, g.out)] for k, (g, _) in geo.items()}
    assert any(min(v) == 1 and max(v) >= 3 for v in nch.values())
    assert any(g.out == (1, 128, 8) for g, _ in geo.values()) and any(g.first == (1, 144, 8) for g, _ in geo.values())
    assert any(16 in (g.first[1], g.hidden[1]) for g, _ in geo.values())


# ------------------------------------------------------------------------------------------------------------------------------
# 2. sampler parity at D != L (GPU)
# ------------------------------------------------------------------------------------------------------------------------------
def _modules(r, seed):
    from sdrm_b200.models import SDRM, VAE
    torch.manual_seed(seed)
    vae = VAE(input_dim=r.I, hidden_dim=r.H, latent_dim=r.L)
    diff = SDRM(N_ITEMS=r.L, EMB_DIM=r.T, LATENT_DIM=r.D, n_hidden_layers=r.nh)
    return diff.cuda().eval(), vae.cuda().eval()


def _engine(diff, vae, T, nd):
    from sdrm_b200.engine import SamplerEngine
    from sdrm_b200.models import make_schedule
    eng = SamplerEngine()
    eng.pack_denoiser(diff, make_schedule(T, device="cuda"), nd)
    eng.pack_decoder(vae)
    return eng


def _last(eng):
    lib = eng.lib
    return (lib.sdrm_last_cluster_size(eng.handle), lib.sdrm_last_split_size(eng.handle), lib.sdrm_last_resident_mode(eng.handle))


def _run(eng, flow, n, **kw):
    """One sdrm_sample on `flow`; asserts that the launch took it, restores the automatic choice, returns (out, flow that ran)."""
    opts, want = _flows()[flow]
    try:
        for k, v in opts.items():
            eng.set_option(k, v)
        out = eng.sample(n, check=True, **kw)
        got = _last(eng)
        assert want is None or got == want, (flow, got, want)
    finally:
        for k in opts:
            eng.set_option(k, 0)
    return out, got


def _flows_of(r, g, s):
    """Every flow the row admits, the automatic launch first (the row's own flows are a subset: test_shape_table_premises)."""
    return ["auto"] + [f for f in _flows() if f != "auto" and _admits(r, f, g, s)]


def _slices(n):
    return sorted({0, (n // 2) // TILE_M * TILE_M + 19, max(0, n - 12)})   # first tile, a middle tile, the ragged last tile


def _where(got, ref):
    """(row, column) of the worst scaled error and the columns whose error exceeds the bar: which layer chunk is wrong"""
    e = (got.double() - ref.double()).abs() / ref.double().abs().clamp_min(1.0)
    i = int(e.argmax())
    bad = torch.nonzero(e.max(0).values > TOL_MAX).flatten().tolist()
    return (i // e.shape[1], i % e.shape[1]), bad[:8], len(bad)


def _auto_want(r, g, s):
    if max(r.L, r.D, r.H) <= SMALL_MAX:
        return (0, 0, 0)                                      # K6
    if _admits(r, "split8", g, s):
        return (1, 8, 0)                                      # a few row tiles of a wide denoiser: clusters of 8
    return None


@pytest.mark.gpu
@pytest.mark.parametrize("r", ROWS, ids=lambda r: r.name)
def test_every_flow_matches_the_oracle(r):
    """In-kernel Philox noise on every flow the row admits: logits and latent against orc.sample_full (fed the numpy restatement
    of the streams) and orc.sample_bf16_emulated on 12-row slices; every K1 flow bit-identical to the automatic launch (K6 vs
    K1 within TOL_K6_K1)."""
    from oracle import philox_ref
    from oracle import sdrm_oracle as orc
    lib = _lib_handle()[1]
    g, s = _chain_geometry(lib, r)
    diff, vae = _modules(r, seed=3)
    eng = _engine(diff, vae, r.T, r.nd)
    seed, off = 0x1234ABCD5678, 1000
    res = {}
    for f in _flows_of(r, g, s):
        lat = torch.empty(r.n, r.L, device="cuda")
        out, got = _run(eng, f, r.n, row_offset=off, seed=seed, latent_out=lat)
        assert torch.isfinite(out).all(), f
        res[f] = (out.cpu(), lat.cpu(), got)
    want = _auto_want(r, g, s)
    assert want is None or res["auto"][2] == want, (res["auto"][2], want)
    # flow identity: K1 flows bit for bit, K6 launches bit for bit, K6 against K1 within its summation-order bar
    k1 = [f for f in res if res[f][2] != (0, 0, 0)]
    k6 = [f for f in res if res[f][2] == (0, 0, 0)]
    for fl in (k1, k6):
        for f in fl[1:]:
            assert torch.equal(res[f][0], res[fl[0]][0]) and torch.equal(res[f][1], res[fl[0]][1]), (fl[0], f)
    if "k6" in res:
        assert rel_fro(res["k6"][0], res[k1[0]][0]) < TOL_K6_K1 and rel_fro(res["k6"][1], res[k1[0]][1]) < TOL_K6_K1
    dsd, vsd = state_dicts(diff, vae)
    worst = dict(fro=0.0, max=0.0, lat=0.0, emu=0.0)
    for start in _slices(r.n):
        rows = min(12, r.n - start)
        xT, z, keep = (torch.from_numpy(a) for a in philox_ref.sampler_noise(seed, off + start, rows, r.L, r.T))
        ref, ref_lat = orc.sample_full(dsd, vsd, r.T, r.nd, xT, z, keep, return_latent=True)
        emu = orc.sample_bf16_emulated(dsd, vsd, r.T, r.nd, xT, z, keep)
        for f, (out, lat, _) in res.items():
            got, got_lat = out[start:start + rows], lat[start:start + rows]
            e = dict(fro=rel_fro(got, ref), max=max_scaled_err(got, ref), lat=rel_fro(got_lat, ref_lat), emu=rel_fro(got, emu))
            for k in worst:
                worst[k] = max(worst[k], e[k])
            assert e["fro"] < TOL and e["max"] < TOL_MAX and e["lat"] < TOL and e["emu"] < TOL_EMU, \
                (f, start, e, "logits", _where(got, ref), "latent", _where(got_lat, ref_lat))
    print(f"{r.name}: auto {res['auto'][2]} flows {[f for f in res if f != 'auto']}: rel-Frobenius {worst['fro']:.2e} "
          f"scaled max {worst['max']:.2e} latent {worst['lat']:.2e} vs bf16 emulation {worst['emu']:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["split_L200_D830", "res_L128_D512", "k6_L40_D64"])
def test_multiresolution_chains_match_the_oracle(name):
    """Per-row start steps in [0, T] (0: the row decodes x_T) against orc.sample_random on every flow that takes them (the
    resident and sub-tile flows run full-resolution chains only); the K1 flows bit for bit."""
    from oracle import philox_ref
    from oracle import sdrm_oracle as orc
    r = ROW[name]
    lib = _lib_handle()[1]
    g, s = _chain_geometry(lib, r)
    diff, vae = _modules(r, seed=8)
    eng = _engine(diff, vae, r.T, r.nd)
    t_np = np.random.RandomState(4).randint(0, r.T + 1, size=r.n).astype(np.int32)
    seed = 321
    flows = [f for f in _flows_of(r, g, s) if f in ("auto", "k6", "single", "pair", "pair_grid", "split8", "split4")]
    outs = {}
    for f in flows:
        out, got = _run(eng, f, r.n, t_start=torch.from_numpy(t_np).cuda(), seed=seed)
        outs[f] = (out.cpu(), got)
    xT, z, keep = (torch.from_numpy(a) for a in philox_ref.sampler_noise(seed, 0, r.n, r.L, r.T))
    dsd, vsd = state_dicts(diff, vae)
    ref = orc.sample_random(dsd, vsd, r.T, r.nd, xT, z, keep, t_np)
    worst = 0.0
    for f, (out, _) in outs.items():
        e = rel_fro(out, ref)
        worst = max(worst, e)
        assert e < TOL and max_scaled_err(out, ref) < TOL_MAX, (f, e, _where(out, ref))
    k1 = [f for f in outs if outs[f][1] != (0, 0, 0)]
    for f in k1[1:]:
        assert torch.equal(outs[f][0], outs[k1[0]][0]), (k1[0], f)
    print(f"{name} multi-resolution: flows {[(f, outs[f][1]) for f in outs]} worst rel-Frobenius {worst:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["split_L72_D1300", "split_L830_D200"])
def test_injected_noise_split_equals_one_cta_per_tile(name):
    """Injected x_T / z / keep tensors: the column split and the one-CTA-per-tile flow give the same rows and latent bit for bit,
    and the rows of the in-kernel streams they restate within MUFU Box-Muller rounding."""
    from oracle import philox_ref
    r = ROW[name]
    diff, vae = _modules(r, seed=13)
    eng = _engine(diff, vae, r.T, r.nd)
    inj = dict(zip(("inj_xT", "inj_z", "inj_keep"),
                   (torch.from_numpy(t).cuda().contiguous() for t in philox_ref.sampler_noise(21, 0, r.n, r.L, r.T))))
    lat = [torch.empty(r.n, r.L, device="cuda") for _ in range(2)]
    a, got = _run(eng, "auto", r.n, seed=0, latent_out=lat[0], **inj)
    assert got == (1, 8, 0), got
    b, _ = _run(eng, "pair", r.n, seed=0, latent_out=lat[1], **inj)
    p, _ = _run(eng, "auto", r.n, seed=21)
    assert torch.equal(a, b) and torch.equal(lat[0], lat[1])
    assert rel_fro(a.cpu(), p.cpu()) < 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["sub_L96_D320", "k6_L64_D24"])
def test_step_grids_and_bf16_rows(name):
    """A strided DDPM grid and a DDIM grid against tests/grid_oracle.py (injected slabs and in-kernel Philox), and bfloat16 rows
    equal to the rounded fp32 rows, on the default chain and on a grid."""
    import grid_oracle as go
    from oracle import philox_ref
    from sdrm_b200.train_SDRM import step_grid
    r = ROW[name]
    lib = _lib_handle()[1]
    g, s = _chain_geometry(lib, r)
    diff, vae = _modules(r, seed=42)
    eng = _engine(diff, vae, r.T, r.nd)
    dsd, vsd = state_dicts(diff, vae)
    n, off, seed = 300, 64, 0x6121D
    flows = [f for f in _flows_of(r, g, s) if f in ("auto", "k6", "single", "pair", "subtiles", "resident")]
    for tau, eta in ((step_grid(r.T, 3).tolist(), None), ([2, 3, r.T], 0.5), (None, None)):
        eng.set_step_grid(tau, eta)
        S = r.T if tau is None else len(tau)
        xT, z, keep = (torch.from_numpy(a) for a in philox_ref.sampler_noise(seed, off, n, r.L, S))
        inj = dict(inj_xT=xT.cuda(), inj_z=z.cuda(), inj_keep=keep.cuda())
        grid = list(range(1, r.T + 1)) if tau is None else tau
        refs = {st: go.sample_grid(dsd, vsd, r.T, r.nd, xT[st:st + 12], z[:, st:st + 12], keep[:, st:st + 12], grid, eta)
                for st in _slices(n)}
        emus = {st: go.sample_bf16_emulated_grid(dsd, vsd, r.T, r.nd, xT[st:st + 12], z[:, st:st + 12], keep[:, st:st + 12], grid,
                                                 eta) for st in _slices(n)}
        for f in flows:
            out_i, _ = _run(eng, f, n, row_offset=off, **inj)
            out_p, _ = _run(eng, f, n, row_offset=off, seed=seed)
            bf, _ = _run(eng, f, n, row_offset=off, seed=seed, out=torch.empty(n, r.I, dtype=torch.bfloat16, device="cuda"))
            assert torch.equal(bf.view(torch.int16), out_p.to(torch.bfloat16).view(torch.int16)), (f, tau, eta)
            for o in (out_i.cpu(), out_p.cpu()):
                for st, ref in refs.items():
                    got = o[st:st + 12]
                    assert rel_fro(got, ref) < TOL and max_scaled_err(got, ref) < TOL_MAX, (f, tau, eta, st, rel_fro(got, ref))
                    assert rel_fro(got, emus[st]) < TOL_EMU, (f, tau, eta, st, rel_fro(got, emus[st]))
    eng.set_step_grid(None)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["res_L512_D136", "k6_L64_D24"])
def test_public_call_at_hidden_width(name):
    """sample_ddpm(n, diff, vae, L) returns the engine's rows; the hidden width in the latent-width argument is an error."""
    from sdrm_b200.train_SDRM import sample_ddpm
    r = ROW[name]
    diff, vae = _modules(r, seed=2)
    out = sample_ddpm(r.n, diff, vae, r.L, r.nd, n_timesteps=r.T, seed=9)
    assert out.shape == (r.n, r.I) and torch.isfinite(out).all()
    ref = _engine(diff, vae, r.T, r.nd).sample(r.n, seed=9, check=True)
    assert torch.equal(out, ref)
    with pytest.raises(ValueError):
        sample_ddpm(r.n, diff, vae, r.D, r.nd, n_timesteps=r.T, seed=9)


# ------------------------------------------------------------------------------------------------------------------------------
# 3. the training step at D != L (GPU)
# ------------------------------------------------------------------------------------------------------------------------------
def _wgrad_splits(M, N, K, clusters):
    """train_gemm.cu wgrad_splits: the split-K factor of a weight-gradient product"""
    nt = (N + 255) // 256
    tiles = (M + 255) // 256 * nt
    kb = (K + 63) // 64
    s = min(max(1, clusters // max(1, tiles)), min(kb, 8))
    per = (kb + s - 1) // s
    return (kb + per - 1) // per


def _train_workspace_bytes(R, L, D, nh, clusters):
    """train_gemm.cu make_layout's total for a given count of resident GEMM pairs"""
    up64 = lambda x: (x + 63) // 64 * 64
    a256 = lambda b: (b + 255) & ~255
    pair = lambda rows, ld: a256(rows * ld * 4)
    Rp, Lp, Dp = up64(R), up64(L), up64(D)
    Wp, Wmax = max(Lp, Dp), max(L, D)
    n_slabs = max(max(nh, 1) * _wgrad_splits(D, D, R, clusters), _wgrad_splits(L, D, R, clusters), _wgrad_splits(D, L, R, clusters))
    parts = [256, pair(R, Lp)] + [R * Dp * 4, pair(R, Dp)] * (nh + 1) + [pair(D, Lp), pair(D, Dp), pair(L, Dp), pair(D, Dp), pair(D, Lp)]
    parts += [R * Wp * 4, pair(R, Wp)] * 2 + [pair(Wmax, Rp), pair(Wmax, Rp), Wp * 16, n_slabs * Wmax * Wp * 4]
    return sum(a256(p) for p in parts)


def _fwd_bwd_report(L, D, T, nh, B, slopes):
    from sdrm_b200.models import SDRM
    from sdrm_b200.training import denoiser_gemms
    torch.manual_seed(L + 3 * D + T)
    net = SDRM(N_ITEMS=L, EMB_DIM=T, LATENT_DIM=D, n_hidden_layers=nh).cuda()
    with torch.no_grad():
        net.dnn[1].weight.fill_(slopes[0])
        if nh > 0:
            net.dnn[3].weight.fill_(slopes[1])
    rows = 3 * B
    x = torch.randn(rows, L, device="cuda") * (torch.rand(rows, L, device="cuda") < 0.5) * 2.0
    t = torch.randint(1, T + 1, (B,), device="cuda").repeat(3)
    g_out = torch.randn(rows, L, device="cuda") / rows

    net.zero_grad()
    out = denoiser_gemms(net, x, t, passes=3)
    (out * g_out).sum().backward()
    got = {k: p.grad.detach().clone() for k, p in net.named_parameters()}

    ref_net = SDRM(N_ITEMS=L, EMB_DIM=T, LATENT_DIM=D, n_hidden_layers=nh).cuda().double()
    ref_net.load_state_dict({k: v.double() for k, v in net.state_dict().items()})
    emb = ref_net.emb_layer(ref_net.timestep_embedding(t, T).double())      # SDRM.forward in float64, layer by layer
    h, prelu_io = torch.cat([x.double(), emb], dim=-1), []
    for m in ref_net.dnn:
        if isinstance(m, torch.nn.PReLU):
            pre, h = h, m(h)
            h.retain_grad()
            prelu_io.append((m, pre, h))
        else:
            h = m(h)
    ref_out = h
    (ref_out * g_out.double()).sum().backward()
    assert (out.double() - ref_out).abs().max().item() <= 2e-5, (out.double() - ref_out).abs().max().item()
    # A PReLU slope's gradient is one sum over every application, row and column of dh * min(pre, 0).  Its rounding error scales
    # with the sum of the terms' magnitudes, not with the sum: when the terms cancel, even a float32 evaluation of the same
    # network misses the float64 value by far more than its usual ~1e-6 (6e-5 of the hidden slope's gradient at L = 830,
    # D = 300, nh = 2 on a B200).  The slopes are judged against the larger of the two scales; every other gradient against its max.
    term_mag, term_sum = {}, {}
    for m, pre, y in prelu_io:
        terms = y.grad * pre.clamp(max=0.0)
        term_mag[id(m.weight)] = term_mag.get(id(m.weight), 0.0) + terms.abs().sum().item()
        term_sum[id(m.weight)] = term_sum.get(id(m.weight), 0.0) + terms.sum().item()
    for m, _, _ in prelu_io:   # (the terms are the slope's gradient)
        assert abs(term_sum[id(m.weight)] - m.weight.grad.item()) <= 1e-9 * term_mag[id(m.weight)]
    mx, fro = {}, {}
    for k, p in ref_net.named_parameters():
        d = got[k].double() - p.grad
        mx[k] = d.abs().max().item() / (max(p.grad.abs().max().item(), term_mag.get(id(p), 0.0)) + 1e-30)
        fro[k] = d.norm().item() / (p.grad.norm().item() + 1e-30)
    cancel = {k: term_mag[id(p)] / (p.grad.abs().item() + 1e-30) for k, p in ref_net.named_parameters() if id(p) in term_mag}
    # the split-K factors of the three weight gradients: the restated layout that reproduces the library's workspace size names
    # the count of resident GEMM pairs, hence the factors (W0 [D, L], Wh [D, D], Wo [L, D])
    from sdrm_b200 import _lib
    ws = _lib.load().sdrm_denoiser_train_workspace_bytes(rows, L, D, nh)
    split = sorted({(_wgrad_splits(D, L, rows, c), _wgrad_splits(D, D, rows, c), _wgrad_splits(L, D, rows, c))
                    for c in range(1, 257) if _train_workspace_bytes(rows, L, D, nh, c) == ws})
    assert split, "restated training layout does not reproduce the library's workspace size"
    print(f"L={L} D={D} T={T} nh={nh} B={B} slopes={slopes}: split-K (W0, Wh, Wo) {split}; worst max|d|/max|grad| "
          f"{max(mx.values()):.2e} ({max(mx, key=mx.get)}), worst rel-Frobenius {max(fro.values()):.2e}; slope-gradient "
          f"cancellation sum|terms| / |sum| {', '.join(f'{k} {v:.0f}' for k, v in cancel.items())}")
    return mx, fro


K5_SHAPES = [(24, 40, 7, 2, 12), (40, 24, 9, 5, 30), (150, 520, 43, 1, 100), (520, 150, 43, 1, 100), (830, 300, 83, 2, 550),
             (150, 1000, 7, 3, 1000)]


@pytest.mark.gpu
@pytest.mark.parametrize("L,D,T,nh,B", K5_SHAPES)
def test_denoiser_fwd_bwd_linear_slopes(L, D, T, nh, B):
    """PReLU slopes = 1 (no kink): every gradient within 2e-4 of its max against float64 autograd -- the transposed images
    WoT [D, L] and WhT, the L- and D-row operand transposes, and three different split-K factors with their slab reductions."""
    mx, _ = _fwd_bwd_report(L, D, T, nh, B, (1.0, 1.0))
    bad = {k: v for k, v in mx.items() if v > 2e-4}
    assert not bad, (bad, mx)


@pytest.mark.gpu
@pytest.mark.parametrize("slopes", [(0.21, 0.33), (-0.5, 1.5)])
@pytest.mark.parametrize("L,D,T,nh,B", K5_SHAPES[:2])
def test_denoiser_fwd_bwd_real_slopes_small(L, D, T, nh, B, slopes):
    mx, _ = _fwd_bwd_report(L, D, T, nh, B, slopes)
    bad = {k: v for k, v in mx.items() if v > 2e-4}
    assert not bad, (bad, mx)


@pytest.mark.gpu
@pytest.mark.parametrize("L,D,T,nh,B", [K5_SHAPES[4], K5_SHAPES[5]])
def test_denoiser_fwd_bwd_real_slopes_large(L, D, T, nh, B):
    """Real slopes among millions of pre-activations: a few sit within rounding distance of the PReLU kink and flip its
    derivative relative to float64, so the layers below the last PReLU take the relative-Frobenius bar; the out layer keeps 2e-4."""
    mx, fro = _fwd_bwd_report(L, D, T, nh, B, (0.21, 0.33))
    last = f"dnn.{2 + 2 * nh}."
    bad = {k: (mx[k], fro[k]) for k in mx if (mx[k] > 2e-4 if k.startswith(last) else fro[k] > 1e-2)}
    assert not bad, (bad, mx, fro)


def _step_case(L, D, T, nh, B, seed):
    from sdrm_b200.models import SDRM
    torch.manual_seed(seed)
    diff = SDRM(N_ITEMS=L, EMB_DIM=T, LATENT_DIM=D, n_hidden_layers=nh).cuda()
    g = torch.Generator().manual_seed(seed)
    return diff, torch.randn(B, L, generator=g) * 0.5, torch.randint(1, T + 1, (B,), generator=g)


def _oracle_loss_and_grads(diff, mu, t, noise, keeps, T):
    from oracle import sdrm_oracle as orc
    ref = copy.deepcopy(diff).cpu().double()
    for p in ref.parameters():
        p.grad = None
    loss, _ = orc.training_loss(ref.state_dict(keep_vars=True), mu.double(), t, noise.double(), torch.as_tensor(keeps), T)
    loss.backward()
    return loss.item(), {k: p.grad for k, p in ref.named_parameters()}


def _step(stepper, mu, t, **inj):
    stepper.net.zero_grad()
    loss = stepper.loss(mu, t, **inj)
    loss.backward()
    return loss.item(), {k: p.grad.detach().clone() for k, p in stepper.net.named_parameters()}


@pytest.mark.gpu
@pytest.mark.parametrize("L,D,T,nh,B,grad_rel", [(24, 40, 7, 2, 17, 2e-4), (200, 520, 43, 2, 301, None)])
def test_production_training_step_matches_oracle(L, D, T, nh, B, grad_rel):
    """DiffusionTrainStep.loss(mu, t) with nothing injected equals the step fed its own streams (noise from a masked noise_inputs
    call, masks from the restatement), and both match the float64 oracle: the loss within 2e-5 and, at the small shape, every
    gradient within 2e-4 of its largest entry.  (At the mid shape the upstream gradients are near-cancelling sums weighed by
    1 / mu_coef^2, which amplifies the GEMM operands' rounding: there the loss and the injected-step identity are checked.)"""
    from oracle import philox_ref
    from oracle import sdrm_oracle as orc
    from sdrm_b200.training import CudaLossBackend, DiffusionTrainStep
    backend = CudaLossBackend()
    nd, mu_coef = 1.0, 0.1
    diff, mu, t = _step_case(L, D, T, nh, B, seed=L + D)
    diff.train()
    ab = orc.make_schedule(T)[2]
    base = 1 << 40 | 777
    stepper = DiffusionTrainStep(diff, ab.cuda(), T, nd, seed=base)
    for step in range(2):
        noise, _, _, _, masks = backend.noise_inputs(mu.cuda(), t.cuda(), ab.float().cuda(), nd, mu_coef, base + step, 0, want_masks=True)
        keeps = philox_ref.train_keep_masks(base + step, 0, B, L)
        assert np.array_equal(masks.cpu().numpy(), keeps)
        loss, grads = _step(stepper, mu.cuda(), t.cuda())
        idx = stepper.step_index
        loss_inj, grads_inj = _step(stepper, mu.cuda(), t.cuda(), inj_noise=noise, inj_masks=torch.from_numpy(keeps).cuda())
        stepper.step_index = idx
        assert abs(loss - loss_inj) <= 1e-6 * abs(loss_inj), (loss, loss_inj)
        for k, gr in grads.items():
            assert (gr - grads_inj[k]).abs().max().item() <= 1e-5 * (grads_inj[k].abs().max().item() + 1e-30), k
        ref_loss, ref_grads = _oracle_loss_and_grads(diff, mu, t, noise.cpu(), keeps, T)
        assert abs(loss - ref_loss) <= 2e-5 * max(1.0, abs(ref_loss)), (loss, ref_loss)
        errs = {k: (gr.cpu().double() - ref_grads[k]).abs().max().item() / (ref_grads[k].abs().max().item() + 1e-12)
                for k, gr in grads.items()}
        print(f"L={L} D={D} B={B} step {step}: loss {loss:.6f} vs oracle {ref_loss:.6f}; worst gradient "
              f"{max(errs.values()):.2e} ({max(errs, key=errs.get)})")
        if grad_rel:
            bad = {k: v for k, v in errs.items() if v > grad_rel}
            assert not bad, bad
