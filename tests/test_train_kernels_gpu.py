"""K2 training-step kernels on the paths a real training step takes.

`DiffusionTrainStep.loss(mu)` calls `sdrm_noise_inputs` with no injected noise and no mask output, which is the interior-block
fast path of `noise_inputs_kernel` whenever the batch starts on a 16-byte boundary of the global stream.  `ScoreMatchingLoss`
passes `pred`, `sx` and `psx` as row slices of one [3B, L] buffer, so an odd-sized minibatch sends `sdrm_loss_stats` and
`sdrm_loss_grad_seeds` through their unaligned loads.  Data-parallel ranks start at row offsets that may put one rank on each
path.  Every case below is compared with the numpy Philox restatement, a float64 recomputation or the float64 oracle, and names
(and asserts) the path it reaches.

Not covered: B * L > 2^31 local elements (the 64-bit row division of the noising kernel needs more than 40 GB of buffers).
"""
import copy

import numpy as np
import pytest
import torch

from conftest import TRAIN_GOLDENS, load_golden
from helpers import modules_from_golden, random_modules
from oracle import philox_ref
from oracle import sdrm_oracle as orc

pytestmark = pytest.mark.gpu

T_SCHED, ND, MU_COEF, SEED = 43, 0.2, 0.1, 0x5EED_1234_ABCD
MU_COEF32 = float(np.float32(MU_COEF))          # the kernel takes mu_coef as a float
SENTINEL = -12345.5


@pytest.fixture(scope="module")
def lib():
    from sdrm_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module")
def backend():
    from sdrm_b200.training import CudaLossBackend
    return CudaLossBackend()


def _ptr(x):
    from sdrm_b200 import _lib
    return _lib.ptr(x)


def _stream():
    from sdrm_b200 import _lib
    return _lib.stream_ptr()


def _check(rc, what):
    from sdrm_b200 import _lib
    _lib.check(rc, what)


def _ab(T=T_SCHED):
    return orc.make_schedule(T)[2].float().cuda()


def _inputs(B, L, seed):
    """mu ~ N(0, 1) and timesteps in [1, T] with t[b] != t[b + 1] everywhere, so a quad that straddles two rows mixes two
    different schedule coefficients."""
    g = torch.Generator().manual_seed(seed)
    mu = torch.randn(B, L, generator=g)
    step = torch.randint(1, T_SCHED, (B,), generator=g)
    t = 1 + torch.cumsum(step, 0) % T_SCHED
    return mu.cuda(), t.cuda()


# ---------------------------------------------------------------------------------------------------------------------------
# A. sdrm_noise_inputs with in-kernel Philox streams
# ---------------------------------------------------------------------------------------------------------------------------
def _offset(L, cls):
    """A row offset of class `cls` for width L, or None when no offset of that class exists for this L."""
    if cls == "off0":
        return 0
    if cls == "q0":      # row_offset * L = 0 (mod 4), != 0 (mod 512): partial head block, fast interior blocks
        cands = [o for o in range(37, 37 + 2048) if (o * L) % 4 == 0 and (o * L) % 512 != 0]
    elif cls == "q2":    # row_offset * L = 2 (mod 4): the batch starts inside a quad; no block takes the fast path
        cands = [o for o in range(37, 37 + 64) if (o * L) % 4 == 2]
    elif cls == "hi32":  # row_offset * L >= 2^32: the Philox counters' high word c1 is non-zero (fast path where L >= 4)
        base = (1 << 32) // L + 3
        cands = [o for o in range(base, base + 2048) if (o * L) % 4 == 0]
        cands = [o for o in cands if (o * L) % 512 != 0] or cands
    else:
        raise ValueError(cls)
    return cands[0] if cands else None


# L < 4 takes the per-element schedule lookup; 830 and 950 are the cfg-1 and cfg-5 latent widths.  B gives a ragged last
# 512-element block (except L = 2048, whose rows are whole blocks) and, where L allows it, B * L % 4 != 0.
WIDTHS = [(1, 2999), (2, 1501), (3, 1001), (4, 777), (5, 613), (20, 157), (24, 131), (150, 37), (830, 13), (950, 11), (2048, 5)]
NOISE_CASES = [pytest.param(L, B, cls, id=f"L{L}-B{B}-{cls}-BLmod4_{(B * L) % 4}")
               for L, B in WIDTHS for cls in ("off0", "q0", "q2", "hi32") if _offset(L, cls) is not None]


def _has_interior_block(g0, total):
    first = -(-g0 // 512) * 512
    return first + 512 <= g0 + total


def _recompute64(mu, t, ab, noise):
    """float64 x_t, x_p and the scale each is bounded by, from the kernel's own fp32 noise and the fp32 schedule."""
    mu64, nz64 = mu.double().cpu(), noise.double().cpu()
    abt = ab.double().cpu()[t.cpu()][:, None]
    sa, om = abt.sqrt(), 1.0 - abt
    xt = sa * mu64 + om * nz64
    xq = mu64 + MU_COEF32 * nz64
    return xt, (sa * mu64).abs() + (om * nz64).abs(), xq, mu64.abs() + (MU_COEF32 * nz64).abs()


@pytest.mark.parametrize("L,B,cls", NOISE_CASES)
def test_noise_inputs_fast_and_general_paths_match_restatement(backend, L, B, cls):
    off = _offset(L, cls)
    g0, total = off * L, B * L
    if cls in ("off0", "q0", "hi32"):
        assert g0 % 4 == 0
    if cls == "q0":
        assert g0 % 512 != 0
    if cls == "q2":
        assert g0 % 4 == 2
    if cls == "hi32":
        assert g0 >= 1 << 32
    fast_reached = g0 % 4 == 0 and L >= 4 and _has_interior_block(g0, total)
    if L >= 4 and g0 % 4 == 0:
        assert fast_reached, "case should reach the fast path"
    mu, t = _inputs(B, L, seed=L * 1000 + B)
    ab = _ab()
    fast = backend.noise_inputs(mu, t, ab, ND, MU_COEF, SEED, off, want_masks=False)
    gen = backend.noise_inputs(mu, t, ab, ND, MU_COEF, SEED, off, want_masks=True)
    # 1. the mask-less call (fast path on interior blocks) and the masked call (general path) produce the same bits
    for k, name in enumerate(("noise", "in_pert", "in_clean", "in_shift")):
        assert torch.equal(fast[k], gen[k]), f"{name}: fast path != general path"
    noise, in_pert, in_clean, in_shift, masks = gen
    # 2. against the restatement: masks exactly, noise to the MUFU Box-Muller tolerance
    keep_ref = philox_ref.train_keep_masks(SEED, off, B, L)
    assert np.array_equal(masks.cpu().numpy(), keep_ref)
    assert abs(keep_ref.mean() - 0.5) < 0.05
    z = philox_ref.train_normals(SEED, off, B, L) * np.float32(ND)
    assert np.allclose(noise.cpu().numpy(), z, rtol=2e-5, atol=2e-6)
    # denoiser inputs from the kernel's own noise, t and ab_t in float64
    xt, xt_scale, xq, xq_scale = _recompute64(mu, t, ab, noise)
    keep = torch.from_numpy(keep_ref).double()
    assert ((in_pert.cpu().double() - 2 * keep[0] * xt).abs() <= 1e-6 * 2 * xt_scale).all()
    assert torch.equal(in_clean.cpu(), (2 * keep[1] * mu.cpu().double()).float())        # 2 * keep * mu is exact in fp32
    assert ((in_shift.cpu().double() - 2 * keep[2] * xq).abs() <= 1e-6 * 2 * xq_scale).all()
    # the fast path writes no masks: its keep bits, read back from the inputs it zeroed, are the restatement's
    for k, (x, undropped) in enumerate(((fast[1], xt), (fast[2], mu.cpu().double()), (fast[3], xq))):
        live = undropped != 0
        assert torch.equal((x.cpu() != 0)[live], keep[k].bool()[live]), f"keep bits of input {k}"
    # quads that straddle two rows with different t are among the checked entries
    if L % 4 != 0 and L >= 4:
        ends = (off + torch.arange(1, B)) * L
        assert bool((ends % 4 != 0).any()) and bool((t[1:] != t[:-1]).all())


SHARD_CASES = [pytest.param(L, B, cls, id=f"L{L}-B{B}-{cls}") for L, B in WIDTHS for cls in ("off0", "hi32")]


@pytest.mark.parametrize("L,B,cls", SHARD_CASES)
def test_noise_inputs_row_shards_concatenate_to_the_whole_launch(backend, L, B, cls):
    """Data-parallel ranks generate their rows at their own row_offset; the union must be the one-GPU launch, bit for bit,
    whichever path each shard's blocks take."""
    from sdrm_b200.distributed import shard_bounds
    off = _offset(L, cls)
    mu, t = _inputs(B, L, seed=L * 7 + B)
    ab = _ab()
    whole = backend.noise_inputs(mu, t, ab, ND, MU_COEF, SEED, off)
    splits = [[0, s, B] for s in sorted({1, 2, 3, B // 2, B // 2 + 1, B - 1}) if 0 < s < B]
    splits.append(sorted({shard_bounds(B, r, 3)[0] for r in range(3)} | {B}))
    aligned_starts = set()
    for bounds in splits:
        parts = []
        for lo, hi in zip(bounds[:-1], bounds[1:]):
            aligned_starts.add(((off + lo) * L) % 4 == 0)
            parts.append(backend.noise_inputs(mu[lo:hi].contiguous(), t[lo:hi].contiguous(), ab, ND, MU_COEF, SEED, off + lo))
        for k in range(4):
            assert torch.equal(torch.cat([p[k] for p in parts]), whole[k]), (bounds, k)
    if L % 4 != 0:
        assert aligned_starts == {True, False}, "the shards should start on both paths"


PLACEMENT_CASES = [pytest.param(L, B, cls, id=f"L{L}-B{B}-{cls}")
                   for L, B, cls in ((1, 2999, "off0"), (5, 613, "q0"), (24, 131, "off0"), (150, 37, "q2"), (950, 11, "hi32"),
                                     (2048, 5, "off0"))]


def _guarded(n, dtype, lead, guard=8):
    """A sentinel-filled buffer and a view of n elements starting `lead` elements after a guard band."""
    fill = SENTINEL if dtype == torch.float32 else 0xA5
    buf = torch.full((guard + lead + n + guard,), fill, dtype=dtype, device="cuda")
    return buf, buf[guard + lead: guard + lead + n], guard + lead


@pytest.mark.parametrize("L,B,cls", PLACEMENT_CASES)
def test_noise_inputs_buffer_placement(lib, backend, L, B, cls):
    """Offset and misaligned pointers the Python backend never produces, and a null noise_out: the same values as the aligned
    call, and not one element written outside the outputs."""
    off = _offset(L, cls)
    n = B * L
    mu, t = _inputs(B, L, seed=L + B)
    ab = _ab()
    ref = backend.noise_inputs(mu, t, ab, ND, MU_COEF, SEED, off, want_masks=True)
    for lead in (1, 0):      # lead 1: every pointer 4 bytes past a 16-byte boundary (general path); 0: aligned, fast path
        mu_buf = torch.zeros(n + 8, device="cuda")
        mu_v = mu_buf[lead: lead + n]
        mu_v.copy_(mu.reshape(-1))
        outs = [_guarded(n, torch.float32, lead) for _ in range(3)]
        mask_buf, mask_v, mask_at = _guarded(3 * n, torch.uint8, 3 * lead)
        want_masks = lead == 1
        assert (mu_v.data_ptr() % 16 == 4 * lead) and all(o[1].data_ptr() % 16 == 4 * lead for o in outs)
        rc = lib.sdrm_noise_inputs(_ptr(mu_v), _ptr(t), _ptr(ab), B, L, ND, MU_COEF, SEED, off, None, None, None,
                                   _ptr(outs[0][1]), _ptr(outs[1][1]), _ptr(outs[2][1]), _ptr(mask_v) if want_masks else None,
                                   _stream())
        _check(rc, "sdrm_noise_inputs")
        for k, (buf, view, at) in enumerate(outs):
            assert torch.equal(view.view(B, L), ref[k + 1]), (lead, k)
            assert (buf[:at] == SENTINEL).all() and (buf[at + n:] == SENTINEL).all(), f"guard written (lead {lead}, output {k})"
        if want_masks:
            assert torch.equal(mask_v.view(3, B, L), ref[4])
        assert (mask_buf[:mask_at] == 0xA5).all() and (mask_buf[mask_at + 3 * n:] == 0xA5).all()


# ---------------------------------------------------------------------------------------------------------------------------
# B. sdrm_loss_stats / sdrm_loss_grad_seeds
# ---------------------------------------------------------------------------------------------------------------------------
def _loss_operands(B, L, seed, mu_lead=1, r_mean=0.0, r_std=0.5):
    """pred, sx, psx as row slices of one [3B, L] buffer (the layout ScoreMatchingLoss passes) and mu as a view `mu_lead`
    elements into its buffer; pred = mu + r with r ~ N(r_mean, r_std)."""
    g = torch.Generator().manual_seed(seed)
    mu_h = torch.randn(B, L, generator=g)
    r = torch.randn(B, L, generator=g) * r_std + r_mean
    buf = torch.empty(3 * B, L, device="cuda")
    buf[:B] = (mu_h + r).cuda()
    buf[B:] = (torch.randn(2 * B, L, generator=g) * 0.5).cuda()
    mu_buf = torch.empty(B * L + 4, device="cuda")
    mu = mu_buf[mu_lead: mu_lead + B * L].view(B, L)
    mu.copy_(mu_h)
    return buf[:B], buf[B:2 * B], buf[2 * B:], mu


def _stats64(pred, sx, psx, mu):
    p, s, q, m = (v.double() for v in (pred, sx, psx, mu))
    r = p - m
    sd = (q - s) / float(np.float32(MU_COEF * MU_COEF))
    return torch.stack([r.sum(), (r * r).sum(), ((sd - r) ** 2).sum(), ((r - s) ** 2).sum()]).cpu(), r.abs().sum().item()


def _check_stats(st, pred, sx, psx, mu):
    ref, abs_r = _stats64(pred, sx, psx, mu)
    st = st.cpu()
    assert abs(st[0].item() - ref[0].item()) <= 1e-6 * abs_r
    for k in (1, 2, 3):
        assert abs(st[k].item() - ref[k].item()) <= 1e-6 * ref[k].item(), k
    assert st[4].item() == pred.numel()


def _check_seeds_vs_oracle(seeds, pred, sx, psx, mu, loss_rtol=1e-5):
    g_pred, g_sx, g_psx, loss = seeds
    o_pred, o_sx, o_psx, o_loss = orc.loss_grad_seeds(pred.cpu(), sx.cpu(), psx.cpu(), mu.cpu())
    assert abs(loss.item() - float(o_loss)) <= loss_rtol * abs(float(o_loss)), (loss.item(), float(o_loss))
    for a, b in ((g_pred, o_pred), (g_sx, o_sx), (g_psx, o_psx)):
        assert (a.cpu().double() - b).abs().max().item() <= 1e-4 * b.abs().max().item()


@pytest.mark.parametrize("B,L", [pytest.param(17, 21, id="17x21-BLmod4_1"), pytest.param(393, 830, id="393x830-BLmod4_2"),
                                 pytest.param(13, 23, id="13x23-BLmod4_3"), pytest.param(17, 20, id="17x20-BLmod4_0-mu_unaligned")])
def test_loss_stats_and_seeds_on_unaligned_slices(backend, B, L):
    pred, sx, psx, mu = _loss_operands(B, L, seed=B * L)
    if (B * L) % 4:
        assert sx.data_ptr() % 16 != 0       # (psx is 16-byte aligned again when B * L % 4 == 2)
    assert mu.data_ptr() % 16 != 0           # every case runs the unaligned loads of both kernels
    st = backend.stats(pred, sx, psx, mu, MU_COEF)
    _check_stats(st, pred, sx, psx, mu)
    seeds = backend.seeds(pred, sx, psx, mu, MU_COEF, st)
    _check_seeds_vs_oracle(seeds, pred, sx, psx, mu)
    # the same data in fresh (16-byte aligned) buffers takes the float4 loads: the same per-quad partial sums, so the
    # statistics agree to fp64 summation order, and the per-element seed formula is the same
    al = [v.clone() for v in (pred, sx, psx, mu)]
    assert all(v.data_ptr() % 16 == 0 for v in al)
    st_a = backend.stats(*al, MU_COEF)
    abs_r = (al[0].double() - al[3].double()).abs().sum().item()
    assert abs(st[0].item() - st_a[0].item()) <= 1e-12 * abs_r
    for k in (1, 2, 3):
        assert abs(st[k].item() - st_a[k].item()) <= 1e-12 * abs(st_a[k].item()), k
    assert st[4].item() == st_a[4].item()
    seeds_u = backend.seeds(pred, sx, psx, mu, MU_COEF, st_a)
    seeds_a = backend.seeds(*al, MU_COEF, st_a)
    for a, b in zip(seeds_u, seeds_a):
        assert torch.equal(a, b)


def test_loss_stats_and_seeds_at_the_train_benchmark_shape(backend):
    """16384 x 950 (bench.py --mode train): every thread loops through the grid-capped launch and many blocks meet in the
    fp64 atomics."""
    B, L = 16384, 950
    pred, sx, psx, mu = _loss_operands(B, L, seed=5, mu_lead=0)
    assert all(v.data_ptr() % 16 == 0 for v in (pred, sx, psx, mu)) and (B * L) % 4 == 0
    st = backend.stats(pred, sx, psx, mu, MU_COEF)
    _check_stats(st, pred, sx, psx, mu)
    seeds = backend.seeds(pred, sx, psx, mu, MU_COEF, st)
    _check_seeds_vs_oracle(seeds, pred, sx, psx, mu)


@pytest.mark.parametrize("B,L", [pytest.param(17, 20, id="17x20-aligned"), pytest.param(17, 21, id="17x21-unaligned"),
                                 pytest.param(393, 830, id="393x830-unaligned"), pytest.param(4096, 950, id="4096x950-aligned")])
def test_loss_variance_of_a_residual_with_a_large_mean(backend, B, L):
    """r = pred - mu with mean 3 and std 0.05: the variance in the loss's denominator must match float64 r.var() to the loss
    tolerance, although sum r^2 is 3600 times N var(r)."""
    pred, sx, psx, mu = _loss_operands(B, L, seed=B + L, mu_lead=1 if (B * L) % 4 else 0, r_mean=3.0, r_std=0.05)
    st = backend.stats(pred, sx, psx, mu, MU_COEF)
    _check_stats(st, pred, sx, psx, mu)
    N = st[4].item()
    var = (st[1].item() - st[0].item() ** 2 / N) / (N - 1)         # what loss_seeds_kernel divides by
    ref = (pred.double() - mu.double()).var().item()
    assert abs(var - ref) <= 1e-5 * ref, (var, ref)
    _check_seeds_vs_oracle(backend.seeds(pred, sx, psx, mu, MU_COEF, st), pred, sx, psx, mu)


def test_loss_grad_seeds_loss_only(lib, backend):
    """Null gradient outputs with loss_out only: the same loss."""
    B, L = 393, 830
    pred, sx, psx, mu = _loss_operands(B, L, seed=11)
    st = backend.stats(pred, sx, psx, mu, MU_COEF)
    loss_full = backend.seeds(pred, sx, psx, mu, MU_COEF, st)[3]
    loss = torch.full((1,), SENTINEL, device="cuda")
    _check(lib.sdrm_loss_grad_seeds(_ptr(pred), _ptr(sx), _ptr(psx), _ptr(mu), B * L, MU_COEF, _ptr(st), None, None, None,
                                    _ptr(loss), _stream()), "sdrm_loss_grad_seeds")
    assert torch.equal(loss, loss_full)


# ---------------------------------------------------------------------------------------------------------------------------
# C. the production training step: in-kernel noise and masks, end to end
# ---------------------------------------------------------------------------------------------------------------------------
def _step_case(name):
    if name in TRAIN_GOLDENS:
        g = load_golden(name)
        diff, _ = modules_from_golden(g, "cuda")
        return diff, g["mu"], g["t"], g["T"], g["nd"]
    # cfg-1-like denoiser width with an odd minibatch (the last minibatch of an epoch)
    B, L, T, nh = 393, 830, 83, 2
    diff, _ = random_modules(40, 32, L, T, nh, seed=8, device="cuda")
    g = torch.Generator().manual_seed(83)
    return diff, torch.randn(B, L, generator=g) * 0.5, torch.randint(1, T + 1, (B,), generator=g), T, 1.0


def _oracle_loss_and_grads(diff, mu, t, noise, keeps, T):
    ref = copy.deepcopy(diff).cpu().double()
    for p in ref.parameters():
        p.grad = None
    full = ref.state_dict(keep_vars=True)
    loss, _ = orc.training_loss(full, mu.double(), t, noise.double(), torch.as_tensor(keeps), T)
    loss.backward()
    return loss.item(), {k: p.grad for k, p in ref.named_parameters()}


def _grads(diff):
    return {k: p.grad.detach().clone() for k, p in diff.named_parameters()}


def _step(stepper, mu, t, **inj):
    stepper.net.zero_grad()
    loss = stepper.loss(mu, t, **inj)
    loss.backward()
    return loss.item(), _grads(stepper.net)


def _check_step(stepper, mu, t, noise, keeps, T, grad_rel, **loss_kw):
    """The step without injection == the same step fed the oracle's noise and masks (the path the goldens pin), and both
    against the float64 oracle: loss within 2e-5 and, where grad_rel is given, each gradient within grad_rel of its largest
    entry."""
    loss, grads = _step(stepper, mu.cuda(), t.cuda(), **loss_kw)
    step_index = stepper.step_index
    loss_inj, grads_inj = _step(stepper, mu.cuda(), t.cuda(), inj_noise=noise.cuda(), inj_masks=torch.from_numpy(keeps).cuda())
    stepper.step_index = step_index
    assert abs(loss - loss_inj) <= 1e-6 * abs(loss_inj), (loss, loss_inj)
    for k, g in grads.items():
        assert (g - grads_inj[k]).abs().max().item() <= 1e-5 * (grads_inj[k].abs().max().item() + 1e-30), k
    ref_loss, ref_grads = _oracle_loss_and_grads(stepper.net, mu, t, noise, keeps, T)
    assert abs(loss - ref_loss) <= 2e-5 * max(1.0, abs(ref_loss)), (loss, ref_loss)
    for k, g in (grads.items() if grad_rel else ()):
        gref = ref_grads[k]
        err = (g.cpu().double() - gref).abs().max().item()
        assert err <= grad_rel * (gref.abs().max().item() + 1e-12), (k, err, gref.abs().max().item())


# At the golden shapes the bars of test_training_step_matches_reference_golden.  At L = 830 the gradients of the layers
# upstream of the loss are near-cancelling sums: (psx - sx) / mu_coef^2 weighs two almost equal branches by +-100, which
# multiplies the rounding of the bf16x3 GEMM operands (~2^-17) by about 100.  Measured on a B200: 7e-4 of the largest entry
# on emb_layer.weight and 5.5e-3 on dnn.0.weight, the same for the step fed the oracle's noise and masks.  There the loss is
# checked against the oracle and the gradients against the injected-noise step, which is what the streams decide.
STEP_CASES = [pytest.param(n, 2e-4, id=n) for n in TRAIN_GOLDENS] + [pytest.param("cfg1like_B393_L830_nh2_T83", None,
                                                                               id="cfg1like_B393_L830_nh2_T83")]


@pytest.mark.parametrize("name,grad_rel", STEP_CASES)
def test_production_training_step_matches_oracle(backend, name, grad_rel):
    """DiffusionTrainStep.loss(mu, t) with nothing injected (the call train_SDRM and bench.py make) against the float64 oracle
    fed with the step's own streams: its noise from a masked noise_inputs call (bit-identical, see above) and its masks from
    the restatement.  The second step draws seed + 1; a step at rank 1's row offset draws that shard's slice of the batch."""
    from sdrm_b200.distributed import shard_bounds
    from sdrm_b200.training import DiffusionTrainStep
    diff, mu, t, T, nd = _step_case(name)
    diff.train()
    B, L = mu.shape
    ab = orc.make_schedule(T)[2]
    base = 1 << 40 | 12345
    mu_d, t_d = mu.cuda(), t.cuda()

    def streams(seed, lo, hi):
        noise, _, _, _, masks = backend.noise_inputs(mu_d[lo:hi].contiguous(), t_d[lo:hi].contiguous(), ab.float().cuda(), nd,
                                                     MU_COEF, seed, lo, want_masks=True)
        keeps = philox_ref.train_keep_masks(seed, lo, hi - lo, L)
        assert np.array_equal(masks.cpu().numpy(), keeps)
        return noise.cpu(), keeps

    stepper = DiffusionTrainStep(diff, ab.cuda(), T, nd, seed=base)
    for step in range(2):
        assert stepper.step_index == step
        noise, keeps = streams(base + step, 0, B)
        _check_step(stepper, mu, t, noise, keeps, T, grad_rel)
    for world in (2, 3):
        lo, hi = shard_bounds(B, 1, world)
        shard = DiffusionTrainStep(diff, ab.cuda(), T, nd, seed=base)
        shard.row_offset = lo
        noise, keeps = streams(base, 0, B)          # the whole batch's streams, sliced to the shard
        _check_step(shard, mu[lo:hi], t[lo:hi], noise[lo:hi], np.ascontiguousarray(keeps[:, lo:hi]), T, grad_rel)


# ---------------------------------------------------------------------------------------------------------------------------
# D. the frozen encoder on non-canonical CSR rows
# ---------------------------------------------------------------------------------------------------------------------------
def test_frozen_encoder_sums_repeated_column_indices():
    """A CSR row may store the same column twice (and explicit zeros).  to_dense() adds them up, so the L2 normalisation is
    that of the summed row; the encoder must see the same row through scipy staging and through a torch CSR tensor."""
    import scipy.sparse as sp
    from sdrm_b200.models import VAE
    from sdrm_b200.training import DeviceCSR, FrozenEncoder
    items, H, L = 300, 96, 16
    rng = np.random.RandomState(4)
    rows = [
        ([5, 5, 9], [1.0, 2.0, 1.0]),          # repeated column: to_dense gives 3 at column 5
        ([3, 3, 3], [1.0, 1.0, 1.0]),          # one column three times
        ([7, 8], [0.0, 1.0]),                  # explicit zero
        ([4, 4], [1.0, -1.0]),                 # entries that cancel: an all-zero row (F.normalize's clamp)
        ([250, 2, 250, 17, 2], [0.5, 1.0, 1.5, 2.0, 1.0]),   # unsorted with repeats
    ]
    for _ in range(11):                        # canonical rows
        cols = np.sort(rng.choice(items, size=rng.randint(1, 40), replace=False))
        rows.append((cols.tolist(), np.ones(len(cols)).tolist()))
    indptr = np.cumsum([0] + [len(c) for c, _ in rows]).astype(np.int64)
    indices = np.concatenate([c for c, _ in rows]).astype(np.int64)
    data = np.concatenate([v for _, v in rows]).astype(np.float32)
    m = sp.csr_matrix((data, indices, indptr), shape=(len(rows), items))
    assert not m.has_canonical_format
    nnz = m.nnz
    dense = torch.from_numpy(m.toarray())
    torch.manual_seed(4)
    vae = VAE(items, H, L).cuda().eval()
    ref_vae = VAE(items, H, L).double().eval()
    ref_vae.load_state_dict({k: v.detach().cpu().double() for k, v in vae.state_dict().items()})
    with torch.no_grad():
        h_ref = torch.tanh(ref_vae.encoder[0](torch.nn.functional.normalize(dense.double(), p=2, dim=1)))
        mu_ref = torch.chunk(ref_vae.encoder[2](h_ref), 2, dim=1)[0]
    enc = FrozenEncoder(vae)
    staged = DeviceCSR(m, "cuda")
    assert m.nnz == nnz                        # the caller's matrix is left as it was
    sel = [4, 0, 3, 1, 2, 9]
    tcsr = torch.sparse_csr_tensor(torch.from_numpy(indptr), torch.from_numpy(indices), torch.from_numpy(data),
                                   size=(len(rows), items))
    for x, want in ((staged.as_torch_csr(), slice(None)), (staged.csr_rows(sel), sel), (tcsr.cuda(), slice(None))):
        assert (enc.hidden(x).cpu().double() - h_ref[want]).abs().max().item() < 2e-6
        assert (enc(x).cpu().double() - mu_ref[want]).abs().max().item() < 5e-6 * max(1.0, mu_ref.abs().max().item())
