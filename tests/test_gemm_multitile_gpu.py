"""K5 (the tcgen05 bf16x3 GEMM, csrc/gemm_x3_kernel.cuh) on launches where every CTA pair runs several output tiles.

`launch_gemm` (csrc/train_gemm.cu) starts min(work, clusters) CTA pairs, work = m_tiles x n_tiles x splits, and cluster c runs
the work items c, c + n_clusters, ...  With one 197 KB CTA per SM there are at most SMs / 2 clusters, so a launch with
work > 2 * (SMs // 2) gives every cluster at least two tiles and cluster 0 at least three, whatever the occupancy query
returns: both TMEM accumulators (columns 0-255 and 256-511), a wrap of the accumulator barrier parities, the smem stage ring
carried from one tile into the next and the per-tile epilogue state (bias rows, the PReLU' prefetch of the next tile, the slope
sum over tiles) all run.  The shapes are those of the cfg-5 training step (16384 rows per GPU, three forwards: 49152 rows,
L = 950, T = 178, nh = 4) and of MultiVAE++ training at cfg-5 width (B = 500, I = 20000, H = 1000, 2L = 1900).  A case that
production runs with fewer tiles than that ("long K": few output tiles, 192 k-blocks each) says so and is exempt.

Every reference is float64 on the GPU.  Run time: 11 s for the file on a B200 at 1000 W.  Device memory, estimated and not
measured: up to about 10 GB (the float64 autograd of the denoiser at 49152 rows).
"""
import copy
import math

import numpy as np
import pytest
import torch

from oracle import philox_ref
from oracle import sdrm_oracle as orc

pytestmark = pytest.mark.gpu

# ---------------------------------------------------------------------------------------------------------------------------
# launch geometry: tile_width, wgrad_splits and the split normalisation of launch_gemm / sdrm_gemm (csrc/train_gemm.cu)
# ---------------------------------------------------------------------------------------------------------------------------


def _cdiv(a, b):
    return -(-a // b)


def _tile_width(N):
    n_tiles = _cdiv(N, 256)
    return max(16, _cdiv(_cdiv(N, n_tiles), 16) * 16), n_tiles


def _normalised_splits(splits, kb):
    """(splits, k-blocks per split) as launch_gemm uses them: no empty split."""
    per = _cdiv(kb, max(1, min(splits, kb)))
    return _cdiv(kb, per), per


def _wgrad_splits(M, N, K, clusters):
    tiles = _cdiv(M, 256) * _tile_width(N)[1]
    kb = _cdiv(K, 64)
    s = min(max(1, clusters // max(1, tiles)), min(kb, 8))
    return _normalised_splits(s, kb)[0]


def _max_clusters():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count // 2


def _plan(M, N, K, splits):
    """(work items, splits, k-blocks per work item) of one sdrm_gemm launch.  splits = 0 (automatic) depends on the number of
    resident clusters; it is taken at its upper bound SMs / 2, which decides the count for every output of more than SMs / 2
    tiles (one split) and for the long-K weight gradients on any count of 64 to 79 clusters."""
    kb = _cdiv(K, 64)
    s, per = _normalised_splits(splits if splits > 0 else _wgrad_splits(M, N, K, _max_clusters()), kb)
    return _cdiv(M, 256) * _tile_width(N)[1] * s, s, per


def _report_work(what, work, multi_tile):
    clusters = _max_clusters()
    print(f"{what}: {work} work items, >= {work / clusters:.1f} tiles per cluster (at most {clusters} clusters)")
    if multi_tile:
        assert work > 2 * clusters, (what, work, clusters)


# ---------------------------------------------------------------------------------------------------------------------------
# the elementwise bar
# ---------------------------------------------------------------------------------------------------------------------------
def _eps(K, splits, passes):
    """Relative bar of one output entry against sum_k |a_k| |b_k| (the matching entry of |A| |B|^T, plus |bias|).

    passes = 3 is compared with the exact float64 product.  x = hi + lo + d with hi = bf16(x), lo = bf16(x - hi):
    |x - hi| <= 2^-8 |x| and |d| <= 2^-8 |x - hi| <= 2^-16 |x|.  bf16x3 keeps hi.hi + hi.lo + lo.hi and drops lo.lo and the
    lo rounding, a.b - kept = lo_a lo_b + d_a b + a d_b (+ smaller): about 3 * 2^-18 of |a||b| per product at typical
    rounding, 3 * 2^-16 at the worst.  These terms have random signs, so their sum over K products is far below either
    figure times sum |a||b|; 2^-15, 2.7 times the typical figure, holds without relying on that cancellation.
    passes = 1 is compared with the float64 product of the bf16-rounded operands, which leaves only the accumulation.
    Accumulation: the products are exact in fp32, and each of the passes * 4 UMMAs (K = 16) of a k-block and each of the
    split-slab additions rounds the fp32 partial sum once; counting each as a truncation (2^-23 of a partial sum that is at
    most sum |a||b|), n independent roundings add sqrt(n) * 2^-23.

    What the bar resolves: an error in a whole tile (a stale accumulator, a skipped or doubled k-block of hi.hi, a missing
    bias) is of the order of the entry itself, 10^3 times eps or more.  A lost hi.lo pass of one k-block is at most
    2^-9 * 64 / K of sum |a||b| (4 eps at K = 950, under eps beyond K = 4096) and with random signs about an eighth of that,
    so it can pass this bar: that, and anything else that changes a tile by less than eps, is left to the bitwise comparison
    of the row blocks (test_gemm_row_blocks_are_bitwise_launch_invariant)."""
    kb = _cdiv(K, 64)
    per = _normalised_splits(splits, kb)[1]
    n_acc = passes * 4 * per + splits
    return (2.0 ** -15 if passes == 3 else 0.0) + math.sqrt(n_acc) * 2.0 ** -23


# test_gemm_nt_matches_float64's bar of max|ref| was set at K <= 5000.  For zero-mean operands max|ref| grows as sqrt(K) while the
# rounding grows with sum |a||b| ~ K, so beyond that the elementwise bar alone applies (on a B200 at 1000 W: 4.3e-5 of max|ref|
# at K = 49152 and 7.8e-5 at K = 20000, with the elementwise ratio at 1.6e-6 and 3.6e-6).
MAX_REF_BAR_K = 6000


def _check_elementwise(got, ref, scale, eps, what, K, passes=3):
    """got within eps * scale of ref everywhere and, for K <= MAX_REF_BAR_K, within the bar of max|ref| of
    test_gemm_nt_matches_float64."""
    assert torch.isfinite(got).all(), what
    err = (got.double() - ref).abs()
    ratio = (err / scale).max().item()
    print(f"{what}: max |err| / (|A||B|^T) = {ratio:.3e} (eps {eps:.3e}), max |err| / max |ref| = "
          f"{err.max().item() / ref.abs().max().item():.3e}")
    assert ratio <= eps, (what, ratio, eps)
    if K <= MAX_REF_BAR_K:
        assert err.max().item() <= (3e-5 if passes == 3 else 2e-5) * max(1.0, ref.abs().max().item()), what
    return ratio


def _bf(x):
    return x.bfloat16().double()


# ---------------------------------------------------------------------------------------------------------------------------
# 1 + 2: sdrm_gemm at multi-tile shapes
# ---------------------------------------------------------------------------------------------------------------------------
def _gemm(A, B, bias, passes, splits, trans_a, trans_b, M, N, K):
    """C = op(A) op(B)^T through the C ABI; with trans_x the tensor passed is the [K, *] transposed storage."""
    from sdrm_b200 import _lib
    lib = _lib.load()
    C = torch.full((M, N), float("nan"), device="cuda")
    need = lib.sdrm_gemm_workspace_bytes(M, N, K, splits)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    rc = lib.sdrm_gemm(_lib.ptr(A), A.stride(0), int(trans_a), _lib.ptr(B), B.stride(0), int(trans_b), _lib.ptr(bias), _lib.ptr(C),
                       C.stride(0), M, N, K, passes, splits, _lib.ptr(ws), need, _lib.stream_ptr())
    _lib.check(rc, "sdrm_gemm")
    _lib.check(lib.sdrm_train_check_device_error(_lib.ptr(ws), _lib.stream_ptr()), "sdrm_gemm (watchdog word)")
    return C


# name: (M, N, K, trans_a, trans_b, bias, splits, multi_tile)
GEMM_CASES = {
    "train-fwd-49152x950x950-bias": (49152, 950, 950, False, False, True, 1, True),        # 192 x 4 = 768 work items
    "train-dgrad-49152x950x950-Bt": (49152, 950, 950, False, True, False, 1, True),        # dY . W: B given transposed
    "train-wgrad-950x950x49152-longK": (950, 950, 49152, True, True, False, 0, False),     # 16 tiles x 4 splits, 192 k-blocks each
    "vae-dec-out-500x20000x1000-bias": (500, 20000, 1000, False, False, True, 1, True),    # 2 x 79 = 158
    "vae-wgrad-20000x1000x500-AtBt": (20000, 1000, 500, True, True, False, 0, True),       # 79 x 4 = 316
    "ragged-38913x1001x777-At-bias": (38913, 1001, 777, True, False, True, 1, True),       # 153 x 4 = 612, every tail
    "splitk-8192x1008x6000-3splits": (8192, 1008, 6000, False, False, False, 3, True),     # 32 x 4 x 3 = 384
}


def _operands(name):
    M, N, K, ta, tb, has_bias, splits, _ = GEMM_CASES[name]
    g = torch.Generator(device="cuda").manual_seed(sum(map(ord, name)))
    A = torch.randn((K, M) if ta else (M, K), device="cuda", generator=g)
    B = torch.randn((K, N) if tb else (N, K), device="cuda", generator=g) / K ** 0.5
    bias = torch.randn(N, device="cuda", generator=g) if has_bias else None
    return A, B, bias


@pytest.mark.parametrize("passes", [3, 1])
@pytest.mark.parametrize("name", list(GEMM_CASES))
def test_gemm_multitile_matches_float64_elementwise(name, passes):
    M, N, K, ta, tb, _, splits, multi_tile = GEMM_CASES[name]
    work, s, per = _plan(M, N, K, splits)
    _report_work(f"{name} passes={passes} ({s} split(s) of {per} k-blocks)", work, multi_tile)
    A, B, bias = _operands(name)
    C = _gemm(A, B, bias, passes, splits, ta, tb, M, N, K)
    a = A.T if ta else A                     # [M, K] views
    b = B if tb else B.T                     # [K, N]
    a64, b64 = (a.double(), b.double()) if passes == 3 else (_bf(a), _bf(b))
    ref = a64 @ b64
    scale = a64.abs() @ b64.abs()
    del a64, b64
    if bias is not None:
        ref += bias.double()
        scale += bias.double().abs()
    _check_elementwise(C, ref, scale, _eps(K, s, passes), name, K, passes)


def _row_blocks(M):
    """256-aligned row blocks: the first, one in the middle and the last (ragged where M % 256 != 0)."""
    m_tiles = _cdiv(M, 256)
    return sorted({(256 * i, min(M, 256 * (i + 1))) for i in (0, m_tiles // 2, m_tiles - 1)})


@pytest.mark.parametrize("passes", [3, 1])
@pytest.mark.parametrize("name", [n for n, c in GEMM_CASES.items() if c[6] > 0])
def test_gemm_row_blocks_are_bitwise_launch_invariant(name, passes):
    """A tile's arithmetic (its k-blocks, their order and the UMMA sequence) does not depend on which cluster runs it, in which
    position, or which TMEM accumulator it lands in.  So rows recomputed as a launch of their own -- where the tile is a
    cluster's first or second instead of its third or later -- must equal the big launch's rows bit for bit: a stale
    accumulator, a barrier phase mix-up or per-tile epilogue state leaking from the previous tile shows here at any size."""
    M, N, K, ta, tb, _, splits, _ = GEMM_CASES[name]
    A, B, bias = _operands(name)
    C = _gemm(A, B, bias, passes, splits, ta, tb, M, N, K)
    for r0, r1 in _row_blocks(M):
        Ab = A[:, r0:r1] if ta else A[r0:r1]
        work = _plan(r1 - r0, N, K, splits)[0]
        Cb = _gemm(Ab, B, bias, passes, splits, ta, tb, r1 - r0, N, K)
        print(f"{name} passes={passes}: rows {r0}:{r1} alone ({work} work items)")
        assert torch.equal(Cb, C[r0:r1]), (name, r0, r1, (Cb - C[r0:r1]).abs().max().item())


# ---------------------------------------------------------------------------------------------------------------------------
# 3: the denoiser forward / backward at the training-benchmark shape
# ---------------------------------------------------------------------------------------------------------------------------
def _denoiser(L, D, T, nh, slopes, seed):
    from sdrm_b200.models import SDRM
    torch.manual_seed(seed)
    net = SDRM(N_ITEMS=L, EMB_DIM=T, LATENT_DIM=D, n_hidden_layers=nh).cuda()
    with torch.no_grad():
        net.dnn[1].weight.fill_(slopes[0])
        if nh > 0:
            net.dnn[3].weight.fill_(slopes[1])
    return net


def _denoiser_inputs(L, T, B, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    rows = 3 * B
    x = torch.randn(rows, L, device="cuda", generator=g) * (torch.rand(rows, L, device="cuda", generator=g) < 0.5) * 2.0
    t = torch.randint(1, T + 1, (B,), device="cuda", generator=g).repeat(3)
    g_out = torch.randn(rows, L, device="cuda", generator=g) / rows
    return x, t, g_out


def _check_train_workspace(out):
    """The watchdog word of the step's workspace (DenoiserGemms keeps the workspace for the backward)."""
    from sdrm_b200 import _lib
    ws = out.grad_fn.saved_tensors[-1]
    assert ws.dtype == torch.uint8
    return lambda: _lib.check(_lib.load().sdrm_train_check_device_error(_lib.ptr(ws), _lib.stream_ptr()), "denoiser (watchdog word)")


def _denoiser_report(L, D, T, nh, B, slopes):
    """max and relative-Frobenius error of every parameter gradient of denoiser_gemms against float64 autograd of SDRM.forward
    (train_SDRM.py:97-103), both on the GPU."""
    from sdrm_b200.training import denoiser_gemms
    net = _denoiser(L, D, T, nh, slopes, L + T + D)
    x, t, g_out = _denoiser_inputs(L, T, B, L + T)
    rows = 3 * B
    for what, M, N, K in (("layer 0", rows, D, L), ("output layer", rows, L, D)):
        _report_work(f"denoiser L={L} D={D} {what} forward", _plan(M, N, K, 1)[0], True)
    print(f"denoiser L={L} D={D}: weight gradients of the hidden layer {_plan(D, D, rows, 0)[:2]} (work items, splits): long K")

    net.zero_grad()
    out = denoiser_gemms(net, x, t, passes=3)
    check_ws = _check_train_workspace(out)
    (out * g_out).sum().backward()
    check_ws()
    got = {k: p.grad.detach().clone() for k, p in net.named_parameters()}

    ref_net = copy.deepcopy(net).double()
    ref_net.zero_grad()
    # the shared PReLU (dnn.3) runs nh times: its slope gradient is the sum of nh sums c_j = sum dh_j * min(pre_j, 0)
    c = []
    shared_prelu = ref_net.dnn[3] if nh > 0 else None

    def keep_slope_sum(_, inp, outp):
        outp.register_hook(lambda gr, pre=inp[0]: c.append((gr * pre.clamp(max=0)).sum().item()))

    hook = shared_prelu.register_forward_hook(keep_slope_sum) if nh > 0 else None
    emb = ref_net.emb_layer(ref_net.timestep_embedding(t, T).double())
    ref_out = ref_net.dnn(torch.cat([x.double(), emb], dim=-1))
    (ref_out * g_out.double()).sum().backward()
    if hook is not None:
        hook.remove()
    out_err = (out.double() - ref_out).abs().max().item()
    del ref_out, emb
    mx, fro = {}, {}
    for k, p in ref_net.named_parameters():
        d = got[k].double() - p.grad
        # gah: each c_j is rounded like any other gradient, and their sum can cancel below every one of them
        scale = sum(abs(v) for v in c) if (nh > 0 and k == "dnn.3.weight") else p.grad.abs().max().item()
        mx[k] = d.abs().max().item() / (scale + 1e-30)
        fro[k] = d.norm().item() / (p.grad.norm().item() + 1e-30)
    print(f"denoiser L={L} D={D} T={T} nh={nh} B={B} slopes={slopes}: output max |err| {out_err:.2e}")
    if nh > 0:
        print(f"  gah = sum of {len(c)} applications {['%.4e' % v for v in c]} = {sum(c):.4e}")
    for k in mx:
        print(f"  {k}: max |err| / max |grad| {mx[k]:.2e}, relative Frobenius {fro[k]:.2e}")
    assert out_err <= 2e-5, out_err
    return mx, fro


DENOISER_LINEAR = [pytest.param(950, 950, 178, 4, 16384, id="cfg5-L950-T178-nh4-B16384"),
                   pytest.param(340, 1000, 50, 2, 8192, id="L340-D1000-T50-nh2-B8192")]


@pytest.mark.parametrize("L,D,T,nh,B", DENOISER_LINEAR)
def test_denoiser_multitile_linear_slopes(L, D, T, nh, B):
    """Slopes = 1 leave no kink, so every gradient must match float64 autograd to 2e-4 of its max, including the slope sums
    ga0 / gah (one double per epilogue warp, summed over all of the warp's tiles before one atomicAdd) and the time-embedding
    table gradient.  gah is held to 2e-4 of sum_j |c_j|, its nh per-application sums: at the benchmark shape they cancel
    (on a B200 the error came to 2.008e-4 of |gah| itself)."""
    mx, _ = _denoiser_report(L, D, T, nh, B, (1.0, 1.0))
    bad = {k: v for k, v in mx.items() if v > 2e-4}
    assert not bad, (bad, mx)


def test_denoiser_multitile_real_slopes():
    """Real slopes at the benchmark shape, with the bars of test_denoiser_fwd_bwd_real_slopes_large: the layers above the last
    PReLU keep 2e-4 of max|grad|; below it a handful of pre-activations within rounding distance of 0 flip PReLU' relative to
    float64, so those gradients are held to 1e-2 relative Frobenius error."""
    L, D, T, nh, B = 950, 950, 178, 4, 16384
    mx, fro = _denoiser_report(L, D, T, nh, B, (0.21, 0.33))
    last = f"dnn.{2 + 2 * nh}."
    bad = {k: (mx[k], fro[k]) for k in mx if (mx[k] > 2e-4 if k.startswith(last) else fro[k] > 1e-2)}
    assert not bad, (bad, mx, fro)


@pytest.mark.parametrize("L,D,T,nh,B", DENOISER_LINEAR)
def test_denoiser_forward_row_blocks_are_bitwise_launch_invariant(L, D, T, nh, B):
    """The forward's rows recomputed as launches of their own (every layer's product, bias-table rows and PReLU epilogue) equal
    the full call's rows bit for bit."""
    from sdrm_b200.training import denoiser_gemms
    net = _denoiser(L, D, T, nh, (0.21, 0.33), L + T + D)
    x, t, _ = _denoiser_inputs(L, T, B, L + T)
    with torch.no_grad():
        full = denoiser_gemms(net, x, t, passes=3)
        for r0, r1 in _row_blocks(x.shape[0]):
            part = denoiser_gemms(net, x[r0:r1], t[r0:r1], passes=3)
            assert torch.equal(part, full[r0:r1]), (r0, r1, (part - full[r0:r1]).abs().max().item())
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------------------------------
# 4: the production training step at the benchmark shape
# ---------------------------------------------------------------------------------------------------------------------------
def _step(stepper, mu, t, **inj):
    stepper.net.zero_grad()
    loss = stepper.loss(mu, t, **inj)
    loss.backward()
    return loss.item(), {k: p.grad.detach().clone() for k, p in stepper.net.named_parameters()}


def test_production_training_step_at_benchmark_shape():
    """DiffusionTrainStep.loss(mu, t) with in-kernel noise and masks (the call of bench.py --mode train, cfg 5: B = 16384,
    L = 950, T = 178, nh = 4, nd = 1) against the float64 oracle on the GPU fed the step's own streams: the loss within 2e-5,
    and the gradients within 1e-5 of the same step fed those streams (upstream of the loss the gradients are near-cancelling
    sums that multiply the GEMM's operand rounding by about 100, see test_production_training_step_matches_oracle)."""
    from sdrm_b200.training import CudaLossBackend, DiffusionTrainStep
    B, L, T, nh, nd, mu_coef = 16384, 950, 178, 4, 1.0, 0.1
    _report_work("training step: forward / data-gradient products", _plan(3 * B, L, L, 1)[0], True)
    diff = _denoiser(L, L, T, nh, (0.25, 0.25), 5)         # nn.PReLU's initial slope
    diff.train()
    g = torch.Generator().manual_seed(16384)
    mu = torch.randn(B, L, generator=g).cuda()
    t = torch.randint(1, T + 1, (B,), generator=g).cuda()
    ab = orc.make_schedule(T)[2]
    seed = 1 << 40 | 77
    backend = CudaLossBackend()
    noise, _, _, _, masks = backend.noise_inputs(mu, t, ab.float().cuda(), nd, mu_coef, seed, 0, want_masks=True)
    keeps = philox_ref.train_keep_masks(seed, 0, B, L)
    assert np.array_equal(masks.cpu().numpy(), keeps)

    stepper = DiffusionTrainStep(diff, ab.cuda(), T, nd, seed=seed)
    loss, grads = _step(stepper, mu, t)
    stepper.step_index = 0
    loss_inj, grads_inj = _step(stepper, mu, t, inj_noise=noise, inj_masks=masks)
    torch.cuda.synchronize()
    assert abs(loss - loss_inj) <= 1e-6 * abs(loss_inj), (loss, loss_inj)
    for k, gk in grads.items():
        rel = (gk - grads_inj[k]).abs().max().item() / (grads_inj[k].abs().max().item() + 1e-30)
        print(f"training step {k}: max |grad - grad(injected streams)| / max |grad| = {rel:.2e}")
        assert rel <= 1e-5, (k, rel)

    ref = copy.deepcopy(diff).double()
    with torch.no_grad():
        ref_loss, _ = orc.training_loss(ref.state_dict(), mu.double(), t, noise.double(), masks, T, mu_coef)
    print(f"training step: loss {loss:.8f}, float64 oracle {ref_loss.item():.8f}")
    assert abs(loss - ref_loss.item()) <= 2e-5 * max(1.0, abs(ref_loss.item())), (loss, ref_loss.item())


# ---------------------------------------------------------------------------------------------------------------------------
# 5: TcLinear at the cfg-5 MultiVAE++ layer shapes
# ---------------------------------------------------------------------------------------------------------------------------
VAE_B = 500
# (layer, in, out, the products with more than two tiles per cluster)
VAE_LAYERS = [("encoder.0", 20000, 1000, ("dx", "dW")), ("encoder.2", 1000, 1900, ()), ("decoder.0", 950, 1000, ()),
              ("decoder.2", 1000, 20000, ("y", "dW"))]


@pytest.mark.parametrize("layer,n_in,n_out,multi", [pytest.param(*c, id=c[0]) for c in VAE_LAYERS])
def test_tc_linear_at_vae_layer_shapes(layer, n_in, n_out, multi):
    """y = x W^T + b, dx = dy W, dW = dy^T x (automatic split-K) and db against float64 F.linear autograd, elementwise."""
    from sdrm_b200.training import TcLinear
    plans = {"y": (VAE_B, n_out, n_in, 1), "dx": (VAE_B, n_in, n_out, 1), "dW": (n_out, n_in, VAE_B, 0)}
    eps = {}
    for what, (M, N, K, splits) in plans.items():
        work, s, _ = _plan(M, N, K, splits)
        _report_work(f"TcLinear {layer} {what} [{M} x {N}, K = {K}]", work, what in multi)
        eps[what] = _eps(K, s, 3)
    torch.manual_seed(n_in + n_out)
    lin = torch.nn.Linear(n_in, n_out).cuda()
    x = torch.randn(VAE_B, n_in, device="cuda", requires_grad=True)
    g = torch.randn(VAE_B, n_out, device="cuda")
    y = TcLinear.apply(x, lin.weight, lin.bias, 3)
    y.backward(g)
    torch.cuda.synchronize()          # a GEMM wait past its watchdog traps: the launch error surfaces here

    x64 = x.detach().double().requires_grad_()
    W64 = lin.weight.detach().double().requires_grad_()
    b64 = lin.bias.detach().double().requires_grad_()
    y64 = torch.nn.functional.linear(x64, W64, b64)
    y64.backward(g.double())
    xa, Wa, ga = x64.detach().abs(), W64.detach().abs(), g.double().abs()
    _check_elementwise(y.detach(), y64.detach(), xa @ Wa.T + b64.detach().abs(), eps["y"], f"{layer} y", n_in)
    _check_elementwise(x.grad, x64.grad, ga @ Wa, eps["dx"], f"{layer} dx", n_out)
    _check_elementwise(lin.weight.grad, W64.grad, ga.T @ xa, eps["dW"], f"{layer} dW", VAE_B)
    # db is torch's fp32 column sum of B entries: sqrt(B) roundings of at most 2^-23 of sum |g|
    _check_elementwise(lin.bias.grad, b64.grad, ga.sum(0), math.sqrt(VAE_B) * 2.0 ** -23, f"{layer} db", VAE_B)


# ---------------------------------------------------------------------------------------------------------------------------
# 6: the library's launch count
# ---------------------------------------------------------------------------------------------------------------------------
TRAIN_KERNELS = ("sdrm_gemm_pair_kernel", "operand_prep_kernel", "slab_reduce_kernel", "table_grad_kernel", "finish_sums_kernel")


@pytest.mark.parametrize("nh", [0, 2])
def test_train_launch_count_matches_profiler(nh):
    """sdrm_train_launch_count (bench.py's gpu_launches of the training step) counts exactly the kernels of the denoiser forward
    and backward that a profiler sees.  The counter is per thread and autograd runs the CUDA backward on a thread of its own,
    so the backward is called here through its graph node, on this thread."""
    from torch.profiler import ProfilerActivity, profile

    from sdrm_b200 import _lib
    from sdrm_b200.training import denoiser_gemms
    lib = _lib.load()
    L, T, B = 24, 7, 12
    net = _denoiser(L, L, T, nh, (0.21, 0.33), 3)
    x, t, g_out = _denoiser_inputs(L, T, B, 3)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        lib.sdrm_train_launch_count(1)
        out = denoiser_gemms(net, x, t, passes=3)
        out.grad_fn.apply(g_out)
        counted = lib.sdrm_train_launch_count(1)
        torch.cuda.synchronize()
    seen = [e.name for e in prof.events()
            if e.device_type == torch.autograd.DeviceType.CUDA and any(k in e.name for k in TRAIN_KERNELS)]
    print(f"nh={nh}: counted {counted}, profiled {len(seen)}")
    assert counted == len(seen), (counted, sorted(seen))
