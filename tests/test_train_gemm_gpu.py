"""GPU parity of K5: the tcgen05 GEMM of the training step (csrc/gemm_x3_kernel.cuh) and the denoiser forward / backward built on it
(C ABI sdrm_gemm_nt, sdrm_denoiser_fwd, sdrm_denoiser_bwd) against float64 torch products / torch autograd of the same module
(reference: SDRM.forward + autograd, train_SDRM.py:97-103, 191-199, 336)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _gemm_nt(A, B, bias, passes, splits, trans_a=False, trans_b=False):
    """C = op(A) op(B)^T; with trans_x the tensor passed is the [K, *] transposed storage."""
    from sdrm_b200 import _lib
    lib = _lib.load()
    M, K = (A.shape[1], A.shape[0]) if trans_a else A.shape
    N = B.shape[1] if trans_b else B.shape[0]
    C = torch.full((M, N), float("nan"), device="cuda")
    need = lib.sdrm_gemm_workspace_bytes(M, N, K, splits)
    ws = torch.empty(need, dtype=torch.uint8, device="cuda")
    rc = lib.sdrm_gemm(_lib.ptr(A), A.stride(0), int(trans_a), _lib.ptr(B), B.stride(0), int(trans_b), _lib.ptr(bias), _lib.ptr(C),
                       C.stride(0), M, N, K, passes, splits, _lib.ptr(ws), need, _lib.stream_ptr())
    _lib.check(rc, "sdrm_gemm")
    _lib.check(lib.sdrm_train_check_device_error(_lib.ptr(ws), _lib.stream_ptr()), "sdrm_gemm (device)")
    return C


@pytest.mark.parametrize("M,N,K,splits", [(36, 24, 24, 1), (300, 200, 150, 1), (1650, 830, 830, 1), (257, 513, 70, 1),
                                           (950, 950, 5000, 4), (40, 24, 300, 3), (830, 1008, 1650, 2)])
@pytest.mark.parametrize("passes", [3, 1])
def test_gemm_nt_matches_float64(M, N, K, splits, passes):
    g = torch.Generator(device="cuda").manual_seed(M * 7 + N * 3 + K)
    A = torch.randn(M, K, device="cuda", generator=g)
    B = torch.randn(N, K, device="cuda", generator=g) / K ** 0.5
    bias = torch.randn(N, device="cuda", generator=g) if splits == 1 else None
    C = _gemm_nt(A, B, bias, passes, splits)
    if passes == 3:
        ref = A.double() @ B.double().T
    else:
        ref = A.bfloat16().double() @ B.bfloat16().double().T
    if bias is not None:
        ref = ref + bias.double()
    assert torch.isfinite(C).all()
    err = (C.double() - ref).abs().max().item()
    # bf16x3 drops the lo.lo term (2^-18 relative per product) and rounds lo to bf16 (2^-17): ~1e-5 of the row scale
    tol = (3e-5 if passes == 3 else 2e-5) * max(1.0, ref.abs().max().item())
    assert err <= tol, (err, tol)


def test_gemm_nt_strided_operands():
    g = torch.Generator(device="cuda").manual_seed(5)
    Abig = torch.randn(100, 90, device="cuda", generator=g)
    Bbig = torch.randn(64, 90, device="cuda", generator=g)
    A, B = Abig[:, :70], Bbig[:, :70]          # leading dimension 90, K = 70 (dnn.0.weight[:, :L] is such a view)
    C = _gemm_nt(A, B, None, 3, 1)
    ref = A.double() @ B.double().T
    assert (C.double() - ref).abs().max().item() <= 3e-5 * ref.abs().max().item()


def _fwd_bwd_report(L, T, nh, B, slopes):
    from sdrm_b200.models import SDRM
    from sdrm_b200.training import denoiser_gemms
    torch.manual_seed(L + T)
    net = SDRM(N_ITEMS=L, EMB_DIM=T, LATENT_DIM=L, n_hidden_layers=nh).cuda()
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

    ref_net = SDRM(N_ITEMS=L, EMB_DIM=T, LATENT_DIM=L, n_hidden_layers=nh).cuda().double()
    ref_net.load_state_dict({k: v.double() for k, v in net.state_dict().items()})
    emb = ref_net.emb_layer(ref_net.timestep_embedding(t, T).double())      # SDRM.forward in float64 (train_SDRM.py:97-103)
    ref_out = ref_net.dnn(torch.cat([x.double(), emb], dim=-1))
    (ref_out * g_out.double()).sum().backward()
    assert (out.double() - ref_out).abs().max().item() <= 2e-5, (out.double() - ref_out).abs().max().item()
    mx, fro = {}, {}
    for k, p in ref_net.named_parameters():
        d = got[k].double() - p.grad
        mx[k] = d.abs().max().item() / (p.grad.abs().max().item() + 1e-30)
        fro[k] = d.norm().item() / (p.grad.norm().item() + 1e-30)
    return mx, fro


# bf16x3 operands carry 16 mantissa bits (hi + bf16(lo)): a product is good to ~1.5e-5 relative, a gradient to ~1e-5 of its terms.
@pytest.mark.parametrize("ta,tb,splits", [(False, True, 1), (True, True, 0), (True, False, 2), (False, False, 0)])
def test_gemm_transposed_operands_and_auto_splits(ta, tb, splits):
    """the three products of a Linear layer: y = x W^T (nt), dx = dy W (B given transposed), dW = dy^T x (both transposed)"""
    g = torch.Generator(device="cuda").manual_seed(11)
    M, N, K = 333, 217, 1200
    A = torch.randn((K, M) if ta else (M, K), device="cuda", generator=g)
    B = torch.randn((K, N) if tb else (N, K), device="cuda", generator=g) / K ** 0.5
    C = _gemm_nt(A, B, None, 3, splits, ta, tb)
    ref = (A.double().T if ta else A.double()) @ (B.double() if tb else B.double().T)
    assert (C.double() - ref).abs().max().item() <= 3e-5 * max(1.0, ref.abs().max().item())


@pytest.mark.parametrize("L,T,nh,B", [(20, 6, 0, 5), (24, 7, 2, 12), (150, 43, 1, 100), (300, 7, 2, 100), (830, 83, 2, 550),
                                      (950, 178, 4, 700)])
def test_denoiser_fwd_bwd_matches_autograd_linear_slopes(L, T, nh, B):
    """PReLU slopes = 1 make the network piecewise-free (no kink), so EVERY gradient must match float64 autograd to 2e-4 of its
    max at every shape: multi-tile outputs, split-K weight-gradient slabs, the transposed operand images, the bias column sums,
    the slope sums (sum of dh * min(pre, 0), non-trivial at slope 1) and the time-embedding table gradient."""
    mx, _ = _fwd_bwd_report(L, T, nh, B, (1.0, 1.0))
    bad = {k: v for k, v in mx.items() if v > 2e-4}
    assert not bad, (bad, mx)


@pytest.mark.parametrize("L,T,nh,B,slopes", [
    pytest.param(20, 6, 0, 5, (0.21, 0.33), id="20-6-0-5"),
    pytest.param(24, 7, 2, 12, (0.21, 0.33), id="24-7-2-12"),
    pytest.param(40, 9, 5, 30, (0.21, 0.33), id="40-9-5-30"),
    pytest.param(20, 6, 0, 5, (-0.5, 1.5), id="20-6-0-5-slopes-0.5,1.5"),    # slopes outside [0, 1] (trained slopes can leave it)
    pytest.param(24, 7, 2, 12, (-0.5, 1.5), id="24-7-2-12-slopes-0.5,1.5"),
    pytest.param(40, 9, 5, 30, (-0.5, 1.5), id="40-9-5-30-slopes-0.5,1.5"),
])
def test_denoiser_fwd_bwd_matches_autograd_small(L, T, nh, B, slopes):
    """Real slopes at small shapes (a pre-activation within rounding distance of 0 -- where fp32-grade and float64 arithmetic
    legitimately pick different sides of the PReLU kink -- is improbable among a few thousand entries): 2e-4 of max|grad|."""
    mx, _ = _fwd_bwd_report(L, T, nh, B, slopes)
    bad = {k: v for k, v in mx.items() if v > 2e-4}
    assert not bad, (bad, mx)


@pytest.mark.parametrize("L,T,nh,B", [(830, 83, 2, 550), (950, 178, 4, 700)])
def test_denoiser_fwd_bwd_real_slopes_large(L, T, nh, B):
    """Real slopes at the cfg-1 / cfg-5 layer shapes: among millions of pre-activations a handful sit within 1e-6 of zero and
    flip PReLU' between 1 and the slope relative to float64 (any fp32 implementation does: one flipped entry moves one row of a
    weight gradient by ~0.75 / sqrt(rows) of its scale), so the bar is the relative Frobenius error; the layers above the last
    PReLU (dnn.{2+2nh}) have no kink upstream and keep the 2e-4 max bar."""
    mx, fro = _fwd_bwd_report(L, T, nh, B, (0.21, 0.33))
    last = f"dnn.{2 + 2 * nh}."
    bad = {k: (mx[k], fro[k]) for k in mx if (mx[k] > 2e-4 if k.startswith(last) else fro[k] > 1e-2)}
    assert not bad, (bad, mx, fro)


def test_bf16_single_pass_mode_is_close():
    from sdrm_b200.models import SDRM
    from sdrm_b200.training import denoiser_gemms
    torch.manual_seed(3)
    L, T, nh, B = 150, 43, 2, 64
    net = SDRM(N_ITEMS=L, EMB_DIM=T, LATENT_DIM=L, n_hidden_layers=nh).cuda()
    x = torch.randn(3 * B, L, device="cuda")
    t = torch.randint(1, T + 1, (B,), device="cuda").repeat(3)
    with torch.no_grad():
        o3 = denoiser_gemms(net, x, t, passes=3)
        o1 = denoiser_gemms(net, x, t, passes=1)
    assert (o3 - o1).abs().max().item() < 3e-2 and (o3 - o1).abs().max().item() > 0
