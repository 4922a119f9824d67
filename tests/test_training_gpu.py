"""GPU parity of K2 (fused noising / loss statistics / gradient seeds) against the oracle and the reference goldens."""
import numpy as np
import pytest
import torch

from conftest import TRAIN_GOLDENS, load_golden
from helpers import modules_from_golden
from oracle import philox_ref
from oracle import sdrm_oracle as orc

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", TRAIN_GOLDENS)
def test_training_step_matches_reference_golden(name):
    """Same weights, same noise / t / dropout masks the reference drew -> same loss and same gradients."""
    from sdrm_b200.training import DiffusionTrainStep
    g = load_golden(name)
    diff, _ = modules_from_golden(g, "cuda")
    diff.train()
    _, _, ab_t = orc.make_schedule(g["T"])
    stepper = DiffusionTrainStep(diff, ab_t.cuda(), g["T"], g["nd"], seed=1)
    diff.zero_grad()
    loss = stepper.loss(g["mu"].cuda(), g["t"].cuda(), inj_noise=g["noise"].cuda().contiguous(),
                        inj_masks=g["keeps"].cuda().contiguous())
    loss.backward()
    ref = g["loss_ref"].item()
    assert abs(loss.item() - ref) <= 2e-5 * max(1.0, abs(ref)), (loss.item(), ref)
    for k, p in diff.named_parameters():
        gref = g["grads_ref"][k]
        scale = gref.abs().max().item() + 1e-12
        assert (p.grad.cpu() - gref).abs().max().item() <= 2e-4 * scale, k   # TF32-free fp32 GEMMs on the GPU vs CPU


def test_noise_inputs_philox_stream_matches_restatement():
    from sdrm_b200.training import CudaLossBackend
    be = CudaLossBackend()
    B, L, T, nd, seed, off = 300, 150, 43, 0.2, 987654321, 5001     # 5001 * 150 is not a multiple of 512: ragged first block
    mu = torch.randn(B, L, device="cuda")
    t = torch.randint(1, T + 1, (B,), device="cuda")
    _, _, ab_t = orc.make_schedule(T)
    noise, in_pert, in_clean, in_shift, masks = be.noise_inputs(mu, t, ab_t.cuda(), nd, 0.1, seed, off, want_masks=True)
    z = philox_ref.train_normals(seed, off, B, L) * np.float32(nd)
    assert np.allclose(noise.cpu().numpy(), z, rtol=2e-5, atol=2e-6)
    assert np.array_equal(masks.cpu().numpy(), philox_ref.train_keep_masks(seed, off, B, L))
    # row sharding does not change the streams: rows [100, 300) generated on their own equal the slice of the whole
    part = be.noise_inputs(mu[100:].contiguous(), t[100:].contiguous(), ab_t.cuda(), nd, 0.1, seed, off + 100, want_masks=True)
    assert torch.equal(part[0], noise[100:]) and torch.equal(part[4], masks[:, 100:])
    x_t = orc.perturb_input(mu.cpu(), t.cpu(), noise.cpu(), ab_t)
    keep = masks.cpu().float()
    assert torch.allclose(in_pert.cpu(), x_t * keep[0] * 2, atol=1e-6)
    assert torch.allclose(in_clean.cpu(), mu.cpu() * keep[1] * 2, atol=1e-6)
    assert torch.allclose(in_shift.cpu(), (mu.cpu() + 0.1 * noise.cpu()) * keep[2] * 2, atol=1e-6)
    assert abs(masks.float().mean().item() - 0.5) < 0.01


@pytest.mark.parametrize("B,L", [(17, 20), (550, 830), (4096, 950)])
def test_loss_stats_and_seeds_vs_oracle(B, L):
    from sdrm_b200.training import CudaLossBackend
    be = CudaLossBackend()
    g = torch.Generator(device="cuda").manual_seed(B)
    pred, sx, psx, mu = (torch.randn(B, L, device="cuda", generator=g) * s for s in (0.5, 0.5, 0.5, 1.0))
    st = be.stats(pred, sx, psx, mu, 0.1)
    r = (pred - mu).double()
    assert abs(st[0].item() - r.sum().item()) <= 1e-6 * r.abs().sum().item()
    assert abs(st[4].item() - B * L) == 0
    g_pred, g_sx, g_psx, loss = be.seeds(pred, sx, psx, mu, 0.1, st)
    o_pred, o_sx, o_psx, o_loss = orc.loss_grad_seeds(pred.cpu(), sx.cpu(), psx.cpu(), mu.cpu())
    assert abs(loss.item() - float(o_loss)) <= 1e-5 * abs(float(o_loss))
    for a, b in ((g_pred, o_pred), (g_sx, o_sx), (g_psx, o_psx)):
        assert (a.cpu().double() - b).abs().max().item() <= 1e-4 * b.abs().max().item()


def test_three_adam_steps_track_the_oracle():
    """A few full optimisation steps (forward, fused loss, backward, Adam) stay on the oracle's trajectory."""
    from sdrm_b200.training import DiffusionTrainStep
    g = load_golden("t_nh2_T7_L24")
    diff, _ = modules_from_golden(g, "cuda")
    ref_mod, _ = modules_from_golden(g, "cpu")
    diff.train(); ref_mod.train()
    _, _, ab_t = orc.make_schedule(g["T"])
    stepper = DiffusionTrainStep(diff, ab_t.cuda(), g["T"], g["nd"], seed=3)
    opt = torch.optim.Adam(diff.parameters(), lr=1e-3, weight_decay=1e-4, eps=1e-8)
    opt_ref = torch.optim.Adam(ref_mod.parameters(), lr=1e-3, weight_decay=1e-4, eps=1e-8)
    gen = torch.Generator().manual_seed(0)
    for step in range(3):
        noise = torch.randn(g["mu"].shape, generator=gen) * g["nd"]
        t = torch.randint(1, g["T"] + 1, (g["mu"].shape[0],), generator=gen)
        keeps = (torch.rand((3,) + tuple(g["mu"].shape), generator=gen) < 0.5).to(torch.uint8)
        opt.zero_grad()
        loss = stepper.loss(g["mu"].cuda(), t.cuda(), inj_noise=noise.cuda(), inj_masks=keeps.cuda())
        loss.backward(); opt.step()
        opt_ref.zero_grad()
        sd = dict(ref_mod.named_parameters())
        full = {k: v for k, v in ref_mod.state_dict(keep_vars=True).items()}
        loss_ref, _ = orc.training_loss(full, g["mu"], t, noise, keeps, g["T"])
        loss_ref.backward(); opt_ref.step()
        assert abs(loss.item() - loss_ref.item()) <= 1e-3 * abs(loss_ref.item())
    for (k, p), (_, q) in zip(diff.named_parameters(), ref_mod.named_parameters()):
        assert torch.allclose(p.detach().cpu(), q.detach(), rtol=2e-3, atol=2e-5), k


@pytest.mark.parametrize("rows,items,H,L,density", [
    (550, 1008, 930, 830, 0.0575),     # cfg 1 ml-100k training batch
    (850, 8582, 40, 40, 0.00115),      # cfg 3 adm
    (530, 729, 550, 400, 0.0133),      # cfg 4 alb
    (37, 300, 2048, 16, 0.2),          # widest hidden layer the kernel takes
])
def test_frozen_encoder_csr_matches_dense_encode(rows, items, H, L, density):
    """K2 `sdrm_encode_csr` (+ the mu half of the second Linear) == VAE.encode(x.to_dense())[0] of the reference-shaped
    module in eval mode (train_SDRM.py:241-250), evaluated in float64 on the CPU.  fp32 gather-sum vs a dense GEMM only
    differ in summation order: 2e-6 absolute on activations bounded by 1."""
    from sdrm_b200.models import VAE
    from sdrm_b200.training import FrozenEncoder
    rng = np.random.RandomState(rows)
    torch.manual_seed(rows)
    vae = VAE(items, H, L).cuda().eval()
    dense = (rng.rand(rows, items) < density).astype(np.float32)
    dense[3] = 0.0                                   # a user without interactions: F.normalize's 1e-12 clamp
    dense[5, :7] = np.array([2.0, 0.5, 3.0, 1.0, 4.0, 0.25, 1.5], dtype=np.float32)   # non-binary values
    xd = torch.from_numpy(dense)
    coo = xd.to_sparse()                             # what sparse_batch_collate yields (dataloaders.py:61-79)
    enc = FrozenEncoder(vae)
    mu = enc(coo.cuda())
    ref_vae = VAE(items, H, L).double().eval()
    ref_vae.load_state_dict({k: v.detach().cpu().double() for k, v in vae.state_dict().items()})
    with torch.no_grad():
        h_ref = torch.tanh(ref_vae.encoder[0](torch.nn.functional.normalize(xd.double(), p=2, dim=1)))
        mu_ref = torch.chunk(ref_vae.encoder[2](h_ref), 2, dim=1)[0]
    assert (enc.hidden(coo.cuda()).cpu().double() - h_ref).abs().max().item() < 2e-6
    assert (mu.cpu().double() - mu_ref).abs().max().item() < 5e-6 * max(1.0, mu_ref.abs().max().item())
    # layouts: CSR and dense inputs take the same kernel
    assert torch.equal(enc(coo.cuda().coalesce().to_sparse_csr()), mu)
    assert torch.equal(enc(xd.cuda()), mu)
    # and the module's own dense encode on the GPU agrees within fp32 GEMM noise
    with torch.no_grad():
        mu_torch = vae.encode(xd.cuda())[0]
    assert (mu - mu_torch).abs().max().item() < 1e-4 * max(1.0, mu_torch.abs().max().item())


@pytest.mark.parametrize("rows,items", [(780, 1008), (200, 8582), (64, 20000), (5, 729), (1, 1), (3, 33)])
def test_multinomial_nll_matches_torch_autograd(rows, items):
    """Fused log-softmax NLL (train_SDRM.py:143) and its gradient against the reference expression in float64."""
    from sdrm_b200.training import multinomial_nll
    g = torch.Generator().manual_seed(rows * 31 + items)
    logits = (torch.randn(rows, items, generator=g) * 3).cuda().requires_grad_(True)
    X = (torch.rand(rows, items, generator=g) < 0.05).float()
    X[0] = 0.0                                              # a row without positives contributes 0 and no gradient
    X = X.cuda()
    loss = multinomial_nll(logits, X)
    (loss * 1.7).backward()                                 # a non-trivial upstream gradient
    ref_in = logits.detach().double().cpu().requires_grad_(True)
    ref = -torch.mean(torch.sum(torch.nn.functional.log_softmax(ref_in, dim=1) * X.double().cpu(), dim=1))
    (ref * 1.7).backward()
    assert abs(loss.item() - ref.item()) <= 2e-6 * max(1.0, abs(ref.item()))
    gscale = ref_in.grad.abs().max().item() + 1e-30
    assert (logits.grad.double().cpu() - ref_in.grad).abs().max().item() <= 5e-6 * gscale
    # strided inputs (a column slice of a wider buffer) take the scalar path and agree
    wide = torch.zeros(rows, items + 5, device="cuda")
    wide[:, :items] = logits.detach()
    v = wide[:, :items].clone().requires_grad_(True)
    loss2 = multinomial_nll(v, X)
    assert abs(loss2.item() - loss.item()) <= 1e-6 * max(1.0, abs(loss.item()))
    # large-magnitude logits (scale 50, |logit| up to ~250): a softmax without the max shift overflows fp32 here.  The fp32
    # row lse of that magnitude carries ~1.5e-5 of rounding, which every softmax term of the gradient inherits.
    big = (torch.randn(rows, items, generator=g) * 50).cuda().requires_grad_(True)
    loss_b = multinomial_nll(big, X)
    (loss_b * 1.7).backward()
    ref_b_in = big.detach().double().cpu().requires_grad_(True)
    ref_b = -torch.mean(torch.sum(torch.nn.functional.log_softmax(ref_b_in, dim=1) * X.double().cpu(), dim=1))
    (ref_b * 1.7).backward()
    assert torch.isfinite(loss_b).item() and torch.isfinite(big.grad).all().item()
    assert abs(loss_b.item() - ref_b.item()) <= 2e-6 * max(1.0, abs(ref_b.item()))
    gscale_b = ref_b_in.grad.abs().max().item() + 1e-30
    assert (big.grad.double().cpu() - ref_b_in.grad).abs().max().item() <= 4e-5 * gscale_b
