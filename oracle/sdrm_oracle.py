"""TEST INFRASTRUCTURE — CPU restatement (the ORACLE) of SDRM's diffusion hot path.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg may import
this module; the product path (sdrm_b200/) never does.

Every function restates, in plain fp32 torch on the CPU and with ALL randomness passed in explicitly,
what /root/reference/train_SDRM.py computes.  Parity pinning: tests/golden/make_golden.py imports the
real reference in the build container, replays its RNG draw order, and stores inputs + the
reference's own outputs; tests/test_oracle_golden.py checks this oracle against those files.

Weights are passed as reference-style state_dicts:
  denoiser: emb_layer.{weight,bias}, dnn.0.{weight,bias}, dnn.1.weight, [dnn.2.{weight,bias}, dnn.3.weight,]
            dnn.{2+2nh}.{weight,bias}                                   (train_SDRM.py:86-95)
  vae:      encoder.{0,2}.{weight,bias}, decoder.{0,2}.{weight,bias}    (train_SDRM.py:210-215)
"""
import math

import numpy as np
import torch
import torch.nn.functional as F


# ------------------------------------------------------------------------------------------------
# schedule (train_SDRM.py:275-276, 297-303)
# ------------------------------------------------------------------------------------------------
def make_schedule(T, beta1=1e-4, beta2=0.02):
    b_t = (beta2 - beta1) * torch.linspace(0, 1, T + 1) + beta1
    a_t = 1 - b_t
    ab_t = torch.cumsum(a_t.log(), dim=0).exp()
    ab_t[0] = 1
    return b_t, a_t, ab_t


# ------------------------------------------------------------------------------------------------
# denoiser (SDRM.forward / timestep_embedding, train_SDRM.py:97-112)
# ------------------------------------------------------------------------------------------------
def n_hidden_of(sd):
    n_lin = len([k for k in sd if k.startswith("dnn.") and k.endswith(".bias")])
    return n_lin - 2


def timestep_embedding(t, dim):
    half = dim // 2
    freqs = torch.exp(-math.log(10_000) * torch.arange(start=0, end=half, dtype=torch.float32, device=t.device) / half)
    args = t[:, None].float() * freqs[None]
    emb = torch.cat([torch.cos(args), torch.sin(args)], dim=-1)
    if dim % 2:
        emb = torch.cat([emb, torch.zeros(emb.shape[0], 1, dtype=emb.dtype, device=emb.device)], dim=-1)   # (dim = 1: emb has no column to copy)
    return emb


def prelu(x, a):
    return torch.where(x > 0, x, a * x)


def denoiser_forward(sd, x, t, keep_mask):
    """eps = SDRM.forward(x, t) with the dropout keep-mask given explicitly (F.dropout p=.5, line 100)."""
    T = sd["emb_layer.weight"].shape[0]
    nh = n_hidden_of(sd)
    w_emb = sd["emb_layer.weight"]
    # the sinusoid is fp32 like the model's; widened to the weights' dtype so that a float64 state_dict runs in float64
    emb = F.linear(timestep_embedding(t, T).to(w_emb.dtype), w_emb, sd["emb_layer.bias"])
    h = torch.cat([x * keep_mask.to(x.dtype) * 2.0, emb], dim=-1)
    h = prelu(F.linear(h, sd["dnn.0.weight"], sd["dnn.0.bias"]), sd["dnn.1.weight"])
    for _ in range(nh):  # the SAME Linear + PReLU nh times (train_SDRM.py:94)
        h = prelu(F.linear(h, sd["dnn.2.weight"], sd["dnn.2.bias"]), sd["dnn.3.weight"])
    last = 2 + 2 * nh
    return torch.tanh(F.linear(h, sd[f"dnn.{last}.weight"], sd[f"dnn.{last}.bias"]))


def posterior_step(x, eps, z_scaled, i, sched):
    """denoise_add_noise (train_SDRM.py:20-25) with z already multiplied by noise_divider."""
    b_t, a_t, ab_t = sched
    noise = b_t.sqrt()[i] * z_scaled
    mean = (x - eps * ((1 - a_t[i]) / (1 - ab_t[i]).sqrt())) / a_t[i].sqrt()
    return mean + noise


def vae_decode(vsd, z):
    h = torch.tanh(F.linear(z, vsd["decoder.0.weight"], vsd["decoder.0.bias"]))
    return F.linear(h, vsd["decoder.2.weight"], vsd["decoder.2.bias"])


def vae_encode_mu(vsd, x):
    """VAE.encode in eval mode returns mu (train_SDRM.py:236-250; is_training == 0)."""
    xn = F.normalize(x, p=2, dim=1)
    h = torch.tanh(F.linear(xn, vsd["encoder.0.weight"], vsd["encoder.0.bias"]))
    out = F.linear(h, vsd["encoder.2.weight"], vsd["encoder.2.bias"])
    mu, _ = torch.chunk(out, 2, dim=1)
    return mu


# ------------------------------------------------------------------------------------------------
# samplers (train_SDRM.py:27-63)
# ------------------------------------------------------------------------------------------------
def sample_full(sd, vsd, T, nd, xT, z, keep, return_latent=False):
    """Full-resolution chain.  z[i] (i>=2) are N(0,1) draws, keep[i] (i>=1) dropout keep masks, [T+1,n,L]."""
    sched = make_schedule(T)
    x = xT.clone()
    n = x.shape[0]
    for i in range(T, 0, -1):
        zz = z[i] * nd if i > 1 else 0
        eps = denoiser_forward(sd, x, torch.full((n,), i, dtype=torch.long), keep[i])
        x = posterior_step(x, eps, zz, i, sched)
    out = vae_decode(vsd, x)
    return (out, x) if return_latent else out


def sample_random(sd, vsd, T, nd, xT, z, keep, t_start, return_latent=False):
    """Multi-resolution mode (train_SDRM.py:37-49) as a lock-step batch: row j runs steps t_start[j]..1."""
    sched = make_schedule(T)
    x = xT.clone()
    n = x.shape[0]
    t_start = torch.as_tensor(t_start, dtype=torch.long)
    for i in range(int(t_start.max()), 0, -1):
        zz = z[i] * nd if i > 1 else torch.zeros_like(x)
        eps = denoiser_forward(sd, x, torch.full((n,), i, dtype=torch.long), keep[i])
        xn = posterior_step(x, eps, zz, i, sched)
        x = torch.where((t_start >= i)[:, None], xn, x)
    out = vae_decode(vsd, x)
    return (out, x) if return_latent else out


# bf16-emulating variant: rounds exactly where the CUDA kernel rounds (operands of every GEMM),
# keeps fp32 accumulation / epilogues, hoists the time-embedding into a bias table, and uses the
# bf16x3 split in the decoder.  Used to separate "kernel bug" from "bf16 effect" in the GPU tests.
def _bf(x):
    return x.to(torch.bfloat16).to(torch.float32)


def bias_table(sd, T):
    L = sd["dnn.0.weight"].shape[1] - T
    temb = timestep_embedding(torch.arange(T + 1), T)
    emb = F.linear(temb, sd["emb_layer.weight"], sd["emb_layer.bias"])
    return F.linear(emb, sd["dnn.0.weight"][:, L:], sd["dnn.0.bias"])  # [T+1, D]


def _split3_linear(x, W, b):
    xh, Wh = _bf(x), _bf(W)
    xl, Wl = _bf(x - xh), _bf(W - Wh)
    return (xh.double() @ Wh.double().T + xh.double() @ Wl.double().T + xl.double() @ Wh.double().T).float() + b


def sample_bf16_emulated(sd, vsd, T, nd, xT, z, keep, t_start=None, return_latent=False):
    b_t, a_t, ab_t = make_schedule(T)
    nh = n_hidden_of(sd)
    L = xT.shape[1]
    tab = bias_table(sd, T)
    W0 = _bf(sd["dnn.0.weight"][:, :L]).double()
    Wo = _bf(sd[f"dnn.{2 + 2 * nh}.weight"]).double()
    bo = sd[f"dnn.{2 + 2 * nh}.bias"]
    x = xT.clone()
    n = x.shape[0]
    ts = torch.full((n,), T, dtype=torch.long) if t_start is None else torch.as_tensor(t_start, dtype=torch.long)
    for i in range(int(ts.max()), 0, -1):
        a = _bf(x * keep[i].float() * 2.0).double()
        h = prelu((a @ W0.T).float() + tab[i], sd["dnn.1.weight"])
        for _ in range(nh):
            h = prelu((_bf(h).double() @ _bf(sd["dnn.2.weight"]).double().T).float() + sd["dnn.2.bias"], sd["dnn.3.weight"])
        eps = torch.tanh((_bf(h).double() @ Wo.T).float() + bo)
        c1 = (1 - a_t[i]) / (1 - ab_t[i]).sqrt()
        c2 = 1.0 / a_t[i].sqrt()
        sg = b_t[i].sqrt() * nd if i > 1 else 0.0
        xn = (x - eps * c1) * c2 + sg * z[i]
        x = torch.where((ts >= i)[:, None], xn, x)
    h = torch.tanh(_split3_linear(x, vsd["decoder.0.weight"], vsd["decoder.0.bias"]))
    out = _split3_linear(h, vsd["decoder.2.weight"], vsd["decoder.2.bias"])
    return (out, x) if return_latent else out


# ------------------------------------------------------------------------------------------------
# training step (train_SDRM.py:321-337, 191-203)
# ------------------------------------------------------------------------------------------------
def perturb_input(x, t, noise, ab_t):
    return ab_t.sqrt()[t, None] * x + (1 - ab_t[t, None]) * noise


def training_loss(sd, mu, t, noise_scaled, keeps, T, mu_coef=0.1):
    """Score-matching loss of one minibatch.  keeps = 3 dropout keep masks (pred, sx, psx); autograd-friendly.  Runs on the
    device of its inputs (a float64 state_dict on the GPU is the oracle at shapes the CPU would take minutes over)."""
    ab_t = make_schedule(T)[2].to(mu.device)
    x_pert = perturb_input(mu, t, noise_scaled, ab_t)
    pred = denoiser_forward(sd, x_pert, t, keeps[0])
    sx = denoiser_forward(sd, mu, t, keeps[1])
    psx = denoiser_forward(sd, mu + mu_coef * noise_scaled, t, keeps[2])
    sd_ = (psx - sx) / (mu_coef ** 2)
    r = pred - mu
    loss = 0.5 * (F.mse_loss(sd_, r) + F.mse_loss(r, sx)) / (1e-8 + r.var())
    return loss, (pred, sx, psx)


def loss_grad_seeds(pred, sx, psx, mu, mu_coef=0.1):
    """Closed-form d loss / d {pred, sx, psx} (SURVEY.md §8a9), fp64."""
    pred, sx, psx, mu = (v.double() for v in (pred, sx, psx, mu))
    N = pred.numel()
    r = pred - mu
    sd_ = (psx - sx) / (mu_coef ** 2)
    V = r.var()
    A = ((sd_ - r) ** 2).mean()
    Bm = ((r - sx) ** 2).mean()
    den = 1e-8 + V
    c = 0.5 / den
    g_sd = 2 * c * (sd_ - r) / N
    g_psx = g_sd / (mu_coef ** 2)
    g_sx = -2 * c * (r - sx) / N - g_sd / (mu_coef ** 2)
    g_pred = c * (-2 * (sd_ - r) + 2 * (r - sx)) / N - 0.5 * (A + Bm) / den ** 2 * 2 * (r - r.mean()) / (N - 1)
    return g_pred, g_sx, g_psx, 0.5 * (A + Bm) / den


# ------------------------------------------------------------------------------------------------
# metrics (utilities.py:116-171)
# ------------------------------------------------------------------------------------------------
def topk_oracle(scores, k):
    """Deterministic top-k: descending score, ties -> lower index (stable argsort of -score); NaN last."""
    s = np.asarray(scores, dtype=np.float32).copy()
    s[np.isnan(s)] = -np.inf
    order = np.argsort(-s, axis=1, kind="stable")
    return order[:, :k].astype(np.int32)


def recall_at_k_oracle(X_pred, heldout, k):
    """utilities.recall_at_k_batch with the deterministic top-k above (np.argpartition ties are
    implementation-defined; the reference result is identical whenever score k and k+1 differ)."""
    idx = topk_oracle(X_pred, k)
    rows = X_pred.shape[0]
    pred_bin = np.zeros(X_pred.shape, dtype=bool)
    pred_bin[np.arange(rows)[:, None], idx] = True
    true_bin = np.asarray(heldout) > 0
    tmp = np.logical_and(true_bin, pred_bin).sum(axis=1).astype(np.float32)
    with np.errstate(invalid="ignore", divide="ignore"):
        return tmp / np.minimum(k, true_bin.sum(axis=1))


def ndcg_at_k_oracle(X_pred, heldout, k):
    """utilities.NDCG_binary_at_k_batch; IDCG counts stored entries like getnnz on a dense->csr matrix."""
    idx = topk_oracle(X_pred, k)
    rows = X_pred.shape[0]
    tp = 1.0 / np.log2(np.arange(2, k + 2))
    held = np.asarray(heldout, dtype=np.float64)
    dcg = (held[np.arange(rows)[:, None], idx] * tp).sum(axis=1)
    idcg = np.array([tp[: min(int(n), k)].sum() for n in (held != 0).sum(axis=1)])
    with np.errstate(invalid="ignore", divide="ignore"):
        return dcg / idcg
