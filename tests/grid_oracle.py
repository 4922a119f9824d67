"""TEST INFRASTRUCTURE — CPU restatement of the fewer-step chains (sdrm_set_step_grid; sample_ddpm's sampling_steps / eta), built
on the oracle of the reference chain (oracle/sdrm_oracle.py): the grid coefficients in float64 rounded once, the fp32 chain on a
grid, and its bf16-emulating twin.  Only tests import it."""
import math

import numpy as np
import torch

from oracle import sdrm_oracle as orc


def grid_coefficients(T, timesteps, nd, eta=None):
    """[S+1, 4] float32 rows {c0, c1, c2, 0} of the chain on timesteps tau_1 < ... < tau_S (tau_0 = 0): step j maps x to
    (x - c0 eps) c1 + c2 z with z ~ N(0, 1); row 0 is zero.  Computed in float64 and rounded to float32 once, except a DDPM
    span of one step, which takes the float32 expressions of the full chain's coefficients (so the full grid reproduces them).
      eta=None, strided DDPM: a' = prod a_t over (tau_{j-1}, tau_j], c0 = (1 - a') / sqrt(1 - ab_{tau_j}), c1 = 1 / sqrt(a'),
               c2 = sqrt(1 - a') nd;
      eta in [0, 1], DDIM: ab_c = ab_{tau_j}, ab_p = ab_{tau_{j-1}} (1 at tau_0), sigma = eta sqrt((1 - ab_p) / (1 - ab_c))
               sqrt(1 - ab_c / ab_p), c1 = sqrt(ab_p / ab_c), c0 = sqrt(1 - ab_c) - sqrt(max(0, 1 - ab_p - sigma^2)) / c1,
               c2 = sigma nd.
    c2 = 0 at j = 1 in both (the reference draws no noise at its last step)."""
    b_t, a_t, ab_t = (v.numpy() for v in orc.make_schedule(T))
    tau = [0] + [int(t) for t in timesteps]
    nd64 = float(np.float32(nd))
    out = np.zeros((len(tau), 4), dtype=np.float32)
    f32 = np.float32
    for j in range(1, len(tau)):
        tc, tp = tau[j], tau[j - 1]
        if eta is None and tc - tp == 1:
            out[j, 0] = (f32(1) - a_t[tc]) / np.sqrt(f32(1) - ab_t[tc])
            out[j, 1] = f32(1) / np.sqrt(a_t[tc])
            out[j, 2] = np.sqrt(b_t[tc]) * f32(nd) if j > 1 else 0.0
            continue
        if eta is None:
            ap = 1.0
            for t in range(tp + 1, tc + 1):
                ap *= float(a_t[t])
            c = ((1 - ap) / math.sqrt(1 - float(ab_t[tc])), 1 / math.sqrt(ap), math.sqrt(1 - ap) * nd64 if j > 1 else 0.0)
        else:
            abc, abp = float(ab_t[tc]), 1.0 if tp == 0 else float(ab_t[tp])
            sigma = float(eta) * math.sqrt((1 - abp) / (1 - abc)) * math.sqrt(max(0.0, 1 - abc / abp))
            c1 = math.sqrt(abp / abc)
            c = (math.sqrt(1 - abc) - math.sqrt(max(0.0, 1 - abp - sigma * sigma)) / c1, c1, sigma * nd64)
        out[j, :3] = np.array(c, dtype=np.float64).astype(np.float32)
    return torch.from_numpy(out)


def sample_grid(sd, vsd, T, nd, xT, z, keep, timesteps, eta=None, t_start=None, return_latent=False):
    """Chain of S steps on the grid `timesteps` (grid_coefficients), full resolution or, with t_start (grid steps s_j in
    [0, S]), multi-resolution as a lock-step batch.  Step j feeds the denoiser timestep tau_j with keep[j] and adds c2 z[j];
    z / keep are [S+1, n, L] (slab j = step j)."""
    cf = grid_coefficients(T, timesteps, nd, eta)
    tau = [0] + [int(t) for t in timesteps]
    x = xT.clone()
    n = x.shape[0]
    s = torch.full((n,), len(tau) - 1, dtype=torch.long) if t_start is None else torch.as_tensor(t_start, dtype=torch.long)
    for j in range(int(s.max()), 0, -1):
        eps = orc.denoiser_forward(sd, x, torch.full((n,), tau[j], dtype=torch.long), keep[j])
        c0, c1, c2 = (float(v) for v in cf[j, :3])
        xn = (x - c0 * eps) * c1
        if c2 != 0.0:
            xn = xn + c2 * z[j]
        x = torch.where((s >= j)[:, None], xn, x)
    out = orc.vae_decode(vsd, x)
    return (out, x) if return_latent else out


def sample_bf16_emulated_grid(sd, vsd, T, nd, xT, z, keep, timesteps, eta=None, t_start=None, return_latent=False):
    """orc.sample_bf16_emulated on a step grid: step j reads row tau_j of the bias table and the grid's coefficients, in the
    kernels' operation order; t_start holds grid steps, z / keep are [S+1, n, L]."""
    nh = orc.n_hidden_of(sd)
    L = xT.shape[1]
    tab = orc.bias_table(sd, T)
    cf = grid_coefficients(T, timesteps, nd, eta)
    tau = [0] + [int(t) for t in timesteps]
    W0 = orc._bf(sd["dnn.0.weight"][:, :L]).double()
    Wo = orc._bf(sd[f"dnn.{2 + 2 * nh}.weight"]).double()
    bo = sd[f"dnn.{2 + 2 * nh}.bias"]
    x = xT.clone()
    n = x.shape[0]
    ts = torch.full((n,), len(tau) - 1, dtype=torch.long) if t_start is None else torch.as_tensor(t_start, dtype=torch.long)
    for i in range(int(ts.max()), 0, -1):
        a = orc._bf(x * keep[i].float() * 2.0).double()
        h = orc.prelu((a @ W0.T).float() + tab[tau[i]], sd["dnn.1.weight"])
        for _ in range(nh):
            h = orc.prelu((orc._bf(h).double() @ orc._bf(sd["dnn.2.weight"]).double().T).float() + sd["dnn.2.bias"], sd["dnn.3.weight"])
        eps = torch.tanh((orc._bf(h).double() @ Wo.T).float() + bo)
        c0, c1, c2 = (float(v) for v in cf[i, :3])
        xn = (x - eps * c0) * c1 + (c2 * z[i] if c2 != 0.0 else 0.0)
        x = torch.where((ts >= i)[:, None], xn, x)
    h = torch.tanh(orc._split3_linear(x, vsd["decoder.0.weight"], vsd["decoder.0.bias"]))
    out = orc._split3_linear(h, vsd["decoder.2.weight"], vsd["decoder.2.bias"])
    return (out, x) if return_latent else out
