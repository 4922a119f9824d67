"""Fewer-step sampling on the host: the step-grid rule, the multi-resolution start-step mapping, argument checking, and the
CPU oracle's grid coefficients (sample_ddpm's sampling_steps / eta; sdrm_set_step_grid)."""
import math

import numpy as np
import pytest
import torch

from oracle import philox_ref
from oracle import sdrm_oracle as orc
import grid_oracle as go
from helpers import random_modules, rel_fro, state_dicts
from sdrm_b200.train_SDRM import grid_start_steps, resolve_step_grid, step_grid


def test_step_grid_rule():
    assert step_grid(7, 7).tolist() == list(range(1, 8))          # S = T: the full chain
    assert step_grid(83, 83).tolist() == list(range(1, 84))
    assert step_grid(7, 1).tolist() == [7]
    assert step_grid(10, 3).tolist() == [4, 7, 10]                 # ceil(j T / S) with S not dividing T
    assert step_grid(178, 89).tolist() == list(range(2, 179, 2))
    for T in (2, 43, 83, 93, 178):
        for S in sorted({1, 2, 10, 25, T // 4, T // 2, T - 1, T} - {0}):
            if S > T:
                continue
            tau = step_grid(T, S)
            assert tau.dtype == np.int32 and len(tau) == S and tau[-1] == T and tau[0] >= 1
            assert (np.diff(tau) > 0).all()
            assert tau.tolist() == [math.ceil(j * T / S) for j in range(1, S + 1)]
    assert step_grid(np.int64(10), np.int32(3)).tolist() == [4, 7, 10]


def test_explicit_grids():
    assert step_grid(9, [1, 2, 5, 9]).tolist() == [1, 2, 5, 9]
    assert step_grid(9, (3,)).tolist() == [3]                      # need not end at T
    assert step_grid(9, np.array([2, 4, 8])).tolist() == [2, 4, 8]
    assert step_grid(9, torch.tensor([1, 6])).tolist() == [1, 6]
    assert step_grid(9, range(1, 10)).tolist() == list(range(1, 10))


@pytest.mark.parametrize("bad", [0, -1, 10, True, 2.5, "3", [], [0, 1], [3, 3], [4, 2], [1, 10], [1.0, 2.0], [True]])
def test_bad_sampling_steps_raise(bad):
    with pytest.raises(ValueError):
        step_grid(9, bad)
    with pytest.raises(ValueError):
        resolve_step_grid(9, bad, None)


@pytest.mark.parametrize("bad", [-0.1, 1.5, float("nan"), float("inf"), True, "0.5", [0.5]])
def test_bad_eta_raises(bad):
    with pytest.raises(ValueError):
        resolve_step_grid(9, None, bad)
    with pytest.raises(ValueError):
        resolve_step_grid(9, 3, bad)


def test_resolve_step_grid():
    assert resolve_step_grid(9) == (None, None)                    # the reference chain, untouched
    tau, eta = resolve_step_grid(9, 3)
    assert tau.tolist() == [3, 6, 9] and eta is None
    tau, eta = resolve_step_grid(9, None, 0)                       # eta alone: DDIM on the full grid
    assert tau.tolist() == list(range(1, 10)) and eta == 0.0 and isinstance(eta, float)
    tau, eta = resolve_step_grid(9, [2, 5], 1)
    assert tau.tolist() == [2, 5] and eta == 1.0


def test_grid_start_steps():
    tau = [4, 7, 10]
    t = np.array([0, 1, 3, 4, 5, 6, 7, 9, 10])
    assert grid_start_steps(t, tau).tolist() == [0, 0, 0, 1, 1, 1, 2, 2, 3]
    assert grid_start_steps(t, tau).dtype == np.int32
    full = np.arange(1, 11)
    rng = np.random.RandomState(0)
    t = rng.randint(1, 10, size=500)
    assert (grid_start_steps(t, full) == t).all()                  # the full grid maps every row to its own step
    s = grid_start_steps(t, [5, 9])
    assert ((s == 0) == (t < 5)).all() and ((s == 2) == (t >= 9)).all()


# ---- the oracle ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("T,nd", [(7, 1.0), (83, 1.0), (43, 0.2)])
def test_full_grid_coefficients_equal_posterior_step(T, nd):
    b_t, a_t, ab_t = orc.make_schedule(T)
    cf = go.grid_coefficients(T, range(1, T + 1), nd)
    assert cf.dtype == torch.float32 and cf.shape == (T + 1, 4)
    assert (cf[0] == 0).all() and (cf[:, 3] == 0).all()
    for i in range(1, T + 1):
        assert cf[i, 0] == (1 - a_t[i]) / (1 - ab_t[i]).sqrt()     # the expression posterior_step uses, bit for bit
        assert abs(float(cf[i, 1]) * float(a_t[i].sqrt()) - 1) < 2e-7
        assert cf[i, 2] == ((b_t[i].sqrt() * nd) if i > 1 else 0.0)
    # posterior_step with these coefficients reproduces the reference update
    x, eps, z = torch.randn(3, 5, 6).unbind(0)
    for i in (1, 2, T):
        ref = orc.posterior_step(x, eps, z * nd if i > 1 else 0, i, (b_t, a_t, ab_t))
        got = (x - cf[i, 0] * eps) * cf[i, 1] + cf[i, 2] * z
        assert torch.allclose(got, ref, rtol=1e-6, atol=1e-6)


def test_strided_ddpm_coefficients():
    T, nd = 10, 0.5
    b_t, a_t, ab_t = (v.double() for v in orc.make_schedule(T))
    cf = go.grid_coefficients(T, [4, 7, 10], nd)
    for j, (tp, tc) in enumerate([(0, 4), (4, 7), (7, 10)], start=1):
        ap = float(torch.prod(a_t[tp + 1:tc + 1]))
        want = [(1 - ap) / math.sqrt(1 - float(ab_t[tc])), 1 / math.sqrt(ap), math.sqrt(1 - ap) * nd if j > 1 else 0.0]
        assert cf[j, :3].tolist() == pytest.approx(want, rel=1e-6)


@pytest.mark.parametrize("eta", [0.0, 0.5, 1.0])
def test_ddim_coefficients(eta):
    T, nd = 20, 1.0
    _, _, ab_t = (v.double() for v in orc.make_schedule(T))
    tau = [1, 3, 8, 20]
    cf = go.grid_coefficients(T, tau, nd, eta)
    assert cf[1, 2] == 0.0                                         # sigma = 0 at the last step (ab_0 = 1)
    if eta == 0.0:
        assert (cf[:, 2] == 0).all()
    x, eps = torch.randn(2, 4, 5, dtype=torch.float64).unbind(0)
    for j in range(1, len(tau) + 1):
        abc, abp = float(ab_t[tau[j - 1]]), 1.0 if j == 1 else float(ab_t[tau[j - 2]])
        sigma = eta * math.sqrt((1 - abp) / (1 - abc)) * math.sqrt(1 - abc / abp)
        assert float(cf[j, 2]) == pytest.approx(sigma * nd, rel=1e-6, abs=1e-12)
        x0 = (x - math.sqrt(1 - abc) * eps) / math.sqrt(abc)    # the DDIM update, noise-free part
        want = math.sqrt(abp) * x0 + math.sqrt(max(0.0, 1 - abp - sigma ** 2)) * eps
        got = (x - float(cf[j, 0]) * eps) * float(cf[j, 1])
        assert torch.allclose(got, want, rtol=1e-5, atol=1e-5)


def test_oracle_full_grid_chain_equals_reference_chain():
    """sample_grid on the explicit full grid is sample_full / sample_random, and the emulated sampler's grid path is its
    default path (the noise slabs of the full grid are the reference's)."""
    I, H, L, T, nh, nd = 50, 24, 20, 6, 1, 0.7
    diff, vae = random_modules(I, H, L, T, nh, seed=4)
    dsd, vsd = state_dicts(diff, vae)
    xT, z, keep = (torch.from_numpy(a) for a in philox_ref.sampler_noise(11, 0, 9, L, T))
    full = orc.sample_full(dsd, vsd, T, nd, xT, z, keep)
    assert rel_fro(go.sample_grid(dsd, vsd, T, nd, xT, z, keep, range(1, T + 1)), full) < 1e-6
    ts = np.array([0, 1, 2, 3, 4, 5, 5, 2, 1])
    rnd = orc.sample_random(dsd, vsd, T, nd, xT, z, keep, ts)
    assert rel_fro(go.sample_grid(dsd, vsd, T, nd, xT, z, keep, range(1, T + 1), t_start=ts), rnd) < 1e-6
    emu = orc.sample_bf16_emulated(dsd, vsd, T, nd, xT, z, keep)
    assert rel_fro(go.sample_bf16_emulated_grid(dsd, vsd, T, nd, xT, z, keep, range(1, T + 1)), emu) < 1e-6
    # a strided grid: the emulation stays near the fp32 oracle
    tau = [2, 3, 6]
    g = go.sample_grid(dsd, vsd, T, nd, xT, z[:4], keep[:4], tau)
    assert rel_fro(go.sample_bf16_emulated_grid(dsd, vsd, T, nd, xT, z[:4], keep[:4], tau), g) < 2e-2
