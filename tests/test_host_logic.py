"""CPU: host-side logic of the drop-in surface (no kernels): module layout, schedule, CLI, sharding maths."""
import numpy as np
import pytest
import torch

from oracle import sdrm_oracle as orc
from sdrm_b200 import distributed as sd_dist
from sdrm_b200.models import SDRM, VAE, make_schedule


def test_state_dict_layout_matches_reference_aliases():
    m = SDRM(N_ITEMS=24, EMB_DIM=7, LATENT_DIM=24, n_hidden_layers=3)
    keys = list(m.state_dict().keys())
    assert keys[:5] == ["emb_layer.weight", "emb_layer.bias", "dnn.0.weight", "dnn.0.bias", "dnn.1.weight"]
    for j in range(3):
        assert f"dnn.{2 + 2 * j}.weight" in keys and f"dnn.{3 + 2 * j}.weight" in keys
    assert "dnn.8.weight" in keys and m.dnn[2] is m.dnn[4] is m.dnn[6]      # ONE shared hidden layer
    assert len(list(m.parameters())) == 10                                   # de-duplicated for Adam
    assert m.dnn[0].weight.shape == (24, 24 + 7) and float(m.dnn[1].weight) == 0.25
    assert len(sd_dist.unique_parameters(m)) == 10


def test_forward_equals_oracle_with_explicit_mask():
    torch.manual_seed(0)
    m = SDRM(N_ITEMS=20, EMB_DIM=6, LATENT_DIM=20, n_hidden_layers=2).eval()
    x, t = torch.randn(9, 20), torch.randint(1, 7, (9,))
    keep = (torch.rand(9, 20) < 0.5)
    ours = m(x, t, keep_mask=keep)
    ref = orc.denoiser_forward({k: v for k, v in m.state_dict().items()}, x, t, keep)
    assert torch.allclose(ours, ref, atol=1e-6)
    assert torch.allclose(m(x * keep * 2.0, t, prescaled=True), ref, atol=1e-6)
    a, b = m(x, t), m(x, t)            # dropout is ALWAYS on, even in eval mode (train_SDRM.py:100)
    assert not torch.equal(a, b)


def test_vae_matches_oracle_and_reference_attrs():
    torch.manual_seed(1)
    v = VAE(input_dim=30, hidden_dim=12, latent_dim=5).eval()
    assert v.model_is_trained is False and v.is_training == 0
    x = (torch.rand(4, 30) < 0.2).float()
    x[:, 0] = 1
    z, kl = v.encode(x)
    vsd = dict(v.state_dict())
    assert torch.allclose(z, orc.vae_encode_mu(vsd, x), atol=1e-6)
    assert torch.allclose(v.decode(z), orc.vae_decode(vsd, z), atol=1e-6)
    assert v.sample(3).shape == (3, 30)


def test_schedule_matches_oracle_bitwise():
    for T in (5, 43, 78, 83, 178):
        for a, b in zip(make_schedule(T, device="cpu"), orc.make_schedule(T)):
            assert torch.equal(a, b)


def test_resolve_steps_variants():
    from sdrm_b200.train_SDRM import _resolve_steps
    m = SDRM(8, 11, 8, 0)
    assert _resolve_steps(m, None, 11) == (11, False)
    assert _resolve_steps(m, "random", 11) == (11, True)
    assert _resolve_steps(m, 11, None) == (11, False)            # hyperparameter_search.py passes T positionally
    assert _resolve_steps(m, None, None) == (11, False)
    with pytest.raises(ValueError):
        _resolve_steps(m, None, 12)


def test_cli_flags_and_defaults_match_reference():
    import main as cli
    p = cli.build_parser()
    a = p.parse_args([])
    expect = dict(dataset="ml-1m", model="svd", augment_training_data=False, SDRM_epochs=100, SDRM_batch_size=500,
                  SDRM_lr=1e-5, SDRM_timesteps=50, SDRM_noise_variance_diminisher=0.5, MLP_hidden_layers=2,
                  VAE_batch_size=500, VAE_hidden_layer_neurons=100, MLP_latent_neurons=100, VAE_lr=1e-5)
    for k, v in expect.items():
        assert getattr(a, k) == v, k
    b = p.parse_args("--dataset ml-100k --model svd --augment-training-data --SDRM-timesteps 83 "
                     "--SDRM-noise-variance-diminisher 1.0 --MLP-hidden-layers 2 --VAE-hidden-layer-neurons 930 "
                     "--MLP-latent-neurons 830".split())
    assert (b.SDRM_timesteps, b.MLP_hidden_layers, b.VAE_hidden_layer_neurons, b.MLP_latent_neurons) == (83, 2, 930, 830)
    x = np.arange(100, dtype=np.float32).reshape(10, 10)
    assert cli.equal_sparsity(x, 0.9).sum() == 10


def test_shard_bounds_cover_rows_exactly():
    for n in (0, 1, 7, 1208, 1000000):
        for world in (1, 2, 3, 4, 8):
            spans = [sd_dist.shard_bounds(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


def test_topk_oracle_agrees_with_argpartition_sets():
    rng = np.random.RandomState(0)
    x = rng.randn(50, 300).astype(np.float32)
    for k in (1, 5, 10, 50):
        ours = orc.topk_oracle(x, k)
        ref = np.argpartition(-x, k, axis=1)[:, :k]
        assert all(set(a) == set(b) for a, b in zip(ours, ref))
    t = np.array([[1.0, 3.0, 3.0, -np.inf, np.nan, 3.0]], dtype=np.float32)
    assert orc.topk_oracle(t, 4).tolist() == [[1, 2, 5, 0]]           # ties -> lower index; NaN/-inf last
