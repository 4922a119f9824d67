"""Host-side model containers with the reference's constructor signatures and state_dict layout.

They hold the parameters (torch owns all memory) and define the maths in plain torch for autograd-based
VAE training; the diffusion hot path (sampling, the SDRM training step) does not run through
`forward` — it goes to the CUDA library via sdrm_b200.engine.

Reference: class SDRM (train_SDRM.py:86-112), class VAE (train_SDRM.py:206-268).
"""
import math

import torch
from torch import nn
from torch.nn import functional as F


def default_device():
    return "cuda" if torch.cuda.is_available() else "cpu"


def make_schedule(timesteps, beta1=1e-4, beta2=0.02, device=None):
    """DDPM schedule exactly as train_SDRM.py:297-303: ab[0] is overwritten with 1, so ab[1] = a0*a1."""
    device = device or default_device()
    b_t = (beta2 - beta1) * torch.linspace(0, 1, timesteps + 1, device=device) + beta1
    a_t = 1 - b_t
    ab_t = torch.cumsum(a_t.log(), dim=0).exp()
    ab_t[0] = 1
    return b_t, a_t, ab_t


class SDRM(nn.Module):
    """MLP denoiser.  NOTE (train_SDRM.py:94): the hidden Linear+PReLU pair is ONE module pair repeated
    n_hidden_layers times, so state_dict has alias keys dnn.2/dnn.4/... that all point at the same tensors."""

    def __init__(self, N_ITEMS, EMB_DIM, LATENT_DIM=200, n_hidden_layers=4):
        super().__init__()
        self.N_ITEMS = N_ITEMS
        self.EMB_DIM = EMB_DIM
        self.LATENT_DIM = LATENT_DIM
        self.n_hidden_layers = n_hidden_layers
        self.emb_layer = nn.Linear(EMB_DIM, EMB_DIM)
        shared = [nn.Linear(LATENT_DIM, LATENT_DIM), nn.PReLU()]
        self.dnn = nn.Sequential(nn.Linear(N_ITEMS + EMB_DIM, LATENT_DIM), nn.PReLU(),
                                 *(shared * n_hidden_layers),
                                 nn.Linear(LATENT_DIM, N_ITEMS), nn.Tanh())

    # -- parameter views used by the engine packer ------------------------------------------------
    def layer_tensors(self):
        d = self.dnn
        nh = self.n_hidden_layers
        out = d[2 + 2 * nh]
        hid = (d[2].weight, d[2].bias, d[3].weight) if nh > 0 else (None, None, None)
        return dict(We=self.emb_layer.weight, be=self.emb_layer.bias, W0=d[0].weight, b0=d[0].bias, a0=d[1].weight,
                    Wh=hid[0], bh=hid[1], ah=hid[2], Wo=out.weight, bo=out.bias)

    def timestep_embedding(self, timesteps, dim):
        half = dim // 2
        freqs = torch.exp(-math.log(10_000) * torch.arange(0, half, dtype=torch.float32, device=timesteps.device) / half)
        args = timesteps[:, None].float() * freqs[None]
        emb = torch.cat([torch.cos(args), torch.sin(args)], dim=-1)
        if dim % 2:
            emb = torch.cat([emb, emb.new_zeros(emb.shape[0], 1)], dim=-1)   # (dim = 1: emb has no column to copy)
        return emb

    def forward(self, x, t, keep_mask=None, prescaled=False):
        """eps_theta(x, t).  Dropout(p=.5) is ALWAYS active like the reference (F.dropout default
        training=True, train_SDRM.py:100); pass keep_mask to make it deterministic, or prescaled=True when
        x already is input * keep * 2 (the fused noising kernel produces it that way)."""
        emb = self.emb_layer(self.timestep_embedding(t, self.EMB_DIM))
        if prescaled:
            pass
        elif keep_mask is None:
            x = F.dropout(x, p=0.5)
        else:
            x = x * keep_mask.to(x.dtype) * 2.0
        return self.dnn(torch.cat([x, emb], dim=-1))


class VAE(nn.Module):
    """MultiVAE-style autoencoder; tanh MLP encoder to (mu, logvar), tanh MLP decoder to item logits."""

    def __init__(self, input_dim, hidden_dim, latent_dim, p_drop=0.5):
        super().__init__()
        self.input_dim, self.hidden_dim, self.latent_dim = input_dim, hidden_dim, latent_dim
        self.encoder = nn.Sequential(nn.Linear(input_dim, hidden_dim), nn.Tanh(), nn.Linear(hidden_dim, latent_dim * 2))
        self.decoder = nn.Sequential(nn.Linear(latent_dim, hidden_dim), nn.Tanh(), nn.Linear(hidden_dim, input_dim))
        self.model_is_trained = False
        self.is_training = 0  # multiplies the reparameterisation noise; 0 => deterministic encode
        self.dropout = nn.Dropout(p=p_drop)
        self.weight_decay = 0
        for m in self.modules():
            if isinstance(m, nn.Linear):
                nn.init.xavier_uniform_(m.weight.data)
                m.bias.data.normal_(0.0, 0.001)

    def reparameterize(self, mu, logvar):
        std = torch.exp(0.5 * logvar)
        eps = torch.randn_like(std)  # drawn even when is_training == 0 (RNG side effect kept, train_SDRM.py:238)
        return mu + self.is_training * eps * std

    def encode(self, x):
        h = self.encoder(self.dropout(F.normalize(x, p=2, dim=1)))
        mu_q, logvar_q = torch.chunk(h, chunks=2, dim=1)
        kl = -0.5 * torch.mean(torch.sum(1 + logvar_q - mu_q.pow(2) - logvar_q.exp(), dim=1))
        return self.reparameterize(mu_q, logvar_q), kl

    def decode(self, z):
        return self.decoder(z)

    def forward(self, x):
        z, kl = self.encode(x)
        return self.decode(z), kl

    def get_l2_reg(self):
        # reference: weight_decay (=0) * sum ||W||^2 built on an uninitialised tensor (trap T6); 0 here.
        reg = torch.zeros((), device=self.decoder[0].weight.device)
        if self.weight_decay > 0:
            for k, m in self.state_dict().items():
                if k.endswith(".weight"):
                    reg = reg + torch.norm(m, p=2) ** 2
        return self.weight_decay * reg

    def sample(self, n_samples):
        z = torch.randn(n_samples, self.latent_dim).to(self.decoder[0].weight.device)
        return self.decode(z).cpu().detach().numpy()
