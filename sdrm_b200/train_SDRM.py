"""Drop-in call surface of the reference's train_SDRM.py, backed by the CUDA library.

Same names, argument order and return values as /root/reference/train_SDRM.py so that main.py,
hyperparameter_search.py and the SVD / MLP / NeuMF benchmarks can switch by changing one import:

    train_SDRM(dl, N_ITEMS, ..., verbose=False) -> (DIFF, variational_ae)       (train_SDRM.py:271-340)
    sample_ddpm(n_sample, diff_net, vae_net, diff_latent_dim, noise_divider=1.0,
                timesteps=None, n_timesteps=None, verbose=False) -> Tensor[n, N_ITEMS] on the device   (27-63)
                (keyword-only extras, among them sampling_steps / eta for a fewer-step chain)
    SDRM, VAE, train_variational_autoencoder, perturb_input, denoise_add_noise, checkpoint, resume

The sampling chain and the diffusion training step run in hand-written sm_100a kernels through the C ABI
(include/sdrm_b200.h).  There is no CPU fallback: without CUDA or the built library these raise.
"""
import os
import time
import weakref

import numpy as np
import torch
import torch.optim as optim
from torch.nn import functional as F

from . import _lib, metrics, recommend, training
from .engine import SamplerEngine
from .models import SDRM, VAE, default_device, make_schedule  # noqa: F401  (re-exported)

DEVICE = default_device()

# The reference keeps the schedule in module globals written by train_SDRM (train_SDRM.py:297-303).
b_t = None
a_t = None
ab_t = None

_ENGINES = weakref.WeakKeyDictionary()


class TrialPruned(Exception):
    """Stand-in for optuna.TrialPruned when optuna is not installed (checkpoint / resume failures)."""


def _pruned():
    try:
        import optuna
        return optuna.TrialPruned()
    except Exception:
        return TrialPruned()


# --------------------------------------------------------------------------------------------------
# small reference-compatible helpers (plain torch; used by callers outside the hot loops)
# --------------------------------------------------------------------------------------------------
def denoise_add_noise(x, t, pred_noise, z=None):
    """x_{t-1} from x_t and eps (train_SDRM.py:20-25), on the module-global schedule."""
    if z is None:
        z = torch.randn_like(x)
    noise = b_t.sqrt()[t] * z
    mean = (x - pred_noise * ((1 - a_t[t]) / (1 - ab_t[t]).sqrt())) / a_t[t].sqrt()
    return mean + noise


def perturb_input(x, t, noise):
    """q(x_t | x_0) as the reference writes it: sqrt(ab) x + (1 - ab) noise (train_SDRM.py:202-203)."""
    return torch.as_tensor(ab_t.sqrt()[t, None] * x + (1 - ab_t[t, None]) * noise, dtype=torch.float)


def resume(model, filename, VAE_DIR_PATH):
    try:
        model.load_state_dict(torch.load(os.path.normpath(os.path.join(VAE_DIR_PATH, filename))))
    except Exception:
        print("Failed to load model parameters from %s" % filename)
        raise _pruned()


def checkpoint(model, filename, VAE_DIR_PATH):
    try:
        torch.save(model.state_dict(), os.path.normpath(os.path.join(VAE_DIR_PATH, filename)))
    except Exception:
        print("Failed to save model parameters to %s" % filename)
        raise _pruned()


# --------------------------------------------------------------------------------------------------
# sampling
# --------------------------------------------------------------------------------------------------
def _resolve_steps(diff_net, timesteps, n_timesteps):
    """main.py passes n_timesteps=T (+ timesteps='random'); hyperparameter_search.py passes the 6th
    positional argument `timesteps` as the int T or 'random' (hyperparameter_search.py:147-160)."""
    random_mode = isinstance(timesteps, str) and timesteps == "random"
    if n_timesteps is not None:
        T = int(n_timesteps)
    elif timesteps is not None and not isinstance(timesteps, str):
        T = int(timesteps)
    else:
        T = int(diff_net.EMB_DIM)
    if T != int(diff_net.EMB_DIM):
        raise ValueError(f"n_timesteps={T} does not match the denoiser's EMB_DIM={diff_net.EMB_DIM} "
                         "(the reference sets EMB_DIM = TIMESTEPS, train_SDRM.py:305)")
    return T, random_mode


def step_grid(T, sampling_steps):
    """Timesteps 1 <= tau_1 < ... < tau_S <= T of a fewer-step chain over the T-step schedule, as an int32 array.

    An int S in [1, T] gives tau_j = ceil(j T / S), so tau_S = T and S = T is the full chain; a sequence of ints is taken as an
    explicit grid and must increase strictly within [1, T]."""
    T = int(T)
    if isinstance(sampling_steps, (bool, np.bool_)):
        raise ValueError(f"sampling_steps must be an int or a sequence of ints, got {sampling_steps!r}")
    if isinstance(sampling_steps, (int, np.integer)):
        S = int(sampling_steps)
        if not 1 <= S <= T:
            raise ValueError(f"sampling_steps={S} must lie in [1, T={T}]")
        j = np.arange(1, S + 1, dtype=np.int64)
        return ((j * T + S - 1) // S).astype(np.int32)
    if isinstance(sampling_steps, torch.Tensor):
        sampling_steps = sampling_steps.tolist()
    try:
        vals = list(sampling_steps)
    except TypeError:
        raise ValueError(f"sampling_steps must be an int or a sequence of ints, got {sampling_steps!r}") from None
    if not vals or not all(isinstance(v, (int, np.integer)) and not isinstance(v, (bool, np.bool_)) for v in vals):
        raise ValueError("an explicit sampling_steps grid must be a non-empty sequence of ints")
    tau = np.asarray(vals, dtype=np.int64)
    if tau[0] < 1 or tau[-1] > T or (np.diff(tau) <= 0).any():
        raise ValueError(f"an explicit sampling_steps grid must increase strictly within [1, T={T}], got {vals}")
    return tau.astype(np.int32)


def grid_start_steps(t, timesteps):
    """Grid step at which a multi-resolution row with start timestep t_j enters a fewer-step chain: s_j = #{k >= 1 : tau_k <= t_j},
    the index of the largest grid timestep not above t_j (0: the row runs no step and decodes x_T).  On the full grid s_j = t_j."""
    return np.searchsorted(np.asarray(timesteps), np.asarray(t), side="right").astype(np.int32)


def resolve_step_grid(T, sampling_steps=None, eta=None):
    """sample_ddpm's sampling_steps / eta -> (timesteps, eta) for SamplerEngine.set_step_grid; (None, None) is the reference
    chain on all T steps.  eta=None is strided DDPM; eta in [0, 1] is DDIM, on the full grid when sampling_steps is None."""
    if eta is not None:
        if isinstance(eta, (bool, np.bool_)) or not isinstance(eta, (int, float, np.integer, np.floating)) or not 0.0 <= float(eta) <= 1.0:
            raise ValueError(f"eta must be a number in [0, 1], got {eta!r}")
        eta = float(eta)
    if sampling_steps is None:
        return (None, None) if eta is None else (step_grid(T, T), eta)
    return step_grid(T, sampling_steps), eta


def _resolve_schedule(diff_net, T, device):
    sched = getattr(diff_net, "sdrm_schedule", None)
    if sched is None and b_t is not None and b_t.numel() == T + 1:
        sched = (b_t, a_t, ab_t)
    if sched is None or sched[0].numel() != T + 1:
        sched = make_schedule(T, device=device)
    return sched


def engine_for(diff_net, device=None):
    eng = _ENGINES.get(diff_net)
    if eng is None:
        eng = SamplerEngine(device)
        _ENGINES[diff_net] = eng
    return eng


def _check_out_dtype(out_dtype, out):
    if out_dtype not in (torch.float32, torch.bfloat16):
        raise ValueError(f"out_dtype must be torch.float32 or torch.bfloat16, got {out_dtype}")
    if out is not None and out.dtype != out_dtype:
        raise ValueError(f"out has dtype {out.dtype} but out_dtype is {out_dtype}")
    return out_dtype


@torch.no_grad()
def sample_ddpm(n_sample, diff_net, vae_net, diff_latent_dim, noise_divider=1.0, timesteps=None, n_timesteps=None,
                verbose=False, *, seed=None, row_offset=0, out=None, return_latent=False, reuse_packed=False, t_rows=None,
                out_dtype=torch.float32, sampling_steps=None, eta=None, topk=None, exclude=None):
    """Reverse diffusion in the VAE latent space + decode -> float32 logits [n_sample, N_ITEMS] on the GPU.

    timesteps='random' is the multi-resolution mode: row j runs only t_j ~ U{1..T-1} steps, t_j drawn from
    NumPy's global RNG exactly like the reference (train_SDRM.py:42).  Keyword-only extras: `seed` keys the
    in-kernel Philox streams (default: drawn from torch's global generator, so torch.manual_seed makes a run
    reproducible), `row_offset` is the global id of row 0 when the rows are sharded over several GPUs, `reuse_packed=True`
    skips re-packing the weights when the parameter tensors are unchanged since the last call (the default re-packs: ~0.1 ms,
    and safe against in-place edits through `.data` that no version counter records), `t_rows` gives the multi-resolution
    chain lengths explicitly (row-sharded callers slice one global draw, sdrm_b200.distributed.sample_ddpm_sharded).
    `out_dtype=torch.bfloat16` returns bfloat16 logits: each one the round-to-nearest-even bfloat16 of the float32 logit the
    default would return for the same seed (half the bytes to keep, copy or gather; the latent stays float32).  An `out` tensor
    must have dtype `out_dtype`.

    Fewer-step sampling (the defaults run the reference's chain on all T steps):
      `sampling_steps=S` (an int in [1, T]) runs S reverse steps on the timesteps tau_j = ceil(j T / S); a sequence of ints is
      an explicit grid 1 <= tau_1 < ... < tau_S <= T.  Step j feeds the denoiser the time embedding of tau_j.
      `eta=None` (strided DDPM) applies denoise_add_noise with the jump's schedule: a' = prod a_t over (tau_{j-1}, tau_j],
      x' = (x - (1 - a') / sqrt(1 - ab_{tau_j}) eps) / sqrt(a') + sqrt(1 - a') noise_divider z.
      `eta` in [0, 1] takes the DDIM update instead (eta = 0: no noise added; eta alone runs DDIM on all T steps).
      Both read the denoiser's output as the noise eps, as the reference's denoise_add_noise does.  SDRM's denoiser applies
      dropout on every forward, so even eta = 0 is random through the keep masks.  With timesteps='random' the drawn t_j maps
      to grid step s_j = #{k : tau_k <= t_j} (grid_start_steps).  Step j draws the random streams of step index j, so x_T is
      the default call's.  Sample quality against S and eta is not characterised here.

    Top-K recommendation (the default returns the dense rows):
      `topk=k` (an int in [1, min(256, N_ITEMS)]) returns `(values [n_sample, k], indices int64 [n_sample, k])` instead of the
      dense logits: per row the k highest logits by descending score, ties to the lower item index, computed on the device from
      the rows this call samples (recommend.recommend_topk; `out` / `out_dtype` still choose the dense buffer and the dtype of
      the values).  `exclude=(indptr, indices)` is the users' history in CSR form (int64[n_sample + 1], int32[nnz], on the
      denoiser's device): row j never recommends an item of indices[indptr[j]:indptr[j + 1]].  With return_latent the result is
      `((values, indices), latent)`.  A row with fewer than k items outside its history raises ValueError after the sampling.
    """
    start_time = time.time()
    out_dtype = _check_out_dtype(out_dtype, out)
    if topk is None and exclude is not None:
        raise ValueError("exclude= needs topk=")
    diff_net.eval()
    vae_net.eval()
    dev = next(diff_net.parameters()).device
    if dev.type != "cuda":
        raise _lib.SdrmError("sample_ddpm: the denoiser must live on a CUDA device (no CPU fallback)")
    T, random_mode = _resolve_steps(diff_net, timesteps, n_timesteps)
    grid = resolve_step_grid(T, sampling_steps, eta)
    lt = diff_net.layer_tensors()
    L = lt["W0"].shape[1] - T
    if int(diff_latent_dim) != L:
        raise ValueError(f"diff_latent_dim={diff_latent_dim} but the denoiser works on {L} latent columns")
    eng = engine_for(diff_net, dev)
    eng.pack_denoiser(diff_net, _resolve_schedule(diff_net, T, dev), noise_divider, force=not reuse_packed)
    eng.pack_decoder(vae_net, force=not reuse_packed)
    eng.set_step_grid(*grid)
    if topk is not None:
        topk = recommend.check_k(topk, eng.I)
        if exclude is None:
            exclude = (torch.zeros(int(n_sample) + 1, dtype=torch.int64, device=dev), torch.empty(0, dtype=torch.int32, device=dev))
        if not isinstance(exclude, (tuple, list)) or len(exclude) != 2:
            raise TypeError("exclude must be a pair (indptr int64[n_sample + 1], indices int32[nnz])")
        exclude = recommend.check_history(exclude[0], exclude[1], int(n_sample))
        if exclude[0].device != dev or exclude[1].device != dev:
            raise ValueError(f"exclude tensors must be on {dev}, the denoiser's device")
    if seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    t_start = row_ids = None
    if random_mode:
        if T < 2:
            raise ValueError("multi-resolution sampling needs at least 2 timesteps")
        t_np = (np.random.randint(1, T, size=int(n_sample)) if t_rows is None else np.asarray(t_rows)).astype(np.int32)
        if t_np.shape != (int(n_sample),):
            raise ValueError("t_rows must have n_sample entries")
        if grid[0] is not None:
            t_np = grid_start_steps(t_np, grid[0])
        order = np.argsort(-t_np, kind="stable").astype(np.int32)  # long chains first: tiles finish together
        t_start = torch.from_numpy(t_np[order])
        row_ids = torch.from_numpy(order)
    latent = torch.empty((n_sample, L), dtype=torch.float32, device=dev) if return_latent else None
    if int(n_sample) == 0:
        empty = torch.empty((0, eng.I), dtype=out_dtype, device=dev)
        if topk is not None:
            empty = (torch.empty((0, topk), dtype=out_dtype, device=dev), torch.empty((0, topk), dtype=torch.int64, device=dev))
        return (empty, latent) if return_latent else empty
    if out is None and out_dtype != torch.float32:
        out = torch.empty((int(n_sample), eng.I), dtype=out_dtype, device=dev)
    samples = eng.sample(int(n_sample), row_offset=int(row_offset), t_start=t_start, row_ids=row_ids, seed=seed,
                         out=out, latent_out=latent)
    if topk is not None:
        samples = recommend.recommend_topk(samples[: int(n_sample), : eng.I], exclude[0], exclude[1], topk)
    if verbose:
        torch.cuda.synchronize(dev)
        print(f"Sampling {n_sample}/{n_sample}, Sampling took {np.round((time.time() - start_time) / 60, 2)} minutes")
    return (samples, latent) if return_latent else samples


@torch.no_grad()
def sample_ddpm_host(n_sample, diff_net, vae_net, diff_latent_dim, noise_divider=1.0, timesteps=None, n_timesteps=None,
                     verbose=False, *, seed=None, row_offset=0, host_out=None, chunk_rows=None, out_dtype=None,
                     sampling_steps=None, eta=None):
    """Full-resolution sample_ddpm whose result is delivered in (pinned) HOST memory — what main.py's
    `.detach().cpu().numpy()` consumes (main.py:171,175).  Rows are generated in chunks of whole CTA waves; the
    device->host copy of chunk c runs on a side stream while chunk c+1 is being computed, so the 4*I bytes per
    user never wait for the chain.  Row content is identical to sample_ddpm(seed=..., row_offset=...).
    A bfloat16 `host_out` or `out_dtype=torch.bfloat16` delivers bfloat16 rows (2*I bytes per user), identical to
    sample_ddpm(..., out_dtype=torch.bfloat16); out_dtype defaults to host_out's dtype, else float32.
    `sampling_steps` / `eta` choose a fewer-step chain exactly as in sample_ddpm."""
    if out_dtype is None:
        out_dtype = host_out.dtype if host_out is not None else torch.float32
    out_dtype = _check_out_dtype(out_dtype, host_out)
    diff_net.eval()
    vae_net.eval()
    dev = next(diff_net.parameters()).device
    if dev.type != "cuda":
        raise _lib.SdrmError("sample_ddpm_host: the denoiser must live on a CUDA device (no CPU fallback)")
    T, random_mode = _resolve_steps(diff_net, timesteps, n_timesteps)
    if random_mode:
        raise NotImplementedError("sample_ddpm_host streams full-resolution rows; use sample_ddpm for timesteps='random'")
    grid = resolve_step_grid(T, sampling_steps, eta)
    L = diff_net.layer_tensors()["W0"].shape[1] - T
    if int(diff_latent_dim) != L:
        raise ValueError(f"diff_latent_dim={diff_latent_dim} but the denoiser works on {L} latent columns")
    eng = engine_for(diff_net, dev)
    eng.pack_denoiser(diff_net, _resolve_schedule(diff_net, T, dev), noise_divider)
    eng.pack_decoder(vae_net)
    eng.set_step_grid(*grid)
    if seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    n_sample = int(n_sample)
    if host_out is None:
        host_out = torch.empty((n_sample, eng.I), dtype=out_dtype, pin_memory=True)
    if chunk_rows is None:
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        # one CTA wave per chunk: the device->host copy of a wave (57 GB/s) is shorter than its compute, so only the LAST
        # chunk's copy is exposed, and a one-wave chunk makes that tail as short as it gets
        chunk_rows = int(os.environ.get("SDRM_HOST_CHUNK_WAVES", "1")) * sms * 128
    bufs = getattr(eng, "_host_bufs", None)
    if bufs is None or bufs[0].shape != (chunk_rows, eng.I) or bufs[0].dtype != out_dtype:
        bufs = [torch.empty((chunk_rows, eng.I), dtype=out_dtype, device=dev) for _ in range(2)]
        eng._host_bufs = bufs
        eng._copy_stream = torch.cuda.Stream(dev)
    copy_stream = eng._copy_stream
    freed = [None, None]
    cur = torch.cuda.current_stream(dev)
    for c, s in enumerate(range(0, n_sample, chunk_rows)):
        e = min(s + chunk_rows, n_sample)
        buf = bufs[c & 1]
        if freed[c & 1] is not None:
            cur.wait_event(freed[c & 1])
        eng.sample(e - s, row_offset=int(row_offset) + s, seed=seed, out=buf)
        ready = torch.cuda.Event()
        ready.record(cur)
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(ready)
            host_out[s:e].copy_(buf[: e - s], non_blocking=True)
            done = torch.cuda.Event()
            done.record(copy_stream)
            freed[c & 1] = done
    copy_stream.synchronize()
    return host_out


# --------------------------------------------------------------------------------------------------
# MultiVAE++ training (adjacent to the hot path; plain torch autograd, GPU metrics for early stopping)
# --------------------------------------------------------------------------------------------------
def train_variational_autoencoder(model, train_data, test_data, epochs, batch_size, lr, early_stop_metric="NDCG@50",
                                  VAE_DIR_PATH="./", verbose=False):
    """Reference: train_SDRM.py:115-188 (multinomial NLL + annealed KL, early stopping on Recall/NDCG@k)."""
    from .data import split_train_test_proportion_from_csr_matrix
    os.makedirs(os.path.normpath(VAE_DIR_PATH), exist_ok=True)
    dev = next(model.parameters()).device
    anneal_cap, anneal_count = 0.2, 0.0
    best_metric, best_epoch, stall = -np.inf, 0, 0
    optimizer = optim.Adam(model.parameters(), lr=lr)
    kind, k = early_stop_metric.split("@")
    k = int(k)
    start_time = time.time()
    on_gpu = dev.type == "cuda"
    # the interaction matrix goes to the device ONCE (CSR); minibatches are row slices densified there (SURVEY 8f-4)
    staged = training.DeviceCSR(train_data, dev) if on_gpu else None
    n_train = train_data.shape[0]
    for epoch in range(epochs):
        losses = []
        model.train()
        model.is_training = 1
        perm = np.random.permutation(n_train)      # same draw as the reference's train_data[np.random.permutation(...)]
        if staged is None:
            train_data = train_data[perm]
        for s in range(0, n_train, batch_size):
            e = min(s + batch_size, n_train)
            anneal = min(anneal_cap, 1.0 * anneal_count / 20_000)
            if staged is not None:
                X = staged.dense_rows(perm[s:e])
            else:
                X = torch.tensor(train_data[s:e].toarray(), dtype=torch.float32, device=dev)
            optimizer.zero_grad()
            if on_gpu:
                output, vae_kl = training.vae_forward_tc(model, X)   # the four Linear layers on the tcgen05 GEMM (fwd + bwd)
            else:
                output, vae_kl = model(X)
            neg_ll = training.multinomial_nll(output, X)   # fused log-softmax NLL (train_SDRM.py:143)
            loss = neg_ll + anneal * vae_kl + model.get_l2_reg()
            losses.append(loss.detach())
            loss.backward()
            optimizer.step()
            anneal_count += 1
        model.eval()
        model.is_training = 0
        vals = []
        valid_train, valid_test = split_train_test_proportion_from_csr_matrix(test_data, batch_size=1000)
        with torch.no_grad():
            for s in range(0, valid_train.shape[0], 500):
                e = min(s + 500, valid_train.shape[0])
                Xtr = torch.tensor(valid_train[s:e].toarray(), dtype=torch.float32, device=dev)
                X_pred, _ = model(Xtr)
                X_pred = X_pred.masked_fill(Xtr != 0, float("-inf"))  # mask_training_examples, utilities.py:116-120
                held = torch.tensor(valid_test[s:e].toarray(), dtype=torch.float32, device=dev)
                if "Recall" in kind:
                    vals.append(metrics.recall_at_k_device(X_pred, held, k))
                else:
                    vals.append(metrics.ndcg_at_k_device(X_pred, held, k))
        avg_metric = np.nanmean(np.concatenate(vals))
        if verbose:
            mean_loss = float(torch.stack(losses).mean())
            print(f"Epoch: {epoch}, Loss: {np.round(mean_loss, 4)}, {early_stop_metric}: {np.round(avg_metric, 4)}", end="\r")
        if avg_metric > best_metric:
            best_metric = max(best_metric, avg_metric)
            checkpoint(model, f"epoch-{epoch}.pth", VAE_DIR_PATH)
            best_epoch, stall = epoch, 0
        else:
            stall += 1
            if stall > 20:
                if verbose:
                    print(f"MultiVAE++ training complete. Early stopping at epoch {epoch}, "
                          f"Training took {np.round((time.time() - start_time) / 60, 2)} minutes")
                break
    resume(model, f"epoch-{best_epoch}.pth", VAE_DIR_PATH)
    model.model_is_trained = True
    model.is_training = 0


# --------------------------------------------------------------------------------------------------
# SDRM training
# --------------------------------------------------------------------------------------------------
def train_SDRM(dl, N_ITEMS, VAE_HIDDEN, VAE_LATENT, VAE_BATCH_SIZE, VAE_LR, DIFF_LATENT, N_HIDDEN_MLP_LAYERS, DIFF_LR,
               DIFF_TRAINING_EPOCHS, TIMESTEPS, noise_divider, VAE_DIR_PATH, TRAIN_PARTIAL_VALID_DATA, VALID_DATA,
               OPTIMIZATION_OBJECTIVE, verbose=False):
    """Reference: train_SDRM.py:271-340.  Returns (DIFF, variational_ae) as nn.Modules on the GPU."""
    global b_t, a_t, ab_t
    if not torch.cuda.is_available():
        raise _lib.SdrmError("train_SDRM needs a CUDA device (sm_100a); there is no CPU fallback")
    dev = torch.device("cuda", torch.cuda.current_device())

    variational_ae = VAE(input_dim=N_ITEMS, hidden_dim=VAE_HIDDEN, latent_dim=VAE_LATENT).to(dev)
    assert variational_ae.model_is_trained is False
    train_variational_autoencoder(variational_ae, train_data=TRAIN_PARTIAL_VALID_DATA, test_data=VALID_DATA, epochs=500,
                                  batch_size=VAE_BATCH_SIZE, lr=VAE_LR, early_stop_metric=OPTIMIZATION_OBJECTIVE,
                                  VAE_DIR_PATH=VAE_DIR_PATH, verbose=verbose)
    assert variational_ae.model_is_trained
    for p in variational_ae.parameters():
        p.requires_grad = False
    variational_ae.eval()

    b_t, a_t, ab_t = make_schedule(TIMESTEPS, device=dev)

    DIFF = SDRM(N_ITEMS=VAE_LATENT, EMB_DIM=TIMESTEPS, LATENT_DIM=DIFF_LATENT, n_hidden_layers=N_HIDDEN_MLP_LAYERS).to(dev)
    DIFF.sdrm_schedule = (b_t, a_t, ab_t)
    DIFF.train()
    diff_optim = torch.optim.Adam(DIFF.parameters(), lr=DIFF_LR, weight_decay=0.0001, eps=1e-8)
    stepper = training.DiffusionTrainStep(DIFF, ab_t, TIMESTEPS, noise_divider)
    encoder = training.FrozenEncoder(variational_ae)   # sparse rows -> mu without densifying the batch (train_SDRM.py:323-324)

    start_time = time.time()
    # The VAE is frozen and its eval-mode encode is deterministic (train_SDRM.py:291-294), so mu of EVERY training row is computed
    # once from the device-resident CSR matrix instead of once per epoch from re-collated host batches; the loader's own batch
    # sampler still decides which rows form each minibatch (SURVEY 8a7 / 8f-4).  Any other iterable `dl` takes the generic path.
    staged = training.stage_loader(dl, dev)
    mu_all = None
    if staged is not None:
        rows_all, batch_sampler = staged
        mu_all = encoder(rows_all.as_torch_csr())
    for ep in range(DIFF_TRAINING_EPOCHS):
        if verbose:
            print(f"SDRM Epoch: {ep + 1}/{DIFF_TRAINING_EPOCHS}", end="\r")
        diff_optim.param_groups[0]["lr"] = DIFF_LR * (1 - ep / DIFF_TRAINING_EPOCHS)
        if mu_all is not None:
            batches = (mu_all[torch.as_tensor(idx, device=dev)] for idx in batch_sampler)
        else:
            batches = (encoder(x) for x, _ in iter(dl))
        for encode_x in batches:
            diff_optim.zero_grad()
            loss = stepper.loss(encode_x)
            loss.backward()
            diff_optim.step()
    if verbose:
        print(f"SDRM training complete, Training took {np.round((time.time() - start_time) / 60, 2)} minutes")
    return DIFF, variational_ae
