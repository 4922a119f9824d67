"""Multi-GPU plumbing (SURVEY.md §8e): one process per GPU, torch.distributed (NCCL over NVLink on the box,
gloo in the CPU tests).  The reference has no distributed code at all; this is new.

Sampling shards naturally: rows are independent and the Philox streams are keyed by the GLOBAL row id, so rank r
simply generates rows [lo_r, hi_r) and, for full-resolution chains, the union is bit-identical to a single-GPU run
(multi-resolution chain lengths are drawn for ALL rows from one seeded generator on every rank, see
sample_ddpm_sharded).  No collective happens during compute; gathering the rows afterwards is optional (fp32 blocks for
dataset-sized problems, bit-packed rows after the global equal-sparsity threshold at scale).

Training is data-parallel with ONE real exchange step: the score-matching loss divides by the variance of the
residual over the GLOBAL minibatch, so the five fp64 partial sums are all-reduced before the gradient seeds are
formed (sdrm_b200.training.ScoreMatchingLoss), and the flat parameter gradient is all-reduced (SUM — the seeds
already carry the global 1/N) before the identical Adam step on every rank.
"""
import torch
import torch.distributed as dist


def shard_bounds(n, rank, world):
    """Contiguous block partition of n rows: the first n % world ranks get one extra row."""
    if world < 1 or not (0 <= rank < world):
        raise ValueError("bad rank / world size")
    base, extra = divmod(int(n), world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def sample_ddpm_sharded(n_sample, diff_net, vae_net, diff_latent_dim, noise_divider=1.0, timesteps=None,
                        n_timesteps=None, *, seed, group=None, gather=False, sparsity=None, sampler=None, out_dtype=None):
    """Each rank samples its contiguous block of the n_sample rows (same `seed` on every rank; the Philox streams are keyed
    by the global row id, so in full-resolution mode the union of the blocks is bit-identical to a single-GPU run).

    timesteps='random' (multi-resolution): the per-row chain lengths t_j come from NumPy's global RNG inside the sampler
    (train_SDRM.py:42); every rank therefore draws the FULL vector of n_sample lengths here from a generator seeded with `seed`
    and uses its slice, so the result does not depend on the world size or on per-process RNG state.

    gather=False      -> (rows of this rank [hi-lo, I] fp32, (lo, hi))
    gather=True       -> the full [n_sample, I] fp32 matrix on every rank (all_gather of equal-size padded blocks: dataset-sized
                         problems only -- 80 GB at the scale-up shape)
    gather="bits"     -> equal-sparsity binarisation with the GLOBAL np.quantile threshold (sparsity = the reference's SPARSITY,
                         main.py:177-178) and an all_gather of the BIT-PACKED rows (32x less NVLink traffic: 312 MB per GPU at the
                         scale-up shape); returns (PackedMatrix of all n_sample rows, (0, n_sample))
    out_dtype=torch.bfloat16 samples bfloat16 rows (the rounded float32 rows, sample_ddpm's out_dtype): gather=False / True then
    return / gather bfloat16 blocks (half the NVLink bytes), and gather="bits" binarises the bfloat16 rows (sparsify.py: ties
    at the threshold can keep a few more ones than the float32 rows would).
    An empty block (more ranks than rows) is legal: the rank still takes part in the collectives."""
    import numpy as np
    if sampler is None:
        from .train_SDRM import sample_ddpm as sampler
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    lo, hi = shard_bounds(n_sample, rank, world)
    kw = {}
    if isinstance(timesteps, str) and timesteps == "random" and n_timesteps is not None:
        t_all = np.random.RandomState(int(seed) & 0x7FFFFFFF).randint(1, int(n_timesteps), size=int(n_sample)).astype(np.int32)
        kw["t_rows"] = t_all[lo:hi]
    if out_dtype is not None:
        kw["out_dtype"] = out_dtype
    rows = sampler(hi - lo, diff_net, vae_net, diff_latent_dim, noise_divider, timesteps=timesteps,
                   n_timesteps=n_timesteps, seed=seed, row_offset=lo, **kw)
    if not gather or world == 1:
        if gather == "bits":
            from .sparsify import equal_sparsity_device
            return equal_sparsity_device(rows, sparsity), (0, n_sample)
        return rows, (lo, hi)
    cap = shard_bounds(n_sample, 0, world)[1]  # largest block
    if gather == "bits":
        from .sparsify import PackedMatrix, equal_sparsity_device
        if sparsity is None:
            raise ValueError("gather='bits' needs the sparsity of the binarisation")
        pm = equal_sparsity_device(rows, sparsity, group=group if group is not None else dist.group.WORLD)   # (sparsify: None = one process)
        wpr = pm.bits.shape[1]
        padded = pm.bits.new_zeros((cap, wpr))
        padded[: hi - lo] = pm.bits
        parts = [torch.empty_like(padded) for _ in range(world)]
        dist.all_gather(parts, padded, group=group)
        ones = pm.ones.clone()
        dist.all_reduce(ones, group=group)
        bits = torch.cat([p[: shard_bounds(n_sample, r, world)[1] - shard_bounds(n_sample, r, world)[0]] for r, p in enumerate(parts)], dim=0)
        return PackedMatrix(bits, pm.n_cols, pm.threshold, ones), (0, n_sample)
    width = rows.shape[1]
    padded = rows.new_zeros((cap, width))
    padded[: hi - lo] = rows
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded, group=group)
    out = torch.cat([p[: shard_bounds(n_sample, r, world)[1] - shard_bounds(n_sample, r, world)[0]]
                     for r, p in enumerate(parts)], dim=0)
    return out, (0, n_sample)


def unique_parameters(module):
    """Parameters de-duplicated by identity (the shared hidden layer appears once, like in Adam's param list)."""
    seen, out = set(), []
    for p in module.parameters():
        if id(p) not in seen:
            seen.add(id(p))
            out.append(p)
    return out


def allreduce_gradients(module, group=None):
    """SUM-all-reduce all gradients as one flat bucket (8-12 MB for the SDRM denoiser: latency-, not bandwidth-bound)."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return
    params = [p for p in unique_parameters(module) if p.grad is not None]
    if not params:
        return
    flat = torch.cat([p.grad.reshape(-1) for p in params])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    off = 0
    for p in params:
        n = p.grad.numel()
        p.grad.copy_(flat[off: off + n].view_as(p.grad))
        off += n


def dp_train_step(stepper, optimizer, mu_global, t_global=None, group=None, inj_noise=None, inj_masks=None):
    """One data-parallel diffusion training step on a GLOBAL minibatch of latents [B, L] known to every rank:
    rank r works on its block of rows; returns the global loss (identical on all ranks).  When t_global is None the step draws
    the WHOLE vector of B timesteps from the CPU generator (like the reference, train_SDRM.py:327) on every rank -- ranks seeded
    alike therefore agree on it -- and each rank uses its slice."""
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    lo, hi = shard_bounds(mu_global.shape[0], rank, world)
    stepper.group = (group if group is not None else dist.group.WORLD) if world > 1 else None
    stepper.row_offset = lo
    optimizer.zero_grad()
    if t_global is None:
        t_global = torch.randint(1, stepper.T + 1, (mu_global.shape[0],))
    if hi == lo:
        raise ValueError(f"data-parallel step: rank {rank} has no row (minibatch of {mu_global.shape[0]} rows on {world} ranks)")
    loss = stepper.loss(mu_global[lo:hi], None if t_global is None else t_global[lo:hi],
                        None if inj_noise is None else inj_noise[lo:hi].contiguous(),
                        None if inj_masks is None else inj_masks[:, lo:hi].contiguous())
    loss.backward()
    allreduce_gradients(stepper.net, group)
    optimizer.step()
    return loss.detach()
