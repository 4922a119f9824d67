"""Synthetic datasets from a saved generator: a checkpoint of the trained SDRM denoiser + VAE, and a CLI that samples N users,
binarises them with the training data's equal-sparsity rule and writes the rows as a sparse CSR matrix (scipy .npz).

    python -m sdrm_b200.synthesize --generator G.pt --users N --out X.npz [--seed S] [--multi-resolution]
        [--sampling-steps S] [--eta E] [--bf16] [--sparsity q] [--activity-from REAL.npz]
    torchrun --nproc_per_node G -m sdrm_b200.synthesize ...      (rows sharded over G GPUs, NCCL set up from the environment)

Every rank samples its block of rows and converts it to CSR on its GPU (sample_ddpm_sharded(gather="csr")); rank 0 writes the
file.  The rows depend on the seed and the flags, not on the number of processes.  --activity-from gives every synthetic user the
number of interactions of a user of REAL.npz instead (sparsify.activity_matched_device).
"""
import argparse
import os
import sys
import time

import torch

from .models import SDRM, VAE, make_schedule

FORMAT = "sdrm_b200.generator"
VERSION = 1


def save_generator(path, diff_net, vae_net, *, noise_divider, sparsity):
    """Write the denoiser and the VAE (constructor arguments and state dicts), the number of timesteps T, noise_divider and the
    training data's sparsity (1 - nnz / (users * items), explicit stored zeros counted, as main.py computes it) to `path`."""
    ckpt = {
        "format": FORMAT, "version": VERSION,
        "sdrm_args": dict(N_ITEMS=int(diff_net.N_ITEMS), EMB_DIM=int(diff_net.EMB_DIM), LATENT_DIM=int(diff_net.LATENT_DIM),
                          n_hidden_layers=int(diff_net.n_hidden_layers)),
        "vae_args": dict(input_dim=int(vae_net.input_dim), hidden_dim=int(vae_net.hidden_dim), latent_dim=int(vae_net.latent_dim),
                         p_drop=float(vae_net.dropout.p)),
        "sdrm_state": {k: v.detach().cpu().clone() for k, v in diff_net.state_dict().items()},
        "vae_state": {k: v.detach().cpu().clone() for k, v in vae_net.state_dict().items()},
        "T": int(diff_net.EMB_DIM), "noise_divider": float(noise_divider), "sparsity": float(sparsity),
    }
    torch.save(ckpt, path)
    return path


def load_generator(path, device):
    """(diff_net, vae_net, meta) from a save_generator file, on `device`, in eval mode.  The diffusion schedule is rebuilt with
    make_schedule(T) as train_SDRM builds it, so the loaded modules sample the same rows as the saved ones for the same seed.
    meta: {"T", "noise_divider", "sparsity", "sdrm_args", "vae_args"}."""
    ckpt = torch.load(path, map_location="cpu", weights_only=True)
    if not isinstance(ckpt, dict) or ckpt.get("format") != FORMAT:
        raise ValueError(f"{path} is not an SDRM generator checkpoint")
    if ckpt.get("version") != VERSION:
        raise ValueError(f"{path}: generator checkpoint version {ckpt.get('version')}, this code reads version {VERSION}")
    diff = SDRM(**ckpt["sdrm_args"])
    diff.load_state_dict(ckpt["sdrm_state"])
    vae = VAE(**ckpt["vae_args"])
    vae.load_state_dict(ckpt["vae_state"])
    vae.model_is_trained = True
    for p in vae.parameters():
        p.requires_grad = False
    diff, vae = diff.to(device).eval(), vae.to(device).eval()
    diff.sdrm_schedule = make_schedule(ckpt["T"], device=device)
    meta = {k: ckpt[k] for k in ("T", "noise_divider", "sparsity", "sdrm_args", "vae_args")}
    return diff, vae, meta


def build_parser():
    p = argparse.ArgumentParser(prog="python -m sdrm_b200.synthesize",
                                description="Sample a synthetic user x item dataset from a saved SDRM generator and write it as "
                                            "a sparse CSR matrix (scipy.sparse.save_npz)")
    p.add_argument("--generator", required=True, help="checkpoint written by save_generator (main.py --save-generator)")
    p.add_argument("--users", required=True, type=int, help="number of synthetic users (rows)")
    p.add_argument("--out", required=True, help="output .npz file")
    p.add_argument("--seed", type=int, default=0, help="seed of the sampler's random streams (default 0)")
    p.add_argument("--multi-resolution", action="store_true", help="M-SDRM rows (random chain lengths) instead of F-SDRM rows")
    p.add_argument("--sampling-steps", type=int, default=None, help="reverse steps of the chain; default: all T")
    p.add_argument("--eta", type=float, default=None, help="DDIM at this noise scale in [0, 1]; default: DDPM")
    p.add_argument("--bf16", action="store_true", help="sample bfloat16 rows and binarise those")
    p.add_argument("--sparsity", type=float, default=None,
                   help="share of zeros of the binarised rows, in [0, 1]; default: the training data's, from the checkpoint")
    p.add_argument("--activity-from", default=None, metavar="REAL.npz",
                   help="scipy sparse matrix of real users x the generator's items: every synthetic user keeps as many items as a "
                        "real user has (matched by rank of the equal-sparsity row sums), at its highest scores")
    return p


def parse_args(argv=None):
    p = build_parser()
    args = p.parse_args(argv)
    if args.users < 1:
        p.error("--users must be at least 1")
    if args.sparsity is not None and not 0.0 <= args.sparsity <= 1.0:
        p.error("--sparsity must lie in [0, 1]")
    if args.eta is not None and not 0.0 <= args.eta <= 1.0:
        p.error("--eta must lie in [0, 1]")
    if args.sampling_steps is not None and args.sampling_steps < 1:
        p.error("--sampling-steps must be at least 1")
    if not args.out.endswith(".npz"):
        p.error("--out must name a .npz file")
    return args


def load_activity(path, n_items):
    """row_activity of the scipy sparse matrix in `path`, which must have the generator's `n_items` columns."""
    import scipy.sparse as sp

    from .sparsify import row_activity
    real = sp.load_npz(path)
    if real.shape[1] != n_items:
        raise ValueError(f"{path}: {real.shape[1]} items, the generator samples {n_items}")
    if real.shape[0] < 1:
        raise ValueError(f"{path} holds no users")
    return row_activity(real)


def synthesize(args, group=None):
    """Sample, binarise and gather args.users rows on this process's GPU (or this rank's share); returns (SparseRows, meta)."""
    from .distributed import sample_ddpm_sharded
    dev = torch.device("cuda", torch.cuda.current_device())
    diff, vae, meta = load_generator(args.generator, dev)
    sparsity = meta["sparsity"] if args.sparsity is None else args.sparsity
    activity = None
    if getattr(args, "activity_from", None):
        activity = load_activity(args.activity_from, meta["vae_args"]["input_dim"])
    rows, _ = sample_ddpm_sharded(args.users, diff, vae, meta["sdrm_args"]["N_ITEMS"], meta["noise_divider"],
                                  timesteps="random" if args.multi_resolution else None, n_timesteps=meta["T"], seed=args.seed,
                                  group=group, gather="csr", sparsity=sparsity,
                                  out_dtype=torch.bfloat16 if args.bf16 else None,
                                  sampling_steps=args.sampling_steps, eta=args.eta, activity=activity)
    return rows, dict(meta, sparsity_used=sparsity)


def main(argv=None):
    args = parse_args(argv)
    import scipy.sparse as sp
    import torch.distributed as dist
    distributed = int(os.environ.get("WORLD_SIZE", "1")) > 1
    if distributed:
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    elif not torch.cuda.is_available():
        from ._lib import SdrmError
        raise SdrmError("sdrm_b200.synthesize needs a CUDA device (no CPU fallback)")
    try:
        start = time.time()
        rows, meta = synthesize(args)
        rank = dist.get_rank() if distributed else 0
        if rank == 0:
            mat = rows.to_scipy()
            sp.save_npz(args.out, mat)
            world = dist.get_world_size() if distributed else 1
            thr = "none (activity-matched)" if rows.threshold is None else repr(float(rows.threshold))
            print(f"synthesize: {mat.shape[0]} users x {mat.shape[1]} items, nnz {mat.nnz} "
                  f"({mat.nnz / max(1, mat.shape[0] * mat.shape[1]):.4%} ones), threshold {thr}, "
                  f"sparsity {meta['sparsity_used']}, {world} GPU(s), {time.time() - start:.2f} s -> {args.out}", flush=True)
        if distributed:
            dist.barrier()
    finally:
        if distributed:
            dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
