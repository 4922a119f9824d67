"""SDRM reproducibility driver with the reference's CLI (reference: main.py:88-377), running the diffusion
hot path on the B200 CUDA library.  Same 13 flags and defaults; `--runs`, `--data-dir`, `--seed` are additions.

    python main.py --dataset ml-100k --model svd --augment-training-data --SDRM-epochs 265 --SDRM-batch-size 550 \
        --SDRM-lr 1e-5 --SDRM-timesteps 83 --SDRM-noise-variance-diminisher 1.0 --MLP-hidden-layers 2 \
        --VAE-batch-size 200 --VAE-hidden-layer-neurons 930 --MLP-latent-neurons 830 --VAE-lr 1e-4
"""
import argparse
import time

import numpy as np

ROWS = ["Recall@1", "Recall@3", "Recall@5", "Recall@10", "Recall@20", "Recall@50",
        "NDCG@1", "NDCG@3", "NDCG@5", "NDCG@10", "NDCG@20", "NDCG@50"]
COLS = ["F-SDRM", "M-SDRM", "MultiVAE++"]


def build_parser():
    p = argparse.ArgumentParser(prog="SDRM Reproducibility", description="Run this file to reproduce results from SDRM paper")
    p.add_argument("--dataset", type=str, default="ml-1m", help="Dataset to run experiments on")
    p.add_argument("--model", type=str, default="svd", help="Model to run experiments on")
    p.add_argument("--augment-training-data", action="store_true", default=False,
                   help="Whether to augment training data with synthetic data")
    p.add_argument("--SDRM-epochs", type=int, default=100, help="Number of epochs to train for")
    p.add_argument("--SDRM-batch-size", type=int, default=500, help="Batch size to use for training SDRM")
    p.add_argument("--SDRM-lr", type=float, default=0.00001, help="Learning rate to use for training SDRM")
    p.add_argument("--SDRM-timesteps", type=int, default=50, help="Number of timesteps to use for training SDRM")
    p.add_argument("--SDRM-noise-variance-diminisher", type=float, default=0.5,
                   help="Noise variance diminisher to use for training SDRM")
    p.add_argument("--SDRM-sampling-steps", type=int, default=None,
                   help="reverse steps of the sampling chain (strided over the training timesteps); default: all of them")
    p.add_argument("--SDRM-eta", type=float, default=None,
                   help="sample with DDIM at this noise scale in [0, 1] instead of DDPM; default: DDPM")
    p.add_argument("--MLP-hidden-layers", type=int, default=2, help="Number of hidden layers to use for training MLP")
    p.add_argument("--VAE-batch-size", type=int, default=500, help="Batch size to use for training VAE")
    p.add_argument("--VAE-hidden-layer-neurons", type=int, default=100,
                   help="Number of hidden layer neurons to use for training VAE")
    p.add_argument("--MLP-latent-neurons", type=int, default=100, help="Number of latent neurons to use for training MLP")
    p.add_argument("--VAE-lr", type=float, default=0.00001, help="Learning rate to use for training VAE")
    # additions (not in the reference)
    p.add_argument("--runs", type=int, default=5, help="number of independent runs (reference: 5)")
    p.add_argument("--data-dir", type=str, default="./data", help="directory holding <dataset>/<dataset>_*.pkl")
    p.add_argument("--seed", type=int, default=None, help="seed torch / numpy for a reproducible run")
    p.add_argument("--privacy-audit", action="store_true", default=False,
                   help="after each run, print how close the binarised synthetic rows come to the training rows (privacy_audit)")
    p.add_argument("--fidelity-audit", action="store_true", default=False,
                   help="after each run, print how closely the binarised synthetic rows resemble the training rows (fidelity_audit)")
    p.add_argument("--save-generator", type=str, default=None, metavar="DIR",
                   help="write each run's trained denoiser + VAE to DIR/run{n}_generator.pt (python -m sdrm_b200.synthesize reads it)")
    p.add_argument("--save-synthetic", type=str, default=None, metavar="DIR",
                   help="write each run's binarised synthetic rows to DIR/run{n}_{F-SDRM,M-SDRM,MultiVAE++}.npz (scipy sparse CSR)")
    p.add_argument("--svd-on-gpu", action="store_true", default=False,
                   help="--model svd: run the SVD evaluator's randomized SVD on the GPU from the binarised rows where they are "
                        "(evaluators.compute_mf_results_gpu) instead of sklearn on dense host rows")
    p.add_argument("--binarise", choices=["equal-sparsity", "activity"], default="equal-sparsity",
                   help="equal-sparsity: the reference's single global threshold; activity: every synthetic row keeps the number "
                        "of interactions of a training user, at its highest scores (sparsify.activity_matched_device, on the GPU)")
    return p


def equal_sparsity(scores, sparsity):
    """Binarise so the synthetic matrix keeps the training sparsity (main.py:177-185).

    CUDA score matrices never leave the GPU as floats: kernel K4 finds np.quantile's threshold with an exact radix select
    and ships 1 bit per entry (sdrm_b200/sparsify.py); the result is identical to the reference's host-side lines.
    Host arrays (VAE.sample returns a NumPy array in the reference too, main.py:183) take the reference's own two lines."""
    return binarise(scores, sparsity)[0]


def binarise(scores, sparsity):
    """equal_sparsity, returning (dense 0/1 rows, the device PackedMatrix of CUDA scores or None for host arrays), so that the
    privacy audit searches the bits already on the GPU instead of uploading the dense frame again."""
    import torch
    if isinstance(scores, torch.Tensor):
        from sdrm_b200.sparsify import equal_sparsity_device
        pm = equal_sparsity_device(scores.detach(), sparsity)
        return pm.numpy(int), pm
    return (scores >= np.quantile(scores.flatten(), sparsity)).astype(int), None


def binarise_activity(scores, sparsity, activity):
    """The activity-matched binarisation (sdrm_b200/sparsify.py activity_matched_device): rows ranked by their equal-sparsity
    row sums take the training users' activities at the same quantile, at their highest scores.  Host arrays (VAE.sample) are
    uploaded as float32.  Returns (dense 0/1 rows, the device PackedMatrix) like binarise."""
    import torch

    from sdrm_b200.sparsify import activity_matched_device
    if not isinstance(scores, torch.Tensor):
        scores = torch.as_tensor(np.asarray(scores, dtype=np.float32), device="cuda")
    pm = activity_matched_device(scores.detach(), sparsity, activity)
    return pm.numpy(int), pm


AUDIT_COLS = ["DCR mean", "DCR p5", "DCR p50", "DCR p95", "exact copies", "copy share", "NNDR median"]


def privacy_audit(binarised, real, baseline=None):
    """Distance to the closest record of every binarised synthetic row set against `real` (the rows the generator was trained
    on, TRAIN_PARTIAL_VALID_DATA), with the real rows against themselves (each row's own index excluded) as the baseline line.
    DCR = 1 - Jaccard similarity of the nearest real row; exact copies have Hamming distance 0; NNDR = DCR of the nearest over
    DCR of the second nearest real row (sdrm_b200.privacy.NearestRows.summary).  Returns (table, baseline summary).

    Read the synthetic lines against the baseline line, not against 0.  Equal sparsity keeps 1 - SPARSITY of the entries, and
    SPARSITY counts the training matrix's explicit stored zeros as interactions, so synthetic rows carry more ones than real
    rows do (10.07 % against 5.75 % of the entries at ml-100k).  That alone lowers their Jaccard similarity to any real row."""
    import pandas as pd

    from sdrm_b200.privacy import nearest_rows
    if baseline is None:
        baseline = nearest_rows(real, real, k=2, exclude_same_index=True).summary()
    rows = {}
    for name, (dense, packed) in binarised.items():
        rows[name] = nearest_rows(packed if packed is not None else dense, real, k=2).summary()
    rows["real vs real (baseline)"] = baseline
    keys = ["dcr_mean", "dcr_p5", "dcr_p50", "dcr_p95", "exact_copies", "exact_copy_share", "nndr_median"]
    table = pd.DataFrame([[s[k] for k in keys] for s in rows.values()], index=list(rows), columns=AUDIT_COLS)
    return table, baseline


FIDELITY_COLS = ["ones/user", "activity KS", "item freq r", "item freq rho", "item TV", "item coverage", "phi PCD",
                 "phi RMSE", "phi corr", "neighbour recall@k"]
FIDELITY_SPLIT_SEED = 123


def fidelity_audit(binarised, real, baseline=None):
    """Fidelity of every binarised synthetic row set to `real` (TRAIN_PARTIAL_VALID_DATA): user activity, item frequencies, the
    pairwise item correlation (phi) and item-neighbour recall (sdrm_b200.fidelity.FidelityReport.summary), with k = 10 nearest
    items (fewer when there are fewer items).  The baseline line compares two random halves of the real rows, split by a
    private generator so the run's global random state is untouched: it is the metrics' noise floor at that sample size.
    Returns (table, baseline summary)."""
    import pandas as pd

    from sdrm_b200.fidelity import compare
    n_items = real.shape[1]
    k = min(10, n_items - 1) if n_items > 1 else None
    if baseline is None:
        perm = np.random.default_rng(FIDELITY_SPLIT_SEED).permutation(real.shape[0])
        half = real.shape[0] // 2
        baseline = compare(real[np.sort(perm[:half])], real[np.sort(perm[half:])], k=k).summary()
    rows = {}
    for name, (dense, packed) in binarised.items():
        rows[name] = compare(real, packed if packed is not None else dense, k=k).summary()
    rows["real split-half (baseline)"] = baseline
    keys = ["ones_per_user_synth", "activity_ks", "item_freq_pearson", "item_freq_spearman", "item_tv", "item_coverage",
            "phi_pcd", "phi_rmse", "phi_corr", "neighbour_recall_at_k"]
    table = pd.DataFrame([[s[k] for k in keys] for s in rows.values()], index=list(rows), columns=FIDELITY_COLS)
    return table, baseline


def save_synthetic(binarised, out_dir, run):
    """Each binarised row set as DIR/run{run}_{name}.npz: the GPU rows through K10 (PackedMatrix.to_sparse, no dense host copy),
    host rows through csr_matrix.  Draws from no random generator."""
    import os

    import scipy.sparse as sp
    os.makedirs(out_dir, exist_ok=True)
    for name, (dense, packed) in binarised.items():
        mat = packed.to_sparse().to_scipy() if packed is not None else sp.csr_matrix(dense)
        sp.save_npz(os.path.join(out_dir, f"run{run}_{name}.npz"), mat)


def main(argv=None):
    args = build_parser().parse_args(argv)
    import pandas as pd
    import torch
    from torch.utils.data import DataLoader

    from sdrm_b200 import evaluators
    from sdrm_b200.data import SparseDataset, load_data, sparse_batch_collate
    from sdrm_b200.train_SDRM import sample_ddpm, train_SDRM

    if args.seed is not None:
        torch.manual_seed(args.seed)
        np.random.seed(args.seed)

    TRAIN_DATA, TRAIN_PARTIAL_VALID_DATA, VALID_DATA = load_data(dataset_name=args.dataset.lower(), data_dir_path=args.data_dir)
    N_USERS, N_ITEMS = TRAIN_DATA.shape
    SPARSITY = 1 - (TRAIN_DATA.nnz / (N_USERS * N_ITEMS))  # counts explicit stored zeros, like the reference (main.py:123)

    ds = SparseDataset(TRAIN_PARTIAL_VALID_DATA, TRAIN_PARTIAL_VALID_DATA)
    sampler = torch.utils.data.sampler.BatchSampler(
        torch.utils.data.sampler.RandomSampler(ds, generator=torch.Generator(device="cpu")),
        batch_size=args.SDRM_batch_size, drop_last=False)
    dl = DataLoader(ds, batch_size=1, collate_fn=sparse_batch_collate, generator=torch.Generator(device="cpu"),
                    sampler=sampler, shuffle=False)

    if args.binarise == "activity":
        from sdrm_b200.sparsify import row_activity
        activity = row_activity(TRAIN_DATA)   # the N_USERS synthetic rows stand in for TRAIN_DATA's users

        def binarise_run(scores, sparsity):
            return binarise_activity(scores, sparsity, activity)
    else:
        def binarise_run(scores, sparsity):
            return binarise(scores, sparsity)

    model = args.model.lower()
    results = {c: [] for c in COLS}
    audit_baseline = None
    fidelity_baseline = None
    for run_n in range(args.runs):
        start_time = time.time()
        print(10 * "#", "Starting run", run_n + 1, 10 * "#")
        SDRM, VAE = train_SDRM(
            dl=dl, N_ITEMS=N_ITEMS, VAE_LATENT=args.MLP_latent_neurons, VAE_HIDDEN=args.VAE_hidden_layer_neurons,
            VAE_LR=args.VAE_lr, VAE_BATCH_SIZE=args.VAE_batch_size, DIFF_LATENT=args.MLP_latent_neurons,
            DIFF_TRAINING_EPOCHS=args.SDRM_epochs, DIFF_LR=args.SDRM_lr, N_HIDDEN_MLP_LAYERS=args.MLP_hidden_layers,
            TIMESTEPS=args.SDRM_timesteps, noise_divider=args.SDRM_noise_variance_diminisher, VAE_DIR_PATH="./temp_vae",
            TRAIN_PARTIAL_VALID_DATA=TRAIN_PARTIAL_VALID_DATA, VALID_DATA=VALID_DATA,
            OPTIMIZATION_OBJECTIVE="Recall@10", verbose=True)
        if args.save_generator:
            import os

            from sdrm_b200.synthesize import save_generator
            os.makedirs(args.save_generator, exist_ok=True)
            save_generator(os.path.join(args.save_generator, f"run{run_n + 1}_generator.pt"), SDRM, VAE,
                           noise_divider=args.SDRM_noise_variance_diminisher, sparsity=SPARSITY)

        print("Sampling Multi-resolution Data")
        M_SDRM = sample_ddpm(N_USERS, SDRM, VAE, args.MLP_latent_neurons, args.SDRM_noise_variance_diminisher,
                             timesteps="random", n_timesteps=args.SDRM_timesteps, verbose=True,
                             sampling_steps=args.SDRM_sampling_steps, eta=args.SDRM_eta)
        print("Sampling Full-resolution Data")
        F_SDRM = sample_ddpm(N_USERS, SDRM, VAE, args.MLP_latent_neurons, args.SDRM_noise_variance_diminisher,
                             n_timesteps=args.SDRM_timesteps, verbose=True,
                             sampling_steps=args.SDRM_sampling_steps, eta=args.SDRM_eta)
        binarised = {
            "M-SDRM": binarise_run(M_SDRM, SPARSITY),
            "F-SDRM": binarise_run(F_SDRM, SPARSITY),
            "MultiVAE++": binarise_run(VAE.sample(N_USERS), SPARSITY),
        }
        synth = {name: pd.DataFrame(dense) for name, (dense, _) in binarised.items()}
        if args.save_synthetic:
            save_synthetic({c: binarised[c] for c in COLS}, args.save_synthetic, run_n + 1)
        if args.privacy_audit:
            audit, audit_baseline = privacy_audit({c: binarised[c] for c in COLS}, TRAIN_PARTIAL_VALID_DATA, audit_baseline)
            print(f"\nPrivacy audit (run {run_n + 1}): distance to the closest training row\n{audit.round(4).to_markdown()}")
        if args.fidelity_audit:
            fid, fidelity_baseline = fidelity_audit({c: binarised[c] for c in COLS}, TRAIN_PARTIAL_VALID_DATA, fidelity_baseline)
            print(f"\nFidelity audit (run {run_n + 1}): synthetic rows against the training rows\n{fid.round(4).to_markdown()}")
        for name, frame in synth.items():
            if model == "svd" and args.svd_on_gpu:
                dense, packed = binarised[name]
                rec, ndcg = evaluators.compute_mf_results_gpu(TRAIN_DATA, VALID_DATA, packed if packed is not None else dense,
                                                              only_synthetic=args.augment_training_data)
            elif model == "svd":
                # NOTE: the flag is passed as only_synthetic=, exactly like the reference (main.py:189-194)
                rec, ndcg = evaluators.compute_mf_results(TRAIN_DATA, VALID_DATA, synthetic_data=frame, nnmf=False,
                                                          only_synthetic=args.augment_training_data)
            elif model == "mlp":
                rows = frame.to_numpy()
                if args.augment_training_data:
                    rows = np.concatenate([TRAIN_PARTIAL_VALID_DATA.toarray(), rows], axis=0)
                rec, ndcg = evaluators.compute_mlp_results(rows, VALID_DATA)
            elif model == "neumf":
                raise RuntimeError("the NeuMF evaluator glue (main.py:216-348 of the reference) is a consumer outside the "
                                   "B200 hot path; run the reference's main.py with `from sdrm_b200.train_SDRM import "
                                   "train_SDRM, sample_ddpm` instead")
            else:
                raise RuntimeError(f"{model} not a valid model. Please selection from SVD, MLP, or NeuMF")
            results[name].append(np.concatenate([rec, ndcg]).reshape(-1, 1))
        print("Run", run_n + 1, "took", round(time.time() - start_time, 2), "seconds")

    def table(fn):
        return pd.DataFrame(np.concatenate([fn(results[c], axis=0) for c in COLS], axis=1), index=ROWS, columns=COLS).round(4)

    print("\nMean\n", table(np.nanmean).to_markdown(), sep="")
    print("\nMax\n", table(np.nanmax).to_markdown(), sep="")
    print("\nStandard Deviation\n", table(np.nanstd).to_markdown(), sep="")
    return {c: np.concatenate(results[c], axis=1) for c in COLS}


if __name__ == "__main__":
    main()
