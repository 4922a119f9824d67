"""End-to-end quality run of THIS repo on the GPU: same loop, hyper-parameters and evaluator settings as tools/ref_e2e.py.

  python tools/our_e2e.py [runs] [only_synth] [out] [json overrides] [--sampling-steps S] [--eta X] [--svd-on-gpu]
                         [--binarise {equal-sparsity,activity}]
--sampling-steps / --eta sample F-SDRM and M-SDRM on a fewer-step chain (sample_ddpm's sampling_steps / eta); default: all T steps.
--svd-on-gpu scores with evaluators.compute_mf_results_gpu from the device bits instead of sklearn; each record names the
evaluator that ran ("svd_evaluator").
--binarise activity gives every synthetic row a training user's number of interactions (sparsify.activity_matched_device)
instead of the equal-sparsity threshold; each record names the binarisation ("binarise")."""
import json, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, pandas as pd, torch
from torch.utils.data import DataLoader
from sdrm_b200 import evaluators
from sdrm_b200.data import SparseDataset, load_data, sparse_batch_collate
from sdrm_b200.train_SDRM import sample_ddpm, train_SDRM

GRID = {}
for flag, key, conv in (("--sampling-steps", "sampling_steps", int), ("--eta", "eta", float)):
    if flag in sys.argv:
        i = sys.argv.index(flag)
        GRID[key] = conv(sys.argv[i + 1])
        del sys.argv[i:i + 2]
BINARISE = "equal-sparsity"
if "--binarise" in sys.argv:
    i = sys.argv.index("--binarise")
    BINARISE = sys.argv[i + 1]
    del sys.argv[i:i + 2]
    if BINARISE not in ("equal-sparsity", "activity"):
        sys.exit(f"--binarise must be equal-sparsity or activity, got {BINARISE}")
SVD_ON_GPU = "--svd-on-gpu" in sys.argv
if SVD_ON_GPU:
    sys.argv.remove("--svd-on-gpu")
runs = int(sys.argv[1]) if len(sys.argv) > 1 else 5
only_synth = (sys.argv[2] == "1") if len(sys.argv) > 2 else True
out_path = sys.argv[3] if len(sys.argv) > 3 else "gpurun_out/e2e_ours_ml100k.jsonl"
A = dict(T=83, B=550, H=930, L=830, nh=2, nd=1.0, epochs=265, lr=2.1e-5, vae_bs=780, vae_lr=6e-4)  # README trial 223
if len(sys.argv) > 4:
    A.update(json.loads(sys.argv[4]))
TRAIN, TPV, VALID = load_data("ml-100k", "baseline/_ref/data")
N_USERS, N_ITEMS = TRAIN.shape
SPARSITY = 1 - (TRAIN.nnz / (N_USERS * N_ITEMS))
ds = SparseDataset(TPV, TPV)
sampler = torch.utils.data.sampler.BatchSampler(torch.utils.data.sampler.RandomSampler(ds, generator=torch.Generator(device="cpu")), batch_size=A["B"], drop_last=False)
dl = DataLoader(ds, batch_size=1, collate_fn=sparse_batch_collate, generator=torch.Generator(device="cpu"), sampler=sampler, shuffle=False)
for run in range(runs):
    t0 = time.time()
    DIFF, VAE = train_SDRM(dl=dl, N_ITEMS=N_ITEMS, VAE_LATENT=A["L"], VAE_HIDDEN=A["H"], VAE_LR=A["vae_lr"], VAE_BATCH_SIZE=A["vae_bs"],
                           DIFF_LATENT=A["L"], DIFF_TRAINING_EPOCHS=A["epochs"], DIFF_LR=A["lr"], N_HIDDEN_MLP_LAYERS=A["nh"], TIMESTEPS=A["T"],
                           noise_divider=A["nd"], VAE_DIR_PATH="/tmp/our_temp_vae", TRAIN_PARTIAL_VALID_DATA=TPV, VALID_DATA=VALID,
                           OPTIMIZATION_OBJECTIVE="Recall@10", verbose=False)
    torch.cuda.synchronize()
    res = {"impl": "sdrm_b200", "run": run, "train_s": round(time.time() - t0, 1), "only_synthetic": only_synth, **GRID,
           "svd_evaluator": "compute_mf_results_gpu" if SVD_ON_GPU else "compute_mf_results", "binarise": BINARISE}
    t1 = time.time()
    from sdrm_b200.sparsify import equal_sparsity_device
    M = sample_ddpm(N_USERS, DIFF, VAE, A["L"], A["nd"], timesteps="random", n_timesteps=A["T"], **GRID)
    torch.cuda.synchronize(); res["sample_random_s"] = round(time.time() - t1, 4); t1 = time.time()
    F = sample_ddpm(N_USERS, DIFF, VAE, A["L"], A["nd"], n_timesteps=A["T"], **GRID)
    torch.cuda.synchronize(); res["sample_full_s"] = round(time.time() - t1, 4)
    V = VAE.sample(N_USERS)
    for name, S in (("F-SDRM", F), ("M-SDRM", M), ("MultiVAE++", V)):
        if BINARISE == "activity":
            from sdrm_b200.sparsify import activity_matched_device, row_activity
            S = S if isinstance(S, torch.Tensor) else torch.as_tensor(np.asarray(S, dtype=np.float32), device="cuda")
            pm = activity_matched_device(S, SPARSITY, row_activity(TRAIN))
            syn = pd.DataFrame(pm.numpy(int))
        elif isinstance(S, torch.Tensor):   # K4: threshold identical to np.quantile, 1 bit per entry to the host
            pm = equal_sparsity_device(S, SPARSITY)
            dense = pm.numpy(int)
            host = S.cpu().numpy()
            assert pm.threshold == np.quantile(host.flatten(), SPARSITY) and (dense == (host >= pm.threshold)).all()
            syn = pd.DataFrame(dense)
        else:
            pm = None
            syn = pd.DataFrame((S >= np.quantile(S.flatten(), SPARSITY)).astype(int))
        t1 = time.time()
        if SVD_ON_GPU:
            rec, ndcg = evaluators.compute_mf_results_gpu(TRAIN, VALID, pm if pm is not None else syn, only_synthetic=only_synth)
        else:
            rec, ndcg = evaluators.compute_mf_results(TRAIN, VALID, synthetic_data=syn, nnmf=False, only_synthetic=only_synth)
        res[f"{name}_svd_s"] = round(time.time() - t1, 3)
        res[name] = {"recall@10": float(rec[3]), "ndcg@10": float(ndcg[3])}
    print(json.dumps(res), flush=True)
    with open(out_path, "a") as fh:
        fh.write(json.dumps(res) + "\n")
