"""Time of one sample_ddpm call against the number of reverse steps (sampling_steps S), for the BASELINE configurations on one GPU:
one JSON line per (configuration, S, sampler).

For each configuration (cfg 1-4: the dataset-sized call of n users; cfg 5: one GPU's shard of 125 000 users) the settings
S in {T, T/2, T/4, 25, 10} (those <= T, duplicates dropped) run as strided DDPM (eta=None) and as DDIM with eta = 0, alternating in
one process; each line carries the median (and all) of --reps device times (CUDA events around the call, the step grid already
set on the handle, the weights packed once), users/s, the time relative to the full chain (S = T, DDPM) and the same ratio
predicted from the algorithmic FLOPs (S * 2 L^2 (2 + nh) for the chain + 2 (L H + H I) for the decode).  The card name and power
limit are read in the same run.

  python tools/step_grid_bench.py [--configs cfg1,...,cfg5] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:   # (the numbers still stand; the card line says why it is missing)
        return f"nvidia-smi failed: {e}"


def settings(T):
    steps = []
    for S in (T, T // 2, T // 4, 25, 10):
        if 1 <= S <= T and S not in steps:
            steps.append(S)
    return [(S, eta) for S in steps for eta in (None, 0.0)]


def flop_ratio(w, S):
    chain = 2 * w["L"] ** 2 * (2 + w["nh"])
    decode = 2 * (w["L"] * w["H"] + w["H"] * w["I"])
    return (S * chain + decode) / (w["T"] * chain + decode)


def run_config(name, reps, card_line):
    import torch
    from bench import WORKLOADS, build_models
    from sdrm_b200.train_SDRM import engine_for, resolve_step_grid, sample_ddpm
    w = WORKLOADS[name]
    dev = torch.device("cuda", 0)
    diff, vae = build_models(w, dev, seed=0)
    n, I, L, T, nd = w["n"], w["I"], w["L"], w["T"], w["nd"]
    out = torch.empty((n, I), dtype=torch.float32, device=dev)
    seed = 1234
    todo = settings(T)
    eng = None

    def call(S, eta, reuse=True):
        return sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, out=out, reuse_packed=reuse, sampling_steps=S, eta=eta)

    call(T, None, reuse=False)                 # packs the weights once
    eng = engine_for(diff)
    for S, eta in todo:                        # warm-up of every setting
        call(S, eta)
    torch.cuda.synchronize()
    times = {k: [] for k in todo}
    for _ in range(reps):
        for S, eta in todo:                    # alternate the settings
            eng.set_step_grid(*resolve_step_grid(T, S, eta))   # (sample_ddpm then finds the grid set: nothing to launch)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            call(S, eta)
            b.record()
            b.synchronize()
            times[(S, eta)].append(a.elapsed_time(b))
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    lines = []
    for (S, eta), ms in med.items():
        lines.append({"config": name, "n": n, "T": T, "S": S, "sampler": "ddpm" if eta is None else "ddim", "eta": eta,
                      "ms_median": round(ms, 3), "ms_all": [round(t, 3) for t in times[(S, eta)]],
                      "users_per_s": round(n / (ms / 1e3)), "time_vs_full": round(ms / med[(T, None)], 4),
                      "flop_model_vs_full": round(flop_ratio(w, S), 4), "reps": reps, "card": card_line})
    return lines


if __name__ == "__main__":
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="cfg1,cfg2,cfg3,cfg4,cfg5")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("step_grid_bench: needs a CUDA device; nothing is measured without one")
    card_line = card()
    fh = open(args.out, "w") if args.out else None
    for name in args.configs.split(","):
        for rec in run_config(name, args.reps, card_line):
            line = json.dumps(rec)
            print(line, flush=True)
            if fh:
                fh.write(line + "\n")
                fh.flush()
