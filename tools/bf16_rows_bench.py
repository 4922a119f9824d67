"""fp32 vs bfloat16 synthetic rows on one GPU, for the BASELINE configurations: one JSON line per configuration.

For each configuration the two output dtypes alternate in the same process:
  * device ms of one sample_ddpm (CUDA events; best and median of --reps),
  * end-to-end users/s of sample_ddpm_host (rows delivered in pinned host memory; host clock around the synchronised call),
  * ms of K4 equal_sparsity_device on the sampled matrix, at the configuration's sparsity,
  * logits bytes written per user by the sampler and read per user by K4 (computed from the shapes),
  * the effect of rounding on the binarisation: ones of the bfloat16 bits vs the fp32 bits of the same seed (ties at the
    threshold add ones) and the Jaccard index of the two bit matrices.
The card name and power limit are read in the same run.

  python tools/bf16_rows_bench.py [--configs cfg1,cfg2,...] [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# Equal-sparsity targets: 1 - density of the training matrix for MovieLens-100k (cfg 1) and -1M (cfg 2), 0.99 elsewhere (as
# bench.py's K4 leg)
SPARSITY = {"cfg1": 0.937, "cfg2": 0.955, "cfg3": 0.99, "cfg4": 0.99, "cfg5": 0.99}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:   # (the numbers still stand; the card line says why it is missing)
        return f"nvidia-smi failed: {e}"


def popcount(words):
    x = words.to(torch.int64) & 0xFFFFFFFF
    x = x - ((x >> 1) & 0x55555555)
    x = (x & 0x33333333) + ((x >> 2) & 0x33333333)
    x = (x + (x >> 4)) & 0x0F0F0F0F
    return int((((x * 0x01010101) & 0xFFFFFFFF) >> 24).sum().item())


def timed_ms(fn, reps):
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[0], ts[len(ts) // 2]


def run_config(name, reps):
    from bench import WORKLOADS, build_models
    from sdrm_b200.sparsify import equal_sparsity_device
    from sdrm_b200.train_SDRM import sample_ddpm, sample_ddpm_host
    w = WORKLOADS[name]
    dev = torch.device("cuda", 0)
    diff, vae = build_models(w, dev, seed=0)
    n, I, L, T, nd = w["n"], w["I"], w["L"], w["T"], w["nd"]
    dtypes = {"fp32": torch.float32, "bf16": torch.bfloat16}
    outs = {k: torch.empty((n, I), dtype=dt, device=dev) for k, dt in dtypes.items()}
    hosts = {k: torch.empty((n, I), dtype=dt, pin_memory=True) for k, dt in dtypes.items()}
    seed = 1234
    res = {k: {"sample_ms": [], "host_users_per_s": [], "k4_ms": []} for k in dtypes}
    for k in dtypes:   # warm-up of every shape the timed window uses
        sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, out=outs[k], out_dtype=dtypes[k])
        sample_ddpm_host(n, diff, vae, L, nd, n_timesteps=T, seed=seed, host_out=hosts[k])
        equal_sparsity_device(outs[k], SPARSITY[name])
    torch.cuda.synchronize()
    for _ in range(reps):
        for k in dtypes:   # alternate the two dtypes
            res[k]["sample_ms"].append(timed_ms(lambda: sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, out=outs[k],
                                                                    out_dtype=dtypes[k], reuse_packed=True), 1)[0])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            sample_ddpm_host(n, diff, vae, L, nd, n_timesteps=T, seed=seed, host_out=hosts[k])
            torch.cuda.synchronize()
            res[k]["host_users_per_s"].append(n / (time.perf_counter() - t0))
            res[k]["k4_ms"].append(timed_ms(lambda: equal_sparsity_device(outs[k], SPARSITY[name]), 1)[0])
    sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, out=outs["fp32"])
    sample_ddpm(n, diff, vae, L, nd, n_timesteps=T, seed=seed, out=outs["bf16"], out_dtype=torch.bfloat16)
    same = bool(torch.equal(outs["bf16"].view(torch.int16), outs["fp32"].to(torch.bfloat16).view(torch.int16)))
    pm32 = equal_sparsity_device(outs["fp32"], SPARSITY[name])
    pm16 = equal_sparsity_device(outs["bf16"], SPARSITY[name])
    ones32, ones16 = int(pm32.ones.item()), int(pm16.ones.item())
    inter, union = popcount(pm32.bits & pm16.bits), popcount(pm32.bits | pm16.bits)
    summary = {}
    for k in dtypes:
        r = res[k]
        s = sorted(r["sample_ms"]); h = sorted(r["host_users_per_s"]); q = sorted(r["k4_ms"])
        summary[k] = {"sample_ms_best": round(s[0], 3), "sample_ms_median": round(s[len(s) // 2], 3),
                      "host_users_per_s_best": round(h[-1]), "host_users_per_s_median": round(h[len(h) // 2]),
                      "k4_ms_best": round(q[0], 3), "k4_ms_median": round(q[len(q) // 2], 3)}
    esize = {"fp32": 4, "bf16": 2}
    passes = {"fp32": 4, "bf16": 3}   # K4: histogram passes + the pack pass, each reading the matrix once
    for k in dtypes:
        summary[k]["logits_bytes_written_per_user"] = esize[k] * I
        summary[k]["k4_bytes_read_per_user"] = passes[k] * esize[k] * I
        summary[k]["d2h_bytes_per_user"] = esize[k] * I
    return {"config": name, "n": n, "items": I, "sparsity": SPARSITY[name], "reps": reps, "card": CARD,
            "bf16_equals_rounded_fp32": same, **summary,
            "binarisation": {"ones_fp32": ones32, "ones_bf16": ones16, "extra_ones_bf16": ones16 - ones32,
                             "extra_ones_fraction": round((ones16 - ones32) / max(ones32, 1), 6),
                             "jaccard": round(inter / max(union, 1), 6),
                             "threshold_fp32": float(pm32.threshold), "threshold_bf16": float(pm16.threshold)}}


if __name__ == "__main__":
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="cfg1,cfg2,cfg3,cfg4,cfg5")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bf16_rows_bench: needs a CUDA device; nothing is measured without one")
    CARD = card()
    fh = open(args.out, "w") if args.out else None
    for name in args.configs.split(","):
        line = json.dumps(run_config(name, args.reps))
        print(line, flush=True)
        if fh:
            fh.write(line + "\n")
            fh.flush()
    if torch.cuda.device_count() < 2:
        print(json.dumps({"multi_gpu_host_leg": "not measured: one GPU in this run", "card": CARD}), flush=True)
