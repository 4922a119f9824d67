"""Top-K recommendation with seen-item exclusion: the CUDA path (recommend.recommend_topk, K7) against the PyTorch path a caller
would otherwise write (scatter -inf into the history positions of the logits in place, then torch.topk).

    python tools/bench_recommend_topk.py [--users 4096 16384 32768] [--items 20000 50000] [--k 10 50 100] [--density 0.01]
                                         [--reps 20] [--out results.jsonl]

One JSON line per (dtype, users, items, k): median milliseconds per call of each path over --reps timed calls (CUDA events around
each call, after 3 warm-up calls), the speedup, and the logit bytes one pass reads over the CUDA path's time.  The logits are
random normal, larger than the 126 MB L2 at every default shape, and the history has `density` of the items per user, drawn
uniformly.  The reference path's (row, item) coordinates are built once outside the timed region, so it is timed at its cheapest.
Every configuration is checked first: the CUDA values equal torch.topk's values on the masked logits (its tie order may differ),
the indices point at those values, and no index is in the user's history.  The GPU's name and power limit head the output.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from sdrm_b200.recommend import recommend_topk


def history(users, n_items, density, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    g_cpu = torch.Generator().manual_seed(seed)   # (torch.binomial runs on the CPU: seeded too, so every dtype sees one history)
    counts = torch.binomial(torch.full((users,), float(n_items)), torch.full((users,), float(density)), generator=g_cpu).long().cuda()
    indptr = torch.zeros(users + 1, dtype=torch.int64, device="cuda")
    indptr[1:] = torch.cumsum(counts, 0)
    nnz = int(indptr[-1])
    # uniform draws with replacement: a row may list an item twice, which the API allows (at 1 % the distinct share stays ~99.5 %)
    indices = torch.randint(0, n_items, (nnz,), generator=g, device="cuda", dtype=torch.int32)
    rows = torch.repeat_interleave(torch.arange(users, device="cuda"), counts)
    return indptr, indices, rows


def timed(fn, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2], ts[0], ts[-1]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # (the query is informative only)
        q = f"nvidia-smi unavailable: {e}"
    return {"gpu": torch.cuda.get_device_name(), "nvidia_smi": q}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, nargs="+", default=[4096, 16384, 32768])
    ap.add_argument("--items", type=int, nargs="+", default=[20000, 50000])
    ap.add_argument("--k", type=int, nargs="+", default=[10, 50, 100])
    ap.add_argument("--dtypes", nargs="+", default=["float32", "bfloat16"])
    ap.add_argument("--density", type=float, default=0.01)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_recommend_topk: no CUDA device; the timings need a B200")
    lines = [json.dumps(gpu_info())]
    print(lines[0], flush=True)
    for dname in a.dtypes:
        dtype = getattr(torch, dname)
        for users in a.users:
            for n_items in a.items:
                logits = torch.randn(users, n_items, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1)).to(dtype)
                indptr, indices, rows = history(users, n_items, a.density, seed=2)
                cols = indices.long()
                work = logits.clone()
                neg_inf = torch.tensor(float("-inf"), dtype=dtype, device="cuda")

                def reference(k):
                    work.index_put_((rows, cols), neg_inf)   # in place: the same work on every call
                    return torch.topk(work, k, dim=1)

                for k in a.k:
                    vals, idx = recommend_topk(logits, indptr, indices, k)
                    rv, _ = reference(k)
                    assert torch.equal(vals, rv), "CUDA top-K values differ from torch.topk on the masked logits"
                    assert torch.equal(logits.gather(1, idx), vals)
                    assert not (work.gather(1, idx) == float("-inf")).logical_and(vals != float("-inf")).any(), "history item returned"
                    ms_cuda = timed(lambda: recommend_topk(logits, indptr, indices, k), a.reps)
                    ms_ref = timed(lambda: reference(k), a.reps)
                    rec = {"dtype": dname, "users": users, "items": n_items, "k": k, "density": a.density,
                           "history_nnz": int(indices.numel()), "cuda_ms": round(ms_cuda[0], 4),
                           "cuda_ms_min_max": [round(ms_cuda[1], 4), round(ms_cuda[2], 4)],
                           "reference_ms": round(ms_ref[0], 4), "reference_ms_min_max": [round(ms_ref[1], 4), round(ms_ref[2], 4)],
                           "speedup": round(ms_ref[0] / ms_cuda[0], 2),
                           "cuda_logit_read_GBps": round(logits.numel() * logits.element_size() / ms_cuda[0] / 1e6, 1)}
                    lines.append(json.dumps(rec))
                    print(lines[-1], flush=True)
                del logits, work, indptr, indices, rows, cols
                torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
