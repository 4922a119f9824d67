"""Activity-matched binarisation on the device: K12 (sdrm_topk_pack) alone, activity_matched_device end to end, and the
equal-sparsity binarisation (equal_sparsity_device, K4) on the same scores, against a PyTorch reference (a stable descending sort
of every row, in row chunks, then rank < k).

    python tools/bench_topk_pack.py [--shapes 843x1008 ...] [--densities 0.01 0.05] [--dtypes float32 bfloat16] [--reps 10]
                                    [--out profiles/topk_pack_b200.jsonl]

Shapes: the dataset configurations (843 x 1 008, 5 429 x 3 125, 9 558 x 8 582, 1 208 x 729) and a cfg-5 shard (125 000 x 20 000).
The scores are random normal; the real activity is a seeded heavy-tailed (log-normal) draw of as many users as rows, scaled to
the mean density and clipped to [0, items], and the equal-sparsity step uses sparsity = 1 - density.  Per configuration: the
K12 bits are first checked against the reference's bits, then the three device paths are timed alternately (CUDA events around
each call, median of --reps after 2 warm-up calls each), the reference over fewer calls.  K12 alone is the kernel launch
without the status read-back; its `hbm_fraction` is the score bytes read once over its time, as a share of 7.7 TB/s.  Shapes
whose scores fit the 126 MB L2 are marked: after the first call they are read from L2.  The GPU's name and power limit head
the output.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from sdrm_b200 import _lib
from sdrm_b200.sparsify import activity_matched_device, activity_targets, equal_sparsity_device, topk_pack

HBM_BYTES_PER_S = 7.7e12
L2_BYTES = 126e6
SHAPES = ["843x1008", "5429x3125", "9558x8582", "1208x729", "125000x20000"]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # (the query is informative only)
        q = f"nvidia-smi unavailable: {e}"
    return {"gpu": torch.cuda.get_device_name(), "nvidia_smi": q}


def activity(rows, n_cols, density, seed):
    x = np.random.default_rng(seed).lognormal(0.0, 1.0, size=rows)
    return np.clip(np.round(x / x.mean() * density * n_cols), 0, n_cols).astype(np.int64)


def reference_bits(S, k, chunk_elems=1 << 28):
    """bool [rows, items] on the device: each row's k highest scores in K7's order (NaN as -inf, -0.0 as +0.0), ties to the
    lower index, by a stable descending sort per row chunk."""
    rows, n_cols = S.shape
    out = torch.empty((rows, n_cols), dtype=torch.bool, device=S.device)
    step = max(1, chunk_elems // n_cols)
    pos = torch.arange(n_cols, device=S.device)
    for r0 in range(0, rows, step):
        x = S[r0:r0 + step].float()
        x = torch.where(torch.isnan(x), torch.full_like(x, float("-inf")), x) + 0.0
        order = torch.sort(x, dim=1, descending=True, stable=True).indices
        keep = pos[None, :] < k[r0:r0 + step, None]
        out[r0:r0 + step] = torch.zeros_like(keep).scatter_(1, order, keep)
    return out


def unpack(bits, n_cols):
    shifts = torch.arange(32, device=bits.device, dtype=torch.int32)
    return ((bits.unsqueeze(-1) >> shifts) & 1).reshape(bits.shape[0], -1)[:, :n_cols].bool()


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def alternate(fns, reps):
    """{name: (median, min, max) ms}, the functions timed in turn within every repetition."""
    for fn in fns.values():
        fn()
        fn()
    torch.cuda.synchronize()
    ts = {name: [] for name in fns}
    for _ in range(reps):
        for name, fn in fns.items():
            ts[name].append(event_ms(fn))
    return {name: (float(np.median(v)), min(v), max(v)) for name, v in ts.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", nargs="+", default=SHAPES)
    ap.add_argument("--densities", type=float, nargs="+", default=[0.01, 0.05])
    ap.add_argument("--dtypes", nargs="+", default=["float32", "bfloat16"])
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--ref-reps", type=int, default=3)
    ap.add_argument("--out", default="profiles/topk_pack_b200.jsonl")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_topk_pack: no CUDA device; the timings need a B200")
    lib = _lib.load()
    lines = [json.dumps(gpu_info())]
    print(lines[0], flush=True)
    for shape in a.shapes:
        rows, n_cols = (int(v) for v in shape.split("x"))
        S32 = torch.randn((rows, n_cols), device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
        for dname in a.dtypes:
            S = S32 if dname == "float32" else S32.to(getattr(torch, dname))
            for density in a.densities:
                act = activity(rows, n_cols, density, seed=int(density * 1e4) + rows)
                sparsity = 1.0 - density
                pm = activity_matched_device(S, sparsity, act)
                k = activity_targets(equal_sparsity_device(S, sparsity).to_sparse().indptr.diff(), act, n_cols)
                ref = reference_bits(S, k)
                same = True
                step = max(1, (1 << 28) // n_cols)
                for r0 in range(0, rows, step):
                    same &= bool(torch.equal(unpack(pm.bits[r0:r0 + step], n_cols), ref[r0:r0 + step]))
                assert same, f"K12 bits differ from the sorted reference at {shape} {dname} {density}"
                del ref
                k32 = k.to(torch.int32).contiguous()
                bits = torch.empty_like(pm.bits)
                count = torch.zeros(1, dtype=torch.int64, device="cuda")
                status = torch.zeros(1, dtype=torch.int32, device="cuda")
                entry = lib.sdrm_topk_pack_bf16 if S.dtype == torch.bfloat16 else lib.sdrm_topk_pack

                def k12():
                    _lib.check(entry(_lib.ptr(S), rows, n_cols, n_cols, _lib.ptr(k32), _lib.ptr(bits), bits.shape[1],
                                     _lib.ptr(count), _lib.ptr(status), _lib.stream_ptr()), "sdrm_topk_pack")
                t = alternate({"k12": k12,
                               "activity_matched": lambda: activity_matched_device(S, sparsity, act),
                               "equal_sparsity": lambda: equal_sparsity_device(S, sparsity)}, a.reps)
                assert torch.equal(bits, pm.bits) and int(status.item()) == 0
                t_ref = alternate({"reference": lambda: reference_bits(S, k)}, a.ref_reps)["reference"]
                score_bytes = rows * n_cols * S.element_size()
                rec = {"dtype": dname, "rows": rows, "items": n_cols, "density": density, "ones": int(pm.ones.item()),
                       "score_bytes": score_bytes, "fits_l2": score_bytes <= L2_BYTES, "bits_equal_reference": same,
                       "k12_ms": round(t["k12"][0], 4), "k12_ms_min_max": [round(t["k12"][1], 4), round(t["k12"][2], 4)],
                       "k12_hbm_fraction": round(score_bytes / (t["k12"][0] * 1e-3) / HBM_BYTES_PER_S, 3),
                       "activity_matched_ms": round(t["activity_matched"][0], 4),
                       "equal_sparsity_ms": round(t["equal_sparsity"][0], 4),
                       "reference_ms": round(t_ref[0], 3),
                       "k12_vs_equal_sparsity": round(t["k12"][0] / t["equal_sparsity"][0], 3)}
                lines.append(json.dumps(rec))
                print(lines[-1], flush=True)
                del pm, bits
            del S
            torch.cuda.empty_cache()
        del S32
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
