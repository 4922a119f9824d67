"""Pairwise item-correlation sums (fidelity.compare, K9) against the same sums in PyTorch on the same GPU.

    python tools/bench_fidelity_audit.py [--shapes ml-100k ml-1m adm scale-up] [--reps 5] [--out results.jsonl]

One JSON line per shape, each carrying the GPU's name, power limit and maximum SM clock read in the same run:
  - k9_ms: median of --reps timed K9 calls (sdrm_fidelity_pair_stats: item statistics, the tile kernel and the slot reduction)
    on prepared item-major images (CUDA events around each call, after 2 warm-up calls).
  - prep_real_ms / prep_synth_ms: the item-major image of each side from bit-packed rows (the PackedMatrix that main.py's
    binarisation leaves on the device), one call each after a warm-up.
  - k8_neighbour_ms: the two K8 item-neighbour searches (k = 10, each item against the items of its own set).
  - torch_ms: the comparator: per chunk of items, an fp32 matmul of the 0/1 item columns (TF32 allowed, still exact: 0/1
    inputs and counts below 2^24), phi and the six sums over i < j in float64.  Its sums must agree with K9's within the test
    tolerance (1e-9 max(1, P) absolute) or the script stops: the comparison is checked, not just timed.
  - int_ops_per_s: 2 (U_real + U_synth) I (I + 1) / 2 over the K9 time, the algorithmic integer operations per second of the
    upper-triangle products; datasheet_share: that over 4.5 POPS, the dense INT8 rate of one B200 on NVIDIA's HGX B200 data
    sheet (72 POPS for 8 GPUs with 2:4 sparsity, a sixteenth of that) -- a data-sheet figure, not a reached one.
  - epilogue_floor_ms: K9 at the same user counts and items but one user per set (one k-block each: nearly no tensor work, every
    pair still through the fp64 epilogue).
Rows are uniform random at the shape's density.  The small shapes' images fit the 126 MB L2 and are re-read from there.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from sdrm_b200 import fidelity, privacy
from sdrm_b200.sparsify import PackedMatrix

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_privacy_audit import INT8_DENSE_OPS, gpu_info, rows, timed  # noqa: E402

SHAPES = {   # real users, synthetic users, items, density
    "ml-100k": (938, 843, 1008, 0.0575),
    "ml-1m": (6034, 5429, 3125, 0.0447),
    "adm": (10621, 9558, 8582, 0.00115),
    "scale-up": (131072, 131072, 20000, 0.01),
}


def pack(X):
    """Bool rows [n, I] as a PackedMatrix (bit j of word w = column 32 w + j)."""
    n, items = X.shape
    wpr = (items + 31) // 32
    bits = torch.empty((n, wpr), dtype=torch.int32, device=X.device)
    shifts = torch.arange(32, device=X.device, dtype=torch.int64)
    for s in range(0, n, 4096):
        e = min(n, s + 4096)
        xp = torch.zeros((e - s, wpr * 32), dtype=torch.int64, device=X.device)
        xp[:, :items] = X[s:e]
        w = (xp.view(e - s, wpr, 32) << shifts).sum(-1)
        bits[s:e] = (w - ((w >> 31) & 1) * (1 << 32)).to(torch.int32)
    return PackedMatrix(bits, items, 0.0, None)


def item_image(pm):
    n, items = pm.shape
    return fidelity._item_image(pm, "bits", n, items, pm.bits.device)


def torch_sums(R, S, chunk):
    """The comparator: phi of both sets from fp32 Gram products, the six sums over i < j in float64."""
    items = R.shape[1]
    stats = []
    for X in (R, S):
        Xf = X.float()
        a = X.sum(0, dtype=torch.int64).double()
        U = float(X.shape[0])
        sq = torch.sqrt(a * (U - a))
        stats.append((Xf, a, U, sq))
    out = torch.zeros(6, dtype=torch.float64, device=R.device)
    cols = torch.arange(items, device=R.device)
    for s in range(0, items, chunk):
        e = min(items, s + chunk)
        phis = []
        for Xf, a, U, sq in stats:
            c = (Xf[:, s:e].T @ Xf).double()
            den = sq[s:e, None] * sq[None, :]
            num = U * c - a[s:e, None] * a[None, :]
            phis.append(torch.where(den > 0, num / torch.where(den > 0, den, torch.ones_like(den)), torch.zeros_like(num)))
        upper = cols[None, :] > torch.arange(s, e, device=R.device)[:, None]
        r, q = phis[0][upper], phis[1][upper]
        d = r - q
        out += torch.stack([(d * d).sum(), r.sum(), q.sum(), (r * r).sum(), (q * q).sum(), (r * q).sum()])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", nargs="+", default=list(SHAPES))
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = True   # the comparator's fastest exact fp32 product
    gpu = gpu_info()
    lines = []
    for name in args.shapes:
        ur, us, items, density = SHAPES[name]
        R, S = rows(ur, items, density, 1), rows(us, items, density, 2)
        pr, ps = pack(R), pack(S)
        prep_r = timed(lambda: item_image(pr), 1, warm=1)
        prep_s = timed(lambda: item_image(ps), 1, warm=1)
        (ri, rio, _), (si, sio, _) = item_image(pr), item_image(ps)
        k9 = lambda: fidelity._pair_stats(ri, rio, ur, si, sio, us, items)   # noqa: E731
        ours = k9().cpu()
        chunk = max(1, min(items, (1 << 28) // items))   # ~2 GB of float64 phi per set and chunk
        ref = torch_sums(R, S, chunk).cpu()
        P = items * (items - 1) / 2
        err = float((ours - ref).abs().max())
        if err > 1e-9 * max(1.0, P):
            raise SystemExit(f"{name}: K9 and the torch comparator disagree by {err} (sums {ours.tolist()} vs {ref.tolist()})")
        k9_ms = timed(k9, args.reps)
        torch_ms = timed(lambda: torch_sums(R, S, chunk), max(1, args.reps // 2), warm=0)   # (warmed by the check)
        k8_ms = timed(lambda: (privacy._search(ri, rio, ri, rio, ur, 10, exclude_same_index=True),
                               privacy._search(si, sio, si, sio, us, 10, exclude_same_index=True)), args.reps, warm=1)
        (r1, r1o, _), (s1, s1o, _) = (item_image(pack(rows(1, items, density, 3))), item_image(pack(rows(1, items, density, 4))))
        floor_ms = timed(lambda: fidelity._pair_stats(r1, r1o, 1, s1, s1o, 1, items), args.reps)
        ops = 2.0 * (ur + us) * items * (items + 1) / 2
        rec = dict(gpu=gpu, shape=name, users_real=ur, users_synth=us, items=items, density=density, k9_ms=round(k9_ms, 4),
                   torch_ms=round(torch_ms, 4), speedup=round(torch_ms / k9_ms, 2), prep_real_ms=round(prep_r, 4),
                   prep_synth_ms=round(prep_s, 4), k8_neighbour_ms=round(k8_ms, 4), int_ops_per_s=ops / (k9_ms * 1e-3),
                   datasheet_share=round(ops / (k9_ms * 1e-3) / INT8_DENSE_OPS, 4), epilogue_floor_ms=round(floor_ms, 4),
                   max_abs_diff=err, sums=ours.tolist())
        print(json.dumps(rec), flush=True)
        lines.append(rec)
        del R, S, pr, ps, ri, si
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for rec in lines:
                fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
