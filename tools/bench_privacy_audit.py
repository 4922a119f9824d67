"""Nearest-rows search (privacy.nearest_rows, K8) against the same search in PyTorch on the same GPU.

    python tools/bench_privacy_audit.py [--shapes ml-100k ml-1m adm scale-up] [--k 1 8] [--reps 5] [--out results.jsonl]

One JSON line per (shape, k), each carrying the GPU's name, power limit and maximum SM clock read in the same run:
  - k8_ms: median of --reps timed calls of the K8 search on prepared operand images (CUDA events around each call, after 2
    warm-up calls); the image preparation is timed separately (prep_ms, both sides, once per row set in an audit).
  - torch_ms: the comparator, in chunks of query rows so the count matrix fits: an fp32 matmul of the 0/1 matrices with fp32
    output (TF32 allowed, still exact: 0/1 inputs and sums below 2^24), u = a + b - c, J in float64 (exact order, see
    tests/privacy_oracle.py), torch.topk, then the entries tied with the k-th J re-picked by lowest index (the tie rule).
    Its indices must equal K8's, and its counts too, or the script stops: the comparison is checked, not just timed.
  - int_ops_per_s: 2 n m n_items / k8 time, the algorithmic integer operations per second; datasheet_share: that over 4.5 POPS,
    the dense INT8 rate of one B200 on NVIDIA's HGX B200 data sheet (72 POPS for 8 GPUs with 2:4 sparsity, a sixteenth of that)
    -- a data-sheet figure, not a reached one.  tensor_floor_ms: the padded product at that rate.
  - epilogue_floor_ms: K8 at the same n, m, k and density but 128 items (one k-block, so almost no tensor work and the same
    number of pairs through the top-k epilogue).  bound: "epilogue" when k8_ms is within 25 % of that floor, else "product" (tensor pipe or operand loads).
Rows are uniform random at the shape's density.  The small shapes' operand images fit the 126 MB L2 and are re-read from there.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from sdrm_b200 import privacy

SHAPES = {   # queries, references, items, density
    "ml-100k": (843, 938, 1008, 0.0575),
    "ml-1m": (5429, 6034, 3125, 0.0447),
    "adm": (9558, 10621, 8582, 0.00115),
    "scale-up": (131072, 131072, 20000, 0.01),
}
INT8_DENSE_OPS = 4.5e15


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # (the query is informative only)
        q = f"nvidia-smi unavailable: {e}"
    return q


def timed(fn, reps, warm=2):
    for _ in range(warm):
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
    return ts[len(ts) // 2]


def rows(n, items, density, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    out = torch.empty((n, items), dtype=torch.bool, device="cuda")
    for s in range(0, n, 8192):   # (chunks keep the fp32 uniforms small at the scale-up shape)
        e = min(n, s + 8192)
        out[s:e] = torch.rand((e - s, items), generator=g, device="cuda") < density
    return out


def images(D):
    n, items = D.shape
    return privacy._image(D, "dense", n, items, D.device)


def torch_search(Q, R, k, chunk):
    """The comparator: the exact answer (J desc, index asc) from an fp32 product and torch.topk."""
    Rf = R.float()
    a, b = Q.sum(1, dtype=torch.int64), R.sum(1, dtype=torch.int64)
    out_i, out_c, out_u = [], [], []
    for s in range(0, Q.shape[0], chunk):
        c = Q[s:s + chunk].float() @ Rf.T
        u = a[s:s + chunk, None].double() + b[None, :].double() - c.double()
        j = torch.where(u == 0, torch.ones_like(u), c.double() / u.clamp_min(1))
        vals, top = torch.topk(j, k, dim=1)
        kth = vals[:, -1:]
        n_gt = (vals > kth).sum(1, keepdim=True)
        # the entries above the k-th J (all among topk's) in (J desc, index asc) order: sort by index, then stably by J
        top = torch.sort(top, dim=1).values
        tv = torch.gather(j, 1, top)
        idx_gt = torch.gather(top, 1, torch.sort(torch.where(tv > kth, tv, -1.0), dim=1, descending=True, stable=True).indices)
        # then the lowest-index columns tied with the k-th J
        eq = j == kth
        rank = torch.cumsum(eq.to(torch.int32), 1) - 1
        want = eq & (rank < (k - n_gt))
        r_i, c_i = torch.nonzero(want, as_tuple=True)
        idx_eq = torch.zeros_like(top)
        idx_eq[r_i, rank[r_i, c_i].long()] = c_i
        pos = torch.arange(k, device=j.device)[None, :]
        idx = torch.where(pos < n_gt, idx_gt, torch.gather(idx_eq, 1, (pos - n_gt).clamp_min(0)))
        out_i.append(idx)
        out_c.append(torch.gather(c, 1, idx).to(torch.int32))
        out_u.append(torch.gather(u, 1, idx).to(torch.int32))
    return torch.cat(out_i), torch.cat(out_c), torch.cat(out_u)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", nargs="+", default=list(SHAPES))
    ap.add_argument("--k", nargs="+", type=int, default=[1, 8])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = True   # the comparator's fastest exact fp32 product
    gpu = gpu_info()
    lines = []
    for name in args.shapes:
        n, m, items, density = SHAPES[name]
        Q, R = rows(n, items, density, 1), rows(m, items, density, 2)
        prep_ms = timed(lambda: (images(Q), images(R)), 1, warm=1)
        (qi, qo), (ri, ro) = images(Q), images(R)
        Qs, Rs = rows(n, 128, density, 3), rows(m, 128, density, 4)
        (qs, qso), (rs, rso) = images(Qs), images(Rs)
        chunk = max(1, min(n, (1 << 31) // (8 * m)))   # ~2 GB of float64 J per chunk
        for k in args.k:
            ours = privacy._search(qi, qo, ri, ro, items, k)
            ref = torch_search(Q, R, k, chunk)
            same = all(torch.equal(x, y) for x, y in zip(ours, ref))
            if not same:
                raise SystemExit(f"{name} k={k}: K8 and the torch comparator disagree")
            k8_ms = timed(lambda: privacy._search(qi, qo, ri, ro, items, k), args.reps)
            torch_ms = timed(lambda: torch_search(Q, R, k, chunk), max(1, args.reps // 2), warm=0)   # (warmed by the check)
            floor_ms = timed(lambda: privacy._search(qs, qso, rs, rso, 128, k), args.reps)
            ops = 2.0 * n * m * items
            pitch = ri.shape[1]
            rec = dict(gpu=gpu, shape=name, n=n, m=m, items=items, density=density, k=k, k8_ms=round(k8_ms, 4),
                       torch_ms=round(torch_ms, 4), speedup=round(torch_ms / k8_ms, 2), prep_ms=round(prep_ms, 4),
                       int_ops_per_s=ops / (k8_ms * 1e-3), datasheet_share=round(ops / (k8_ms * 1e-3) / INT8_DENSE_OPS, 4),
                       tensor_floor_ms=round(2.0 * n * m * pitch / INT8_DENSE_OPS * 1e3, 4),
                       epilogue_floor_ms=round(floor_ms, 4), bound="epilogue" if k8_ms <= 1.25 * floor_ms else "product",
                       equal_to_torch=same)
            print(json.dumps(rec), flush=True)
            lines.append(rec)
        del Q, R, qi, ri
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for rec in lines:
                fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
