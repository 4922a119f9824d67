"""Bits -> CSR (K10, sparsify.packed_to_csr) against the same conversion in PyTorch on the same GPU, and the cost of CSR against bits
when synthetic rows leave the device.

    python tools/bench_sparse_rows.py [--shapes ml-100k ml-1m adm cfg5-shard] [--reps 7] [--e2e-reps 3] [--out results.jsonl]

One JSON line per shape, each carrying the GPU's name, power limit and maximum SM clock read in the same run.  The scores are
uniform random float32 [rows, items] binarised by equal_sparsity_device at sparsity 1 - density:
  - indptr_ms / indices_ms: medians of --reps timed calls of the two K10 entries (CUDA events, after 2 warm-up calls);
    to_sparse_ms: PackedMatrix.to_sparse() as a user calls it (both entries, allocation and the one nnz read-back).
  - k10_bytes: the bytes the algorithm must move, the bits read twice (once per entry) + 4 nnz + 8 (rows + 1) written;
    k10_gbs = k10_bytes over indptr_ms + indices_ms, hbm_share = that over 7.7 TB/s (one B200 on NVIDIA's HGX B200 data sheet
    -- a data-sheet figure, not a reached one).  The small shapes' bits fit the 126 MB L2 and are re-read from there.
  - torch_ms: the comparator (unpack the bits with shifts, torch.nonzero, indptr from the row sums).  Its indptr and indices must
    equal K10's, or the script stops.
  - esd_ms: equal_sparsity_device on the same scores; k10_over_esd = (indptr_ms + indices_ms) / esd_ms.  esd_walk: "device",
    or "host" where NumPy's float32 virtual index puts the two order statistics two ranks apart (ml-1m: 18 856 250 scores),
    which the device walk does not take.
At the cfg-5 shard (125 000 x 20 000 at 1 % ones, bench.py's cfg5 generator with random weights) one more line times a whole step
with a host clock around work that ends in a synchronise, alternating the two ways out, --e2e-reps times each (medians):
  csr:  sample_ddpm + equal_sparsity_device + to_sparse() + to_scipy() (pinned buffers, one synchronise)
  bits: sample_ddpm + equal_sparsity_device + the bits copied into a pinned buffer
with the bytes each moves device -> host per user.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from sdrm_b200 import _lib
from sdrm_b200.sparsify import equal_sparsity_device, quantile_plan

SHAPES = {   # rows, items, density of ones
    "ml-100k": (938, 1008, 0.0575),
    "ml-1m": (6034, 3125, 0.0447),
    "adm": (10621, 8582, 0.00115),
    "cfg5-shard": (125000, 20000, 0.01),
}
HBM_BYTES_PER_S = 7.7e12
CFG5 = dict(n=125000, I=20000, H=1000, L=950, T=178, nh=4, nd=1.0)   # bench.py WORKLOADS["cfg5"]


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


def scores(rows, items, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    out = torch.empty((rows, items), dtype=torch.float32, device="cuda")
    for s in range(0, rows, 16384):
        e = min(rows, s + 16384)
        out[s:e] = torch.rand((e - s, items), generator=g, device="cuda")
    return out


def torch_csr(bits, n_cols):
    """The comparator: unpack the bits with shifts, then nonzero for the indices and a cumulative sum of the row counts."""
    shifts = torch.arange(32, dtype=torch.int32, device=bits.device)
    dense = ((bits.unsqueeze(-1) >> shifts) & 1).to(torch.bool).reshape(bits.shape[0], -1)[:, :n_cols]
    indptr = torch.zeros(bits.shape[0] + 1, dtype=torch.int64, device=bits.device)
    torch.cumsum(dense.sum(1), 0, out=indptr[1:])
    return indptr, torch.nonzero(dense)[:, 1].to(torch.int32)


def kernel_line(name, rows, items, density, reps, gpu):
    lib = _lib.load()
    S = scores(rows, items, 1)
    q = 1.0 - density
    # NumPy forms the quantile's virtual index in float32, so past 2^24 scores its two order statistics can lie two ranks
    # apart; the device walk (sdrm_select_begin) takes adjacent ranks only, and such a shape goes through the host walk
    prev_i, nxt_i, _ = quantile_plan(rows * items, q)
    host_walk = nxt_i - prev_i > 1
    pm = equal_sparsity_device(S, q, host_walk=host_walk)
    bits, wpr = pm.bits, pm.bits.shape[1]
    sr = pm.to_sparse()
    ref_ptr, ref_idx = torch_csr(bits, items)
    same = torch.equal(ref_ptr, sr.indptr) and torch.equal(ref_idx, sr.indices)
    if not same:
        raise SystemExit(f"{name}: K10 and the torch comparator disagree")
    del ref_ptr, ref_idx
    st = _lib.stream_ptr()
    ws_bytes = lib.sdrm_packed_csr_workspace_bytes(rows)
    ws = torch.empty(max(1, (ws_bytes + 7) // 8), dtype=torch.int64, device="cuda")
    indptr, indices = torch.empty_like(sr.indptr), torch.empty_like(sr.indices)

    def run_indptr():
        _lib.check(lib.sdrm_packed_csr_indptr(_lib.ptr(bits), wpr, rows, items, _lib.ptr(indptr), _lib.ptr(ws), ws_bytes, st))

    def run_indices():
        _lib.check(lib.sdrm_packed_csr_indices(_lib.ptr(bits), wpr, rows, items, _lib.ptr(sr.indptr), _lib.ptr(indices), st))
    indptr_ms = timed(run_indptr, reps)
    indices_ms = timed(run_indices, reps)
    if not (torch.equal(indptr, sr.indptr) and torch.equal(indices, sr.indices)):
        raise SystemExit(f"{name}: repeated K10 calls disagree")
    to_sparse_ms = timed(pm.to_sparse, reps)
    torch_ms = timed(lambda: torch_csr(bits, items), max(3, reps // 2))
    esd_ms = timed(lambda: equal_sparsity_device(S, q, host_walk=host_walk), max(3, reps // 2))
    nnz = sr.nnz
    k10_bytes = 2 * rows * wpr * 4 + 4 * nnz + 8 * (rows + 1)
    k10_ms = indptr_ms + indices_ms
    rec = dict(gpu=gpu, shape=name, rows=rows, items=items, density=density, nnz=nnz, threshold=float(pm.threshold),
               indptr_ms=round(indptr_ms, 4), indices_ms=round(indices_ms, 4), k10_ms=round(k10_ms, 4),
               to_sparse_ms=round(to_sparse_ms, 4), k10_bytes=k10_bytes, k10_gbs=round(k10_bytes / (k10_ms * 1e-3) / 1e9, 1),
               hbm_share=round(k10_bytes / (k10_ms * 1e-3) / HBM_BYTES_PER_S, 4), torch_ms=round(torch_ms, 4),
               speedup_vs_torch=round(torch_ms / k10_ms, 2), esd_ms=round(esd_ms, 4), esd_walk="host" if host_walk else "device", k10_over_esd=round(k10_ms / esd_ms, 4),
               l2_resident=rows * wpr * 4 < 126e6, equal_to_torch=same)
    del S, pm, bits, sr, indptr, indices, ws
    torch.cuda.empty_cache()
    return rec


def e2e_line(reps, gpu):
    import bench
    from sdrm_b200.train_SDRM import sample_ddpm
    w = CFG5
    diff, vae = bench.build_models(w, torch.device("cuda"), seed=0)
    n, q = w["n"], 0.99

    def step(seed):
        S = sample_ddpm(n, diff, vae, w["L"], w["nd"], n_timesteps=w["T"], seed=seed)
        return equal_sparsity_device(S, q)

    def csr(seed):
        t0 = time.perf_counter()
        mat = step(seed).to_sparse().to_scipy()
        return time.perf_counter() - t0, 4 * mat.nnz + 8 * (n + 1), mat

    def bits(seed):
        t0 = time.perf_counter()
        pm = step(seed)
        host = torch.empty(pm.bits.shape, dtype=torch.int32, pin_memory=True)
        host.copy_(pm.bits, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return time.perf_counter() - t0, host.numel() * 4, host

    csr(100), bits(100)   # warm-up
    t_csr, t_bits = [], []
    for r in range(reps):
        tc, b_csr, mat = csr(200 + r)
        tb, b_bits, host = bits(200 + r)
        # the two ways out carry the same rows
        dense_nnz = int(np.unpackbits(host.numpy().view(np.uint8), axis=1, bitorder="little")[:, : w["I"]].sum())
        if dense_nnz != mat.nnz:
            raise SystemExit("e2e: the CSR and the bit-packed rows of one step disagree")
        t_csr.append(tc)
        t_bits.append(tb)
    med = lambda v: sorted(v)[len(v) // 2] * 1e3
    return dict(gpu=gpu, shape="cfg5-shard e2e step", rows=n, items=w["I"], sparsity=q, nnz=mat.nnz,
                csr_step_ms=round(med(t_csr), 2), bits_step_ms=round(med(t_bits), 2),
                csr_bytes_per_user=round(b_csr / n, 1), bits_bytes_per_user=round(b_bits / n, 1), reps=reps,
                note="sample + equal_sparsity_device + (CSR: to_sparse + to_scipy | bits: pinned copy), host clock, one GPU")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", nargs="+", default=list(SHAPES))
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--e2e-reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    gpu = gpu_info()
    lines = []
    for name in args.shapes:
        rec = kernel_line(name, *SHAPES[name], args.reps, gpu)
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    if args.e2e_reps > 0:
        rec = e2e_line(args.e2e_reps, gpu)
        print(json.dumps(rec), flush=True)
        lines.append(rec)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            for rec in lines:
                fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
