"""The SVD evaluator on the GPU (evaluators.compute_mf_results_gpu, products on K11) against sklearn on the host.

    python tools/bench_svd_evaluator.py [--shapes ml-100k alb adm ml-1m-like scale-up] [--reps 3] [--out results.jsonl]

One JSON line per shape and only_synthetic setting, each carrying the GPU's name, power limit and maximum SM clock read in the
same run.  Rows are seeded random 0/1 rows at the shape's density (train and test rows at the real density, synthetic rows at
the higher density equal sparsity gives them).  The evaluator's matrix is [train; test_data; synthetic] (only_synthetic=False,
2 U + V rows) or [synthetic; test_data] (only_synthetic=True, U + V rows).
  - gpu_ms: compute_mf_results_gpu as a caller runs it (split, row assembly, SVD, scoring, metrics), host clock around a call that
    ends in host arrays; median of --reps calls after one warm-up call.
  - k11_ms: the K11 products of one call (2 n_iter + 2 products at w = 30 on M / Mt, one at w = 20 on the test rows) replayed
    back to back between two CUDA events; median of --reps replays.  The rest of gpu_ms is the 30-column QR / SVD plumbing,
    the split on the host, uploads, K3 metrics and launch overheads.
  - sk_dense_s / sk_csr_s: sklearn's SVD step on the host, TruncatedSVD(20, n_iter=100).fit_transform of the whole matrix and
    inverse_transform of the V scored rows, on the dense int64 matrix (today's path) and on the same rows as scipy CSR.  The
    evaluator itself reconstructs every row; timing only the scored rows favours sklearn.  Dense is not run for scale-up
    (21 GB).  One call each.
  - max_rel_diff: max |GPU score - sklearn score| / max |sklearn score| over the scored block (finite entries), against the dense
    run where there is one, else the CSR run; metrics_equal: recall and ndcg (rounded means) of both blocks through the same
    metrics are equal.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import scipy.sparse as sp
import torch

from sdrm_b200 import evaluators, metrics, svd
from sdrm_b200.data import split_train_test_proportion_from_csr_matrix

SHAPES = {   # U (train users = synthetic users), V (test users), items, real density, synthetic density, only_synthetic settings
    "ml-100k": (843, 95, 1008, 0.0575, 0.1007, (False, True)),
    "alb": (1200, 152, 729, 0.03, 0.05, (False, True)),
    "adm": (9500, 1179, 8582, 0.00115, 0.002, (False, True)),
    "ml-1m-like": (5700, 600, 3125, 0.045, 0.045, (False, True)),
    "scale-up": (130072, 1000, 20000, 0.01, 0.01, (True,)),
}


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # (the query is informative only)
        return f"nvidia-smi unavailable: {e}"


def random_rows(rng, n, n_items, density):
    counts = rng.binomial(n_items, density, size=n)
    keys = np.unique(np.repeat(np.arange(n, dtype=np.int64), counts) * n_items + rng.integers(0, n_items, int(counts.sum())))
    return sp.csr_matrix((np.ones(keys.size, dtype=np.int64), (keys // n_items, keys % n_items)), shape=(n, n_items))


def sklearn_block(train, testing, synth, only, dense):
    from sklearn.decomposition import TruncatedSVD
    test_data, valid = split_train_test_proportion_from_csr_matrix(testing, batch_size=1000, random_seed=123)
    head = synth if only else train
    combined = sp.vstack([head, test_data] + ([] if only else [synth]), format="csr")
    X = combined.toarray().astype(np.int64) if dense else combined.astype(np.float64)
    lo, V = head.shape[0], test_data.shape[0]
    t0 = time.perf_counter()
    mf = TruncatedSVD(n_components=20, n_iter=100)
    Xt = mf.fit_transform(X)
    block = mf.inverse_transform(Xt[lo: lo + V])
    dt = time.perf_counter() - t0
    block[test_data.nonzero()] = -np.inf
    return block, valid, dt, combined.shape


def k11_replay(train, testing, synth, only, reps):
    test_data, _ = split_train_test_proportion_from_csr_matrix(testing, batch_size=1000, random_seed=123)
    test = svd.device_rows(test_data)
    parts = [svd.device_rows(synth), test] if only else [svd.device_rows(train), test, svd.device_rows(synth)]
    M = svd.vstack_rows(parts)
    Mt = svd.transpose_rows(M)
    A, At = (Mt, M) if M.shape[0] < M.shape[1] else (M, Mt)
    qa = torch.randn(A.shape[1], 30, dtype=torch.float64, device="cuda")
    qb = torch.randn(A.shape[0], 30, dtype=torch.float64, device="cuda")
    vt = torch.randn(M.shape[1], 20, dtype=torch.float64, device="cuda")
    status = torch.zeros(1, dtype=torch.int32, device="cuda")

    def products():
        for _ in range(svd.N_ITER + 1):
            svd.spmm(A, qa, status)
            svd.spmm(At, qb, status)
        svd.spmm(test, vt, status)
    products()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        products()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    svd.check_status(status)
    return float(np.median(times)), M.nnz


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", nargs="+", default=list(SHAPES))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_svd_evaluator needs a CUDA device")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    gpu = gpu_info()
    for name in a.shapes:
        U, V, n_items, dens, sdens, onlys = SHAPES[name]
        rng = np.random.default_rng(2024)
        train, testing, synth = (random_rows(rng, U, n_items, dens), random_rows(rng, V, n_items, dens),
                                 random_rows(rng, U, n_items, sdens))
        for only in onlys:
            evaluators.compute_mf_results_gpu(train, testing, synth, only)          # warm-up
            times = []
            for _ in range(a.reps):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                rec, ndcg = evaluators.compute_mf_results_gpu(train, testing, synth, only)
                torch.cuda.synchronize()
                times.append((time.perf_counter() - t0) * 1e3)
            k11_ms, nnz = k11_replay(train, testing, synth, only, a.reps)
            block, _ = evaluators.mf_scores_gpu(train, testing, synth, only)
            block = block.cpu().numpy()
            sk_dense = None
            if name != "scale-up":
                ref, valid, sk_dense, shape = sklearn_block(train, testing, synth, only, True)
            ref_csr, valid, sk_csr, shape = sklearn_block(train, testing, synth, only, False)
            if sk_dense is None:
                ref = ref_csr
            fin = np.isfinite(ref)
            assert (np.isfinite(block) == fin).all()
            diff = float(np.abs(block[fin] - ref[fin]).max() / np.abs(ref[fin]).max())
            both = metrics.recall_ndcg_multi_k(ref, valid, evaluators.K_LIST)
            rec_ref = np.array([np.round(np.nanmean(both[k][0]), 4) for k in evaluators.K_LIST])
            ndcg_ref = np.array([np.round(np.nanmean(both[k][1]), 4) for k in evaluators.K_LIST])
            gpu_ms = float(np.median(times))
            line = {"gpu": gpu, "shape": name, "only_synthetic": only, "rows": shape[0], "items": shape[1], "nnz": nnz,
                    "gpu_ms": round(gpu_ms, 2), "k11_ms": round(k11_ms, 3), "k11_products": 2 * svd.N_ITER + 3,
                    "sk_dense_s": None if sk_dense is None else round(sk_dense, 3), "sk_csr_s": round(sk_csr, 3),
                    "speedup_vs_csr": round(sk_csr * 1e3 / gpu_ms, 1), "max_rel_diff": diff,
                    "metrics_equal": bool((rec == rec_ref).all() and (ndcg == ndcg_ref).all()),
                    "recall@10": float(rec[3]), "ndcg@10": float(ndcg[3])}
            print(json.dumps(line), flush=True)
            if a.out:
                with open(a.out, "a") as fh:
                    fh.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
