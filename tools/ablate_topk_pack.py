"""Where K12 (sdrm_topk_pack, row_select.cu) spends its time: the kernel timed whole and cut short after its first parts.

    python tools/ablate_topk_pack.py [--shapes 125000x20000 9558x8582] [--dtypes float32 bfloat16] [--density 0.01] [--reps 10]
                                     [--out profiles/topk_pack_ablation_b200.jsonl]

row_select.cu is compiled three times into a temporary directory (with errors.cu, nothing else) with SDRM_TOPK_ABLATE =
0 (the kernel as shipped), 1 (the staging pass alone: each row copied once from global into shared memory) and 2 (staging and
the radix select, no pack pass).  The three libraries are loaded side by side and timed alternately on the same scores and
per-row k (CUDA events around each launch, median of --reps after two warm-up launches each).  The pack pass costs the difference
between 0 and 2, the select the difference between 2 and 1.  The k come from a seeded log-normal activity at --density of the
items, assigned to the rows in random order.  The GPU's name and power limit head the output.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from sdrm_b200 import _lib
from sdrm_b200.csrc import build as csrc_build

HBM_BYTES_PER_S = 7.7e12
VARIANTS = {0: "whole kernel", 1: "staging alone", 2: "staging + select"}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # (the query is informative only)
        q = f"nvidia-smi unavailable: {e}"
    return {"gpu": torch.cuda.get_device_name(), "nvidia_smi": q}


def build_variants(tmp):
    nvcc = csrc_build._nvcc()
    libs = {}
    for v in VARIANTS:
        out = os.path.join(tmp, f"libk12_ablate{v}.so")
        srcs = [os.path.join(csrc_build.HERE, s) for s in ("row_select.cu", "errors.cu")]
        subprocess.run([nvcc] + csrc_build.FLAGS + [f"-DSDRM_TOPK_ABLATE={v}", "-shared", "-o", out] + srcs +
                       ["-lcudart_static", "-lpthread", "-ldl", "-lrt"], check=True)
        lib = C.CDLL(out)
        for name in ("sdrm_topk_pack", "sdrm_topk_pack_bf16"):
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = _lib.SIGNATURES[name]
        libs[v] = lib
    return libs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", nargs="+", default=["125000x20000", "9558x8582"])
    ap.add_argument("--dtypes", nargs="+", default=["float32", "bfloat16"])
    ap.add_argument("--density", type=float, default=0.01)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default="profiles/topk_pack_ablation_b200.jsonl")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("ablate_topk_pack: no CUDA device; the timings need a B200")
    lines = [json.dumps(gpu_info())]
    print(lines[0], flush=True)
    with tempfile.TemporaryDirectory(prefix="k12_ablate_") as tmp:
        libs = build_variants(tmp)
        for shape in a.shapes:
            rows, n_cols = (int(v) for v in shape.split("x"))
            S32 = torch.randn((rows, n_cols), device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
            x = np.random.default_rng(rows).lognormal(0.0, 1.0, size=rows)
            k = np.clip(np.round(x / x.mean() * a.density * n_cols), 0, n_cols).astype(np.int32)
            k32 = torch.from_numpy(k).cuda()
            for dname in a.dtypes:
                S = S32 if dname == "float32" else S32.to(getattr(torch, dname))
                bits = torch.empty((rows, (n_cols + 31) // 32), dtype=torch.int32, device="cuda")
                count = torch.zeros(1, dtype=torch.int64, device="cuda")
                status = torch.zeros(1, dtype=torch.int32, device="cuda")

                def launch(v):
                    lib = libs[v]
                    entry = lib.sdrm_topk_pack_bf16 if dname == "bfloat16" else lib.sdrm_topk_pack
                    rc = entry(_lib.ptr(S), rows, n_cols, n_cols, _lib.ptr(k32), _lib.ptr(bits), bits.shape[1], _lib.ptr(count),
                               _lib.ptr(status), _lib.stream_ptr())
                    assert rc == 0, f"variant {v} failed ({rc})"
                for v in VARIANTS:
                    launch(v)
                    launch(v)
                torch.cuda.synchronize()
                ts = {v: [] for v in VARIANTS}
                for _ in range(a.reps):
                    for v in VARIANTS:
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        launch(v)
                        e1.record()
                        e1.synchronize()
                        ts[v].append(e0.elapsed_time(e1))
                score_bytes = rows * n_cols * S.element_size()
                rec = {"dtype": dname, "rows": rows, "items": n_cols, "density": a.density, "score_bytes": score_bytes}
                for v, name in VARIANTS.items():
                    ms = float(np.median(ts[v]))
                    rec[name.replace(" + ", "_").replace(" ", "_") + "_ms"] = round(ms, 4)
                    rec[name.replace(" + ", "_").replace(" ", "_") + "_hbm_fraction"] = round(score_bytes / (ms * 1e-3) / HBM_BYTES_PER_S, 3)
                lines.append(json.dumps(rec))
                print(lines[-1], flush=True)
                del bits
            del S, S32
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
