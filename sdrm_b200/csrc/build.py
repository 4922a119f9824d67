"""Build libsdrm_b200.so (sm_100a only) in-tree with nvcc.  Used by __graft_entry__.build()."""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "libsdrm_b200.so")
SOURCES = ["errors.cu", "engine_host.cu", "engine_bf16.cu", "metrics.cu", "train_kernels.cu", "train_gemm.cu", "sparsify.cu"]
HEADERS = ["ptx_sm100.cuh", "philox.cuh", "layer_engine.cuh", "layer_engine_kernel.cuh", "engine_launch.cuh", "gemm_x3_kernel.cuh", "small_chain_kernel.cuh", "host_util.h",
           "../../include/sdrm_b200.h"]
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=default", "--expt-relaxed-constexpr",
]


def _nvcc():
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; the SDRM CUDA library cannot be built")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(HERE, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force=False, verbose=False, extra_flags=(), out=None):
    """extra_flags / out: tuning variants (e.g. -DSDRM_NSTG_PAIR=6 -> another .so selected with SDRM_B200_LIB)."""
    global LIB
    if out:
        LIB = os.path.join(HERE, out)
        force = True
    if not force and not needs_build():
        return LIB
    nvcc = _nvcc()
    objs = []
    procs = []
    for s in SOURCES:
        src = os.path.join(HERE, s)
        if not os.path.exists(src):
            continue
        obj = os.path.join(HERE, s.replace(".cu", ".o" if not out else "." + out + ".o"))
        cmd = [nvcc] + FLAGS + list(extra_flags) + (["-Xptxas", "-v"] if verbose else []) + ["-dc" if False else "-c", src, "-o", obj]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for s, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError(f"nvcc failed on {s}")
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart_static", "-lpthread", "-ldl", "-lrt"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed")
    return LIB


if __name__ == "__main__":
    extra = [a for a in sys.argv[1:] if a.startswith("-D")]
    outs = [a[6:] for a in sys.argv[1:] if a.startswith("--out=")]
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, extra_flags=extra, out=outs[0] if outs else None))
