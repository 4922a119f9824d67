#!/usr/bin/env python
"""Headline benchmark: synthetic users / second through the FULL T-step reverse chain + VAE decode.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg5] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one sample_ddpm-equivalent pass over one batch of users (SURVEY.md §8d).  Default workload is the
configuration BASELINE.json quotes its target on: the synthetic scale-up (T=178, VAE 1000/950, 4 hidden layers,
20 000 items), 1 M users over 8 GPUs = 125 000 users per GPU, weak scaling (per-GPU work fixed).
`value`   : device-timed, output stays in HBM.
`e2e`     : through the public API with the rows delivered into pinned HOST memory (D2H inside the timed region).
`roofline`: tensor-pipe fraction of the persistent kernel vs the measured sustained bf16 peak.
`cpu_baseline`: the reference's own sample_ddpm (unmodified files under the git-ignored baseline/_ref/, staged by build()) on
               the box's host cores; the oracle port only if the reference is not on the box.
`--impl reference` times that CPU implementation alone with all host threads (rank 0 only) and adds `eager_cuda`: the same
               reference code with DEVICE='cuda' (PyTorch eager) on this box's GPU.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: n per GPU, items, vae hidden, latent, T, hidden layers, noise divider
    "cfg1": dict(n=843, I=1008, H=930, L=830, T=83, nh=2, nd=1.0, desc="ml-100k SVD augment"),
    "cfg2": dict(n=5429, I=3125, H=490, L=340, T=78, nh=1, nd=1.0, desc="ml-1m MLP augment"),
    "cfg3": dict(n=9558, I=8582, H=40, L=40, T=93, nh=5, nd=1.0, desc="ADM NeuMF augment"),
    "cfg4": dict(n=1208, I=729, H=550, L=400, T=43, nh=0, nd=0.2, desc="ALB MLP augment"),
    "cfg5": dict(n=125000, I=20000, H=1000, L=950, T=178, nh=4, nd=1.0,
                 desc="synthetic scale-up 1M users x 20k items over 8 GPUs (125k users/GPU)"),
}


def flops_per_user(w):
    """Algorithmic FLOPs (SURVEY.md §8d): T*2*L^2*(2+nh) + 2*(L*H + H*I); time embedding hoisted, bf16x3 credited once."""
    return w["T"] * 2 * w["L"] ** 2 * (2 + w["nh"]) + 2 * (w["L"] * w["H"] + w["H"] * w["I"])


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            p = json.load(fh)
        return dict(tflops=p.get("bf16_tflops_sustained", 1413.8), hbm=p.get("hbm_gbs", 6535.7), source="measured")
    return dict(tflops=1590.0, hbm=6650.0, source="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            parts = [p.strip() for p in r.split(",")]
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except Exception:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank's host threads (and so the first-touch placement of its pinned buffers) to the NUMA node its GPU hangs
    off: with 8 ranks copying 10 GB of rows per step into host memory, buffers that all land on one socket halve the aggregate
    device->host rate.  Returns a short description for the JSON line (None when sysfs does not say)."""
    try:
        import torch
        prop = torch.cuda.get_device_properties(local_rank)
        bus = f"{prop.pci_domain_id:04x}:{prop.pci_bus_id:02x}:{prop.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as fh:
            node = int(fh.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as fh:
            spec = fh.read().strip()
        cpus = set()
        for part in spec.split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return {"gpu": bus, "numa_node": node, "cpus": len(allowed)}
    except Exception:
        return None


def build_models(w, device, seed=0):
    import torch
    from sdrm_b200.models import SDRM, VAE
    torch.manual_seed(seed)  # reference initialisers; timing is weight-independent (random-init, synthetic data)
    vae = VAE(input_dim=w["I"], hidden_dim=w["H"], latent_dim=w["L"]).to(device).eval()
    diff = SDRM(N_ITEMS=w["L"], EMB_DIM=w["T"], LATENT_DIM=w["L"], n_hidden_layers=w["nh"]).to(device).eval()
    return diff, vae


def _reference_module():
    """The reference's OWN train_SDRM module (unmodified files staged under the git-ignored baseline/_ref/ by build(), imported
    through oracle/refstub.py's optuna / bottleneck stubs), or None when it is not available on this box."""
    try:
        from oracle import refstub
        if not refstub.reference_available():
            return None
        return refstub.import_reference()
    except Exception as exc:   # fall back to the oracle port
        sys.stderr.write(f"reference import failed ({exc!r}); timing the oracle port instead\n")
        return None


def reference_rate(w, rows, device, threads=None, repeats=1):
    """users/s of the reference's own sample_ddpm (train_SDRM.py:27-63, full mode) on `device` ('cpu' or 'cuda'): its module
    global DEVICE and schedule globals are set the way its train_SDRM() sets them (297-303); models are the reference's own
    classes, random-init (timing is weight-independent)."""
    import torch
    from oracle import sdrm_oracle as orc
    ref = _reference_module()
    if ref is None:
        return None
    if threads:
        torch.set_num_threads(threads)
    ref.DEVICE = device
    b_t, a_t, ab_t = orc.make_schedule(w["T"])
    ref.b_t, ref.a_t, ref.ab_t = b_t.to(device), a_t.to(device), ab_t.to(device)
    torch.manual_seed(0)
    vae = ref.VAE(input_dim=w["I"], hidden_dim=w["H"], latent_dim=w["L"]).to(device).eval()
    diff = ref.SDRM(N_ITEMS=w["L"], EMB_DIM=w["T"], LATENT_DIM=w["L"], n_hidden_layers=w["nh"]).to(device).eval()
    best = None
    for _ in range(repeats):
        if device != "cpu":
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = ref.sample_ddpm(rows, diff, vae, w["L"], w["nd"], n_timesteps=w["T"])
        if device != "cpu":
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    assert tuple(out.shape) == (rows, w["I"])
    del out
    return rows / best, best


def cpu_reference_rate(w, rows, threads, repeats=1):
    """(users/s, seconds, kind): the reference's own sample_ddpm on the host cores when it is staged on this box (kind
    'reference'), else the CPU restatement (oracle, kind 'port'); RNG draws inside the timed region like the reference."""
    import torch
    r = reference_rate(w, rows, "cpu", threads, repeats)
    if r is not None:
        return r[0], r[1], "reference"
    from oracle import sdrm_oracle as orc
    torch.set_num_threads(threads)
    diff, vae = build_models(w, "cpu")
    dsd = {k: v.detach() for k, v in diff.state_dict().items()}
    vsd = {k: v.detach() for k, v in vae.state_dict().items()}
    T, L = w["T"], w["L"]
    best = None
    with torch.no_grad():
        for _ in range(repeats):
            t0 = time.perf_counter()
            sched = orc.make_schedule(T)
            x = torch.randn(rows, L)
            for i in range(T, 0, -1):
                z = torch.randn_like(x) * w["nd"] if i > 1 else 0
                keep = torch.empty_like(x).bernoulli_(0.5)
                eps = orc.denoiser_forward(dsd, x, torch.full((rows,), i, dtype=torch.long), keep)
                x = orc.posterior_step(x, eps, z, i, sched)
            out = orc.vae_decode(vsd, x)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    assert out.shape == (rows, w["I"])
    return rows / best, best, "port"


def _cpu_sample_text(kind, rows, w):
    src = "the reference's own train_SDRM.sample_ddpm (baseline/_ref, unmodified)" if kind == "reference" else "oracle/sdrm_oracle.py (port)"
    return f"{rows} users x full T={w['T']} chain + decode per step, {src}, torch CPU, RNG draws inside the timed region"


def run_reference(args, w, rank):
    if rank != 0:
        return
    import torch
    threads = os.cpu_count() or 1
    rows = args.cpu_rows or max(64, min(4096, int(2.0e12 / flops_per_user(w))))
    for _ in range(args.warmup):
        cpu_reference_rate(w, max(8, rows // 8), threads)
    t_all, kind = 0.0, "port"
    for _ in range(args.steps):
        rate, dt, kind = cpu_reference_rate(w, rows, threads)
        t_all += dt
    value = rows * args.steps / t_all
    # second stated baseline (BASELINE.md §4 item 4): the SAME reference code with DEVICE='cuda' -- PyTorch eager / cuBLAS fp32
    # on this box's GPU 0, a bounded sample of the workload
    eager = None
    if torch.cuda.is_available() and _reference_module() is not None and not args.no_eager:
        try:
            erows = args.eager_rows or min(w["n"], 32768)
            reference_rate(w, max(128, erows // 8), "cuda")
            r = reference_rate(w, erows, "cuda", repeats=2)
            eager = {"value": r[0], "unit": "users/s", "rows_per_step": erows, "seconds": r[1],
                     "what": "reference train_SDRM.sample_ddpm unmodified, DEVICE='cuda' (PyTorch eager, fp32 cuBLAS), GPU 0, output left on the device"}
        except Exception as exc:
            eager = {"error": repr(exc)[:200]}
    line = {
        "impl": "reference", "metric": "synthetic users/sec (full reverse diffusion + decode)", "value": value,
        "unit": "users/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t_all / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic (random-init weights of the named shape, torch CPU RNG)",
        "config": {"workload": args.workload, **{k: w[k] for k in ("I", "H", "L", "T", "nh", "nd")},
                   "rows_per_step": rows, "note": "bounded sample of the workload on host cores"},
        "cpu_baseline": {"value": value, "unit": "users/s", "cores": threads, "kind": kind, "sample": _cpu_sample_text(kind, rows, w)},
        "e2e": {"value": value, "unit": "users/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "eager_cuda": eager,
    }
    emit(line)


DUMP_BYTES = 60 << 20   # stays under 64 MB in either unit (10^6 or 2^20 bytes), .npy headers included


def dump_outputs(path, out, rank, world, row_offset):
    """Write what the last timed step returned, the float32 logits [n, I] of this rank, to `path` so that two builds can be
    compared output for output: `logits.npy` holds whole rows (all of them when every rank's rows fit in DUMP_BYTES, else a
    fixed seeded sample) and `logits_rows.npy` their global row ids; with several ranks each file gets a `_rank<r>` suffix."""
    import numpy as np
    import torch
    n, I = out.shape
    k = min(n, DUMP_BYTES // world // (4 * I + 8))
    rows = np.sort(np.random.default_rng(0).choice(n, size=k, replace=False)) if k < n else np.arange(n)
    logits = out.index_select(0, torch.from_numpy(rows).to(out.device)).cpu().numpy()
    suffix = f"_rank{rank}" if world > 1 else ""
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, f"logits{suffix}.npy"), logits.astype(np.float32, copy=False))
    np.save(os.path.join(path, f"logits_rows{suffix}.npy"), (rows + row_offset).astype(np.float64))


def run_ours(args, w, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from sdrm_b200.train_SDRM import engine_for, sample_ddpm, sample_ddpm_host

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n = args.rows or w["n"]
    diff, vae = build_models(w, dev)
    row_offset = rank * n
    out = torch.empty((n, w["I"]), dtype=torch.float32, device=dev)

    def step(seed):
        # device-timed leg: the weights do not change between the steps, so the packed images are reused (reuse_packed);
        # the e2e leg below uploads and re-packs them every step
        sample_ddpm(n, diff, vae, w["L"], w["nd"], n_timesteps=w["T"], seed=seed, row_offset=row_offset, out=out, reuse_packed=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    from sdrm_b200 import _lib as _l
    eng = engine_for(diff, dev)
    eng.set_option(_l.OPT_CLUSTER, args.cluster)
    eng.set_option(_l.OPT_SUBTILES, args.subtiles)
    eng.set_option(_l.OPT_NO_DISCARD, int(os.environ.get("SDRM_NO_DISCARD", "0")))   # A/B of the dead-buffer discard
    eng.set_option(_l.OPT_RESIDENT, int(os.environ.get("SDRM_NO_RESIDENT", "0")))   # A/B of the resident (latency) mode
    if int(os.environ.get("SDRM_DEBUG_FLAGS", "0")):    # perf experiments (tools/ablate.sh): -DSDRM_PERF_DEBUG builds only
        eng.set_option(_l.OPT_DEBUG_FLAGS, int(os.environ["SDRM_DEBUG_FLAGS"]))
    for i in range(args.warmup):
        step(1000 + i)
    barrier()
    from sdrm_b200 import _lib
    _lib.check(eng.lib.sdrm_check_device_error(eng.handle, _lib.stream_ptr()), "warmup")
    launches_per_step = eng.launch_count()

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    ev[0].record()
    for i in range(args.steps):
        step(2000 + i)
        ev[i + 1].record()
    barrier()
    clock_info = clocks.stop() if rank == 0 else None
    total_ms = ev[0].elapsed_time(ev[-1])
    step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(args.steps)]
    t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    value = world * n * args.steps / (total_ms * 1e-3)
    if args.dump_outputs:   # before the e2e leg below, which overwrites `out`
        dump_outputs(args.dump_outputs, out, rank, world, row_offset)

    # ---- end to end through the public call with HOST buffers: every step uploads the trained weights from pinned host
    #      memory (the checkpoint a caller holds), re-packs them, samples, and delivers the rows into pinned host memory
    #      (what main.py's .cpu().numpy() consumes)
    e2e = None
    if not args.no_e2e:
        host = torch.empty((n, w["I"]), dtype=torch.float32, pin_memory=True)
        params = [p for p in list(diff.parameters()) + list(vae.decoder.parameters())]
        host_w = [p.detach().cpu().pin_memory() for p in params]
        h2d_bytes = sum(t.numel() * t.element_size() for t in host_w)

        def e2e_step(seed):
            for p, hw in zip(params, host_w):
                p.data.copy_(hw, non_blocking=True)   # H2D; bumps the tensor version, so the engine re-packs the weights
            sample_ddpm_host(n, diff, vae, w["L"], w["nd"], n_timesteps=w["T"], seed=seed, row_offset=row_offset, host_out=host)

        e2e_step(5)
        barrier()
        t0 = time.perf_counter()
        for i in range(args.e2e_steps):
            e2e_step(3000 + i)
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        e2e = {"value": world * n * args.e2e_steps / float(dt.item()), "unit": "users/s", "h2d_bytes_per_step": h2d_bytes,
               "d2h_bytes_per_step": n * w["I"] * 4, "steps": args.e2e_steps, "host_numa_binding": numa,
               "d2h_gbs_aggregate": world * n * w["I"] * 4 * args.e2e_steps / float(dt.item()) / 1e9,
               "note": "per step: weights H2D from pinned memory + re-pack, sample_ddpm_host (chunked chain+decode, the D2H of "
                       "chunk c overlaps chunk c+1), rows land in pinned host memory; wall clock incl. all copies"}
        del host
        # ---- the same pipeline followed by the reference's next step (main.py:177-178: equal-sparsity binarisation), with K4
        #      on the device: global quantile over all ranks (one 2048-bin histogram all-reduce per radix pass over NCCL)
        #      and 1 bit per entry into pinned host memory.  Reported beside e2e; the headline e2e stays the fp32 logits.
        try:
            from sdrm_b200.sparsify import equal_sparsity_device
            grp = dist.group.WORLD if world > 1 else None
            host_bits = torch.empty((n, (w["I"] + 31) // 32), dtype=torch.int32, pin_memory=True)

            def packed_step(seed):
                for p, hw in zip(params, host_w):
                    p.data.copy_(hw, non_blocking=True)
                sample_ddpm(n, diff, vae, w["L"], w["nd"], n_timesteps=w["T"], seed=seed, row_offset=row_offset, out=out)
                pm = equal_sparsity_device(out, 0.99, group=grp)
                host_bits.copy_(pm.bits, non_blocking=True)
                torch.cuda.synchronize(dev)

            packed_step(7)
            barrier()
            t0 = time.perf_counter()
            for i in range(args.e2e_steps):
                packed_step(4000 + i)
            barrier()
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            e2e["packed"] = {"value": world * n * args.e2e_steps / float(dt.item()), "unit": "users/s",
                             "d2h_bytes_per_step": host_bits.numel() * 4, "sparsity": 0.99,
                             "note": "sample_ddpm + equal_sparsity_device (global np.quantile threshold) + bit-packed rows to pinned host memory"}
        except Exception as exc:   # the headline numbers must survive a failure of the optional leg
            e2e["packed"] = {"error": repr(exc)[:200]}

    if rank == 0:
        peaks = measured_peaks()
        F = flops_per_user(w)
        kernel_ms = statistics.mean(step_ms)  # one persistent kernel per step
        achieved = F * n / (kernel_ms * 1e-3) / 1e12
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath) and args.workload == "cfg5":
            with open(tpath) as fh:
                tj = json.load(fh)
            traffic = tj["dram_bytes_per_user"] * n   # one launch processes n users
            traffic_src = tj["source"]
        roofline = {"bound": "tensor", "achieved": achieved, "peak": peaks["tflops"], "unit": "TFLOP/s",
                    "frac": achieved / peaks["tflops"], "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peaks["source"] + " sustained bf16",
                    "kernel": "sdrm_small_chain_kernel (K6)" if int(eng.lib.sdrm_last_cluster_size(eng.handle)) == 0 else "sdrm_layer_engine_kernel (K1)",
                    "kernel_ms": kernel_ms, "flops_per_user": F,
                    "hbm_min_bytes_per_user": 4 * w["I"],
                    "hbm_frac_of_logits_write": (4 * w["I"] * n / (kernel_ms * 1e-3) / 1e9) / peaks["hbm"]}
        cpu = None
        if not args.no_cpu and world == 1:   # reported on rank 0 at N=1 only
            threads = os.cpu_count() or 1
            rows = args.cpu_rows or max(64, min(4096, int(2.0e12 / F)))
            rate, dt, kind = cpu_reference_rate(w, rows, threads)
            cpu = {"value": rate, "unit": "users/s", "cores": threads, "kind": kind, "seconds": dt, "sample": _cpu_sample_text(kind, rows, w)}
        secondary = None
        if world == 1 and not args.no_secondary:
            try:
                secondary = secondary_kernels(args, w, dev, diff, vae, out, peaks)
            except Exception as exc:   # the headline line must survive a failure of the side measurements
                secondary = {"error": repr(exc)[:200]}
        line = {
            "metric": "synthetic users/sec (full reverse diffusion + decode)", "value": value, "unit": "users/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic (random-init weights of the named shape, in-kernel Philox noise)",
            "config": {"workload": args.workload, "desc": w["desc"], "users_per_gpu": n,
                       **{k: w[k] for k in ("I", "H", "L", "T", "nh", "nd")},
                       "l2": "each step writes n*I*4 bytes of logits (>> 126 MB L2 for cfg5); no reuse across steps",
                       "precision": "bf16 operands / fp32 accumulate in the chain, bf16x3 split in the decoder"},
            "clocks": clock_info, "e2e": e2e, "cluster": int(eng.lib.sdrm_last_cluster_size(eng.handle)), "resident": int(eng.lib.sdrm_last_resident_mode(eng.handle)), "subtiles": args.subtiles, "gpu_launches": launches_per_step * args.steps,
            "roofline": roofline, "cpu_baseline": cpu, "secondary": secondary,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()



def secondary_kernels(args, w, dev, diff, vae, out, peaks):
    """The other kernels of the path, timed in the same process on the logits the timed steps left in `out` (rank 0, one GPU):
    multi-resolution sampling (train_SDRM.py:37-49), K3 top-k (utilities.py:149-171), K4 equal-sparsity binarisation
    (main.py:177-185) and K2 forward noising (train_SDRM.py:191-199).  CUDA events, 3 repetitions after one warm-up, best."""
    import numpy as np
    import torch
    from sdrm_b200 import metrics
    from sdrm_b200.sparsify import equal_sparsity_device
    from sdrm_b200.train_SDRM import sample_ddpm
    from sdrm_b200.training import CudaLossBackend

    def best_ms(fn, reps=3):
        fn()
        ms = []
        for _ in range(reps):
            torch.cuda.synchronize(dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize(dev)
            ms.append(a.elapsed_time(b))
        return min(ms)

    res = {}
    n, I = out.shape
    # multi-resolution mode: row j runs t_j ~ U{1..T-1} steps (rows sorted by chain length; CTA pairs since the third r02 session)
    n_r = min(n, 148 * 128)
    np.random.seed(0)
    ms = best_ms(lambda: sample_ddpm(n_r, diff, vae, w["L"], w["nd"], timesteps="random", n_timesteps=w["T"], seed=5, out=out[:n_r], reuse_packed=True))
    res["sample_ddpm_random"] = {"users_per_s": n_r / (ms * 1e-3), "ms": ms, "rows": n_r, "note": "timesteps='random': mean chain length T/2; CTA pairs, a pair runs the longer of its two tiles' chains"}
    # refill `out` with full-resolution logits for the score consumers below
    sample_ddpm(n, diff, vae, w["L"], w["nd"], n_timesteps=w["T"], seed=6, out=out, reuse_packed=True)
    # (the chain kernel leaves the board at its power cap with the SM clock near 1.2 GHz; the HBM-bound kernels below are timed
    # after a pause, i.e. at the clocks they see when they are not queued right behind 280 ms of tensor work)
    torch.cuda.synchronize(dev)
    time.sleep(1.0)
    rows = min(n, 65536)
    for k in (10, 50):
        ms = best_ms(lambda: metrics.topk_device(out[:rows], k))
        gbs = 4.0 * rows * I / (ms * 1e-3) / 1e9
        res[f"topk_k{k}"] = {"ms": ms, "GBps": gbs, "frac_of_hbm_peak": gbs / peaks["hbm"], "rows": rows, "items": I}
    ms = best_ms(lambda: equal_sparsity_device(out, 0.99))
    res["equal_sparsity_pack"] = {"ms": ms, "rows": n, "items": I, "passes_GBps": 4.0 * 4.0 * n * I / (ms * 1e-3) / 1e9,
                                  "note": "3 radix-select histogram passes + threshold/pack pass over the fp32 scores, end to end incl. the device walk"}
    # K2: forward noising of a [B, L] latent minibatch (1 read, 4 writes)
    B = 262144
    mu = torch.randn(B, w["L"], device=dev)
    t = torch.randint(1, w["T"] + 1, (B,), device=dev)
    from sdrm_b200.models import make_schedule
    _, _, ab_t = make_schedule(w["T"], device=dev)
    be = CudaLossBackend()
    ms = best_ms(lambda: be.noise_inputs(mu, t, ab_t, w["nd"], 0.1, 11, 0))
    gbs = 5.0 * 4.0 * B * w["L"] / (ms * 1e-3) / 1e9
    res["noise_inputs"] = {"ms": ms, "GBps": gbs, "frac_of_hbm_peak": gbs / peaks["hbm"], "rows": B, "L": w["L"]}
    # BASELINE.json configs 1-4 (dataset-sized calls, the latency regime): one sample_ddpm of all N_USERS rows at the full T
    from sdrm_b200 import _lib
    from sdrm_b200.train_SDRM import engine_for
    lib = _lib.load()
    ds = {}
    for name in ("cfg1", "cfg2", "cfg3", "cfg4"):
        wd = WORKLOADS[name]
        d2, v2 = build_models(wd, dev)
        o2 = torch.empty(wd["n"], wd["I"], device=dev)
        ms = best_ms(lambda: sample_ddpm(wd["n"], d2, v2, wd["L"], wd["nd"], n_timesteps=wd["T"], seed=3, out=o2, reuse_packed=True), reps=5)
        hdl = engine_for(d2, dev).handle
        split, resident, cluster = lib.sdrm_last_split_size(hdl), lib.sdrm_last_resident_mode(hdl), lib.sdrm_last_cluster_size(hdl)
        flow = (f"column split, clusters of {split}" if split else "small-chain kernel (K6)" if cluster == 0 else
                "resident tile" if resident else "streaming pairs" if cluster == 2 else "single CTAs")
        ds[name] = {"ms": ms, "users_per_s": wd["n"] / (ms * 1e-3), "rows": wd["n"], "items": wd["I"], "T": wd["T"], "flow": flow}
        del d2, v2, o2
    res["dataset_configs"] = ds
    return res


def train_flops_per_row(w):
    """Algorithmic FLOPs of one diffusion training step per minibatch row (train_SDRM.py:331-337): three denoiser forwards,
    their weight gradients, and the data gradients of every layer but the first (nothing upstream of layer 0 needs one);
    the hoisted time-embedding table (two [T+1, T] products) is not counted; bf16x3 products are credited once."""
    L, nh = w["L"], w["nh"]
    return 3 * 2 * L * L * ((2 + nh) + (2 + nh) + (1 + nh))


def run_train(args, w, rank, world, local_rank):
    """`--mode train`: one diffusion training step (fused noising, 3 forwards, score-matching loss, backward, Adam) per
    minibatch of B latent rows per GPU at the workload's layer shape; data-parallel over `world` GPUs exactly like
    sdrm_b200.distributed.dp_train_step (5-scalar statistics all-reduce + flat gradient all-reduce over NCCL)."""
    import torch
    import torch.distributed as dist
    from sdrm_b200 import distributed as sd
    from sdrm_b200.models import make_schedule
    from sdrm_b200.training import DiffusionTrainStep

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B = args.rows or args.train_batch
    diff, _ = build_models(dict(w, I=64, H=64), dev)     # the VAE is not part of the step (mu is an input)
    diff.train()
    _, _, ab_t = make_schedule(w["T"], device=dev)
    group = dist.group.WORLD if world > 1 else None

    def make(passes):
        st = DiffusionTrainStep(diff, ab_t, w["T"], w["nd"], group=group, seed=77, gemm_passes=passes)
        st.row_offset = rank * B
        opt = torch.optim.Adam(diff.parameters(), lr=1e-5, weight_decay=1e-4, eps=1e-8)
        return st, opt

    torch.manual_seed(1 + rank)
    mu_host = torch.randn(B, w["L"]).pin_memory()
    mu = mu_host.to(dev)

    def step(st, opt, src):
        opt.zero_grad(set_to_none=False)
        loss = st.loss(src if src.is_cuda else src.to(dev, non_blocking=True))
        loss.backward()
        sd.allreduce_gradients(diff, group)
        opt.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(passes, steps, src):
        st, opt = make(passes)
        for _ in range(args.warmup):
            step(st, opt, src)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            loss = step(st, opt, src)
        e1.record()
        if not src.is_cuda:
            float(loss.item())     # e2e: the loss scalar comes back to the host (train_SDRM.py:335)
        barrier()
        wall = time.perf_counter() - t0
        ms = torch.tensor([e0.elapsed_time(e1), wall * 1e3], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms[0].item()), float(ms[1].item()), float(loss.item())

    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    from sdrm_b200 import _lib as _l
    _l.load().sdrm_train_launch_count(1)
    ms3, _, loss3 = timed(3, args.steps, mu)
    # our kernels inside the timed steps: the GEMM-side launches are counted by the library (warm-up steps included, hence the
    # scaling), plus noise_inputs, loss_stats and loss_grad_seeds of every step
    launches = int(_l.load().sdrm_train_launch_count(1)) * args.steps // (args.steps + args.warmup) + 3 * args.steps
    clock_info = clocks.stop() if rank == 0 else None
    ms1, _, _ = timed(1, args.steps, mu)
    ms0, _, loss0 = timed(0, args.steps, mu)
    _, wall_e2e, _ = timed(3, max(args.e2e_steps, 5), mu_host)
    e2e_steps = max(args.e2e_steps, 5)
    if rank == 0:
        peaks = measured_peaks()
        F = train_flops_per_row(w) * B
        rows_s = world * B * args.steps / (ms3 * 1e-3)
        ach = F * args.steps / (ms3 * 1e-3) / 1e12
        line = {
            "metric": "diffusion training rows/sec (noising + 3 forwards + loss + backward + Adam)", "value": rows_s, "unit": "rows/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms3 / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16x3 (fp32-grade split products), fp32 accumulate",
            "data": "synthetic (random-init denoiser of the named shape, N(0,1) latents, in-kernel Philox noise / t)",
            "config": {"workload": args.workload + "-train", "rows_per_gpu": B, **{k: w[k] for k in ("L", "T", "nh", "nd")},
                       "l2": "every step streams > 1 GB of activations (rows x L x 4 B per layer, >> 126 MB L2)"},
            "clocks": clock_info,
            "e2e": {"value": world * B * e2e_steps / (wall_e2e * 1e-3), "unit": "rows/s", "h2d_bytes_per_step": B * w["L"] * 4,
                    "d2h_bytes_per_step": 4, "steps": e2e_steps,
                    "note": "latent minibatch uploaded from pinned host memory every step, loss scalar read back; wall clock"},
            "gpu_launches": launches,
            "roofline": {"bound": "tensor", "achieved": ach, "peak": peaks["tflops"], "unit": "TFLOP/s", "frac": ach / peaks["tflops"],
                         "traffic": None, "kernel": "sdrm_gemm_pair_kernel (bf16x3: executes 3x the credited products)",
                         "flops_per_row": train_flops_per_row(w), "peak_source": peaks["source"] + " sustained bf16"},
            "variants": {"bf16x3_ms_per_step": ms3 / args.steps, "bf16_single_pass_ms_per_step": ms1 / args.steps,
                         "torch_cublas_fp32_ms_per_step": ms0 / args.steps, "loss_bf16x3": loss3, "loss_torch": loss0},
            "cpu_baseline": None,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line goes to the real stdout; everything else (NCCL banners, warnings) was moved to stderr."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)   # libraries that print to fd 1 (NCCL version banner) must not pollute the JSON contract
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--mode", choices=["sample", "train"], default="sample", help="train: one diffusion training step per minibatch")
    ap.add_argument("--train-batch", type=int, default=16384, help="--mode train: minibatch rows per GPU")
    ap.add_argument("--workload", choices=sorted(WORKLOADS), default="cfg5")
    ap.add_argument("--rows", type=int, default=None, help="override users per GPU")
    ap.add_argument("--cpu-rows", type=int, default=None, help="rows of the CPU baseline sample")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the side measurements (random mode, K3, K4, K2) of the default run")
    ap.add_argument("--no-eager", action="store_true", help="--impl reference: skip the eager-CUDA run of the reference")
    ap.add_argument("--eager-rows", type=int, default=None, help="--impl reference: rows of the eager-CUDA sample")
    ap.add_argument("--cluster", type=int, default=0, help="force single CTAs (1), tcgen05 CTA pairs (2) or column-split clusters (4, 8); 0 = auto")
    ap.add_argument("--subtiles", type=int, default=0, help="row tiles a CTA pair interleaves (1, 2); 0 = auto")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the logits of the last step (a fixed sample of rows, <= 64 MB) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.mode != "sample"):
        ap.error("--dump-outputs writes the output of the sampling path (--impl ours --mode sample)")
    w = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if args.impl == "reference":
        run_reference(args, w, rank)
        return
    if world != args.gpus and args.gpus > 1:
        raise SystemExit(f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})")
    if args.mode == "train":
        run_train(args, w, rank, world, local_rank)
        return
    run_ours(args, w, rank, world, local_rank)


if __name__ == "__main__":
    main()
