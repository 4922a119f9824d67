"""GPU, NCCL, world_size 2 (skipped on a one-GPU box): data-parallel diffusion training with the CUDA loss kernels and the tcgen05
training GEMMs under a process group (global statistics all-reduce + flat gradient all-reduce, SURVEY 8e), row-sharded sampling,
and the bit-packed gather of the synthetic rows -- against the single-process reference golden / a single-GPU run."""
import os
import socket
import tempfile

import pytest
import torch

from conftest import load_golden

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        import sys
        sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
        from helpers import modules_from_golden, random_modules
        from oracle import sdrm_oracle as orc
        from sdrm_b200 import distributed as sdd
        from sdrm_b200.training import DiffusionTrainStep
        g = load_golden("t_nh2_T7_L24")
        diff, _ = modules_from_golden(g, dev)
        diff.train()
        _, _, ab_t = orc.make_schedule(g["T"])
        stepper = DiffusionTrainStep(diff, ab_t.to(dev), g["T"], g["nd"], seed=1)      # CudaLossBackend + tcgen05 GEMMs
        opt = torch.optim.SGD(diff.parameters(), lr=0.0)
        loss = sdd.dp_train_step(stepper, opt, g["mu"].to(dev), g["t"].to(dev), inj_noise=g["noise"].to(dev), inj_masks=g["keeps"].to(dev))
        grads = {k: p.grad.detach().cpu() for k, p in diff.named_parameters()}
        # row-sharded sampling + bit-packed gather vs what a single GPU produces for all rows
        n, I, H, L, T, nh, nd = 301, 190, 48, 72, 6, 1, 1.0
        dn, vae = random_modules(I, H, L, T, nh, seed=3, device=dev)
        rows, span = sdd.sample_ddpm_sharded(n, dn, vae, L, nd, n_timesteps=T, seed=55, gather=True)
        pm, _ = sdd.sample_ddpm_sharded(n, dn, vae, L, nd, n_timesteps=T, seed=55, gather="bits", sparsity=0.9)
        rnd, _ = sdd.sample_ddpm_sharded(n, dn, vae, L, nd, timesteps="random", n_timesteps=T, seed=56, gather=True)
        torch.save((rank, float(loss), grads, rows.cpu(), span, pm.bits.cpu(), float(pm.threshold), int(pm.ones.item()), rnd.cpu()),
                   os.path.join(out_dir, f"rank{rank}.pt"))
    except Exception:
        import traceback
        with open(os.path.join(out_dir, f"rank{rank}.err"), "w") as fh:
            fh.write(traceback.format_exc())
        raise
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_rank_nccl_training_and_sharded_sampling():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import numpy as np
    import torch.multiprocessing as mp
    from helpers import random_modules
    from sdrm_b200.sparsify import equal_sparsity_device
    from sdrm_b200.train_SDRM import sample_ddpm
    world = 2
    ctx = mp.get_context("spawn")
    port = _free_port()
    out_dir = tempfile.mkdtemp(prefix="sdrm_dp_gpu_")
    procs = [ctx.Process(target=_worker, args=(r, world, port, out_dir)) for r in range(world)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(280)
    for r, p in enumerate(procs):
        err = os.path.join(out_dir, f"rank{r}.err")
        assert p.exitcode == 0, open(err).read() if os.path.exists(err) else f"rank {r} exit code {p.exitcode}"
    res = [torch.load(os.path.join(out_dir, f"rank{r}.pt"), weights_only=False) for r in range(world)]
    g = load_golden("t_nh2_T7_L24")
    # single-GPU truth for the sampling part
    n, I, H, L, T, nh, nd = 301, 190, 48, 72, 6, 1, 1.0
    dn, vae = random_modules(I, H, L, T, nh, seed=3, device="cuda")
    whole = sample_ddpm(n, dn, vae, L, nd, n_timesteps=T, seed=55)
    pm1 = equal_sparsity_device(whole, 0.9)
    t_all = np.random.RandomState(56).randint(1, T, size=n).astype(np.int32)
    rnd1 = sample_ddpm(n, dn, vae, L, nd, timesteps="random", n_timesteps=T, seed=56, t_rows=t_all)
    for rank, loss, grads, rows, span, bits, thr, ones, rnd in res:
        assert abs(loss - g["loss_ref"].item()) <= 2e-5 * abs(g["loss_ref"].item())
        for k, gref in g["grads_ref"].items():
            assert (grads[k] - gref).abs().max().item() <= 2e-4 * (gref.abs().max().item() + 1e-12), (rank, k)
        assert span == (0, n) and torch.equal(rows, whole.cpu())
        assert thr == float(pm1.threshold) and ones == int(pm1.ones.item()) and torch.equal(bits, pm1.bits.cpu())
        assert torch.equal(rnd, rnd1.cpu())
