"""Python owner of one sdrm_handle: packs the denoiser / decoder weights into the CUDA library and runs
the persistent reverse-diffusion kernel.  All tensors are torch-owned; the handle only keeps its packed
copies (include/sdrm_b200.h).  No CPU path: a CPU tensor or a missing library raises.
"""
import ctypes as C

import torch

from . import _lib


def _f32c(t):
    if t is None:
        return None
    if t.dtype != torch.float32 or not t.is_contiguous():
        t = t.detach().to(torch.float32).contiguous()
    return t.detach()


class SamplerEngine:
    def __init__(self, device=None):
        if not torch.cuda.is_available():
            raise _lib.SdrmError("SDRM sampling needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        h = C.c_void_p()
        _lib.check(self.lib.sdrm_create(C.byref(h), self.device.index or 0), "sdrm_create")
        self.handle = h
        self._den_key = None
        self._dec_key = None
        self._ws = None
        self._grid = None          # (timesteps, eta) of the step grid set on the handle; None = the full chain
        self.T = self.L = self.I = None

    def __del__(self):
        try:
            if getattr(self, "handle", None):
                self.lib.sdrm_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    # ---------------------------------------------------------------------------------------------
    # Weight packing.  The packed images are rebuilt on EVERY call by default: the pack kernels cost ~0.1 ms, and no host-side
    # key can see an in-place edit through `.data` (EMA swaps, `p.data.copy_()`, a new module allocated at recycled addresses
    # with the same version counters), which would silently sample from stale weights.  A caller that guarantees unchanged
    # weights between calls (e.g. main.py's two samplings of one trained model) may opt into reuse with `reuse_packed=True`;
    # `invalidate()` drops the cached key.  Nothing here reads device memory on the host (no hidden synchronisation).
    @staticmethod
    def _key(tensors, extra):
        return tuple((t.data_ptr(), t._version, tuple(t.shape)) for t in tensors if t is not None) + tuple(extra)

    def invalidate(self):
        self._den_key = None
        self._dec_key = None

    def pack_denoiser(self, diff_net, schedule, noise_divider, force=True):
        """diff_net: sdrm_b200.models.SDRM (or any module with the same layer_tensors()); schedule = (b_t,a_t,ab_t).
        force=False skips the re-pack when the parameter tensors (address, version counter, shape) and the schedule tensors
        are the ones packed last time."""
        lt = diff_net.layer_tensors()
        T = diff_net.EMB_DIM
        D, in_dim = lt["W0"].shape
        L = in_dim - T
        nh = diff_net.n_hidden_layers
        for s_ in schedule:
            if s_.numel() != T + 1:
                raise ValueError(f"schedule tensors must have T+1={T + 1} entries, got {s_.numel()}")
        key = self._key(list(lt.values()) + list(schedule), (float(noise_divider), T, L, D, nh))
        if not force and key == self._den_key:
            return
        sched = torch.cat([s_.detach().to(self.device, torch.float32).reshape(-1) for s_ in schedule]).contiguous()
        ts = {k: (_f32c(v.to(self.device)) if v is not None else None) for k, v in lt.items()}
        st = _lib.stream_ptr()
        rc = self.lib.sdrm_denoiser_pack(
            self.handle, _lib.ptr(ts["We"]), _lib.ptr(ts["be"]), _lib.ptr(ts["W0"]), _lib.ptr(ts["b0"]),
            _lib.ptr(ts["a0"]), _lib.ptr(ts["Wh"]), _lib.ptr(ts["bh"]), _lib.ptr(ts["ah"]), _lib.ptr(ts["Wo"]),
            _lib.ptr(ts["bo"]), _lib.ptr(sched), T, L, D, nh, float(noise_divider), st)
        _lib.check(rc, "sdrm_denoiser_pack")
        self._keepalive_den = (ts, sched)
        self._den_key = key
        self._grid = None          # (the pack resets the handle to the full chain)
        self.T, self.L = T, L

    @property
    def steps(self):
        """Reverse steps of the next sample(): S of the step grid, else T."""
        return self.T if self._grid is None else len(self._grid[0])

    def set_step_grid(self, timesteps=None, eta=None):
        """Run the chain on the timesteps 1 <= tau_1 < ... < tau_S <= T (a sequence of ints) instead of all T: strided DDPM when
        eta is None, DDIM with noise scale eta in [0, 1] otherwise (include/sdrm_b200.h, sdrm_set_step_grid).  timesteps=None
        restores the full chain.  Stays set until the next call or the next pack of the denoiser; a call that repeats the grid
        already set launches nothing.  t_start entries of sample() are then grid steps in [0, S], and injected z / keep slabs
        are [S+1, n, L]."""
        if self._den_key is None:
            raise _lib.SdrmError("pack_denoiser must be called before set_step_grid")
        grid = None if timesteps is None else (tuple(int(t) for t in timesteps), None if eta is None else float(eta))
        if grid == self._grid:
            return
        if grid is None:
            rc = self.lib.sdrm_set_step_grid(self.handle, None, 0, 0, 0.0, _lib.stream_ptr())
        else:
            tau, e = grid
            arr = (C.c_int32 * len(tau))(*tau)
            rc = self.lib.sdrm_set_step_grid(self.handle, arr, len(tau), 0 if e is None else 1, 0.0 if e is None else e,
                                             _lib.stream_ptr())
        _lib.check(rc, "sdrm_set_step_grid")
        self._grid = grid

    def pack_decoder(self, vae_net, force=True):
        W1, b1 = vae_net.decoder[0].weight, vae_net.decoder[0].bias
        W2, b2 = vae_net.decoder[2].weight, vae_net.decoder[2].bias
        H, L = W1.shape
        I = W2.shape[0]
        key = self._key([W1, b1, W2, b2], (L, H, I))
        if not force and key == self._dec_key:
            return
        ts = [_f32c(t.to(self.device)) for t in (W1, b1, W2, b2)]
        rc = self.lib.sdrm_decoder_pack(self.handle, *[_lib.ptr(t) for t in ts], L, H, I, _lib.stream_ptr())
        _lib.check(rc, "sdrm_decoder_pack")
        self._keepalive_dec = ts
        self._dec_key = key
        self.I = I

    # ---------------------------------------------------------------------------------------------
    def workspace(self, n):
        need = self.lib.sdrm_sample_workspace_bytes(self.handle, n)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._ws, need

    def sample(self, n, row_offset=0, t_start=None, row_ids=None, seed=0, out=None, latent_out=None, inj_xT=None, inj_z=None,
               inj_keep=None, check=False):
        """Run the chain + decode for n rows; returns logits [n, I] on the device, fp32 unless `out` is a bfloat16 tensor: then
        every logit is the round-to-nearest-even bfloat16 of the fp32 value (sdrm_sample_bf16), at half the bytes."""
        if self._den_key is None or self._dec_key is None:
            raise _lib.SdrmError("pack_denoiser / pack_decoder must be called before sample")
        if out is None:
            out = torch.empty((n, self.I), dtype=torch.float32, device=self.device)
        if out.device.type != "cuda":
            raise _lib.SdrmError("out must be a CUDA tensor (no CPU fallback)")
        if (out.dtype not in (torch.float32, torch.bfloat16) or out.dim() != 2 or out.stride(1) != 1 or out.shape[0] < n
                or out.shape[1] < self.I):
            raise ValueError("out must be float32 or bfloat16 [>=n, >=I] with unit column stride")
        if n == 0:
            return out
        ws, need = self.workspace(n)
        if t_start is not None:
            if t_start.numel() != n:
                raise ValueError("t_start must have n entries")
            if t_start.device.type == "cpu" and t_start.numel() and (int(t_start.min()) < 0 or int(t_start.max()) > self.steps):
                raise ValueError(f"t_start entries must lie in [0, {self.steps}] (the chain's steps)")   # (device tensors are clamped by the kernel)
            t_start = t_start.to(self.device, torch.int32).contiguous()
        if row_ids is not None:
            row_ids = row_ids.to(self.device, torch.int32).contiguous()
            if row_ids.numel() != n:
                raise ValueError("row_ids must have n entries")
        for name, t, dt in (("inj_xT", inj_xT, torch.float32), ("inj_z", inj_z, torch.float32),
                            ("inj_keep", inj_keep, torch.uint8)):
            if t is not None and (t.dtype != dt or not t.is_contiguous() or t.device != self.device):
                raise ValueError(f"{name} must be a contiguous {dt} tensor on {self.device}")
        entry = self.lib.sdrm_sample_bf16 if out.dtype == torch.bfloat16 else self.lib.sdrm_sample
        rc = entry(self.handle, n, row_offset, _lib.ptr(t_start), _lib.ptr(row_ids), seed & (2 ** 64 - 1),
                   _lib.ptr(latent_out), _lib.ptr(out), out.stride(0), _lib.ptr(inj_xT),
                   _lib.ptr(inj_z), _lib.ptr(inj_keep), _lib.ptr(ws), need, _lib.stream_ptr())
        _lib.check(rc, "sdrm_sample_bf16" if out.dtype == torch.bfloat16 else "sdrm_sample")
        if check:
            _lib.check(self.lib.sdrm_check_device_error(self.handle, _lib.stream_ptr()), "sdrm_sample (device)")
        return out

    def set_option(self, option, value):
        """Per-handle tuning option (include/sdrm_b200.h enum sdrm_option; _lib.OPT_*).  0 = automatic."""
        _lib.check(self.lib.sdrm_set_option(self.handle, int(option), int(value)), "sdrm_set_option")

    def launch_count(self):
        return int(self.lib.sdrm_last_launch_count(self.handle))
