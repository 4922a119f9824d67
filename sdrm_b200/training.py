"""The diffusion training step (reference: train_SDRM.py:321-337 + score_matching_loss 191-199).

Per minibatch of latents mu = VAE.encode(x):
  1. K2 `sdrm_noise_inputs`  : noise, x_t = sqrt(ab_t) mu + (1-ab_t) noise, x_p = mu + .1 noise and the three
                               dropout-scaled denoiser inputs, one fused pass (in-kernel Philox);
  2. the three denoiser forwards run as ONE [3B, L] batch through the shared MLP (rows are independent, so
     this is the same arithmetic); every dense product of the forward AND the backward runs on the hand-written
     tcgen05 GEMM (`DenoiserGemms` -> C ABI `sdrm_denoiser_fwd/bwd`, bf16x3 split operands, fp32 accumulate);
  3. K2 `sdrm_loss_stats` + `sdrm_loss_grad_seeds`: five fp64 partial sums -> (optional all-reduce over the
     data-parallel group: the loss divides by the GLOBAL-batch variance, SURVEY.md §8e) -> scalar loss and
     the closed-form gradient seeds, wrapped in a torch.autograd.Function.
"""
import torch

from . import _lib


class CudaLossBackend:
    """Calls the C ABI.  Tests may substitute an object with the same three methods."""

    def __init__(self):
        self.lib = _lib.load()

    def noise_inputs(self, mu, t, ab_t, nd, mu_coef, seed, row_offset, inj_noise=None, inj_masks=None, want_masks=False):
        B, L = mu.shape
        outs = [torch.empty_like(mu) for _ in range(4)]
        masks = torch.empty((3, B, L), dtype=torch.uint8, device=mu.device) if want_masks else None
        rc = self.lib.sdrm_noise_inputs(_lib.ptr(mu), _lib.ptr(t), _lib.ptr(ab_t), B, L, float(nd), float(mu_coef),
                                        seed & (2 ** 64 - 1), int(row_offset), _lib.ptr(inj_noise), _lib.ptr(inj_masks),
                                        _lib.ptr(outs[0]), _lib.ptr(outs[1]), _lib.ptr(outs[2]), _lib.ptr(outs[3]),
                                        _lib.ptr(masks), _lib.stream_ptr())
        _lib.check(rc, "sdrm_noise_inputs")
        return outs[0], outs[1], outs[2], outs[3], masks

    def stats(self, pred, sx, psx, mu, mu_coef):
        st = torch.zeros(5, dtype=torch.float64, device=pred.device)
        rc = self.lib.sdrm_loss_stats(_lib.ptr(pred), _lib.ptr(sx), _lib.ptr(psx), _lib.ptr(mu), pred.numel(),
                                      float(mu_coef), _lib.ptr(st), _lib.stream_ptr())
        _lib.check(rc, "sdrm_loss_stats")
        return st

    def seeds(self, pred, sx, psx, mu, mu_coef, stats):
        g = [torch.empty_like(pred) for _ in range(3)]
        loss = torch.empty(1, dtype=torch.float32, device=pred.device)
        rc = self.lib.sdrm_loss_grad_seeds(_lib.ptr(pred), _lib.ptr(sx), _lib.ptr(psx), _lib.ptr(mu), pred.numel(),
                                           float(mu_coef), _lib.ptr(stats), _lib.ptr(g[0]), _lib.ptr(g[1]), _lib.ptr(g[2]),
                                           _lib.ptr(loss), _lib.stream_ptr())
        _lib.check(rc, "sdrm_loss_grad_seeds")
        return g[0], g[1], g[2], loss


class MultinomialNLL(torch.autograd.Function):
    """neg_ll = -mean_r(sum_j log_softmax(logits)[r, j] * X[r, j])  (reference train_SDRM.py:143, MultiVAE++ training step)
    as two fused passes (kernels `sdrm_multinomial_nll_fwd/bwd`): the [B, I] log_softmax and its autograd temporaries are
    never materialised; forward reads logits and X once, backward writes the logits gradient once."""

    @staticmethod
    def forward(ctx, logits, X):
        if logits.device.type != "cuda":
            raise _lib.SdrmError("multinomial_nll: logits must be a CUDA tensor (no CPU fallback)")
        lib = _lib.load()
        logits = logits if (logits.dtype == torch.float32 and logits.stride(1) == 1) else logits.float().contiguous()
        X = X if (X.dtype == torch.float32 and X.stride(1) == 1) else X.float().contiguous()
        rows, n_items = logits.shape
        if X.shape != logits.shape:
            raise ValueError("logits and X must have the same [rows, items] shape")
        lse, sx, dot = (torch.empty(rows, dtype=torch.float32, device=logits.device) for _ in range(3))
        _lib.check(lib.sdrm_multinomial_nll_fwd(_lib.ptr(logits), _lib.ptr(X), rows, n_items, logits.stride(0), X.stride(0),
                                                _lib.ptr(lse), _lib.ptr(sx), _lib.ptr(dot), _lib.stream_ptr()),
                   "sdrm_multinomial_nll_fwd")
        ctx.save_for_backward(logits, X, lse, sx)
        return -(dot - sx * lse).mean()

    @staticmethod
    def backward(ctx, grad_out):
        logits, X, lse, sx = ctx.saved_tensors
        lib = _lib.load()
        rows, n_items = logits.shape
        grad = torch.empty_like(logits, memory_format=torch.contiguous_format)
        g = grad_out.detach().to(torch.float32).contiguous()
        _lib.check(lib.sdrm_multinomial_nll_bwd(_lib.ptr(logits), _lib.ptr(X), rows, n_items, logits.stride(0), X.stride(0),
                                                _lib.ptr(lse), _lib.ptr(sx), _lib.ptr(g), 1.0 / rows, _lib.ptr(grad),
                                                grad.stride(0), _lib.stream_ptr()), "sdrm_multinomial_nll_bwd")
        return grad, None


def multinomial_nll(logits, X):
    return MultinomialNLL.apply(logits, X)


class FrozenEncoder:
    """mu = VAE.encode(x)[0] of the FROZEN, eval-mode VAE for sparse interaction batches (train_SDRM.py:291-294, 323-324).

    The reference densifies every minibatch (`x.to_dense()`: [B, I] floats, 29 MB per step at adm) and runs the first
    encoder Linear as a dense GEMM over mostly-zero columns.  Here the first layer is kernel `sdrm_encode_csr` (gather-sum
    of the row's items over W_e1^T, L2-normalisation and tanh fused); the small second layer [B, H] x [H, L] stays a library
    GEMM and only its mu half is computed (logvar and the KL term are discarded by the caller, is_training == 0).
    The reference's eval-mode encode also draws an unused randn_like(std); that RNG side effect is not reproduced.
    """

    def __init__(self, vae):
        self.lib = _lib.load()
        lin1, lin2 = vae.encoder[0], vae.encoder[2]
        L = vae.latent_dim
        self.n_items, self.H, self.L = lin1.weight.shape[1], lin1.weight.shape[0], L
        self.W1T = lin1.weight.detach().t().contiguous().float()      # [I, H]; the VAE is frozen: transposed once
        self.b1 = lin1.bias.detach().contiguous().float()
        self.W2mu = lin2.weight.detach()[:L].t().contiguous().float() # [H, L]
        self.b2mu = lin2.bias.detach()[:L].contiguous().float()

    def hidden(self, x):
        dev = self.W1T.device
        if dev.type != "cuda":
            raise _lib.SdrmError("FrozenEncoder: the VAE must live on a CUDA device (no CPU fallback)")
        if x.layout == torch.sparse_csr:
            # a torch CSR tensor may store one column twice in a row; to_dense() adds such entries, and the kernel's L2 norm
            # must be that of the sum, so the entries are summed first (to_sparse_coo() marks its result coalesced as is)
            coo = x.to_sparse_coo()
            csr = torch.sparse_coo_tensor(coo.indices(), coo.values(), coo.shape).coalesce().to_sparse_csr()
        elif x.layout == torch.sparse_coo:
            csr = x.coalesce().to_sparse_csr()
        else:
            csr = x.to_sparse_csr()
        csr = csr.to(dev)
        if csr.shape[1] != self.n_items:
            raise ValueError(f"batch has {csr.shape[1]} items, the encoder expects {self.n_items}")
        indptr = csr.crow_indices().to(torch.int64).contiguous()
        indices = csr.col_indices().to(torch.int64).contiguous()
        values = csr.values().to(torch.float32).contiguous()
        rows = csr.shape[0]
        out = torch.empty((rows, self.H), dtype=torch.float32, device=dev)
        _lib.check(self.lib.sdrm_encode_csr(_lib.ptr(indptr), _lib.ptr(indices), _lib.ptr(values), rows, self.n_items,
                                            _lib.ptr(self.W1T), _lib.ptr(self.b1), self.H, _lib.ptr(out), _lib.stream_ptr()),
                   "sdrm_encode_csr")
        return out

    @torch.no_grad()
    def __call__(self, x):
        return torch.addmm(self.b2mu, self.hidden(x), self.W2mu)


class DenoiserGemms(torch.autograd.Function):
    """eps_theta for the batched [3B, L] rows with every dense product on the hand-written tcgen05 GEMM
    (C ABI `sdrm_denoiser_fwd` / `sdrm_denoiser_bwd`, csrc/train_gemm.cu).  Reference: SDRM.forward (train_SDRM.py:97-103)
    called three times by score_matching_loss (191-199) and differentiated by autograd (336).

    The time embedding enters as a hoisted table (table[i] = W0[:, L:] (We temb(i) + be) + b0, built by the caller in torch
    so that autograd carries d table back to We, be, W0[:, L:] and b0): layer 0 is a K = L product plus a gathered bias row.
    """

    @staticmethod
    def forward(ctx, x, t, table, W0, a0, Wh, bh, ah, Wo, bo, L, nh, passes):
        lib = _lib.load()
        if x.device.type != "cuda":
            raise _lib.SdrmError("DenoiserGemms: CUDA tensors required (no CPU fallback)")
        x = x.detach().contiguous().float()
        t = t.detach().to(torch.int64).contiguous()
        rows, D = x.shape[0], W0.shape[0]
        tens = [v.detach() if v is not None else None for v in (table, W0, a0, Wh, bh, ah, Wo, bo)]
        table_, W0_, a0_, Wh_, bh_, ah_, Wo_, bo_ = [v.contiguous().float() if v is not None else None for v in tens]
        need = lib.sdrm_denoiser_train_workspace_bytes(rows, L, D, nh)
        if need == 0:
            raise _lib.SdrmError("sdrm_denoiser_train_workspace_bytes failed: " + lib.sdrm_last_error().decode())
        ws = torch.empty(need, dtype=torch.uint8, device=x.device)
        out = torch.empty((rows, L), dtype=torch.float32, device=x.device)
        st = _lib.stream_ptr()
        rc = lib.sdrm_denoiser_fwd(_lib.ptr(x), _lib.ptr(t), _lib.ptr(table_), table_.stride(0), _lib.ptr(W0_), W0_.stride(0),
                                   _lib.ptr(a0_), _lib.ptr(Wh_), _lib.ptr(bh_), _lib.ptr(ah_), _lib.ptr(Wo_), _lib.ptr(bo_),
                                   rows, L, D, nh, passes, _lib.ptr(out), _lib.ptr(ws), need, st)
        _lib.check(rc, "sdrm_denoiser_fwd")
        ctx.save_for_backward(x, t, out, a0_, Wh_, ah_, Wo_, ws)
        ctx.dims = (rows, L, D, nh, passes, table_.shape[0] - 1, W0.shape[1])
        return out

    @staticmethod
    def backward(ctx, g_out):
        lib = _lib.load()
        x, t, out, a0, Wh, ah, Wo, ws = ctx.saved_tensors
        rows, L, D, nh, passes, T, w0_cols = ctx.dims
        g_out = g_out.detach().contiguous().float()
        order = torch.argsort(t, stable=True).contiguous()
        offsets = torch.zeros(T + 2, dtype=torch.int64, device=t.device)
        offsets[1:] = torch.cumsum(torch.bincount(t, minlength=T + 1), 0)
        dev = x.device
        gW0 = torch.empty((D, L), dtype=torch.float32, device=dev)
        gTable = torch.empty((T + 1, D), dtype=torch.float32, device=dev)
        ga0 = torch.empty(1, dtype=torch.float32, device=dev)
        gWo = torch.empty((L, D), dtype=torch.float32, device=dev)
        gbo = torch.empty(L, dtype=torch.float32, device=dev)
        gWh = gbh = gah = None
        if nh > 0:
            gWh = torch.empty((D, D), dtype=torch.float32, device=dev)
            gbh = torch.empty(D, dtype=torch.float32, device=dev)
            gah = torch.empty(1, dtype=torch.float32, device=dev)
        rc = lib.sdrm_denoiser_bwd(_lib.ptr(g_out), _lib.ptr(out), _lib.ptr(x), _lib.ptr(order), _lib.ptr(offsets), T, _lib.ptr(a0),
                                   _lib.ptr(Wh), _lib.ptr(ah), _lib.ptr(Wo), rows, L, D, nh, passes, _lib.ptr(gW0), _lib.ptr(gTable),
                                   _lib.ptr(ga0), _lib.ptr(gWh), _lib.ptr(gbh), _lib.ptr(gah), _lib.ptr(gWo), _lib.ptr(gbo),
                                   _lib.ptr(ws), ws.numel(), _lib.stream_ptr())
        _lib.check(rc, "sdrm_denoiser_bwd")
        gW0_full = torch.zeros((D, w0_cols), dtype=torch.float32, device=dev)
        gW0_full[:, :L] = gW0
        return None, None, gTable, gW0_full, ga0, gWh, gbh, gah, gWo, gbo, None, None, None


def denoiser_gemms(net, x, t, passes=3):
    """SDRM.forward(x, t, prescaled=True) with the Linear layers on the tcgen05 GEMM; differentiable wrt net's parameters."""
    lt = net.layer_tensors()
    T = net.EMB_DIM
    L = lt["W0"].shape[1] - T
    steps = torch.arange(T + 1, device=x.device)
    emb = net.emb_layer(net.timestep_embedding(steps, T))                       # [T+1, T]   (tiny: stays in torch / autograd)
    table = torch.nn.functional.linear(emb, lt["W0"][:, L:], lt["b0"])         # [T+1, D]
    return DenoiserGemms.apply(x, t, table, lt["W0"], lt["a0"], lt["Wh"], lt["bh"], lt["ah"], lt["Wo"], lt["bo"],
                               L, net.n_hidden_layers, int(passes))


# --------------------------------------------------------------------------------------------------------------------
# torch.nn.Linear on the tcgen05 GEMM (MultiVAE++ training step, SURVEY.md 8f-3; reference train_SDRM.py:136-150, 210-215)
# --------------------------------------------------------------------------------------------------------------------
def _tc_gemm(A, trans_a, B, trans_b, bias, M, N, K, passes, splits):
    lib = _lib.load()
    need = lib.sdrm_gemm_workspace_bytes(M, N, K, splits)
    ws = torch.empty(need, dtype=torch.uint8, device=A.device)
    C_ = torch.empty((M, N), dtype=torch.float32, device=A.device)
    rc = lib.sdrm_gemm(_lib.ptr(A), A.stride(0), int(trans_a), _lib.ptr(B), B.stride(0), int(trans_b), _lib.ptr(bias), _lib.ptr(C_),
                       C_.stride(0), M, N, K, passes, splits, _lib.ptr(ws), need, _lib.stream_ptr())
    _lib.check(rc, "sdrm_gemm")
    return C_


class TcLinear(torch.autograd.Function):
    """y = x W^T + b with the forward product and both backward products (dx = dy W, dW = dy^T x) on the hand-written tcgen05
    GEMM (C ABI `sdrm_gemm`, bf16x3 split operands by default); db is a column sum."""

    @staticmethod
    def forward(ctx, x, W, b, passes):
        if x.device.type != "cuda":
            raise _lib.SdrmError("TcLinear: CUDA tensors required (no CPU fallback)")
        x_ = x.detach().float()
        x_ = x_ if x_.stride(-1) == 1 and x_.dim() == 2 else x_.reshape(-1, x.shape[-1]).contiguous()
        W_ = W.detach().float()
        W_ = W_ if W_.stride(1) == 1 else W_.contiguous()
        b_ = b.detach().float().contiguous() if b is not None else None
        M, K = x_.shape
        N = W_.shape[0]
        y = _tc_gemm(x_, False, W_, False, b_, M, N, K, passes, 1)
        ctx.save_for_backward(x_, W_)
        ctx.passes = passes
        ctx.has_bias = b is not None
        return y

    @staticmethod
    def backward(ctx, g):
        x_, W_ = ctx.saved_tensors
        g = g.detach().float()
        g = g if g.stride(1) == 1 else g.contiguous()
        M, K = x_.shape
        N = W_.shape[0]
        gx = gW = gb = None
        if ctx.needs_input_grad[0]:
            gx = _tc_gemm(g, False, W_, True, None, M, K, N, ctx.passes, 1)          # [M, K] = g [M, N] . W [N, K]
        if ctx.needs_input_grad[1]:
            gW = _tc_gemm(g, True, x_, True, None, N, K, M, ctx.passes, 0)           # [N, K] = g^T [N, M] . x [M, K]
        if ctx.has_bias and ctx.needs_input_grad[2]:
            gb = g.sum(0)
        return gx, gW, gb, None


def tc_linear(x, layer, passes=3):
    return TcLinear.apply(x, layer.weight, layer.bias, int(passes))


def vae_forward_tc(vae, X, passes=3):
    """VAE.forward (encode + reparameterise + decode + KL, train_SDRM.py:236-256) with the four Linear layers on the tcgen05
    GEMM; the elementwise pieces (normalise, dropout, tanh, KL, reparameterisation) stay torch ops under autograd.
    Same RNG draws as VAE.forward: the dropout mask, then randn_like(std)."""
    h = vae.dropout(torch.nn.functional.normalize(X, p=2, dim=1))
    h = torch.tanh(tc_linear(h, vae.encoder[0], passes))
    h = tc_linear(h, vae.encoder[2], passes)
    mu_q, logvar_q = torch.chunk(h, chunks=2, dim=1)
    kl = -0.5 * torch.mean(torch.sum(1 + logvar_q - mu_q.pow(2) - logvar_q.exp(), dim=1))
    z = vae.reparameterize(mu_q, logvar_q)
    d = torch.tanh(tc_linear(z, vae.decoder[0], passes))
    return tc_linear(d, vae.decoder[2], passes), kl


# --------------------------------------------------------------------------------------------------------------------
# device-resident CSR staging of the interaction matrix (SURVEY.md 8f-4; reference dataloaders.py:46-79, train_SDRM.py:136, 323)
# --------------------------------------------------------------------------------------------------------------------
class DeviceCSR:
    """The interaction matrix uploaded ONCE as CSR (int64 indptr / indices, fp32 values); minibatches are row-index slices
    taken on the device.  The reference converts every minibatch from scipy to a torch COO tensor on the host
    (`torch.LongTensor(tuple of ndarrays)`, dataloaders.py:54), ships it and densifies it."""

    def __init__(self, csr, device):
        csr = csr.tocsr()
        if not csr.has_canonical_format:   # repeated (row, column) entries are summed once here, like to_dense() would
            csr = csr.copy()
            csr.sum_duplicates()
        self.shape = csr.shape
        self.host_indptr = csr.indptr.astype("int64")
        self.indptr = torch.from_numpy(self.host_indptr).to(device)
        self.indices = torch.from_numpy(csr.indices.astype("int64")).to(device)
        self.values = torch.from_numpy(csr.data.astype("float32")).to(device)
        self.device = torch.device(device)

    def as_torch_csr(self):
        return torch.sparse_csr_tensor(self.indptr, self.indices, self.values, size=self.shape)

    def _gather(self, rows):
        """positions of the stored entries of `rows` (host int array / list): (row id inside the batch, position in indices)"""
        import numpy as np
        rows = np.asarray(rows, dtype=np.int64)
        lens = self.host_indptr[rows + 1] - self.host_indptr[rows]          # host copy of indptr: no device sync for the sizes
        total = int(lens.sum())
        r_dev = torch.from_numpy(rows).to(self.device)
        lens_dev = torch.from_numpy(lens).to(self.device)
        row_of = torch.repeat_interleave(torch.arange(len(rows), device=self.device), lens_dev, output_size=total)
        start_excl = torch.cumsum(lens_dev, 0) - lens_dev
        pos = self.indptr[r_dev][row_of] + (torch.arange(total, device=self.device) - start_excl[row_of])
        return row_of, pos, lens_dev

    def dense_rows(self, rows):
        """dense fp32 [len(rows), I] batch built on the device (duplicates add up, like to_dense() of a COO tensor)"""
        row_of, pos, _ = self._gather(rows)
        out = torch.zeros((len(rows), self.shape[1]), dtype=torch.float32, device=self.device)
        out.index_put_((row_of, self.indices[pos]), self.values[pos], accumulate=True)
        return out

    def csr_rows(self, rows):
        row_of, pos, lens_dev = self._gather(rows)
        indptr = torch.zeros(len(rows) + 1, dtype=torch.int64, device=self.device)
        indptr[1:] = torch.cumsum(lens_dev, 0)
        return torch.sparse_csr_tensor(indptr, self.indices[pos], self.values[pos], size=(len(rows), self.shape[1]))


def stage_loader(dl, device):
    """If `dl` is a torch DataLoader over a sdrm_b200.data.SparseDataset driven by a BatchSampler (what main.py builds,
    main.py:126-135), return (DeviceCSR of the whole dataset, the batch sampler): iterating the sampler yields exactly the
    index batches that iterating `dl` would have collated, without the per-batch host conversion.  Otherwise None."""
    ds = getattr(dl, "dataset", None)
    sampler = getattr(dl, "sampler", None)
    if ds is None or sampler is None or not hasattr(ds, "get_all_data") or not hasattr(sampler, "batch_size"):
        return None
    data, _ = ds.get_all_data()
    if not hasattr(data, "tocsr"):
        return None
    return DeviceCSR(data, device), sampler


class ScoreMatchingLoss(torch.autograd.Function):
    """loss = 0.5 (mean((sd-r)^2) + mean((r-sx)^2)) / (1e-8 + var(r)),  r = pred - mu, sd = (psx - sx)/mu_coef^2,
    with means / variance over the GLOBAL batch when `group` is a process group."""

    @staticmethod
    def forward(ctx, pred, sx, psx, mu, mu_coef, backend, group):
        pred, sx, psx, mu = (v.contiguous() for v in (pred, sx, psx, mu))
        stats = backend.stats(pred, sx, psx, mu, mu_coef)
        if group is not None:
            import torch.distributed as dist
            dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
        g_pred, g_sx, g_psx, loss = backend.seeds(pred, sx, psx, mu, mu_coef, stats)
        ctx.save_for_backward(g_pred, g_sx, g_psx)
        return loss.reshape(())

    @staticmethod
    def backward(ctx, grad_out):
        g_pred, g_sx, g_psx = ctx.saved_tensors
        return grad_out * g_pred, grad_out * g_sx, grad_out * g_psx, None, None, None, None


class DiffusionTrainStep:
    """Builds the loss of one minibatch; the caller does zero_grad / backward / optimizer.step like the reference."""

    def __init__(self, diff_net, ab_t, timesteps, noise_divider, mu_coef=0.1, group=None, backend=None, seed=None, gemm_passes=3):
        self.net = diff_net
        # dense layers: 3 = bf16x3 products on the tcgen05 GEMM (fp32-grade), 1 = plain bf16 operands, 0 = torch / cuBLAS
        # (kept for comparison runs and for the CPU test backend)
        self.gemm_passes = int(gemm_passes)
        self.ab_t = ab_t.detach().to(torch.float32).contiguous()
        self.T = int(timesteps)
        self.nd = float(noise_divider)
        self.mu_coef = mu_coef
        self.group = group
        self.backend = backend if backend is not None else CudaLossBackend()
        self.base_seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if seed is None else int(seed)
        self.step_index = 0
        self.row_offset = 0  # data-parallel ranks set this to their first global row of the minibatch

    def loss(self, mu, t=None, inj_noise=None, inj_masks=None):
        if isinstance(self.backend, CudaLossBackend) and mu.device.type != "cuda":
            raise _lib.SdrmError("the SDRM training step needs CUDA tensors (no CPU fallback)")
        mu = mu.detach().to(torch.float32).contiguous()
        B = mu.shape[0]
        if t is None:
            # CPU generator then .to(device), like the reference (train_SDRM.py:327)
            t = torch.randint(1, self.T + 1, (B,)).to(mu.device)
        t = t.to(mu.device, torch.int64).contiguous()
        seed = self.base_seed + self.step_index
        self.step_index += 1
        _, in_pert, in_clean, in_shift, _ = self.backend.noise_inputs(
            mu, t, self.ab_t.to(mu.device), self.nd, self.mu_coef, seed, self.row_offset, inj_noise, inj_masks)
        x3 = torch.cat([in_pert, in_clean, in_shift], dim=0)
        if self.gemm_passes and isinstance(self.backend, CudaLossBackend):
            out3 = denoiser_gemms(self.net, x3, t.repeat(3), self.gemm_passes)
        else:
            out3 = self.net(x3, t.repeat(3), prescaled=True)
        pred, sx, psx = out3[:B], out3[B:2 * B], out3[2 * B:]
        return ScoreMatchingLoss.apply(pred, sx, psx, mu, self.mu_coef, self.backend, self.group)
