"""Test-side restatement of the fidelity audit (sdrm_b200/fidelity.py, K9) on dense 0/1 matrices, in float64 torch.

Item and user ones are column and row sums; the pair counts c = X^T X are exact in float64 (counts <= 2^20).  phi follows the
definition: (U c_ij - a_i a_j) / (sqrt(v_i) sqrt(v_j)), v = a (U - a), and 0 where v_i = 0 or v_j = 0.  The six sums run over
the pairs i < j."""
import numpy as np
import torch

from sdrm_b200.fidelity import FidelityReport


def _dense(X, device):
    t = torch.as_tensor(np.asarray(X) if not isinstance(X, torch.Tensor) else X)
    return (t != 0).to(device=device, dtype=torch.float64)


def phi_matrix(X, device="cpu"):
    """float64 [I, I] phi of the item columns of X [U, I]."""
    Xt = _dense(X, device)
    U = Xt.shape[0]
    a = Xt.sum(0)
    c = Xt.T @ Xt
    v = a * (U - a)
    num = U * c - a[:, None] * a[None, :]
    den = torch.sqrt(v)[:, None] * torch.sqrt(v)[None, :]
    return torch.where(den > 0, num / torch.where(den > 0, den, torch.ones_like(den)), torch.zeros_like(num))


def pair_sums(R, S, device="cpu"):
    """float64 [6]: sum d^2, sum phiR, sum phiS, sum phiR^2, sum phiS^2, sum phiR phiS over i < j (d = phiR - phiS)."""
    pr, ps = phi_matrix(R, device), phi_matrix(S, device)
    iu = torch.triu_indices(pr.shape[0], pr.shape[0], offset=1, device=pr.device)
    r, s = pr[iu[0], iu[1]], ps[iu[0], iu[1]]
    d = r - s
    return torch.stack([(d * d).sum(), r.sum(), s.sum(), (r * r).sum(), (s * s).sum(), (r * s).sum()]).cpu()


def report(R, S, k=None, device="cpu"):
    """The FidelityReport compare(R, S, k) should give, with host tensors (neighbours from the K8 test oracle)."""
    Rt, St = _dense(R, device), _dense(S, device)
    nb_r = nb_s = None
    if k is not None:
        from privacy_oracle import nearest_oracle
        from sdrm_b200.privacy import NearestRows
        nb = []
        for X in (Rt, St):
            idx, c, u = nearest_oracle(X.T, X.T, k, exclude_same_index=True, device=device)
            nb.append(NearestRows(idx, c, u, X.sum(0).to(torch.int32).cpu()))
        nb_r, nb_s = nb
    return FidelityReport(Rt.sum(0).to(torch.int32).cpu(), St.sum(0).to(torch.int32).cpu(), Rt.sum(1).to(torch.int32).cpu(),
                          St.sum(1).to(torch.int32).cpu(), pair_sums(Rt, St, device), nb_r, nb_s)
