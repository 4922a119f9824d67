"""Test-side restatement of the nearest-rows search (sdrm_b200/privacy.py, K8) on dense 0/1 matrices.

c = Q @ R^T in float64 is exact (counts <= 2^20 < 2^53).  J = c / u is then taken in float64: IEEE division is correctly rounded,
so equal fractions give equal doubles, and two different fractions with u <= 2^21 differ by at least 2^-42 relative, far above
the 2^-53 rounding, so the float64 order is the exact rational order.  u = 0 gives J = 1; an excluded pair gets J = -1 and sorts
last.  A stable descending sort keeps equal J in index order (ties to the lower index)."""
import numpy as np
import torch


def nearest_oracle(Q, R, k, exclude_same_index=False, q_index_offset=0, device="cpu", chunk=1024):
    """Q [n, I], R [m, I] 0/1 (any dtype, nonzero = 1) -> (index int64 [n, k], c int32 [n, k], u int32 [n, k])."""
    Qt = (torch.as_tensor(np.asarray(Q) if not isinstance(Q, torch.Tensor) else Q) != 0).to(device=device, dtype=torch.float64)
    Rt = (torch.as_tensor(np.asarray(R) if not isinstance(R, torch.Tensor) else R) != 0).to(device=device, dtype=torch.float64)
    a, b = Qt.sum(1), Rt.sum(1)
    m = Rt.shape[0]
    out_i, out_c, out_u = [], [], []
    for s in range(0, Qt.shape[0], chunk):
        c = Qt[s:s + chunk] @ Rt.T
        u = a[s:s + chunk, None] + b[None, :] - c
        j = torch.where(u == 0, torch.ones_like(u), c / u.clamp_min(1))
        if exclude_same_index:
            rows = torch.arange(s, s + c.shape[0], device=device) + q_index_offset
            hit = rows < m
            j[torch.nonzero(hit).flatten(), rows[hit]] = -1.0
        order = torch.sort(j, dim=1, descending=True, stable=True).indices[:, :k]
        out_i.append(order.cpu())
        out_c.append(torch.gather(c, 1, order).to(torch.int32).cpu())
        out_u.append(torch.gather(u, 1, order).to(torch.int32).cpu())
    if not out_i:
        z = torch.zeros((0, k), dtype=torch.int32)
        return z.long(), z, z
    return torch.cat(out_i), torch.cat(out_c), torch.cat(out_u)


def random_rows(rng, rows, items, density):
    return (rng.random((rows, items)) < density).astype(np.uint8)
