"""fp64 autograd reference of the start gradient of the rollout scores (sb_rollout_score_grad_ics' grad_x0) — TEST
INFRASTRUCTURE ONLY.

The per-pair SSE is `rollout_fp64_ref.sse64`; the pairs are independent, so the gradient of their sum with respect to
x0 (N, d) is the per-pair ∂sse[n]/∂x0[n]. Nothing here imports the product. Callers hand in the fp32 tensors the kernel
sees; they are cast exactly to fp64.
"""
import torch

from rollout_fp64_ref import sse64


def grad_x0_64(x0, W, lib, dt, steps_per_row, y, method, rows=None):
    """(per-pair SSE (M, N), ∂sse[m, n]/∂x0 of the pair (M, N, d)), fp64. W (M, d, K); x0 (N, d) shared by the models or
    (M, N, d) per model; rows None or (M, N) rows compared per pair."""
    W = W.detach().to(torch.float64)
    M = W.shape[0]
    x0 = x0.detach().to(torch.float64)
    y = y.detach().to(torch.float64)
    sse, grads = [], []
    for m in range(M):
        xm = (x0[m] if x0.dim() == 3 else x0).clone().requires_grad_(True)
        s = sse64(xm, W[m], lib, dt, steps_per_row, y, method, None if rows is None else rows[m])
        if s.requires_grad:
            (g,) = torch.autograd.grad(s.sum(), (xm,))
        else:
            g = torch.zeros_like(xm)
        sse.append(s.detach())
        grads.append(g.detach())
    return torch.stack(sse), torch.stack(grads)


def windows(x, R):
    """(n_traj, T, d) -> (n_traj·T/R, R, d): every trajectory's consecutive, non-overlapping windows of R rows."""
    n, T, d = x.shape
    assert T % R == 0
    return x.reshape(n * (T // R), R, d)
