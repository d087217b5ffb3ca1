"""fp64 autograd reference of the rollout-score gradient (sb_rollout_score_grad) — TEST INFRASTRUCTURE ONLY.

Plain PyTorch in float64 through the odeint recurrence (`model_utils.py:236-253`): Euler x + dt·h(x), or RK4 with stages
x, x + dt/2·k1, x + dt/2·k2, x + dt·k3 and x + dt/6·(((k1 + 2k2) + 2k3) + k4), h(x) = Θ(x)Wᵀ with Θ from `theta64`
(pinned to the oracle's column order). Nothing here imports the product. Callers hand in the fp32 tensors the kernel
sees; they are cast exactly to fp64.
"""
import torch

from symreg_fp64_ref import theta64


def step64(x, W, lib, dt, method):
    h = lambda q: theta64(q, *lib) @ W.T
    k1 = h(x)
    if method == "euler":
        return x + dt * k1
    k2 = h(x + dt / 2 * k1)
    k3 = h(x + dt / 2 * k2)
    k4 = h(x + dt * k3)
    return x + dt / 6 * (((k1 + 2 * k2) + 2 * k3) + k4)


def sse64(x0, W, lib, dt, steps_per_row, y, method, rows=None):
    """Per-IC SSE Σ_{r < rows[n]} ‖x_{(r+1)·spr} − y[r, n]‖² (rows[n] = all rows of y when None), fp64 (N,).
    x0 (N, d), W (d, K), y (n_rows, N, d)."""
    n_rows = y.shape[0]
    rows = torch.full((x0.shape[0],), n_rows, dtype=torch.long, device=x0.device) if rows is None else rows.long()
    x = x0
    out = torch.zeros(x0.shape[0], dtype=torch.float64, device=x0.device)
    for r in range(int(rows.max()) if rows.numel() else 0):
        # a pair that has stopped continues from 0 outside the graph: its own state may overflow, and 0·inf in the
        # backward of the batched step would leak NaN into the other pairs' gradient
        x = torch.where((rows > r).unsqueeze(1), x, torch.zeros_like(x).detach())
        for _ in range(steps_per_row):
            x = step64(x, W, lib, dt, method)
        e = ((x - y[r]) ** 2).sum(-1)
        out = out + torch.where(rows > r, e, torch.zeros_like(e))
    return out


def grad64(x0, W, lib, dt, steps_per_row, y, method, rows=None):
    """(per-IC SSE (N,), ∂/∂W of its sum (d, K)), fp64. W is one model (d, K)."""
    W64 = W.detach().to(torch.float64).requires_grad_(True)
    s = sse64(x0.detach().to(torch.float64), W64, lib, dt, steps_per_row, y.detach().to(torch.float64), method, rows)
    if not s.requires_grad:
        return s.detach(), torch.zeros_like(W64).detach()
    (g,) = torch.autograd.grad(s.sum(), (W64,))
    return s.detach(), g
