"""fp64 forward-mode reference of the Gauss–Newton information of the rollout scores (sb_rollout_score_gn) — TEST
INFRASTRUCTURE ONLY.

The compared states of `rollout_fp64_ref.step64`'s recurrence and their Jacobian, by `torch.func.jacfwd`, with
respect to the listed entries of W (flat d×K indices, −1 = padding) and to the start. The pairs are independent, so one
start direction shared by every pair gives each pair's own ∂x_r/∂x0. Nothing here imports the product. Callers hand in
the fp32 tensors the kernel sees; they are cast exactly to fp64.
"""
import torch
from torch.func import jacfwd

from rollout_fp64_ref import step64


def jac64(x0, W, idx, lib, dt, steps_per_row, n_rows, method):
    """(states (n_rows, N, d), Jθ (n_rows, N, d, P), Jx (n_rows, N, d, d)), fp64. x0 (N, d), W (d, K), idx (P,)."""
    x0 = x0.detach().to(torch.float64)
    W = W.detach().to(torch.float64)
    d, K = W.shape
    idx = torch.as_tensor(idx, dtype=torch.long, device=W.device)
    P = idx.numel()
    live = idx >= 0
    E = torch.zeros(d * K, P, dtype=torch.float64, device=W.device)
    E[idx[live], torch.arange(P, device=W.device)[live]] = 1.0
    base = W.reshape(-1) * (1.0 - E.sum(1))                 # the listed entries come from theta
    theta0 = torch.where(live, W.reshape(-1)[idx.clamp_min(0)], torch.zeros(P, dtype=torch.float64, device=W.device))

    def f(theta, s):
        Wm = (base + E @ theta).view(d, K)
        x = x0 + s
        out = []
        for _ in range(n_rows):
            for _ in range(steps_per_row):
                x = step64(x, Wm, lib, dt, method)
            out.append(x)
        return torch.stack(out)

    s0 = torch.zeros(d, dtype=torch.float64, device=W.device)
    X = f(theta0, s0)
    Jt, Jx = jacfwd(f, argnums=(0, 1))(theta0, s0)
    return X, Jt, Jx


def gn64(x0, W, idx, lib, dt, steps_per_row, y, method, rows=None):
    """The outputs of sb_rollout_score_gn for ONE model, fp64: dict of jtj (P, P), jtr (P,), jtj_px (N, P, d),
    jtj_xx (N, d, d), jtr_x (N, d), each pair summed over its rows r < rows[n] (all rows of y when None)."""
    n_rows = y.shape[0]
    y = y.detach().to(torch.float64)
    X, Jt, Jx = jac64(x0, W, idx, lib, dt, steps_per_row, n_rows, method)
    N = X.shape[1]
    rows = torch.full((N,), n_rows, dtype=torch.long, device=X.device) if rows is None else rows.long().to(X.device)
    keep = torch.arange(n_rows, device=X.device)[:, None] < rows[None, :]          # (n_rows, N)
    k3 = keep[:, :, None]
    # rows past a pair's last one may hold non-finite states: select, never multiply, them away
    Jt = torch.where(k3[..., None], Jt, torch.zeros_like(Jt))
    Jx = torch.where(k3[..., None], Jx, torch.zeros_like(Jx))
    e = torch.where(k3, X - y, torch.zeros_like(X))
    return {"jtj": torch.einsum('rnip,rniq->pq', Jt, Jt), "jtr": torch.einsum('rnip,rni->p', Jt, e),
            "jtj_px": torch.einsum('rnip,rnij->npj', Jt, Jx), "jtj_xx": torch.einsum('rnij,rnik->njk', Jx, Jx),
            "jtr_x": torch.einsum('rnij,rni->nj', Jx, e)}
