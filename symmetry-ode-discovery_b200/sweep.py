"""Seed sweeps in ONE process (SURVEY §8f item 4).

The reference repeats every experiment for seeds 0..49 by starting `python main.py --seed i --config ...` fifty times
(`run_scripts/*.sh`; each start pays ≈ 18 s of imports and data loading for a fit that takes a fraction of that) and
then aggregates the per-seed `.npz` files with `evaluation/eval_eq.py:38-85`. Here the seeds of a sweep run back to
back in one process on data that is already on the device — the LBFGS fit of every seed on the closed-form objective of
its own subsample (one data pass per seed, `train_SIGED_lbfgs(cached_gram=True)`) — and, under `torchrun`, are dealt
round-robin to the ranks (seeds are independent: no collective on the data path, one gather of the results).

`evaluate` and `aggregate` restate the reference's metrics (`eval_eq.py:7-34`, `:38-85`): per-equation "correct form"
(mask equals the truth's support), MSE over the truth's non-zero coefficients, success counts and RMSE mean (std).
What a seed controls follows `main.py:25-77`: the shuffled subsample of the training set that LBFGS sees
(`lbfgs_subsample`) and the random initial coefficients. The draws themselves are this module's own (the reference's
draw order runs through its autoencoder / GAN constructors, which are not part of this repository), so sweeps are
statistically, not seed-for-seed, comparable with the reference's.
"""
from __future__ import annotations

import io
from contextlib import redirect_stdout
from typing import Callable, Dict, Iterable, List, Optional

import numpy as np
import torch
import torch.distributed as dist

__all__ = ["evaluate", "aggregate", "run_seed_sweep", "lbfgs_fit", "BatchedLBFGS", "batched_lbfgs_fits",
           "run_seed_sweep_batched", "param_map"]


def evaluate(regressor, truth) -> Dict[str, np.ndarray]:
    """`eval_sindy_regressor` (`eval_eq.py:7-34`): masked coefficients, per-equation correct form and MSE over the
    truth's support, and both over all equations."""
    with torch.no_grad():
        coef = regressor.get_Xi() if regressor.constraint else regressor.Xi
        coef = coef.detach().cpu().numpy()
        mask = regressor.mask.bool().cpu().numpy()
    truth = np.asarray(truth, dtype=np.float64)
    coef = np.where(mask, coef, 0.0)
    truth_mask = truth != 0
    correct = np.array([float(np.all(mask[i] == truth_mask[i])) for i in range(coef.shape[0])])
    mse = np.array([np.mean((coef[i, truth_mask[i]] - truth[i, truth_mask[i]]) ** 2) for i in range(coef.shape[0])])
    return {"coefficients": coef, "correct_form": correct, "mse": mse, "correct_form_all": bool(np.all(correct)),
            "mse_all": float(np.mean(mse))}


def aggregate(results: Iterable[Dict], mse_multiplier: float = 1.0, verbose: bool = True) -> Dict:
    """`aggregate_results` (`eval_eq.py:38-85`) on in-memory results: success counts per equation and jointly, RMSE
    mean and std over the successful runs and over all runs (the reference prints these lines; so does this)."""
    results = list(results)
    cf = np.stack([r["correct_form"] for r in results])
    cf_all = np.array([bool(r["correct_form_all"]) for r in results])
    rmse = np.sqrt(np.stack([r["mse"] for r in results]))
    rmse_all = np.sqrt(np.array([r["mse_all"] for r in results]))
    out = {"runs": len(results), "success": cf.sum(0).astype(int), "success_all": int(cf_all.sum()),
           "rmse": [], "rmse_any": []}

    def stats(v):
        return (float(np.mean(v) * mse_multiplier), float(np.std(v) * mse_multiplier)) if len(v) else (float("nan"),) * 2

    for i in range(cf.shape[1]):
        out["rmse"].append(stats(rmse[cf[:, i] > 0, i]))
        out["rmse_any"].append(stats(rmse[:, i]))
    out["rmse_all"] = stats(rmse_all[cf_all])
    out["rmse_all_any"] = stats(rmse_all)
    if verbose:
        print(f'Loaded results from {out["runs"]} runs.')
        for i, s in enumerate(out["success"]):
            print(f'Equation {i} success rate = {s}/{out["runs"]}')
        print(f'Joint success rate = {out["success_all"]}/{out["runs"]}')
        for i in range(cf.shape[1]):
            print(f'Equation {i} RMSE = {out["rmse"][i][0]:.4f} ({out["rmse"][i][1]:.4f})')
            print(f'Equation {i} RMSE (any) = {out["rmse_any"][i][0]:.4f} ({out["rmse_any"][i][1]:.4f})')
        print(f'All equations RMSE = {out["rmse_all"][0]:.4f} ({out["rmse_all"][1]:.4f})')
        print(f'All equations RMSE (any) = {out["rmse_all_any"][0]:.4f} ({out["rmse_all_any"][1]:.4f})')
    return out


def lbfgs_fit(regressor, x, dx, lr_sindy=0.1, w_sindy_reg=0.0, st_freq=50, threshold=0.05, num_epochs=200, **kwargs):
    """The fit of `main.py` with `--sindy_optimizer lbfgs` and no sym-reg (`train_SIGED_lbfgs`, data-space branch) on
    the closed-form objective of this batch: one data pass, then K×K algebra per closure."""
    import train
    ident = torch.nn.Identity()
    train.train_SIGED_lbfgs(
        train_loader=[(x, dx)], test_loader=[(x, dx)], num_epochs=num_epochs, device=x.device, log_interval=10 ** 9,
        save_interval=10 ** 9, save_dir=None, autoencoder=ident, generator=ident, regressor=regressor,
        regressor_dst=None, use_latent=False, distill_latent=False, lr_sindy=lr_sindy, w_sindy_z=0.0, w_sindy_x=1.0,
        sindy_reg_type='l1' if w_sindy_reg > 0 else 'none', w_sindy_reg=w_sindy_reg, sym_reg_type='i', w_sym_reg=0.0,
        st_freq=st_freq, threshold=threshold, int_t=0.1, int_dt=0.01, print_eq=False, cached_gram=True)


def run_seed_sweep(x: torch.Tensor, dx: torch.Tensor, truth, seeds: Iterable[int], make_regressor: Callable[[], object],
                   fit: Callable = lbfgs_fit, subsample: float = 0.5, group=None, quiet: bool = True,
                   **fit_kwargs) -> Optional[List[Dict]]:
    """Fit one regressor per seed on a shuffled `subsample` of (x, dx) (`main.py:33-37`: the single LBFGS batch) and
    evaluate it against `truth`. x, dx: (N, d) CUDA tensors. Under torch.distributed the seeds are dealt round-robin to
    the ranks and the per-seed results are gathered on every rank in seed order. Returns the list of result dicts
    (each with its 'seed')."""
    seeds = list(seeds)
    distributed = dist.is_available() and dist.is_initialized()
    rank = dist.get_rank(group) if distributed else 0
    world = dist.get_world_size(group) if distributed else 1
    xf, dxf = x.reshape(-1, x.shape[-1]), dx.reshape(-1, dx.shape[-1])
    n = xf.shape[0]
    take = max(1, int(n * subsample))
    mine = []
    for s in seeds[rank::world]:
        torch.manual_seed(int(s))
        np.random.seed(int(s))
        idx = torch.randperm(n, device=xf.device)[:take]
        xb, dxb = xf[idx].contiguous(), dxf[idx].contiguous()
        regressor = make_regressor()
        sink = io.StringIO()
        with redirect_stdout(sink) if quiet else _nullcontext():
            fit(regressor, xb, dxb, **fit_kwargs)
        res = evaluate(regressor, truth)
        res["seed"] = int(s)
        mine.append(res)
    if not distributed or world == 1:
        return mine
    gathered = [None] * world
    dist.all_gather_object(gathered, mine, group=group)
    return sorted((r for part in gathered for r in part), key=lambda r: seeds.index(r["seed"]))


# --------------------------------------------------------------------------------------------------------------------
# all seeds as ONE batched LBFGS problem (SURVEY §8f-4)
# --------------------------------------------------------------------------------------------------------------------
class BatchedLBFGS:
    """torch.optim.LBFGS (no line search; defaults max_iter=20, history_size=100, tolerance_grad=1e-7,
    tolerance_change=1e-9 — what `train.py:630` constructs) for S independent problems of P parameters at once: every
    quantity of the optimiser carries a leading problem axis, the two-loop recursion runs over the stacked histories with
    per-problem validity masks, and the early exits of the serial loop (`gtd > -tolerance_change`, optimality, step and
    loss changes below tolerance) become per-problem `active` masks — no host synchronisation inside a step.
    `closure(x)` maps the (S, P) parameters to (loss (S,), grad (S, P)). `reset(which)` is the reference's
    "fresh optimiser" after thresholding (`train.py:717,723`) for the problems selected by the boolean mask."""

    def __init__(self, x: torch.Tensor, lr: float, max_iter: int = 20, history_size: int = 100,
                 tolerance_grad: float = 1e-7, tolerance_change: float = 1e-9):
        self.x = x
        S, P = x.shape
        dev, dt = x.device, x.dtype
        self.lr, self.max_iter, self.H = float(lr), int(max_iter), int(history_size)
        self.tg, self.tc = float(tolerance_grad), float(tolerance_change)
        self.n_iter = torch.zeros(S, dtype=torch.long, device=dev)
        self.d = torch.zeros(S, P, dtype=dt, device=dev)
        self.t = torch.zeros(S, dtype=dt, device=dev)
        self.H_diag = torch.ones(S, dtype=dt, device=dev)
        self.prev_g = torch.zeros(S, P, dtype=dt, device=dev)
        self.prev_loss = torch.zeros(S, dtype=dt, device=dev)
        self.old_y = torch.zeros(S, self.H, P, dtype=dt, device=dev)
        self.old_s = torch.zeros(S, self.H, P, dtype=dt, device=dev)
        self.ro = torch.zeros(S, self.H, dtype=dt, device=dev)
        self.hist = torch.zeros(S, dtype=torch.long, device=dev)
        self._hist_bound = 0      # host-side upper bound of hist.max(): avoids a device read per iteration

    def reset(self, which: torch.Tensor):
        self.n_iter[which] = 0
        self.hist[which] = 0
        self.H_diag[which] = 1.0
        if bool(which.all()):
            self._hist_bound = 0

    def push(self, y: torch.Tensor, sv: torch.Tensor, upd: torch.Tensor, ys: torch.Tensor):
        """Appends the curvature pair (s = sv, y) with ys = yᵀs to the history of the problems selected by `upd`
        (dropping their oldest pair when the history is full) and sets their initial Hessian scale to ys / yᵀy."""
        S = y.shape[0]
        full = upd & (self.hist == self.H)
        if self._hist_bound >= self.H and bool(full.any()):       # limited memory: drop the oldest pair
            self.old_y[full] = torch.roll(self.old_y[full], -1, 1)
            self.old_s[full] = torch.roll(self.old_s[full], -1, 1)
            self.ro[full] = torch.roll(self.ro[full], -1, 1)
            self.hist[full] -= 1
        pos = self.hist.clamp(max=self.H - 1)
        u = torch.arange(S, device=y.device)[upd]
        self.old_y[u, pos[u]] = y[u]
        self.old_s[u, pos[u]] = sv[u]
        self.ro[u, pos[u]] = 1.0 / ys[u]
        self.H_diag = torch.where(upd, ys / (y * y).sum(1).clamp_min(torch.finfo(y.dtype).tiny), self.H_diag)
        self.hist += upd.long()
        self._hist_bound = min(self.H, self._hist_bound + 1)

    def direction(self, g: torch.Tensor) -> torch.Tensor:
        """−H·g for every problem: the two-loop recursion over its stored pairs (entries past a problem's own history
        count are masked out), with H₀ = H_diag·I."""
        q = -g
        al = []
        for i in range(self._hist_bound - 1, -1, -1):
            valid = (i < self.hist)
            a_i = torch.where(valid, (self.old_s[:, i] * q).sum(1) * self.ro[:, i], torch.zeros_like(self.t))
            q = q - a_i.unsqueeze(1) * self.old_y[:, i]
            al.append(a_i)
        al.reverse()
        r = q * self.H_diag.unsqueeze(1)
        for i in range(self._hist_bound):
            valid = (i < self.hist)
            b_i = (self.old_y[:, i] * r).sum(1) * self.ro[:, i]
            r = r + torch.where(valid, al[i] - b_i, torch.zeros_like(b_i)).unsqueeze(1) * self.old_s[:, i]
        return r

    @torch.no_grad()
    def step(self, closure, enabled: Optional[torch.Tensor] = None):
        """One `optimizer.step(closure)` for every enabled problem; returns the loss of the first evaluation."""
        x = self.x
        S, P = x.shape
        loss, g = closure(x)
        first_loss = loss.clone()
        active = torch.ones(S, dtype=torch.bool, device=x.device) if enabled is None else enabled.clone()
        active &= ~(g.abs().amax(1) <= self.tg)                       # optimal condition before the loop
        for it in range(1, self.max_iter + 1):
            self.n_iter += active.long()
            first = active & (self.n_iter == 1)
            later = active & (self.n_iter > 1)
            # ---- memory update and two-loop recursion (problems past their first iteration) ----
            y = g - self.prev_g
            sv = self.d * self.t.unsqueeze(1)
            ys = (y * sv).sum(1)
            self.push(y, sv, later & (ys > 1e-10), ys)
            d_new = torch.where(first.unsqueeze(1), -g, self.direction(g))
            self.d = torch.where(active.unsqueeze(1), d_new, self.d)
            self.prev_g = torch.where(active.unsqueeze(1), g, self.prev_g)
            self.prev_loss = torch.where(active, loss, self.prev_loss)
            # ---- step length ----
            t_first = torch.minimum(torch.ones_like(self.t), 1.0 / g.abs().sum(1)) * self.lr
            self.t = torch.where(first, t_first, torch.where(later, torch.full_like(self.t, self.lr), self.t))
            gtd = (g * self.d).sum(1)
            active &= ~(gtd > -self.tc)
            x += torch.where(active.unsqueeze(1), self.d * self.t.unsqueeze(1), torch.zeros_like(x))
            if it == self.max_iter:
                break
            new_loss, new_g = closure(x)
            loss = torch.where(active, new_loss, loss)
            g = torch.where(active.unsqueeze(1), new_g, g)
            opt = g.abs().amax(1) <= self.tg
            small_step = (self.d * self.t.unsqueeze(1)).abs().amax(1) <= self.tc
            small_change = (loss - self.prev_loss).abs() < self.tc
            active &= ~(opt | small_step | small_change)
        return first_loss


def batched_lbfgs_fits(G, b, yy, n, xi0, lr_sindy=0.1, st_freq=50, threshold=0.05, num_epochs=200, tol=1e-3,
                       param_map=None, groups=None):
    """The LBFGS phase of `train_SIGED_lbfgs` (`train.py:692-766`, data-space branch, no sym-reg, L1 weight 0) for S
    seeds at once on the closed-form objective of every seed's own subsample.
    G (S,K,K), b (S,K,d), yy (S,) fp64 sufficient statistics; n (S,) sample counts; xi0 (S,P) initial parameters.
    param_map (d·K, P) maps the parameters to vec(Ξ) (None: identity, P = d·K; the equivariance-constrained regressor
    passes [Q | unit columns of the free constants]); groups: list of index ranges = the parameter tensors whose update
    norms the reference adds up (`train.py:701-708`). Returns (parameters (S,P), masks (S,d,K), epochs run (S,))."""
    S = xi0.shape[0]
    K, d = b.shape[1], b.shape[2]
    dev = xi0.device
    x = xi0.clone().to(torch.float32)
    A = None if param_map is None else param_map.to(dev, torch.float64)
    groups = groups or [(0, x.shape[1])]
    mask = torch.ones(S, d, K, dtype=torch.float32, device=dev)
    nd = (n.to(torch.float64) * d).view(S)

    def xi_of(p):
        v = p.double() if A is None else p.double() @ A.T
        return v.view(S, d, K)

    def closure(p):
        W = xi_of(p) * mask.double()
        WG = torch.einsum('sik,skl->sil', W, G)
        quad = (WG * W).sum((1, 2)) - 2.0 * torch.einsum('sik,ski->s', W, b) + yy
        gW = 2.0 * (WG - b.transpose(1, 2)) * mask.double() / nd.view(S, 1, 1)
        gp = gW.reshape(S, d * K) if A is None else gW.reshape(S, d * K) @ A
        return (quad / nd).to(torch.float32), gp.to(torch.float32)

    def moved(p, q):
        return sum(torch.linalg.vector_norm(p[:, a:e] - q[:, a:e], dim=1) for a, e in groups)

    opt = BatchedLBFGS(x, lr_sindy)
    prev, since = x.clone(), x.clone()
    n_iters = torch.zeros(S, dtype=torch.long, device=dev)
    running = torch.ones(S, dtype=torch.bool, device=dev)
    epochs = torch.zeros(S, dtype=torch.long, device=dev)
    for epoch in range(num_epochs):
        n_iters += running.long()
        opt.step(closure, running)
        epochs += running.long()
        nan = torch.isnan(x).any(1)
        running &= ~nan                                              # `train.py:696-699`: NaN -> exit training
        still = moved(x, prev) < tol
        final = running & still & (moved(x, since) < tol)            # converged twice: done
        thr_a = running & still & ~final
        thr_b = running & ~still & (st_freq > 0) & (n_iters % max(st_freq, 1) == 0)
        do_thr = thr_a | thr_b
        if bool(do_thr.any()):
            keep = (xi_of(x).abs() > threshold).float() * mask
            mask = torch.where(do_thr.view(S, 1, 1), keep, mask)
            opt.reset(do_thr)
            n_iters = torch.where(do_thr, torch.zeros_like(n_iters), n_iters)
            since = torch.where(thr_a.unsqueeze(1), x, since)
        running &= ~final
        prev = torch.where(running.unsqueeze(1), x, prev)
        if not bool(running.any()):
            break
    return x, mask, epochs


def param_map(reg):
    """(A, groups) of an equivariance-constrained regressor: vec(Ξ) = A·[β, const] (d·K × (nb + d), fp64; the constant
    columns are zero unless the regressor allows a free constant) and the parameter index ranges of β and const."""
    d, K = reg.latent_dim, reg.library.K
    Q = reg.Q.detach().to(torch.float64)                          # vec(Ξ) (equation-major) = layout(Q β) [+ constants]
    nb = Q.shape[1]
    cols = []
    for j in range(nb):                                            # Ξ is LINEAR in β: read the map off unit vectors
        e = torch.zeros(nb, dtype=reg.beta.dtype, device=reg.beta.device)
        e[j] = 1.0
        flat = reg.Q @ e
        Xi = flat.view(d, -1) if reg.use_kron_product else flat.view(-1, d).transpose(0, 1)
        cols.append(Xi.reshape(-1).double())
    groups = [(0, nb)]
    if reg.allow_constant:
        for i in range(d):
            c = torch.zeros(d * K, dtype=torch.float64, device=Q.device)
            c[i * K] = 1.0
            cols.append(c)
    groups.append((nb, nb + d))                                    # `const` is a parameter even when unused (sindy.py:59-60)
    A = torch.stack(cols, dim=1)
    if not reg.allow_constant:
        A = torch.cat([A, torch.zeros(d * K, d, dtype=torch.float64, device=A.device)], dim=1)
    return A, groups


def run_seed_sweep_batched(x: torch.Tensor, dx: torch.Tensor, truth, seeds: Iterable[int],
                           make_regressor: Callable[[], object], subsample: float = 0.5, lr_sindy=0.1, st_freq=50,
                           threshold=0.05, num_epochs=200, draw: Optional[Callable] = None) -> List[Dict]:
    """`run_seed_sweep` with all seeds fitted as ONE batched LBFGS problem (SURVEY §8f-4): per seed the shuffled
    subsample and the initial parameters are drawn exactly like `run_seed_sweep` does (or by `draw(seed, n, take) ->
    (indices, regressor)`), one statistics pass per seed forms (G, b, Σẋ²), then `batched_lbfgs_fits` advances every
    seed's optimiser, thresholding schedule and convergence test in lock-step tensor operations. Same results as the
    one-after-the-other sweep (tests/test_gpu_train_loops.py), without S × (optimiser + closure) Python overhead."""
    seeds = list(seeds)
    xf, dxf = x.reshape(-1, x.shape[-1]), dx.reshape(-1, dx.shape[-1])
    n = xf.shape[0]
    take = max(1, int(n * subsample))
    regs, stats = [], []
    for s in seeds:
        if draw is not None:
            idx, regressor = draw(int(s), n, take)
        else:
            torch.manual_seed(int(s))
            np.random.seed(int(s))
            idx = torch.randperm(n, device=xf.device)[:take]
            regressor = make_regressor()
        regs.append(regressor)
        stats.append(regressor.sufficient_statistics(xf[idx].contiguous(), dxf[idx].contiguous()))
    G = torch.stack([q["G"] for q in stats])
    b = torch.stack([q["b"] for q in stats])
    yy = torch.stack([q["yy"].reshape(()) for q in stats])
    nn_ = torch.tensor([float(q["n"]) for q in stats], dtype=torch.float64, device=G.device)
    reg0 = regs[0]
    d, K = reg0.latent_dim, reg0.library.K
    if reg0.constraint:
        A, groups = param_map(reg0)
        p0 = torch.stack([torch.cat([r.beta.detach().reshape(-1), r.const.detach().reshape(-1)]) for r in regs])
    else:
        A, groups = None, None
        p0 = torch.stack([r.Xi.detach().reshape(-1) for r in regs])
    params, masks, _ = batched_lbfgs_fits(G, b, yy, nn_, p0, lr_sindy, st_freq, threshold, num_epochs, param_map=A,
                                          groups=groups)
    out = []
    for i, (s, r) in enumerate(zip(seeds, regs)):
        with torch.no_grad():
            if r.constraint:
                nb = r.beta.numel()
                r.beta.data = params[i, :nb].clone()
                r.const.data = params[i, nb:].view(-1, 1).clone()
            else:
                r.Xi.data = params[i].view(d, K).clone()
            r.mask.data = masks[i].clone()
        res = evaluate(r, truth)
        res["seed"] = int(s)
        out.append(res)
    return out


class _nullcontext:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False
