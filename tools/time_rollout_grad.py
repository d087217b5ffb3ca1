"""Timing of the rollout-score gradient (sb_rollout_score_grad) against the scorer it extends (sb_rollout_score) and
against what a user has without it: fp32 torch autograd through a batched RK4 over all models on the GPU.

Shapes:
  cfg-like  d=2, p=2 (K=6):   40 models x 20 ICs x 99 rows x 10 steps
  large     d=3, p=5 (K=56):  64 models x 4096 ICs x 2000 steps (200 rows of 10 steps)
The autograd path keeps every stage of every step for backward; at the large shape that does not fit in memory
(≈ 0.7 GB per step), so it is timed over a reduced number of steps and that time is reported with the step count.
Also one whole sindy.refine_path at the cfg-like shape (40 candidates, max_iter 50). Every timing is CUDA events around
repeated calls after a warm-up, with the window at least 1 s. The card's name, power limit and maximum SM clock are read
(read-only) at the start.

  python tools/time_rollout_grad.py [output file, default profiles/r05_time_rollout_grad.txt]
"""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "symmetry-ode-discovery_b200"), os.path.join(ROOT, "tools")]
from sindy_b200 import native  # noqa: E402
from time_rollout_score import gpu_identity, stable_models, timed  # noqa: E402


def autograd_rk4(x0, W, E, dt, spr, y):
    """Σ SSE over all models and ICs by fp32 torch RK4 (x0 excluded, rows every spr steps), and its gradient."""
    Wg = W.detach().clone().requires_grad_(True)
    M = W.shape[0]
    x = x0.unsqueeze(0).expand(M, -1, -1)

    def h(q):
        th = torch.prod(q.unsqueeze(-2) ** E, -1)                       # (M, N, K)
        return torch.einsum('mnk,mik->mni', th, Wg)

    loss = x.new_zeros(())
    for r in range(y.shape[0]):
        for _ in range(spr):
            k1 = h(x)
            k2 = h(x + dt / 2 * k1)
            k3 = h(x + dt / 2 * k2)
            k4 = h(x + dt * k3)
            x = x + dt / 6 * (((k1 + 2 * k2) + 2 * k3) + k4)
        loss = loss + ((x - y[r]) ** 2).sum()
    (g,) = torch.autograd.grad(loss, (Wg,))
    return g


def main():
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r05_time_rollout_grad.txt")
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say(f"gpu: {gpu_identity()}")
    for name, (d, p), M, N, n_rows, spr, dt, ag_rows in (("cfg-like", (2, 2), 40, 20, 99, 10, 0.002, 99),
                                                         ("large", (3, 5), 64, 4096, 200, 10, 0.001, 2)):
        lib = native.Library(d, p)
        W = stable_models(lib, M, 1)
        g = torch.Generator(device="cuda").manual_seed(2)
        x0 = torch.rand(N, d, device="cuda", generator=g) - 0.5
        y = torch.randn(n_rows, N, d, device="cuda", generator=g) * 0.1
        sse, valid, grad = native.rollout_score_grad(x0, W, lib, dt, spr, y)
        sse0, valid0 = native.rollout_score(x0, W, lib, dt, spr, y)
        same = bool(torch.equal(sse, sse0) and torch.equal(valid, valid0))
        g_ms, g_reps = timed(lambda: native.rollout_score_grad(x0, W, lib, dt, spr, y))
        s_ms, s_reps = timed(lambda: native.rollout_score(x0, W, lib, dt, spr, y))
        E = lib.exponents().cuda().float()
        ya = y[:ag_rows].contiguous()
        ga = autograd_rk4(x0, W, E, dt, spr, ya)
        _, _, gk = native.rollout_score_grad(x0, W, lib, dt, spr, ya)
        rel = float((ga.double() - gk).abs().max() / gk.abs().max())
        a_ms, a_reps = timed(lambda: autograd_rk4(x0, W, E, dt, spr, ya))
        steps, a_steps = n_rows * spr, ag_rows * spr
        say(f"{name}: lib (d={d}, p={p}) K={lib.K}  {M} models x {N} ICs x {n_rows} rows x {spr} steps  "
            f"(all pairs valid: {bool((valid == n_rows).all())}, sse/valid bitwise equal to rollout_score: {same})")
        say(f"   rollout_score_grad: {g_ms:.3f} ms ({g_reps} calls)")
        say(f"   rollout_score:      {s_ms:.3f} ms ({s_reps} calls)  -> gradient / score = {g_ms / s_ms:.2f}")
        if a_steps == steps:
            say(f"   torch fp32 autograd RK4: {a_ms:.3f} ms ({a_reps} calls)  -> gradient kernel is "
                f"{a_ms / g_ms:.1f}x faster  (max rel. diff of the gradients {rel:.1e})")
        else:
            say(f"   torch fp32 autograd RK4 does not fit in memory at {steps} steps (every stage kept for backward); "
                f"at {a_steps} steps ({ag_rows} rows): {a_ms:.3f} ms ({a_reps} calls) = {a_ms / a_steps:.3f} ms per step "
                f"against {g_ms / steps:.4f} ms per step of the gradient kernel at {steps} steps  -> "
                f"{(a_ms / a_steps) / (g_ms / steps):.0f}x per step  (max rel. diff of the gradients at {a_steps} steps "
                f"{rel:.1e})")
        if name == "cfg-like":
            import sindy
            truth = torch.zeros(d, lib.K, device="cuda")
            truth[0, 2], truth[1, 1], truth[1, 2] = 1.0, -1.0, -0.1
            xs, _, _ = native.rollout(x0, truth, lib, dt, steps, stride=spr, want_last=False)
            xf = torch.cat([x0.unsqueeze(0), xs], 0).transpose(0, 1).contiguous()
            xf = xf + 0.01 * torch.randn(xf.shape, device="cuda", generator=g)
            gm = torch.Generator().manual_seed(4)
            masks = (torch.rand(M, d, lib.K, generator=gm) > 0.4).cuda() | (truth != 0)
            xi = (truth + 0.05 * torch.randn(M, d, lib.K, generator=gm).cuda()) * masks
            cand = {"thresholds": torch.linspace(0, 1, M, dtype=torch.float64), "xi": xi, "mask": masks}
            sindy.refine_path(lib, cand, xf, dt, steps_per_row=spr)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = sindy.refine_path(lib, cand, xf, dt, steps_per_row=spr)
            torch.cuda.synchronize()
            r_ms = (time.perf_counter() - t0) * 1e3
            say(f"   refine_path, {M} candidates, max_iter 50: {r_ms:.1f} ms wall clock, iterations "
                f"{int(out['iterations'].min())}..{int(out['iterations'].max())}, SSE ratio after/before median "
                f"{float((out['sse_after'] / out['sse_before']).median()):.3f}")
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
