"""Timing of the Gauss–Newton information of the rollout scores (sb_rollout_score_gn) against the scorer
(sb_rollout_score) and the adjoint gradient (sb_rollout_score_grad) at the same shapes, and against what a user has
without it: fp32 torch.func.jacfwd through a batched RK4.

Shapes (those of tools/time_rollout_grad.py):
  cfg-like  d=2, p=2 (K=6):   40 models x 20 ICs x 99 rows x 10 steps, every coefficient listed (12), with starts
  large     d=3, p=5 (K=56):  64 models x 4096 ICs x 200 rows x 10 steps, 20 listed coefficients per model + 3 starts,
                              and the dense 168 + 3
jacfwd is timed at the cfg-like shape over a reduced number of rows (it keeps one tangent per listed coefficient for
every pair and stage), and its time is reported with the row count. Every timing is CUDA events around repeated calls
after a warm-up, with the window at least 1 s. The card's name, power limit and maximum SM clock are read (read-only)
at the start. The ratio to the gradient kernel is set against the operation count:
  tangent work per stage and pair  ≈ n'·2d² (J_h·S) + d reverse library sweeps (J_h) + the scorer's right-hand side,
  F update per compared row        ≈ n'²·d per pair,  n' = listed coefficients + starts.

  python tools/time_rollout_gn.py [output file, default profiles/r07_time_rollout_gn.txt]
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "symmetry-ode-discovery_b200"), os.path.join(ROOT, "tools")]
from sindy_b200 import native  # noqa: E402
from time_rollout_score import gpu_identity, stable_models, timed  # noqa: E402


def jacfwd_rk4(x0, W, idx, E, dt, spr, n_rows):
    """Σ over pairs of JᵀJ of the listed coefficients by fp32 torch.func.jacfwd through a batched RK4 (all models)."""
    from torch.func import jacfwd, vmap
    M, d, K = W.shape

    def states(theta, Wm):
        Wf = Wm.reshape(-1).index_put((idx,), theta).view(d, K)
        x = x0

        def h(q):
            return torch.prod(q.unsqueeze(-2) ** E, -1) @ Wf.T

        out = []
        for _ in range(n_rows):
            for _ in range(spr):
                k1 = h(x)
                k2 = h(x + dt / 2 * k1)
                k3 = h(x + dt / 2 * k2)
                k4 = h(x + dt * k3)
                x = x + dt / 6 * (((k1 + 2 * k2) + 2 * k3) + k4)
            out.append(x)
        return torch.stack(out)

    def info(Wm):
        J = jacfwd(states)(Wm.reshape(-1)[idx], Wm)                      # (rows, N, d, P)
        return torch.einsum('rnip,rniq->pq', J, J)

    return vmap(info)(W)


def main():
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r07_time_rollout_gn.txt")
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say(f"gpu: {gpu_identity()}")
    for name, (d, p), M, N, n_rows, spr, dt, lists in (("cfg-like", (2, 2), 40, 20, 99, 10, 0.002, (12,)),
                                                       ("large", (3, 5), 64, 4096, 200, 10, 0.001, (20, 168))):
        lib = native.Library(d, p)
        W = stable_models(lib, M, 1)
        g = torch.Generator(device="cuda").manual_seed(2)
        x0 = torch.rand(N, d, device="cuda", generator=g) - 0.5
        y = torch.randn(n_rows, N, d, device="cuda", generator=g) * 0.1
        s_ms, s_reps = timed(lambda: native.rollout_score(x0, W, lib, dt, spr, y))
        g_ms, g_reps = timed(lambda: native.rollout_score_grad(x0, W, lib, dt, spr, y, x0_grad=True))
        sse0, valid0 = native.rollout_score(x0, W, lib, dt, spr, y)
        say(f"{name}: lib (d={d}, p={p}) K={lib.K}  {M} models x {N} ICs x {n_rows} rows x {spr} steps  "
            f"(all pairs valid: {bool((valid0 == n_rows).all())})")
        say(f"   rollout_score:                      {s_ms:.3f} ms ({s_reps} calls)")
        say(f"   rollout_score_grad (W and x0):      {g_ms:.3f} ms ({g_reps} calls)")
        _, _, gw, gx0 = native.rollout_score_grad(x0, W, lib, dt, spr, y, x0_grad=True)
        for n_list in lists:
            gen = torch.Generator().manual_seed(3)
            prm = torch.stack([torch.randperm(d * lib.K, generator=gen)[:n_list] for _ in range(M)]).to(torch.int32)
            prm = prm.cuda()
            out = native.rollout_score_gn(x0, W, prm, lib, dt, spr, y, x0_blocks=True)
            same = bool(torch.equal(out["sse"], sse0) and torch.equal(out["valid_rows"], valid0))
            gl = torch.gather(gw.reshape(M, -1), 1, prm.long())
            fr = max(float((2 * out["jtr"] - gl).abs().max() / gl.abs().max()),
                     float((2 * out["jtr_x"] - gx0).abs().max() / gx0.abs().max()))
            n_ms, n_reps = timed(lambda: native.rollout_score_gn(x0, W, prm, lib, dt, spr, y, x0_blocks=True))
            n_cols = n_list + d
            say(f"   rollout_score_gn, {n_list} coefficients + {d} starts ({n_cols} tangent columns): {n_ms:.3f} ms "
                f"({n_reps} calls)  -> / score {n_ms / s_ms:.1f}, / gradient {n_ms / g_ms:.1f}  (sse/valid bitwise "
                f"equal to rollout_score: {same}; 2·g against the adjoint gradient: rel {fr:.1e})")
            # operation count per pair: tangents J_h·S per stage, the F update per compared row
            stages = n_rows * spr * 4
            say(f"      per pair: tangent work ≈ {stages} stages x {n_cols}·2d² = {stages * n_cols * 2 * d * d:.3e}, "
                f"F update ≈ {n_rows} rows x {n_cols}²·d = {n_rows * n_cols * n_cols * d:.3e}")
        if name == "cfg-like":
            E = lib.exponents().cuda().float()
            idx = torch.arange(d * lib.K, device="cuda")
            jr = 20
            ya = y[:jr].contiguous()
            ref = jacfwd_rk4(x0, W, idx, E, dt, spr, jr)
            mine = native.rollout_score_gn(x0, W, idx.to(torch.int32), lib, dt, spr, ya)["jtj"]
            rel = float((ref.double() - mine).abs().max() / mine.abs().max())
            a_ms, a_reps = timed(lambda: jacfwd_rk4(x0, W, idx, E, dt, spr, jr))
            k_ms, k_reps = timed(lambda: native.rollout_score_gn(x0, W, idx.to(torch.int32), lib, dt, spr, ya))
            say(f"   torch fp32 jacfwd RK4 at {jr} rows (12 coefficients, no starts): {a_ms:.3f} ms ({a_reps} calls) "
                f"against rollout_score_gn {k_ms:.3f} ms at the same size -> {a_ms / k_ms:.0f}x  (max rel. diff of "
                f"JᵀJ {rel:.1e})")
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
