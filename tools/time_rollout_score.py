"""Timing of the fused multi-model rollout scorer (sb_rollout_score) against the loop it replaces: per model one
native.rollout that stores the trajectory, then an fp64 torch reduction of the squared error against the observed rows.

Shapes:
  cfg-like  d=2, p=2:  40 models x 20 ICs x 99 rows x 10 steps  (a 40-threshold path scored on a cfg's validation set)
  large     d=3, p=5:  64 models x 4096 ICs x 2000 steps (200 rows of 10 steps)
For the large shape the scorer's IC-steps/s are set next to rollout_rk4_multi_kernel integrating one model from
64 x 4096 ICs for the same 2000 steps (no trajectory stored): the same total work in one launch. Every timing is CUDA
events around repeated calls after a warm-up, with the window at least 1 s; the outputs of the two scoring paths are
compared. The card's name, power limit and maximum SM clock are read (read-only) at the start.

  python tools/time_rollout_score.py [output file, default profiles/r04_time_rollout_score.txt]
"""
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "symmetry-ode-discovery_b200")]
from sindy_b200 import native  # noqa: E402


def gpu_identity():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=30).stdout.strip().splitlines()
    return out[torch.cuda.current_device()] if out else "unknown"


def timed(fn, min_window=1.0):
    """ms per call: warm-up, then as many calls as fill at least `min_window` seconds between two CUDA events."""
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    reps = max(3, math.ceil(min_window * 1e3 / max(a.elapsed_time(b), 1e-3)))
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps, reps


def stable_models(lib, M, seed):
    """Small random models with a damping diagonal: no pair leaves the bounds, so every pair runs every step."""
    g = torch.Generator().manual_seed(seed)
    W = 0.02 * torch.randn(M, lib.dim, lib.K, generator=g)
    for i in range(lib.dim):
        W[:, i, 1 + i] -= 0.5
    return W.cuda()


def loop_scores(x0, W, lib, dt, spr, y):
    out = []
    for m in range(W.shape[0]):
        traj, _, _ = native.rollout(x0, W[m], lib, dt, y.shape[0] * spr, stride=spr, want_last=False)
        out.append(((traj.double() - y.double()) ** 2).sum(dim=(0, 2)))
    return torch.stack(out)


def main():
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r04_time_rollout_score.txt")
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say(f"gpu: {gpu_identity()}")
    for name, (d, p), M, N, n_rows, spr, dt in (("cfg-like", (2, 2), 40, 20, 99, 10, 0.002),
                                                 ("large", (3, 5), 64, 4096, 200, 10, 0.001)):
        lib = native.Library(d, p)
        W = stable_models(lib, M, 1)
        g = torch.Generator(device="cuda").manual_seed(2)
        x0 = torch.rand(N, d, device="cuda", generator=g) - 0.5
        y = torch.randn(n_rows, N, d, device="cuda", generator=g) * 0.1
        sse, valid = native.rollout_score(x0, W, lib, dt, spr, y)
        ref = loop_scores(x0, W, lib, dt, spr, y)
        rel = ((sse - ref).abs() / ref.abs()).max().item()
        f_ms, f_reps = timed(lambda: native.rollout_score(x0, W, lib, dt, spr, y))
        l_ms, l_reps = timed(lambda: loop_scores(x0, W, lib, dt, spr, y))
        work = M * N * n_rows * spr
        say(f"{name}: lib (d={d}, p={p}) K={lib.K}  {M} models x {N} ICs x {n_rows} rows x {spr} steps  "
            f"(all pairs valid: {bool((valid == n_rows).all())}, max rel. diff fused vs loop {rel:.1e})")
        say(f"   fused rollout_score: {f_ms:.3f} ms ({f_reps} calls)  {work / f_ms / 1e6:.3f} G IC-steps/s")
        say(f"   loop ({M} x rollout + fp64 torch reduction): {l_ms:.3f} ms ({l_reps} calls)  -> fused is "
            f"{l_ms / f_ms:.2f}x faster")
        if name == "large":
            x1 = torch.rand(M * N, d, device="cuda", generator=g) - 0.5
            n_steps = n_rows * spr
            m_ms, m_reps = timed(lambda: native.rollout(x1, W[0], lib, dt, n_steps, stride=n_steps, want_traj=False))
            m_rate = M * N * n_steps / m_ms / 1e6
            say(f"   rollout_rk4_multi_kernel, one model, {M * N} ICs x {n_steps} steps: {m_ms:.3f} ms ({m_reps} calls)"
                f"  {m_rate:.3f} G IC-steps/s  -> fused reaches {work / f_ms / 1e6 / m_rate:.2f} of it")
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
