"""Timing of start estimation in the rollout scores: per-model starts (sb_rollout_score_ics), the start gradient and the
start-only kernel variant (sb_rollout_score_grad_ics), and the legacy entry points they forward to.

Shapes (those of time_rollout_score.py / time_rollout_grad.py):
  cfg-like  d=2, p=2 (K=6):   40 models x 20 ICs x 99 rows x 10 steps
  large     d=3, p=5 (K=56):  64 models x 4096 ICs x 2000 steps (200 rows of 10 steps)
1. sb_rollout_score and sb_rollout_score_grad of this tree against a build of the parent commit (--parent-lib, a
   libsindy_b200.so built from it; the two libraries are loaded side by side), outputs compared bitwise on the same
   inputs and the timings taken alternately, three rounds each, medians reported.
2. rollout_score from per-model starts (copies of the shared set) against shared starts.
3. rollout_score_grad: W gradient only, W and start gradients, start gradient only (the start-only variant).
4. One sindy.refine_path(fit_ic=True) and one sindy.score_path(fit_ic=True) at the cfg-like shape, 40 candidates.
Every kernel timing is CUDA events around repeated calls after a warm-up, the window at least 1 s; the card's name,
power limit and maximum SM clock are read (read-only) at the start.

  python tools/time_rollout_ic.py [output file, default profiles/r06_time_rollout_ic.txt] [--parent-lib PATH]
"""
import ctypes
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "symmetry-ode-discovery_b200"), os.path.join(ROOT, "tools")]
from sindy_b200 import native  # noqa: E402
from time_rollout_score import gpu_identity, stable_models, timed  # noqa: E402


def legacy_calls(cdll):
    """sb_rollout_score / sb_rollout_score_grad of one loaded library, on the binding's argument conventions."""
    for name in ("sb_rollout_score", "sb_rollout_score_grad_workspace_bytes", "sb_rollout_score_grad"):
        fn = getattr(cdll, name)
        fn.restype, fn.argtypes = native._SIGNATURES[name]

    def score(x0, W, lib, dt, spr, y):
        M, N = W.shape[0], x0.shape[0]
        sse = torch.empty(M, N, dtype=torch.float64, device="cuda")
        valid = torch.empty(M, N, dtype=torch.int32, device="cuda")
        st = cdll.sb_rollout_score(x0.data_ptr(), N, ctypes.byref(lib.c()), W.data_ptr(), M, dt, spr, y.shape[0],
                                   native.SB_RK4, y.data_ptr(), 0.0, sse.data_ptr(), valid.data_ptr(),
                                   native._stream(x0.device))
        assert st == 0, st
        return sse, valid

    def grad(x0, W, lib, dt, spr, y, ws):
        M, N = W.shape[0], x0.shape[0]
        sse = torch.empty(M, N, dtype=torch.float64, device="cuda")
        valid = torch.empty(M, N, dtype=torch.int32, device="cuda")
        g = torch.empty(M, lib.dim, lib.K, dtype=torch.float64, device="cuda")
        st = cdll.sb_rollout_score_grad(x0.data_ptr(), N, ctypes.byref(lib.c()), W.data_ptr(), M, dt, spr, y.shape[0],
                                        native.SB_RK4, y.data_ptr(), 0.0, sse.data_ptr(), valid.data_ptr(),
                                        g.data_ptr(), ws.data_ptr(), ws.numel(), native._stream(x0.device))
        assert st == 0, st
        return sse, valid, g

    return score, grad


def main():
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    args = sys.argv[1:]
    parent = None
    if "--parent-lib" in args:
        i = args.index("--parent-lib")
        parent = args[i + 1]
        del args[i:i + 2]
    path = args[0] if args else os.path.join(ROOT, "profiles", "r06_time_rollout_ic.txt")
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say(f"gpu: {gpu_identity()}")
    new = legacy_calls(native.load())
    old = legacy_calls(ctypes.CDLL(os.path.abspath(parent))) if parent else None
    say(f"parent build: {parent if parent else 'not given: no legacy comparison'}")
    for name, (d, p), M, N, n_rows, spr, dt in (("cfg-like", (2, 2), 40, 20, 99, 10, 0.002),
                                                ("large", (3, 5), 64, 4096, 200, 10, 0.001)):
        lib = native.Library(d, p)
        W = stable_models(lib, M, 1)
        g = torch.Generator(device="cuda").manual_seed(2)
        x0 = torch.rand(N, d, device="cuda", generator=g) - 0.5
        y = torch.randn(n_rows, N, d, device="cuda", generator=g) * 0.1
        nb = int(native.load().sb_rollout_score_grad_workspace_bytes(N, ctypes.byref(lib.c()), M, spr, n_rows))
        ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
        say(f"{name}: lib (d={d}, p={p}) K={lib.K}  {M} models x {N} ICs x {n_rows} rows x {spr} steps, RK4")
        if old:
            a, b = new[0](x0, W, lib, dt, spr, y), old[0](x0, W, lib, dt, spr, y)
            same_s = all(torch.equal(u, v) for u, v in zip(a, b))
            a, b = new[1](x0, W, lib, dt, spr, y, ws), old[1](x0, W, lib, dt, spr, y, ws)
            same_g = all(torch.equal(u, v) for u, v in zip(a, b))
            say(f"   legacy entry points against the parent build: sse/valid bitwise equal {same_s}, "
                f"sse/valid/grad bitwise equal {same_g}")
            for label, fn in (("sb_rollout_score", lambda c: c[0](x0, W, lib, dt, spr, y)),
                              ("sb_rollout_score_grad", lambda c: c[1](x0, W, lib, dt, spr, y, ws))):
                tn, to = [], []
                for _ in range(3):
                    tn.append(timed(lambda: fn(new))[0])
                    to.append(timed(lambda: fn(old))[0])
                mn, mo = statistics.median(tn), statistics.median(to)
                say(f"   {label}: this tree {mn:.3f} ms, parent {mo:.3f} ms (medians of 3 alternating rounds; "
                    f"this tree {min(tn):.3f}..{max(tn):.3f}, parent {min(to):.3f}..{max(to):.3f})  -> "
                    f"{(mn / mo - 1) * 100:+.1f} %")
        copies = x0.expand(M, N, d).contiguous()
        s_ms = timed(lambda: native.rollout_score(x0, W, lib, dt, spr, y))[0]
        p_ms = timed(lambda: native.rollout_score(copies, W, lib, dt, spr, y))[0]
        same = all(torch.equal(u, v) for u, v in zip(native.rollout_score(x0, W, lib, dt, spr, y),
                                                       native.rollout_score(copies, W, lib, dt, spr, y)))
        say(f"   rollout_score shared starts {s_ms:.3f} ms, per-model starts {p_ms:.3f} ms ({(p_ms / s_ms - 1) * 100:+.1f} %,"
            f" outputs bitwise equal {same})")
        gw = timed(lambda: native.rollout_score_grad(x0, W, lib, dt, spr, y))[0]
        gb = timed(lambda: native.rollout_score_grad(copies, W, lib, dt, spr, y, x0_grad=True))[0]
        gi = timed(lambda: native.rollout_score_grad(copies, W, lib, dt, spr, y, x0_grad=True, w_grad=False))[0]
        full = native.rollout_score_grad(copies, W, lib, dt, spr, y, x0_grad=True)
        only = native.rollout_score_grad(copies, W, lib, dt, spr, y, x0_grad=True, w_grad=False)
        same = torch.equal(full[0], only[0]) and torch.equal(full[1], only[1]) and torch.equal(full[3], only[3])
        say(f"   rollout_score_grad: W gradient {gw:.3f} ms, W + start gradients {gb:.3f} ms "
            f"({(gb / gw - 1) * 100:+.1f} %), start gradient only (start-only variant) {gi:.3f} ms "
            f"-> {gb / gi:.2f}x faster than the full variant (sse/valid/grad_x0 bitwise equal {same})")
        if name == "cfg-like":
            import sindy
            truth = torch.zeros(d, lib.K, device="cuda")
            truth[0, 2], truth[1, 1], truth[1, 2] = 1.0, -1.0, -0.1
            xs, _, _ = native.rollout(x0, truth, lib, dt, n_rows * spr, stride=spr, want_last=False)
            xf = torch.cat([x0.unsqueeze(0), xs], 0).transpose(0, 1).contiguous()
            xf = xf + 0.01 * torch.randn(xf.shape, device="cuda", generator=g)
            gm = torch.Generator().manual_seed(4)
            masks = (torch.rand(M, d, lib.K, generator=gm) > 0.4).cuda() | (truth != 0)
            xi = (truth + 0.05 * torch.randn(M, d, lib.K, generator=gm).cuda()) * masks
            cand = {"thresholds": torch.linspace(0, 1, M, dtype=torch.float64), "xi": xi, "mask": masks}
            for fit_ic in (False, True):
                sindy.refine_path(lib, cand, xf, dt, steps_per_row=spr, fit_ic=fit_ic)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = sindy.refine_path(lib, cand, xf, dt, steps_per_row=spr, fit_ic=fit_ic)
                torch.cuda.synchronize()
                r_ms = (time.perf_counter() - t0) * 1e3
                say(f"   refine_path(fit_ic={fit_ic}), {M} candidates, max_iter 50: {r_ms:.1f} ms wall clock, "
                    f"iterations {int(out['iterations'].min())}..{int(out['iterations'].max())}, SSE ratio "
                    f"after/before median {float((out['sse_after'] / out['sse_before']).median()):.3f}")
            for fit_ic in (False, True):
                sindy.score_path(lib, out, xf, dt, steps_per_row=spr, fit_ic=fit_ic)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                sc = sindy.score_path(lib, out, xf, dt, steps_per_row=spr, fit_ic=fit_ic)
                torch.cuda.synchronize()
                r_ms = (time.perf_counter() - t0) * 1e3
                say(f"   score_path(fit_ic={fit_ic}), {M} candidates{', ic_iter 20' if fit_ic else ''}: {r_ms:.1f} ms "
                    f"wall clock, median sse {float(sc['sse'].median()):.4g}")
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
