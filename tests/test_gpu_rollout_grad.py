"""GPU checks of the rollout-score gradient (sb_rollout_score_grad) and the trajectory refit (sindy.refine_path): scores
bitwise equal to sb_rollout_score, gradients against the fp64 autograd reference at short and long horizons, exact
zeros, divergence and truncation, bitwise determinism across batches and model order, and refits on synthetic and
golden data."""
import os

import numpy as np
import pytest
import torch

from rollout_fp64_ref import grad64

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DATA = os.path.join(ROOT, "tests", "golden", "data")

# the specialised shapes of SB_SPEC_SHAPES (config 3's (2, 2) + exp among them) and two runtime-table libraries
LIBS = [(2, 2, 0, 0), (2, 3, 0, 0), (3, 2, 0, 0), (3, 3, 0, 0), (3, 5, 0, 0), (2, 2, 0, 1), (2, 2, 1, 0), (4, 2, 0, 0)]


@pytest.fixture(scope="module")
def nat():
    from sindy_b200 import native
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    native.load()
    return native


def models(lib, M, seed, scale=0.3):
    g = torch.Generator().manual_seed(seed)
    W = scale * (6.0 / lib.K) ** 0.5 * torch.randn(M, lib.dim, lib.K, generator=g)
    W[:, :, 0] *= 0.1
    return W.cuda()


def ics(N, d, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(N, d, generator=g) - 0.5).cuda()


def _ref(x0, W, spec, dt, spr, y, method, rows=None):
    d, p, s, e = spec
    return torch.stack([grad64(x0, W[m], (d, p, bool(s), bool(e)), dt, spr, y, method,
                               None if rows is None else rows[m])[1] for m in range(W.shape[0])])


def _rel(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


@pytest.mark.parametrize("method", ["rk4", "euler"])
@pytest.mark.parametrize("spec", LIBS)
def test_scores_bitwise_and_gradient_against_fp64(nat, spec, method):
    d, p, s, e = spec
    lib = nat.Library(d, p, bool(s), bool(e))
    N, dt = 300, 0.01                                   # 300 ICs: a partly filled last block
    W = models(lib, 3, 10 * d + p)
    # for 2000 steps (t = 20) the random models are damped so that no pair leaves the bounds
    damped = 0.1 * W
    for i in range(d):
        damped[:, i, 1 + i] -= 0.5
    x0 = ics(N, d, 7)
    for n_rows, spr, tol in ((1, 1, 1e-4), (7, 3, 1e-4), (20, 100, 1e-3)):
        if n_rows == 20:
            W = damped
        y = torch.randn(n_rows, N, d, device="cuda") * 0.5
        sse0, valid0 = nat.rollout_score(x0, W, lib, dt, spr, y, method)
        sse, valid, g = nat.rollout_score_grad(x0, W, lib, dt, spr, y, method)
        assert torch.equal(sse, sse0) and torch.equal(valid, valid0)
        assert torch.all(valid == n_rows)
        err = _rel(g, _ref(x0, W, spec, dt, spr, y, method))
        print(f"{spec} {method} {n_rows}x{spr} steps: rel max-norm error {err:.2e}")
        # 2000 steps cross 63 checkpoint segments, the last one partial; the fp32 adjoint's rounding grows with the
        # horizon, hence the looser bound there
        assert err < tol, err


def test_own_trajectory_gives_exactly_zero(nat):
    lib = nat.Library(3, 3)
    W = models(lib, 2, 1)
    x0 = ics(200, 3, 2)
    traj, _, _ = nat.rollout(x0, W[0], lib, 0.01, 40 * 5, stride=5, method="rk4", want_last=False)
    sse, valid, g = nat.rollout_score_grad(x0, W, lib, 0.01, 5, traj, "rk4")
    assert torch.all(sse[0] == 0) and torch.all(g[0] == 0)
    assert torch.all(sse[1] > 0) and bool((g[1] != 0).any())


@pytest.mark.parametrize("blowup", [None, 50.0])
def test_divergent_pairs_truncate_the_gradient(nat, blowup):
    """ẋ0 = x0² (+ a small linear term in ẋ1): from x0 = 1 the solution leaves every bound at t = 1, from 0.5 at t = 2,
    from −1 it decays, and from 40 it leaves the bound of 50 within the first row. Each pair's gradient is that of its
    SSE over the rows it compared: the same bits as a run whose objective ends there, the fp64 reference truncated at
    the kernel's valid rows, and exactly nothing for a pair that stops at row 0; the batch is the sum of its pairs."""
    lib = nat.Library(2, 2)
    W = torch.zeros(1, 2, lib.K, device="cuda")
    W[0, 0, 3] = 1.0
    W[0, 1, 1] = 0.1
    x0 = torch.tensor([[1.0, 0.2], [0.5, 0.1], [-1.0, 0.3], [40.0, 0.0]], device="cuda")
    dt, spr, n_rows = 0.01, 5, 48
    y = torch.full((n_rows, 4, 2), 0.1, device="cuda")
    sse, valid, g = nat.rollout_score_grad(x0, W, lib, dt, spr, y, "rk4", blowup=blowup)
    sse0, valid0 = nat.rollout_score(x0, W, lib, dt, spr, y, "rk4", blowup=blowup)
    assert torch.equal(sse, sse0) and torch.equal(valid, valid0)
    v = valid[0].long().cpu()
    assert int(v[2]) == n_rows and int(v[0]) < n_rows and int(v[1]) < n_rows
    if blowup is not None:
        assert int(v[3]) == 0
    traj, _, _ = nat.rollout(x0, W[0], lib, dt, n_rows * spr, stride=spr, method="rk4", want_last=False)
    per = []
    for n in range(4):
        vn = int(v[n])
        xn, yn = x0[n:n + 1].contiguous(), y[:, n:n + 1].contiguous()
        _, valid_n, gn = nat.rollout_score_grad(xn, W, lib, dt, spr, yn, "rk4", blowup=blowup)
        assert int(valid_n) == vn
        per.append(gn)
        if vn == 0:
            assert torch.all(gn == 0)
            continue
        _, valid_t, gt = nat.rollout_score_grad(xn, W, lib, dt, spr, yn[:vn].contiguous(), "rk4", blowup=blowup)
        assert int(valid_t) == vn and torch.equal(gt, gn)
        err = _rel(gn, _ref(xn, W, (2, 2, 0, 0), dt, spr, yn, "rk4", rows=[v[n:n + 1].cuda()]))
        peak = float(traj[:vn, n].abs().max())
        print(f"blowup={blowup} x0={x0[n].tolist()}: {vn} rows, largest compared |x| {peak:.3g}, rel max-norm error "
              f"{err:.2e}")
        # Without the bound a pair runs into the finite-time blow-up and compares states far from the data; there the
        # fp32 trajectory's own rounding, amplified by the blow-up, separates it from the fp64 reference's by ~1e-4
        # relative, and the gradient with it. Moderate states keep the short-horizon accuracy.
        assert err < (1e-4 if peak <= 100.0 else 1e-3), err
    assert _rel(g, torch.stack(per).sum(0)) < 1e-12


def test_a_model_has_the_same_bits_in_every_batch(nat):
    lib = nat.Library(3, 5)
    M, N, spr, n_rows, dt = 200, 257, 2, 5, 0.01
    W = models(lib, M, 11, scale=0.05)
    x0 = ics(N, 3, 12)
    y = torch.randn(n_rows, N, 3, device="cuda") * 0.3
    sse, valid, g = nat.rollout_score_grad(x0, W, lib, dt, spr, y, "rk4")
    again = nat.rollout_score_grad(x0, W, lib, dt, spr, y, "rk4")
    assert torch.equal(sse, again[0]) and torch.equal(valid, again[1]) and torch.equal(g, again[2])
    perm = torch.randperm(M, generator=torch.Generator().manual_seed(0)).cuda()
    _, _, gp = nat.rollout_score_grad(x0, W[perm], lib, dt, spr, y, "rk4")
    assert torch.equal(gp, g[perm])
    m = 137
    _, _, alone = nat.rollout_score_grad(x0, W[m:m + 1], lib, dt, spr, y, "rk4")
    assert torch.equal(alone[0], g[m])
    _, _, part = nat.rollout_score_grad(x0, W[100:150], lib, dt, spr, y, "rk4")
    assert torch.equal(part[m - 100], g[m])


# ---- refine_path ------------------------------------------------------------------------------------------------------
def test_refine_path_synthetic(nat):
    import sindy
    lib = nat.Library(2, 3)
    truth = torch.zeros(2, lib.K)
    truth[0, 2] = 1.0                                    # ẋ0 = x1
    truth[1, 1], truth[1, 2], truth[1, 6] = -1.0, -0.1, -0.5   # ẋ1 = −x0 − 0.1 x1 − 0.5 x0³ (column 6 = x0³)
    g = torch.Generator().manual_seed(3)
    n_traj, T, spr, dt = 12, 60, 5, 0.01
    x0 = (torch.rand(n_traj, 2, generator=g) * 2 - 1).cuda()
    traj, _, _ = nat.rollout(x0, truth.cuda(), lib, dt, (T - 1) * spr, stride=spr, method="rk4", want_last=False)
    x = torch.cat([x0.unsqueeze(0), traj], 0).transpose(0, 1).contiguous()
    x = x + 0.01 * torch.randn(x.shape, generator=g).cuda()
    mask = truth != 0
    full = torch.ones_like(mask)
    start = truth * (1 + 0.2 * torch.randn(truth.shape, generator=g))
    start_full = start + 0.05 * torch.randn(truth.shape, generator=g)
    path = {"thresholds": torch.tensor([0.1, 0.0], dtype=torch.float64),
            "xi": torch.stack([start * mask, start_full]).cuda(), "mask": torch.stack([mask, full]).cuda()}
    out = sindy.refine_path(lib, path, x, dt, steps_per_row=spr, max_iter=40)
    assert torch.equal(out["mask"], path["mask"])
    assert torch.all(out["xi"][~out["mask"]] == 0)
    assert torch.all(out["sse_after"] <= out["sse_before"])
    e0 = float((path["xi"][0].cpu() - truth).norm())
    e1 = float((out["xi"][0].cpu() - truth).norm())
    print(f"true support: |Ξ − truth| {e0:.3e} -> {e1:.3e}, sse {out['sse_before'].tolist()} -> "
          f"{out['sse_after'].tolist()}, iterations {out['iterations'].tolist()}")
    assert e1 < 0.2 * e0


def _golden(name):
    return torch.load(os.path.join(DATA, f"{name}-gp-x.pt")), torch.load(os.path.join(DATA, f"{name}-gp-dx.pt"))


def test_refine_path_constrained_stays_in_the_constraint_space(nat):
    import sindy
    import sweep
    x, dx = _golden("dosc-train-noise20")
    torch.manual_seed(0)
    so2 = torch.tensor([[0.0, 1.0], [-1.0, 0.0]])
    reg = sindy.SINDyRegression(2, 2, False, False, L_list=[so2], threshold=0.05, device="cuda",
                                constrain_constant=False)
    path = sindy.stlsq_path(reg, x.reshape(-1, 2).cuda(), dx.reshape(-1, 2).cuda(), np.logspace(-3, 0, 8))
    xf = x[:6].cuda()
    out = sindy.refine_path(reg, path, xf, 0.002, steps_per_row=100, max_iter=10)
    assert torch.equal(out["mask"], path["mask"]) and torch.all(out["sse_after"] <= out["sse_before"])
    A, _ = sweep.param_map(reg)
    for i in range(out["xi"].shape[0]):
        p = torch.cat([out["beta"][i].reshape(-1), out["const"][i].reshape(-1)]).double()
        want = ((A @ p).view(2, -1) * out["mask"][i]).float()
        assert torch.allclose(out["xi"][i], want, atol=1e-6)
        sindy.apply_candidate(reg, out, i)
        assert torch.allclose(reg.get_Xi() * reg.mask, out["xi"][i], atol=1e-6)


@pytest.mark.parametrize("case", [("growth", "noise05", 10), ("dosc", "noise20", 100)])
def test_refit_then_score_on_golden_data(nat, golden, case):
    import sindy
    system, noise, spr = case
    x, dx = _golden(f"{system}-train-{noise}")
    xv = torch.load(os.path.join(DATA, f"{system}-val-{noise}-gp-x.pt")).cuda()
    reg = sindy.SINDyRegression(2, 2, False, False, threshold=0.05, device="cuda", constrain_constant=True)
    path = sindy.stlsq_path(reg, x.reshape(-1, 2).cuda(), dx.reshape(-1, 2).cuda(), np.logspace(-3, 0, 40))
    out = sindy.refine_path(reg, path, x.cuda(), 0.002, steps_per_row=spr)
    assert torch.equal(out["mask"], path["mask"])
    assert torch.all(out["sse_after"] <= out["sse_before"])
    truth = golden("model")[f"truth_{system}"] != 0
    is_truth = torch.from_numpy(np.all(path["mask"].cpu().numpy() == truth, axis=(1, 2)))
    for name, p in (("before", path), ("after", out)):
        sc = sindy.score_path(reg, p, xv, 0.002, steps_per_row=spr)
        i = sc["chosen"]
        a = sc["aicc"]
        print(f"{system}/{noise} {name} refit: chosen k={int(sc['k'][i])} truth={bool(is_truth[i])} "
              f"AICc(truth)={float(a[is_truth].min()) if is_truth.any() else float('nan'):.1f} "
              f"AICc(best other)={float(a[~is_truth].min()):.1f}")
