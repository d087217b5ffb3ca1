"""GPU checks of start estimation: the per-model-start and start-gradient entry points (sb_rollout_score_ics,
sb_rollout_score_grad_ics) bitwise against the shared-start ones and against themselves, ∂sse/∂x0 against the fp64
autograd reference, truncation and determinism, and refine_path / score_path with fit_ic on synthetic, constrained,
golden and seeded raw-noise data."""
import os

import numpy as np
import pytest
import torch

from rollout_ic_fp64_ref import grad_x0_64

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DATA = os.path.join(ROOT, "tests", "golden", "data")

# the libraries of test_gpu_rollout_grad.py: every specialised shape and two runtime-table libraries
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


def ics(N, d, seed, M=None):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(*((M,) if M else ()), N, d, generator=g) - 0.5).cuda()


def _rel(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-300))


@pytest.mark.parametrize("method", ["rk4", "euler"])
@pytest.mark.parametrize("spec", LIBS)
def test_start_gradient_bitwise_and_against_fp64(nat, spec, method):
    d, p, s, e = spec
    lib = nat.Library(d, p, bool(s), bool(e))
    N, M, dt = 300, 3, 0.01
    W = models(lib, M, 10 * d + p)
    damped = 0.1 * W
    for i in range(d):
        damped[:, i, 1 + i] -= 0.5
    x0 = ics(N, d, 7)
    xm = ics(N, d, 8, M=M)
    for n_rows, spr, tol in ((1, 1, 1e-4), (7, 3, 1e-4), (20, 100, 1e-3)):
        if n_rows == 20:
            W = damped
        y = torch.randn(n_rows, N, d, device="cuda") * 0.5
        sse0, valid0 = nat.rollout_score(x0, W, lib, dt, spr, y, method)
        sse_l, valid_l, g_l = nat.rollout_score_grad(x0, W, lib, dt, spr, y, method)
        # the new entry points with shared starts are the legacy ones
        sse, valid, g, gx = nat.rollout_score_grad(x0, W, lib, dt, spr, y, method, x0_grad=True)
        assert torch.equal(sse, sse_l) and torch.equal(valid, valid_l) and torch.equal(g, g_l)
        assert torch.equal(sse, sse0) and torch.equal(valid, valid0)
        # per-model starts that are copies of the shared set
        copies = x0.expand(M, N, d).contiguous()
        s2, v2 = nat.rollout_score(copies, W, lib, dt, spr, y, method)
        assert torch.equal(s2, sse0) and torch.equal(v2, valid0)
        s3, v3, g3, gx3 = nat.rollout_score_grad(copies, W, lib, dt, spr, y, method, x0_grad=True)
        assert torch.equal(s3, sse) and torch.equal(v3, valid) and torch.equal(g3, g) and torch.equal(gx3, gx)
        # the start-only variant: same sse, valid and grad_x0 bits
        s4, v4, g4, gx4 = nat.rollout_score_grad(copies, W, lib, dt, spr, y, method, x0_grad=True, w_grad=False)
        assert g4 is None and torch.equal(s4, sse) and torch.equal(v4, valid) and torch.equal(gx4, gx)
        assert torch.all(valid == n_rows)
        # distinct per-model starts: model m as if run alone from its own starts
        sm, vm, gm, gxm = nat.rollout_score_grad(xm, W, lib, dt, spr, y, method, x0_grad=True)
        for m in range(M):
            a = nat.rollout_score_grad(xm[m], W[m:m + 1], lib, dt, spr, y, method, x0_grad=True)
            assert torch.equal(a[0][0], sm[m]) and torch.equal(a[1][0], vm[m]) and torch.equal(a[3][0], gxm[m])
            b = nat.rollout_score(xm[m], W[m:m + 1], lib, dt, spr, y, method)
            assert torch.equal(b[0][0], sm[m])
        # against the reference with distinct per-model starts (shared starts are their copies, bit for bit, above)
        err = _rel(gxm, grad_x0_64(xm, W, (d, p, bool(s), bool(e)), dt, spr, y, method)[1])
        print(f"{spec} {method} {n_rows}x{spr} steps: grad_x0 rel max-norm error {err:.2e}")
        # the tolerances of test_gpu_rollout_grad.py's W gradient (the same fp32 adjoint, read at step 0); measured on a
        # B200: at most 1.8e-6 at 20 x 100 steps, 7.5e-7 at 7 x 3 steps
        assert err < tol, err


@pytest.mark.parametrize("blowup", [None, 50.0])
def test_truncated_pairs(nat, blowup):
    """The system of test_gpu_rollout_grad.py's truncation test: ẋ0 = x0² leaves every bound from x0 = 1 and 0.5, and
    from 40 leaves the bound of 50 within the first row. A pair's start gradient is that of the run whose objective
    ends at its valid rows, and exactly zero for a pair that stops at row 0."""
    lib = nat.Library(2, 2)
    W = torch.zeros(1, 2, lib.K, device="cuda")
    W[0, 0, 3] = 1.0
    W[0, 1, 1] = 0.1
    x0 = torch.tensor([[1.0, 0.2], [0.5, 0.1], [-1.0, 0.3], [40.0, 0.0]], device="cuda")
    dt, spr, n_rows = 0.01, 5, 48
    y = torch.full((n_rows, 4, 2), 0.1, device="cuda")
    sse, valid, _, gx = nat.rollout_score_grad(x0, W, lib, dt, spr, y, "rk4", blowup=blowup, x0_grad=True)
    v = valid[0].long().cpu()
    assert int(v[2]) == n_rows and int(v[0]) < n_rows and int(v[1]) < n_rows
    if blowup is not None:
        assert int(v[3]) == 0 and torch.all(gx[0, 3] == 0)
    for n in range(4):
        vn = int(v[n])
        xn, yn = x0[n:n + 1].contiguous(), y[:, n:n + 1].contiguous()
        if vn == 0:
            continue
        _, valid_t, _, gt = nat.rollout_score_grad(xn, W, lib, dt, spr, yn[:vn].contiguous(), "rk4", blowup=blowup,
                                                   x0_grad=True, w_grad=False)
        assert int(valid_t) == vn and torch.equal(gt[0, 0], gx[0, n])


def test_start_gradient_is_deterministic(nat):
    lib = nat.Library(3, 5)
    M, N, spr, n_rows, dt = 200, 257, 2, 5, 0.01
    W = models(lib, M, 11, scale=0.05)
    x0 = ics(N, 3, 12)
    y = torch.randn(n_rows, N, 3, device="cuda") * 0.3
    _, _, _, gx = nat.rollout_score_grad(x0, W, lib, dt, spr, y, "rk4", x0_grad=True)
    again = nat.rollout_score_grad(x0, W, lib, dt, spr, y, "rk4", x0_grad=True)[3]
    assert torch.equal(gx, again)
    perm = torch.randperm(M, generator=torch.Generator().manual_seed(0)).cuda()
    assert torch.equal(nat.rollout_score_grad(x0, W[perm], lib, dt, spr, y, "rk4", x0_grad=True)[3], gx[perm])
    assert torch.equal(nat.rollout_score_grad(x0, W[100:150], lib, dt, spr, y, "rk4", x0_grad=True)[3], gx[100:150])
    # one writer per element and no sum: an IC split gives the same bits, unlike the W gradient
    lo = nat.rollout_score_grad(x0[:100], W, lib, dt, spr, y[:, :100].contiguous(), "rk4", x0_grad=True)[3]
    hi = nat.rollout_score_grad(x0[100:], W, lib, dt, spr, y[:, 100:].contiguous(), "rk4", x0_grad=True,
                                w_grad=False)[3]
    assert torch.equal(torch.cat([lo, hi], 1), gx)


# ---- refine_path / score_path -----------------------------------------------------------------------------------------
def _synthetic(nat, seed=3, noise=0.01):
    """The system of test_gpu_rollout_grad.py's test_refine_path_synthetic, with seeded noise on every row, row 0
    included. Returns (lib, truth, path, x, x0_true)."""
    lib = nat.Library(2, 3)
    truth = torch.zeros(2, lib.K)
    truth[0, 2] = 1.0
    truth[1, 1], truth[1, 2], truth[1, 6] = -1.0, -0.1, -0.5
    g = torch.Generator().manual_seed(seed)
    n_traj, T, spr, dt = 12, 60, 5, 0.01
    x0 = (torch.rand(n_traj, 2, generator=g) * 2 - 1).cuda()
    traj, _, _ = nat.rollout(x0, truth.cuda(), lib, dt, (T - 1) * spr, stride=spr, method="rk4", want_last=False)
    x = torch.cat([x0.unsqueeze(0), traj], 0).transpose(0, 1).contiguous()
    x = x + noise * torch.randn(x.shape, generator=g).cuda()
    mask = truth != 0
    full = torch.ones_like(mask)
    start = truth * (1 + 0.2 * torch.randn(truth.shape, generator=g))
    start_full = start + 0.05 * torch.randn(truth.shape, generator=g)
    path = {"thresholds": torch.tensor([0.1, 0.0], dtype=torch.float64),
            "xi": torch.stack([start * mask, start_full]).cuda(), "mask": torch.stack([mask, full]).cuda()}
    return lib, truth, path, x, x0


def test_refine_path_estimates_the_starts(nat):
    import sindy
    lib, truth, path, x, x0_true = _synthetic(nat)
    spr, dt = 5, 0.01
    fixed = sindy.refine_path(lib, path, x, dt, steps_per_row=spr, max_iter=40)
    fit = sindy.refine_path(lib, path, x, dt, steps_per_row=spr, max_iter=40, fit_ic=True)
    assert torch.equal(fit["sse_before"], fixed["sse_before"])
    assert torch.equal(fit["mask"], path["mask"]) and torch.all(fit["xi"][~fit["mask"]] == 0)
    assert torch.all(fit["sse_after"] <= fit["sse_before"])
    assert fit["x0"].shape == (2, 12, 2)
    e_fixed = float((fixed["xi"][0].cpu() - truth).norm())
    e_fit = float((fit["xi"][0].cpu() - truth).norm())
    d_row0 = float((x[:, 0] - x0_true).norm(dim=1).mean())
    d_fit = float((fit["x0"][0] - x0_true).norm(dim=1).mean())
    print(f"true support: |Ξ − truth| fixed start {e_fixed:.3e}, fitted starts {e_fit:.3e}; mean |x0 − truth| row 0 "
          f"{d_row0:.3e}, x̂0 {d_fit:.3e}; iterations {fit['iterations'].tolist()}")
    assert e_fit < e_fixed
    assert d_fit < d_row0
    # window = T is no window at all, bit for bit
    again = sindy.refine_path(lib, path, x, dt, steps_per_row=spr, max_iter=5, window=60)
    base = sindy.refine_path(lib, path, x, dt, steps_per_row=spr, max_iter=5)
    for key in ("xi", "sse_before", "sse_after", "iterations"):
        assert torch.equal(again[key], base[key]), key
    win = sindy.refine_path(lib, path, x, dt, steps_per_row=spr, max_iter=5, window=20, fit_ic=True)
    assert win["x0"].shape == (2, 36, 2) and torch.all(win["sse_after"] <= win["sse_before"])


def _golden(name):
    return torch.load(os.path.join(DATA, f"{name}-gp-x.pt")), torch.load(os.path.join(DATA, f"{name}-gp-dx.pt"))


def test_refine_path_constrained_with_starts(nat):
    import sindy
    import sweep
    x, dx = _golden("dosc-train-noise20")
    torch.manual_seed(0)
    so2 = torch.tensor([[0.0, 1.0], [-1.0, 0.0]])
    reg = sindy.SINDyRegression(2, 2, False, False, L_list=[so2], threshold=0.05, device="cuda",
                                constrain_constant=False)
    path = sindy.stlsq_path(reg, x.reshape(-1, 2).cuda(), dx.reshape(-1, 2).cuda(), np.logspace(-3, 0, 8))
    xf = x[:6].cuda()
    out = sindy.refine_path(reg, path, xf, 0.002, steps_per_row=100, max_iter=10, fit_ic=True)
    assert torch.equal(out["mask"], path["mask"]) and torch.all(out["sse_after"] <= out["sse_before"])
    A, _ = sweep.param_map(reg)
    for i in range(out["xi"].shape[0]):
        p = torch.cat([out["beta"][i].reshape(-1), out["const"][i].reshape(-1)]).double()
        want = ((A @ p).view(2, -1) * out["mask"][i]).float()
        assert torch.allclose(out["xi"][i], want, atol=1e-6)


def _check_scores(fixed, fit):
    """score_path(fit_ic=True) against fixed starts: every candidate's sse at most its fixed-start sse, and diverged a
    subset of the fixed-start diverged."""
    ok = ~fixed["diverged"]
    assert torch.all(fit["sse"][ok] <= fixed["sse"][ok])
    assert not bool((fit["diverged"] & ~fixed["diverged"]).any())
    assert torch.equal(fit["k"], fixed["k"])


def _report(tag, sc, is_truth):
    i = sc["chosen"]
    a = sc["aicc"]
    truth = float(a[is_truth].min()) if is_truth.any() else float("nan")
    print(f"{tag}: chosen k={int(sc['k'][i]) if i is not None else -1} "
          f"truth={bool(is_truth[i]) if i is not None else False} AICc(truth)={truth:.1f} "
          f"AICc(best other)={float(a[~is_truth].min()):.1f}")


def _select(nat, golden, system, x, dx, xv, spr, tag):
    import sindy
    reg = sindy.SINDyRegression(2, 2, False, False, threshold=0.05, device="cuda", constrain_constant=True)
    path = sindy.stlsq_path(reg, x.reshape(-1, 2).cuda(), dx.reshape(-1, 2).cuda(), np.logspace(-3, 0, 40))
    truth = golden("model")[f"truth_{system}"] != 0
    is_truth = torch.from_numpy(np.all(path["mask"].cpu().numpy() == truth, axis=(1, 2)))
    xc = x.cuda()
    for fit_ic in (False, True):
        out = sindy.refine_path(reg, path, xc, 0.002, steps_per_row=spr, fit_ic=fit_ic)
        assert torch.equal(out["mask"], path["mask"]) and torch.all(out["sse_after"] <= out["sse_before"])
        for p, stage in ((path, "before"), (out, "after")):
            fixed = sindy.score_path(reg, p, xv, 0.002, steps_per_row=spr)
            fit = sindy.score_path(reg, p, xv, 0.002, steps_per_row=spr, fit_ic=True)
            _check_scores(fixed, fit)
            assert fit["x0"].shape == (len(p["thresholds"]), xv.shape[0], 2)
            _report(f"{tag} refit({'fit_ic' if fit_ic else 'fixed'}) {stage}, fixed-start score", fixed, is_truth)
            _report(f"{tag} refit({'fit_ic' if fit_ic else 'fixed'}) {stage}, fit_ic score", fit, is_truth)


@pytest.mark.parametrize("case", [("growth", "noise05", 10), ("dosc", "noise20", 100)])
def test_selection_with_starts_on_golden_data(nat, golden, case):
    system, noise, spr = case
    x, dx = _golden(f"{system}-train-{noise}")
    xv = torch.load(os.path.join(DATA, f"{system}-val-{noise}-gp-x.pt")).cuda()
    _select(nat, golden, system, x, dx, xv, spr, f"{system}/{noise} GP")


@pytest.mark.parametrize("case", [("growth", 0.05, 10), ("dosc", 0.20, 100)])
def test_selection_with_starts_on_raw_noise(nat, golden, case):
    """The same two systems on seeded raw-noise trajectories (the sizes, row spacing and noise level of the golden
    sets, starts drawn uniformly over the golden starts' range): the threshold path from GP derivatives of that draw,
    refit and scores on its raw rows."""
    from data_utils import systems
    from data_utils.ode import gen_data
    from data_utils.smoothing import num_diff_gp
    system, sigma, spr = case
    ref_x, _ = _golden(f"{system}-train-noise{int(round(sigma * 100)):02d}")
    ref_v = torch.load(os.path.join(DATA, f"{system}-val-noise{int(round(sigma * 100)):02d}-gp-x.pt"))
    lo, hi = ref_x[:, 0].min(0).values.numpy(), ref_x[:, 0].max(0).values.numpy()
    ode, T = getattr(systems, system)(), ref_x.shape[1]
    np.random.seed(1234)

    def draw(n):
        return gen_data(ode, lambda k: np.random.uniform(lo, hi, (k, 2)), n_ics=n, dt=0.002, num_steps=T * spr,
                        subsample_rate=spr, noise=sigma, smoothing=None)[0]

    x, xv = draw(ref_x.shape[0]), draw(ref_v.shape[0])
    seq = np.ascontiguousarray(np.transpose(x, (1, 0, 2)))
    dx, _ = num_diff_gp(seq, 0.002 * spr, noise_level=sigma, std_base=np.std(seq, axis=(0, 1)))
    x = torch.as_tensor(x, dtype=torch.float32)
    dx = torch.as_tensor(np.transpose(dx, (1, 0, 2)), dtype=torch.float32)
    _select(nat, golden, system, x, dx, torch.as_tensor(xv, dtype=torch.float32).cuda(), spr,
            f"{system}/σ={sigma} raw")


def test_score_path_window_none_is_window_t(nat):
    import sindy
    lib, truth, path, x, _ = _synthetic(nat)
    a = sindy.score_path(lib, path, x, 0.01, steps_per_row=5)
    b = sindy.score_path(lib, path, x, 0.01, steps_per_row=5, window=60)
    for key in ("sse", "diverged", "aicc", "n_obs"):
        assert (a[key] == b[key]) if key == "n_obs" else torch.equal(a[key], b[key]), key
    w = sindy.score_path(lib, path, x, 0.01, steps_per_row=5, window=20, fit_ic=True, ic_iter=10)
    assert w["n_obs"] == 36 * 20 * 2 and w["k_ic"] == 36 * 2 and w["x0"].shape == (2, 36, 2)
