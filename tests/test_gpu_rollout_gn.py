"""GPU checks of the Gauss–Newton information of the rollout scores (sb_rollout_score_gn) and of
sindy.coefficient_covariance: the scores bitwise against the scorer, F / g against the fp64 forward-mode reference,
forward against reverse (the adjoint gradient kernel), padding, truncation, determinism, the column cap, the calibration
of the standard errors over seeded noise draws, the constrained parameter map and a report on golden data."""
import math
import os

import numpy as np
import pytest
import torch

from rollout_gn_fp64_ref import gn64
from test_gpu_rollout_ic import LIBS, _golden

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DATA = os.path.join(ROOT, "tests", "golden", "data")


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


def _params(dK, n, seed, M):
    """M rows of n distinct indices into d·K (n ≤ dK) and one padding slot each."""
    g = torch.Generator().manual_seed(seed)
    rows = [torch.cat([torch.randperm(dK, generator=g)[:n], torch.tensor([-1])]) for _ in range(M)]
    return torch.stack(rows).to(torch.int32).cuda()


@pytest.mark.parametrize("method", ["rk4", "euler"])
@pytest.mark.parametrize("spec", LIBS)
def test_information_bitwise_scores_and_against_fp64(nat, spec, method):
    d, p, s, e = spec
    lib = nat.Library(d, p, bool(s), bool(e))
    lt = (d, p, bool(s), bool(e))
    N, M, dt = 40, 2, 0.01
    W = models(lib, M, 10 * d + p)
    damped = 0.1 * W
    for i in range(d):
        damped[:, i, 1 + i] -= 0.5
    x0 = ics(N, d, 7)
    xm = ics(N, d, 8, M=M)
    prm = _params(d * lib.K, min(d * lib.K, 12), d + p, M)
    for n_rows, spr, tol in ((1, 1, 1e-4), (7, 3, 1e-4), (20, 100, 1e-3)):
        if n_rows == 20:
            W = damped
        y = torch.randn(n_rows, N, d, device="cuda") * 0.5
        # the scores: bit-identical to the scorer, shared and per-model starts
        sse0, valid0 = nat.rollout_score(x0, W, lib, dt, spr, y, method)
        out = nat.rollout_score_gn(x0, W, prm, lib, dt, spr, y, method)
        assert torch.equal(out["sse"], sse0) and torch.equal(out["valid_rows"], valid0)
        ssem, validm = nat.rollout_score(xm, W, lib, dt, spr, y, method)
        gx = nat.rollout_score_gn(xm, W, prm, lib, dt, spr, y, method, x0_blocks=True)
        assert torch.equal(gx["sse"], ssem) and torch.equal(gx["valid_rows"], validm)
        assert torch.all(validm == n_rows)
        # the θ sums do not depend on whether the start blocks are asked for (same n_params) up to the grouping
        errs = {}
        for m in range(M):
            ref = gn64(xm[m], W[m], prm[m], lt, dt, spr, y, method)
            for key in ("jtj", "jtr", "jtj_px", "jtj_xx", "jtr_x"):
                errs[key] = max(errs.get(key, 0.0), _rel(gx[key][m], ref[key]))
        # forward against reverse: 2·g_θ is the adjoint's ∂sse/∂W on the listed entries, 2·g_x its ∂sse/∂x0
        _, _, gw, gx0 = nat.rollout_score_grad(xm, W, lib, dt, spr, y, method, x0_grad=True)
        live = prm >= 0
        g_list = torch.gather(gw.reshape(M, -1), 1, prm.clamp_min(0).long())
        fr = max(_rel(2 * gx["jtr"][live], g_list[live]), _rel(2 * gx["jtr_x"], gx0))
        print(f"{spec} {method} {n_rows}x{spr} steps: rel max-norm error " +
              " ".join(f"{k} {v:.2e}" for k, v in errs.items()) + f"; forward vs reverse {fr:.2e}")
        assert max(errs.values()) < tol, errs
        assert fr < 1e-5, fr
        # F_θθ is symmetric bit for bit
        assert torch.equal(gx["jtj"], gx["jtj"].transpose(1, 2))


@pytest.mark.parametrize("blowup", [None, 50.0])
def test_padding_and_truncated_pairs(nat, blowup):
    """The system of test_gpu_rollout_ic.py's truncation test (ẋ0 = x0² leaves every bound from x0 = 1 and 0.5; from
    40 it leaves the bound of 50 within the first row). A pair contributes the rows it reports; padded indices give
    exact-zero rows and columns; a pair with valid_rows = 0 gets exact zeros."""
    lib = nat.Library(2, 2)
    W = torch.zeros(1, 2, lib.K, device="cuda")
    W[0, 0, 3] = 1.0
    W[0, 1, 1] = 0.1
    x0 = torch.tensor([[1.0, 0.2], [0.5, 0.1], [-1.0, 0.3], [40.0, 0.0]], device="cuda")
    dt, spr, n_rows = 0.01, 5, 48
    y = torch.full((n_rows, 4, 2), 0.1, device="cuda")
    prm = torch.tensor([[3, -1, 7, 1, -1]], dtype=torch.int32, device="cuda")
    out = nat.rollout_score_gn(x0, W, prm, lib, dt, spr, y, "rk4", blowup=blowup, x0_blocks=True)
    sse, valid = nat.rollout_score(x0, W, lib, dt, spr, y, "rk4", blowup=blowup)
    assert torch.equal(out["sse"], sse) and torch.equal(out["valid_rows"], valid)
    v = valid[0].long().cpu()
    assert int(v[2]) == n_rows and int(v[0]) < n_rows and int(v[1]) < n_rows
    pad = (prm[0] < 0).nonzero().flatten()
    assert torch.all(out["jtj"][0, pad] == 0) and torch.all(out["jtj"][0, :, pad] == 0)
    assert torch.all(out["jtr"][0, pad] == 0) and torch.all(out["jtj_px"][0, :, pad] == 0)
    if blowup is not None:
        assert int(v[3]) == 0
        for key in ("jtj_px", "jtj_xx", "jtr_x"):
            assert torch.all(out[key][0, 3] == 0), key
    ref = gn64(x0, W[0], prm[0], (2, 2, False, False), dt, spr, y, "rk4", rows=v)
    # without a bound the last rows of the escaping pairs are within a few steps of overflow, where the tangents grow
    # like x0² and fp32 loses digits: the tolerance of the long horizon
    tol = 1e-4 if blowup is not None else 1e-3
    for key in ("jtj", "jtr", "jtj_px", "jtj_xx", "jtr_x"):
        err = _rel(out[key][0], ref[key])
        print(f"blowup={blowup} {key}: rel max-norm error {err:.2e}")
        assert err < tol, (key, err)
    # a pair's own blocks are its rows alone: the same bits as a run that ends at its valid rows
    for n in range(4):
        vn = int(v[n])
        if vn == 0:
            continue
        alone = nat.rollout_score_gn(x0[n:n + 1].contiguous(), W, prm, lib, dt, spr, y[:vn, n:n + 1].contiguous(),
                                     "rk4", blowup=blowup, x0_blocks=True)
        for key in ("jtj_px", "jtj_xx", "jtr_x"):
            assert torch.equal(alone[key][0, 0], out[key][0, n]), key


def test_information_is_deterministic(nat):
    lib = nat.Library(3, 5)
    M, N, spr, n_rows, dt = 200, 257, 2, 5, 0.01
    W = models(lib, M, 11, scale=0.05)
    x0 = ics(N, 3, 12)
    y = torch.randn(n_rows, N, 3, device="cuda") * 0.3
    prm = _params(3 * lib.K, 20, 13, M)
    xm = ics(N, 3, 14, M=M)
    for x, xb in ((x0, False), (xm, True)):
        a = nat.rollout_score_gn(x, W, prm, lib, dt, spr, y, "rk4", x0_blocks=xb)
        again = nat.rollout_score_gn(x, W, prm, lib, dt, spr, y, "rk4", x0_blocks=xb)
        perm = torch.arange(M - 1, -1, -1, device="cuda")
        rev = nat.rollout_score_gn(x[perm] if xb else x, W[perm], prm[perm], lib, dt, spr, y, "rk4", x0_blocks=xb)
        part = nat.rollout_score_gn(x[100:150] if xb else x, W[100:150], prm[100:150], lib, dt, spr, y, "rk4",
                                    x0_blocks=xb)
        alone = nat.rollout_score_gn(x[7:8] if xb else x, W[7:8], prm[7:8], lib, dt, spr, y, "rk4", x0_blocks=xb)
        for key in a:
            assert torch.equal(a[key], again[key]), key
            assert torch.equal(rev[key], a[key][perm]), key
            assert torch.equal(part[key], a[key][100:150]), key
            assert torch.equal(alone[key], a[key][7:8]), key


def test_full_candidate_with_starts_and_the_cap(nat):
    """(3,5)'s densest candidate, all 168 coefficients and 3 starts (171 tangent columns), runs and agrees with the
    adjoint; a list above the cap is a ValueError from the binding."""
    lib = nat.Library(3, 5)
    W = models(lib, 2, 21, scale=0.05)
    x0 = ics(64, 3, 22, M=2)
    y = torch.randn(4, 64, 3, device="cuda") * 0.3
    prm = torch.arange(168, dtype=torch.int32, device="cuda").expand(2, -1)
    out = nat.rollout_score_gn(x0, W, prm, lib, 0.01, 3, y, "rk4", x0_blocks=True)
    _, _, gw, gx0 = nat.rollout_score_grad(x0, W, lib, 0.01, 3, y, "rk4", x0_grad=True)
    err = max(_rel(2 * out["jtr"], gw.reshape(2, -1)), _rel(2 * out["jtr_x"], gx0))
    print(f"(3,5) dense + starts: forward vs reverse {err:.2e}")
    assert err < 1e-5
    assert torch.isfinite(out["jtj"]).all() and torch.equal(out["jtj"], out["jtj"].transpose(1, 2))
    over = torch.cat([prm, prm[:, :6]], 1)
    with pytest.raises(ValueError):
        nat.rollout_score_gn(x0, W, over, lib, 0.01, 3, y, "rk4", x0_blocks=True)
    with pytest.raises(ValueError):
        nat.rollout_score_gn(x0, W, torch.cat([prm, prm[:, :9]], 1), lib, 0.01, 3, y, "rk4")


# ---- coefficient_covariance ------------------------------------------------------------------------------------------
def _calibration_system(nat):
    """test_gpu_rollout_ic.py::_synthetic's system and starts: ẋ0 = x1, ẋ1 = −x0 − 0.1·x1 − 0.5·x0³, 12 trajectories
    of 60 rows, 5 RK4 steps of 0.01 apart."""
    lib = nat.Library(2, 3)
    truth = torch.zeros(2, lib.K)
    truth[0, 2] = 1.0
    truth[1, 1], truth[1, 2], truth[1, 6] = -1.0, -0.1, -0.5
    g = torch.Generator().manual_seed(3)
    n_traj, T, spr, dt = 12, 60, 5, 0.01
    x0 = (torch.rand(n_traj, 2, generator=g) * 2 - 1).cuda()
    traj, _, _ = nat.rollout(x0, truth.cuda(), lib, dt, (T - 1) * spr, stride=spr, method="rk4", want_last=False)
    clean = torch.cat([x0.unsqueeze(0), traj], 0).transpose(0, 1).contiguous()
    return lib, truth, clean, spr, dt


def test_standard_errors_are_calibrated(nat):
    """100 seeded noise draws (σ = 0.01 on every row, row 0 included) of one system: per live coefficient the spread of
    the refit estimates against the median predicted stderr, and the coverage of the 95 % normal intervals."""
    import sindy
    lib, truth, clean, spr, dt = _calibration_system(nat)
    mask = truth != 0
    est, se = [], []
    for k in range(100):
        g = torch.Generator().manual_seed(1000 + k)
        x = clean + 0.01 * torch.randn(clean.shape, generator=g).cuda()
        path = {"thresholds": torch.tensor([0.1], dtype=torch.float64), "xi": (truth * mask).unsqueeze(0).cuda(),
                "mask": mask.unsqueeze(0).cuda()}
        fit = sindy.refine_path(lib, path, x, dt, steps_per_row=spr, max_iter=200, tol=1e-12, fit_ic=True)
        cc = sindy.coefficient_covariance(lib, fit, x, dt, steps_per_row=spr, fit_ic=True)
        assert bool(cc["identifiable"][0]) and not bool(cc["diverged"][0])
        est.append(fit["xi"][0].cpu().double()[mask])
        se.append(cc["stderr"][0][mask])
    est, se = torch.stack(est), torch.stack(se)
    sd = est.std(0)
    ratio = sd / se.median(0).values
    cover = float(((est - truth[mask].double()).abs() <= 1.96 * se).double().mean())
    print(f"calibration over 100 draws: empirical sd / median stderr per coefficient {ratio.tolist()}; "
          f"95 % interval coverage {cover:.3f} of {est.numel()}")
    assert torch.all(ratio >= 0.75) and torch.all(ratio <= 1.33), ratio
    assert 0.90 <= cover <= 0.99, cover


def test_constrained_covariance_lies_in_the_parameter_range(nat):
    """The SO(2) dosc regressor of test_gpu_rollout_ic.py::test_refine_path_constrained_with_starts: the covariance of
    vec(Ξ) lies in the range of the parameter map restricted to the live coefficients, diag(mask)·A."""
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
    cc = sindy.coefficient_covariance(reg, out, xf, 0.002, steps_per_row=100, fit_ic=True)
    A, _ = sweep.param_map(reg)
    A = A.cpu()
    n_checked = 0
    for i in range(out["xi"].shape[0]):
        if not bool(cc["identifiable"][i]) or bool(cc["diverged"][i]) or not bool(out["mask"][i].any()):
            continue
        Am = A * out["mask"][i].reshape(-1, 1).cpu().double()
        proj = torch.eye(A.shape[0], dtype=torch.float64) - Am @ torch.linalg.pinv(Am)
        c = cc["cov"][i]
        err = float((proj @ c).abs().max() / c.abs().max())
        print(f"candidate {i}: {int(out['mask'][i].sum())} live, |(I − A A⁺) cov| / |cov| = {err:.1e}, "
              f"cond {float(cc['cond'][i]):.2e}")
        assert err < 1e-10
        assert torch.all(c[~out["mask"][i].reshape(-1).cpu()] == 0)
        n_checked += 1
    assert n_checked > 0


@pytest.mark.parametrize("case", [("growth", "noise05", 10), ("dosc", "noise20", 100)])
def test_golden_report(nat, case):
    """stlsq_path → refine_path(fit_ic) → score_path(fit_ic) on golden data; the AICc-chosen candidate's coefficients
    with their standard errors."""
    import sindy
    system, noise, spr = case
    x, dx = _golden(f"{system}-train-{noise}")
    xv = torch.load(os.path.join(DATA, f"{system}-val-{noise}-gp-x.pt")).cuda()
    reg = sindy.SINDyRegression(2, 2, False, False, threshold=0.05, device="cuda", constrain_constant=True)
    path = sindy.stlsq_path(reg, x.reshape(-1, 2).cuda(), dx.reshape(-1, 2).cuda(), np.logspace(-3, 0, 40))
    xc = x.cuda()
    out = sindy.refine_path(reg, path, xc, 0.002, steps_per_row=spr, fit_ic=True)
    sc = sindy.score_path(reg, out, xv, 0.002, steps_per_row=spr, fit_ic=True)
    i = sc["chosen"]
    assert i is not None
    cc = sindy.coefficient_covariance(reg, out, xc, 0.002, steps_per_row=spr, fit_ic=True)
    m = out["mask"][i].cpu()
    xi, se = out["xi"][i].cpu().double(), cc["stderr"][i]
    names = [f"x{j}' θ{k}" for j in range(2) for k in range(reg.library.K)]
    rows = [f"{names[q]} = {float(xi.reshape(-1)[q]):+.5f} ± {float(se.reshape(-1)[q]):.2e}"
            for q in torch.nonzero(m.reshape(-1)).flatten().tolist()]
    print(f"{system}/{noise} AICc choice ({int(m.sum())} terms, sigma2 {float(cc['sigma2'][i]):.3e}, cond "
          f"{float(cc['cond'][i]):.2e}): " + "; ".join(rows))
    assert bool(cc["identifiable"][i]) and not bool(cc["diverged"][i])
    assert torch.isfinite(se[m]).all() and torch.all(se[m] > 0)
