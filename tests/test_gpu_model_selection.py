"""GPU checks of model selection along the STLSQ threshold path: sb_rollout_score against sb_rollout (bitwise states,
every kernel family), an independent fp64 NumPy RK4, divergence handling, bitwise determinism across batches, model
order and repeats; stlsq_path / WSINDyWrapper.solve_path against the per-threshold solves; and the end-to-end
selection on the golden growth and damped-oscillator data."""
import copy
import os

import numpy as np
import pytest
import torch

from oracle import sindy_oracle as O

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
    """Random models, scaled by 1/sqrt(K / 6) so that none leaves the unit box within the tests' horizons."""
    g = torch.Generator().manual_seed(seed)
    W = scale * (6.0 / lib.K) ** 0.5 * torch.randn(M, lib.dim, lib.K, generator=g)
    W[:, :, 0] *= 0.1
    return W.cuda()


def ics(N, d, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(N, d, generator=g) - 0.5).cuda()


def reference(nat, x0, W, lib, dt, spr, y, method):
    """fp64 SSE over native.rollout's stored rows, one model at a time."""
    out = []
    for m in range(W.shape[0]):
        traj, _, _ = nat.rollout(x0, W[m], lib, dt, y.shape[0] * spr, stride=spr, method=method, want_last=False)
        out.append(((traj.double() - y.double()) ** 2).sum(dim=(0, 2)))
    return torch.stack(out)


# the specialised shapes of SB_SPEC_SHAPES (config 3's (2, 2) + exp among them) and two runtime-table libraries
LIBS = [(2, 2, 0, 0), (2, 3, 0, 0), (3, 2, 0, 0), (3, 3, 0, 0), (3, 5, 0, 0), (2, 2, 0, 1), (2, 2, 1, 0), (4, 2, 0, 0)]


@pytest.mark.parametrize("method", ["rk4", "euler"])
@pytest.mark.parametrize("spec", LIBS)
def test_scores_are_sums_over_the_rollout_trajectories(nat, spec, method):
    d, p, s, e = spec
    lib = nat.Library(d, p, bool(s), bool(e))
    N, spr, n_rows, dt = 300, 3, 7, 0.01          # 300 ICs: a partly filled last block, one IC of a pair without partner
    W = models(lib, 3, 10 * d + p)
    x0 = ics(N, d, 7)
    y = torch.randn(n_rows, N, d, device="cuda") * 0.5
    sse, valid = nat.rollout_score(x0, W, lib, dt, spr, y, method)
    ref = reference(nat, x0, W, lib, dt, spr, y, method)
    assert sse.dtype == torch.float64 and valid.dtype == torch.int32 and sse.shape == (3, N)
    assert torch.all(valid == n_rows)
    assert torch.all((sse - ref).abs() <= 1e-12 * ref.abs())
    # against model 0's own trajectory the states must agree bit for bit: the SSE is exactly zero
    traj, _, _ = nat.rollout(x0, W[0], lib, dt, n_rows * spr, stride=spr, method=method, want_last=False)
    sse0, _ = nat.rollout_score(x0, W, lib, dt, spr, traj, method)
    assert torch.all(sse0[0] == 0)
    assert torch.all(sse0[1:] > 0)


def test_float64_numpy_rk4_agrees(nat):
    lib = nat.Library(3, 3)
    N, spr, n_rows, dt = 40, 4, 25, 0.005
    W = models(lib, 2, 3, scale=0.2)
    x0 = ics(N, 3, 4)
    g = np.random.default_rng(5)
    rows, ref_sse = [], []
    for m in range(2):
        Wm = W[m].double().cpu().numpy()
        f = lambda z: O.theta(z, 3) @ Wm.T
        x = x0.double().cpu().numpy()
        traj = []
        for s in range(1, n_rows * spr + 1):
            k1 = f(x); k2 = f(x + dt / 2 * k1); k3 = f(x + dt / 2 * k2); k4 = f(x + dt * k3)
            x = x + dt / 6 * (k1 + 2 * k2 + 2 * k3 + k4)
            if s % spr == 0:
                traj.append(x)
        rows.append(np.stack(traj))
    y = rows[0] + 0.05 * g.standard_normal(rows[0].shape)
    for m in range(2):
        ref_sse.append(((rows[m] - y) ** 2).sum(axis=(0, 2)))
    sse, valid = nat.rollout_score(x0, W, lib, dt, spr, torch.from_numpy(y).float().cuda(), "rk4")
    ref = np.stack(ref_sse)
    assert np.all(valid.cpu().numpy() == n_rows)
    np.testing.assert_allclose(sse.cpu().numpy(), ref, rtol=1e-5)


@pytest.mark.parametrize("blowup", [None, 50.0])
@pytest.mark.parametrize("spec", [(1, 2), (2, 2)])
def test_divergent_pairs_stop_at_the_first_bad_row(nat, spec, blowup):
    """ẋ = x² from x0 = 1 leaves every bound at t = 1; x0 = 0.5 at t = 2, x0 = −1 decays. Integrated to t = 2.4."""
    d, p = spec
    lib = nat.Library(d, p)
    W = torch.zeros(1, d, lib.K, device="cuda")
    W[0, 0, d + 1] = 1.0                                   # column x0·x0
    x0 = torch.zeros(4, d, device="cuda")
    x0[:, 0] = torch.tensor([1.0, 0.5, -1.0, 2.0])
    dt, spr, n_rows = 0.01, 5, 48
    y = torch.zeros(n_rows, 4, d, device="cuda")
    sse, valid = nat.rollout_score(x0, W, lib, dt, spr, y, "rk4", blowup=blowup)
    traj, _, _ = nat.rollout(x0, W[0], lib, dt, n_rows * spr, stride=spr, method="rk4", want_last=False)
    bad = ~torch.isfinite(traj).all(-1)
    if blowup is not None:
        bad |= (traj.abs() > blowup).any(-1)
    for n in range(4):
        rows = torch.nonzero(bad[:, n]).flatten()
        first = int(rows[0]) if rows.numel() else n_rows
        assert int(valid[0, n]) == first, n
        want = (traj[:first, n].double() ** 2).sum()
        assert float(sse[0, n]) == pytest.approx(float(want), rel=1e-12)
    assert int(valid[0, 2]) == n_rows and int(valid[0, 0]) < n_rows and int(valid[0, 3]) < int(valid[0, 0])


def test_a_pair_has_the_same_bits_in_every_batch(nat):
    lib = nat.Library(3, 5)
    M, N, spr, n_rows, dt = 200, 257, 2, 5, 0.01
    W = models(lib, M, 11, scale=0.05)
    x0 = ics(N, 3, 12)
    y = torch.randn(n_rows, N, 3, device="cuda") * 0.3
    sse, valid = nat.rollout_score(x0, W, lib, dt, spr, y, "rk4")
    again, again_v = nat.rollout_score(x0, W, lib, dt, spr, y, "rk4")
    assert torch.equal(sse, again) and torch.equal(valid, again_v)
    perm = torch.randperm(M, generator=torch.Generator().manual_seed(0)).cuda()
    ps, _ = nat.rollout_score(x0, W[perm], lib, dt, spr, y, "rk4")
    assert torch.equal(ps, sse[perm])
    m, n = 137, 200
    alone, _ = nat.rollout_score(x0[n:n + 1], W[m:m + 1], lib, dt, spr, y[:, n:n + 1].contiguous(), "rk4")
    assert torch.equal(alone[0, 0], sse[m, n])
    part, _ = nat.rollout_score(x0[150:], W[100:150], lib, dt, spr, y[:, 150:].contiguous(), "rk4")
    assert torch.equal(part[m - 100, n - 150], sse[m, n])


def test_invalid_arguments(nat):
    lib = nat.Library(2, 2)
    x0, W, y = ics(4, 2, 0), models(lib, 2, 0), torch.zeros(3, 4, 2, device="cuda")
    with pytest.raises(ValueError):
        nat.rollout_score(x0, W, lib, 0.01, 0, y)
    with pytest.raises(ValueError):
        nat.rollout_score(x0, W, lib, -0.01, 1, y)
    with pytest.raises(ValueError):
        nat.rollout_score(x0, W, lib, 0.01, 1, y[:, :3].contiguous())
    with pytest.raises(ValueError):
        nat.rollout_score(x0, W, lib, 0.01, 1, y, "midpoint")
    with pytest.raises(nat.SindyB200Error):
        nat.rollout_score(x0, W[:, :, :5].contiguous(), nat.Library(2, 6), 0.01, 1, y)


# ---- the threshold path ----------------------------------------------------------------------------------------------
def _train(name):
    x = torch.load(os.path.join(DATA, f"{name}-gp-x.pt"))
    dx = torch.load(os.path.join(DATA, f"{name}-gp-dx.pt"))
    return x, dx


def _loop(reg, solve, thresholds):
    """Per-threshold solves on a copy of the regressor: (masks, Ξ⊙mask, residuals)."""
    masks, xis, res = [], [], []
    for t in thresholds:
        r = copy.deepcopy(reg)
        res.append(solve(r, float(t)))
        masks.append(r.mask > 0)
        xis.append((r._current_Xi() * r.mask).detach())
    return torch.stack(masks), torch.stack(xis), res


def _assert_path(path, masks, xis):
    assert torch.equal(path["mask"], masks)
    scale = xis.abs().amax(dim=(1, 2), keepdim=True).clamp_min(1e-30)
    assert torch.all((path["xi"] - xis).abs() <= 1e-6 * scale)
    assert torch.equal(path["n_terms"], masks.flatten(1).sum(1))


def _state(reg):
    return [p.detach().clone() for p in reg.parameters()] + [reg.mask.clone()]


THRESHOLDS = np.concatenate([[0.0], np.logspace(-4, 0.5, 24)])


@pytest.mark.parametrize("case", ["dosc-train-noise20", "growth-train-noise05", "lorenz", "rank_deficient"])
def test_stlsq_path_equals_per_threshold_solves(nat, golden, case):
    import sindy
    if case == "lorenz":
        g = golden("stlsq")
        x, y, d, p = torch.from_numpy(g["lorenz_x"]), torch.from_numpy(g["lorenz_y"]), 3, 3
    elif case == "rank_deficient":
        # x1 = 2·x0: every support holding both x0 and x1 (or x0² and x0·x1 ...) is singular, small ones are not
        t = torch.linspace(-1, 1, 500, dtype=torch.float64)
        x = torch.stack([t, 2 * t], 1).float()
        y = torch.stack([-0.5 * t + 0.3 * t * t, 0.1 + t], 1).float()
        d, p = 2, 2
    else:
        x, y = _train(case)
        d, p = 2, 2
    x, y = x.reshape(-1, d).cuda(), y.reshape(-1, d).cuda()
    reg = sindy.SINDyRegression(d, p, False, False, threshold=0.05, device="cuda", constrain_constant=True)
    before = _state(reg)
    path = sindy.stlsq_path(reg, x, y, THRESHOLDS, 0.0, 5)
    after = _state(reg)
    assert all(torch.equal(a, b) for a, b in zip(before, after))
    masks, xis, res = _loop(reg, lambda r, t: sindy.solve_SINDy(r, x, y, 0.0, t, 5), THRESHOLDS)
    _assert_path(path, masks, xis)
    np.testing.assert_allclose(path["residual"].cpu().numpy(), torch.stack(res).cpu().numpy(), rtol=1e-5, atol=1e-12)


@pytest.mark.parametrize("cc", [True, False])
def test_constrained_stlsq_path_equals_per_threshold_solves(nat, cc):
    import sindy
    x, y = _train("dosc-train-noise20")
    x, y = x.reshape(-1, 2).cuda(), y.reshape(-1, 2).cuda()
    torch.manual_seed(0)
    so2 = torch.tensor([[0.0, 1.0], [-1.0, 0.0]])
    reg = sindy.SINDyRegression(2, 2, False, False, L_list=[so2], threshold=0.05, device="cuda", constrain_constant=cc)
    reg.Xi = reg.Xi.detach()          # Ξ = reshape(Q·β) is recomputed from β on use; a non-leaf tensor cannot be deep-copied
    before = _state(reg)
    thr = np.logspace(-3, 0, 12)
    path = sindy.stlsq_path(reg, x, y, thr)
    assert all(torch.equal(a, b) for a, b in zip(before, _state(reg)))
    masks, xis, _ = _loop(reg, lambda r, t: sindy.solve_SINDy(r, x, y, 0.0, t, 5), thr)
    _assert_path(path, masks, xis)
    i = int(np.argmax(path["n_terms"].cpu().numpy() < 12))
    sindy.apply_candidate(reg, path, i)
    assert torch.equal(reg.mask > 0, path["mask"][i])
    assert torch.allclose(reg.get_Xi() * reg.mask, path["xi"][i], atol=1e-6)


@pytest.mark.parametrize("family", ["trig", "poly"])
@pytest.mark.parametrize("pooled", [False, True])
def test_wsindy_solve_path_equals_the_loop_of_solve(nat, family, pooled):
    import sindy
    x, _ = _train("growth-train-noise05")
    x = (x[:8] if pooled else x[0]).cuda()
    dt = 0.02
    T = x.shape[-2]
    t = torch.arange(T, dtype=torch.float32) * dt
    reg = sindy.SINDyRegression(2, 2, False, False, threshold=0.05, device="cuda", constrain_constant=True)
    wr = sindy.WSINDyWrapper(reg, t, T * dt, num_test_funcs=20, test_func_family=family, device="cuda")
    thr = np.logspace(-3, 0, 16)
    before = _state(reg)
    path = wr.solve_path(x, 0.01, thr, max_iter=5)
    assert all(torch.equal(a, b) for a, b in zip(before, _state(reg)))

    def loop(r, th):
        w2 = copy.copy(wr)
        w2.regressor = r
        r.reset_mask()
        for _ in range(5):
            res, conv = w2.solve(x, 0.01, th)
            if conv:
                break
        return res

    masks, xis, res = _loop(reg, loop, thr)
    _assert_path(path, masks, xis)
    np.testing.assert_allclose(path["residual"].cpu().numpy(), np.array(res), rtol=1e-6)


# ---- end to end ------------------------------------------------------------------------------------------------------
def test_growth_selection_finds_the_true_support(nat, golden):
    """growth/noise05: train → threshold path → simulation scores on the validation set (sampled every 10 steps of
    0.002). AICc ranks the true support first (the cfg's own threshold gets equation 1 wrong)."""
    import sindy
    x, dx = _train("growth-train-noise05")
    xv = torch.load(os.path.join(DATA, "growth-val-noise05-gp-x.pt")).cuda()
    reg = sindy.SINDyRegression(2, 2, False, False, threshold=0.05, device="cuda", constrain_constant=True)
    path = sindy.stlsq_path(reg, x.reshape(-1, 2).cuda(), dx.reshape(-1, 2).cuda(), np.logspace(-3, 0, 40))
    sc = sindy.score_path(reg, path, xv, 0.002, steps_per_row=10)
    i = sc["chosen"]
    truth = golden("model")["truth_growth"] != 0
    assert np.array_equal(path["mask"][i].cpu().numpy(), truth)
    assert sc["n_obs"] == 20 * 99 * 2 and int(sc["k"][i]) == 3
    # the float64 prototype's numbers: AICc −28488 for the truth, −28046 for the runner-up
    assert sc["aicc"][i].item() == pytest.approx(-28487.7, abs=2.0)
    others = sc["aicc"][~torch.from_numpy(np.all(path["mask"].cpu().numpy() == truth, axis=(1, 2)))]
    assert others.min().item() == pytest.approx(-28046.3, abs=2.0)
    sindy.apply_candidate(reg, path, i)
    assert torch.equal(reg.mask > 0, path["mask"][i])


def test_dosc_selection_is_the_argmin_of_the_reported_criterion(nat):
    import sindy
    x, dx = _train("dosc-train-noise20")
    xv = torch.load(os.path.join(DATA, "dosc-val-noise20-gp-x.pt")).cuda()
    reg = sindy.SINDyRegression(2, 2, False, False, threshold=0.05, device="cuda", constrain_constant=True)
    thr = np.logspace(-3, 0, 40)
    path = sindy.stlsq_path(reg, x.reshape(-1, 2).cuda(), dx.reshape(-1, 2).cuda(), thr)
    for crit in ("aic", "aicc", "bic"):
        sc = sindy.score_path(reg.library, path, xv, 0.002, steps_per_row=100, criterion=crit)
        c = sc[crit].numpy()
        i = sc["chosen"]
        assert c[i] == c.min()
        tied = np.flatnonzero(c == c.min())
        k = sc["k"].numpy()
        assert k[i] == k[tied].min() and thr[i] == thr[tied][k[tied] == k[i]].max()
        n = sc["n_obs"]
        want = sindy.information_criteria(sc["sse"], n, sc["k"].double())[crit]
        finite = ~sc["diverged"]
        assert torch.allclose(sc[crit][finite], want[finite], rtol=1e-12, atol=0)
