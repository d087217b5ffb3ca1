"""Host-side checks of start estimation in the trajectory refit and the simulation scores (no GPU): the fp64 start
gradient reference against central differences, window splitting and the observation / parameter counts, argument
validation of the new keywords before any device work, and the status codes of the new C entry points."""
import ctypes

import pytest
import torch

from rollout_fp64_ref import sse64
from rollout_ic_fp64_ref import grad_x0_64, windows


def _case(seed, M=2, N=5, d=2, K=6):
    g = torch.Generator().manual_seed(seed)
    W = 0.1 * torch.randn(M, d, K, generator=g, dtype=torch.float64)
    W[:, 0, 1] -= 0.5                                    # damped, so that the long horizon (t = 10) stays moderate
    W[:, 1, 2] -= 0.5
    x0 = torch.rand(M, N, d, generator=g, dtype=torch.float64) - 0.5
    return W, x0, g


@pytest.mark.parametrize("method", ["euler", "rk4"])
@pytest.mark.parametrize("horizon", [(1, 1), (7, 3), (20, 25)])
@pytest.mark.parametrize("truncate", [False, True])
@pytest.mark.parametrize("per_model", [False, True])
def test_reference_start_gradient_matches_central_differences(method, horizon, truncate, per_model):
    n_rows, spr = horizon
    lib = (2, 2, False, False)
    W, x0, g = _case(n_rows * 10 + spr)
    if not per_model:
        x0 = x0[0]
    y = 0.4 * torch.randn(n_rows, 5, 2, generator=g, dtype=torch.float64)
    rows = torch.tensor([[n_rows, 0, max(n_rows - 1, 0), 1, n_rows]] * 2) if truncate else None
    dt = 0.02
    s, gx = grad_x0_64(x0, W, lib, dt, spr, y, method, rows)
    assert s.shape == (2, 5) and gx.shape == (2, 5, 2)
    h = 1e-6
    for m in range(2):
        xm = x0[m] if per_model else x0
        rm = None if rows is None else rows[m]
        fd = torch.zeros_like(xm)
        for n in range(5):
            for j in range(2):
                xp, xq = xm.clone(), xm.clone()
                xp[n, j] += h
                xq[n, j] -= h
                fd[n, j] = (sse64(xp, W[m], lib, dt, spr, y, method, rm)[n]
                            - sse64(xq, W[m], lib, dt, spr, y, method, rm)[n]) / (2 * h)
        assert torch.allclose(gx[m], fd, rtol=1e-6, atol=1e-8), (gx[m] - fd).abs().max()
    if truncate:
        # a pair that stops at row 0 has no start gradient
        assert torch.all(gx[:, 1] == 0) and torch.all(s[:, 1] == 0)


def test_window_splitting_and_counts():
    import sindy
    from sindy_b200.native import Library
    lib = Library(2, 2)
    x = torch.arange(3 * 12 * 2, dtype=torch.float32).reshape(3, 12, 2)
    xw, _ = sindy._check_rollout_args(lib, x, "x", 0.01, 1, "rk4", None, window=4)
    assert xw.shape == (9, 4, 2) and torch.equal(xw, windows(x, 4))
    # consecutive and non-overlapping: window j of trajectory i is rows 4j..4j+3, each row exactly once
    assert torch.equal(xw[3 * 1 + 2], x[1, 8:12])
    assert torch.equal(torch.sort(xw.reshape(-1)).values, torch.sort(x.reshape(-1)).values)
    same, _ = sindy._check_rollout_args(lib, x, "x", 0.01, 1, "rk4", None, window=12)
    assert torch.equal(same, x)
    # fixed starts compare rows 1..R−1; with start estimation row 0 is one more residual and each start d parameters
    assert sindy._obs_counts(9, 4, 2, False) == (9 * 3 * 2, 0)
    assert sindy._obs_counts(9, 4, 2, True) == (9 * 4 * 2, 9 * 2)
    n, k_ic = sindy._obs_counts(3, 12, 2, True)
    crit = sindy.information_criteria(torch.tensor([2.0]), n, torch.tensor([4.0]) + k_ic)
    assert float(crit["aic"]) == pytest.approx(n * torch.log(torch.tensor(2.0 / n)).item() + 2 * (4 + 6))


def _path(P=3, d=2, K=6):
    return {"thresholds": torch.linspace(0.1, 0.3, P, dtype=torch.float64), "xi": torch.zeros(P, d, K),
            "mask": torch.ones(P, d, K, dtype=torch.bool)}


BAD_KEYWORDS = [dict(fit_ic=1), dict(fit_ic="yes"), dict(fit_ic=None), dict(window=1), dict(window=3),
                dict(window=2.0), dict(window=True), dict(window=0), dict(window=20)]


@pytest.mark.parametrize("kw", BAD_KEYWORDS)
def test_refine_path_rejects_bad_start_keywords(kw):
    import sindy
    from sindy_b200.native import Library
    with pytest.raises(ValueError):
        sindy.refine_path(Library(2, 2), _path(), torch.zeros(4, 10, 2), 0.01, **kw)


@pytest.mark.parametrize("kw", BAD_KEYWORDS + [dict(ic_iter=0), dict(ic_iter=2.5), dict(ic_iter=True)])
def test_score_path_rejects_bad_start_keywords(kw):
    import sindy
    from sindy_b200.native import Library
    with pytest.raises(ValueError):
        sindy.score_path(Library(2, 2), _path(), torch.zeros(4, 10, 2), 0.01, **kw)


def test_per_model_starts_are_checked():
    from sindy_b200 import native
    orig = native._require_cuda
    native._require_cuda = lambda t, name: None
    try:
        lib = native.Library(2, 2)
        ok = dict(x0=torch.zeros(2, 4, 2), W=torch.zeros(2, 2, 6), lib=lib, dt=0.01, steps_per_row=1,
                  y_obs=torch.zeros(3, 4, 2), method="rk4", blowup=None)
        x0, per_model = native._score_args(**ok)[:2]
        assert per_model and x0.shape == (2, 4, 2)
        assert not native._score_args(**{**ok, "x0": torch.zeros(4, 2)})[1]
        for bad in (dict(x0=torch.zeros(3, 4, 2)), dict(x0=torch.zeros(2, 4, 3)), dict(x0=torch.zeros(2, 5, 2))):
            with pytest.raises(ValueError):
                native._score_args(**{**ok, **bad})
        with pytest.raises(ValueError):
            native.rollout_score_grad(**ok, x0_grad=False, w_grad=False)
    finally:
        native._require_cuda = orig


def test_c_entry_points_validate_without_a_device():
    from sindy_b200 import native
    lib = native.load()
    L = native._CLibrary(2, 2, 0, 0)
    one = ctypes.c_void_p(16)
    need = lib.sb_rollout_score_grad_workspace_bytes(8, ctypes.byref(L), 2, 1, 3)

    def grad(per=1, grad=one, gx=one, nb=need, x0=one):
        return lib.sb_rollout_score_grad_ics(x0, per, 8, ctypes.byref(L), one, 2, 0.01, 1, 3, 1, one, 0.0, one, one,
                                             grad, gx, one, nb, None)

    def score(per=1):
        return lib.sb_rollout_score_ics(one, per, 8, ctypes.byref(L), one, 2, 0.01, 1, 3, 1, one, 0.0, one, one, None)

    for per in (2, -1, 1 << 20):
        assert grad(per=per) == -1 and b"x0_per_model" in lib.sb_last_error()
        assert score(per=per) == -1 and b"x0_per_model" in lib.sb_last_error()
    assert grad(grad=None, gx=None) == -1 and b"both NULL" in lib.sb_last_error()
    assert grad(nb=need - 1) == -4 and b"workspace too small" in lib.sb_last_error()
    assert grad(gx=None, nb=need - 1) == -4 and grad(grad=None, nb=need - 1) == -4
    assert grad(x0=None) == -1 and b"x0 is NULL" in lib.sb_last_error()
