"""Host-side checks of the rollout-score gradient and the trajectory refit (no GPU): the fp64 reference against central
finite differences, argument validation of native.rollout_score_grad and sindy.refine_path before any device work, the C
entry point's checks, and the factored L-BFGS direction against BatchedLBFGS's own step."""
import ctypes

import pytest
import torch

from rollout_fp64_ref import grad64, sse64


def _case(seed, d=2, K=6, N=5):
    g = torch.Generator().manual_seed(seed)
    W = 0.3 * torch.randn(d, K, generator=g, dtype=torch.float64)
    x0 = torch.rand(N, d, generator=g, dtype=torch.float64) - 0.5
    return W, x0, g


@pytest.mark.parametrize("method", ["euler", "rk4"])
@pytest.mark.parametrize("horizon", [(1, 1), (3, 4), (7, 3)])
@pytest.mark.parametrize("truncate", [False, True])
def test_reference_gradient_matches_central_differences(method, horizon, truncate):
    n_rows, spr = horizon
    lib = (2, 2, False, False)
    W, x0, g = _case(n_rows * 10 + spr)
    y = 0.4 * torch.randn(n_rows, x0.shape[0], 2, generator=g, dtype=torch.float64)
    rows = torch.tensor([n_rows, 0, max(n_rows - 1, 0), 1, n_rows]) if truncate else None
    dt = 0.05
    s, gW = grad64(x0, W, lib, dt, spr, y, method, rows)
    assert s.shape == (5,)
    h = 1e-6
    fd = torch.zeros_like(W)
    for i in range(W.shape[0]):
        for k in range(W.shape[1]):
            Wp, Wm = W.clone(), W.clone()
            Wp[i, k] += h
            Wm[i, k] -= h
            fd[i, k] = (sse64(x0, Wp, lib, dt, spr, y, method, rows).sum()
                        - sse64(x0, Wm, lib, dt, spr, y, method, rows).sum()) / (2 * h)
    assert torch.allclose(gW, fd, rtol=1e-6, atol=1e-8), (gW - fd).abs().max()
    if truncate:
        # a pair that stops at row 0 contributes nothing
        assert float(s[1]) == 0.0


def test_reference_sin_exp_columns():
    lib = (2, 1, True, True)
    W, x0, g = _case(3, K=7)
    y = 0.4 * torch.randn(4, 5, 2, generator=g, dtype=torch.float64)
    _, gW = grad64(x0, W, lib, 0.05, 2, y, "rk4")
    h = 1e-6
    Wp, Wm = W.clone(), W.clone()
    Wp[1, 5] += h
    Wm[1, 5] -= h
    fd = (sse64(x0, Wp, lib, 0.05, 2, y, "rk4").sum() - sse64(x0, Wm, lib, 0.05, 2, y, "rk4").sum()) / (2 * h)
    assert float(gW[1, 5]) == pytest.approx(float(fd), rel=1e-6)


def test_rollout_score_grad_refuses_cpu_tensors():
    from sindy_b200 import native
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        native.rollout_score_grad(torch.zeros(4, 2), torch.zeros(2, 2, 6), native.Library(2, 2), 0.01, 1,
                                  torch.zeros(3, 4, 2))


def test_shared_checks_reject_bad_arguments():
    """_score_args holds the checks rollout_score and rollout_score_grad share; without a device they are reached by
    patching out the device check."""
    from sindy_b200 import native
    orig = native._require_cuda
    native._require_cuda = lambda t, name: None
    try:
        lib = native.Library(2, 2)
        ok = dict(x0=torch.zeros(4, 2), W=torch.zeros(2, 2, 6), lib=lib, dt=0.01, steps_per_row=1,
                  y_obs=torch.zeros(3, 4, 2), method="rk4", blowup=None)
        native._score_args(**ok)
        for bad in (dict(steps_per_row=0), dict(steps_per_row=True), dict(dt=0.0), dict(dt=float("nan")),
                    dict(method="midpoint"), dict(blowup=0.0), dict(y_obs=torch.zeros(3, 3, 2)),
                    dict(y_obs=torch.zeros(0, 4, 2)), dict(W=torch.zeros(2, 2, 5)), dict(x0=torch.zeros(4, 3))):
            with pytest.raises(ValueError):
                native._score_args(**{**ok, **bad})
    finally:
        native._require_cuda = orig


def _path(P=3, d=2, K=6):
    return {"thresholds": torch.linspace(0.1, 0.3, P, dtype=torch.float64), "xi": torch.zeros(P, d, K),
            "mask": torch.ones(P, d, K, dtype=torch.bool)}


@pytest.mark.parametrize("kw", [
    dict(x_fit=torch.zeros(4, 10)),
    dict(x_fit=torch.zeros(4, 10, 3)),
    dict(x_fit=torch.zeros(4, 1, 2)),
    dict(x_fit=torch.full((4, 10, 2), float("inf"))),
    dict(steps_per_row=0),
    dict(steps_per_row=1.5),
    dict(dt=0.0),
    dict(method="midpoint"),
    dict(blowup=-1.0),
    dict(max_iter=0),
    dict(max_iter=2.5),
    dict(tol=-1.0),
    dict(path={**_path(), "xi": torch.zeros(3, 2, 5)}),
    dict(path={**_path(), "mask": torch.ones(3, 2, 5, dtype=torch.bool)}),
    dict(regressor="not a library"),
])
def test_refine_path_argument_errors(kw):
    import sindy
    from sindy_b200.native import Library
    args = dict(regressor=Library(2, 2), path=_path(), x_fit=torch.zeros(4, 10, 2), dt=0.01)
    args.update(kw)
    with pytest.raises(ValueError):
        sindy.refine_path(**args)


def test_c_entry_point_validates_without_a_device():
    from sindy_b200 import native
    lib = native.load()
    L = native._CLibrary(2, 2, 0, 0)
    one = ctypes.c_void_p(16)
    need = lib.sb_rollout_score_grad_workspace_bytes(8, ctypes.byref(L), 2, 1, 3)
    # 3 steps: one checkpoint of 2 models × 8 ICs × 2 floats; one block of ICs: 2 partial rows of 2·6 doubles
    assert need == 256 + 2 * 8 * 2 * 4

    def call(x0=one, n=8, lb=ctypes.byref(L), w=one, m=2, dt=0.01, spr=1, rows=3, meth=1, y=one, sse=one, valid=one,
             grad=one, ws=one, nb=need):
        return lib.sb_rollout_score_grad(x0, n, lb, w, m, dt, spr, rows, meth, y, 0.0, sse, valid, grad, ws, nb, None)

    assert call(x0=None) == -1 and b"x0 is NULL" in lib.sb_last_error()
    assert call(y=None) == -1 and call(sse=None) == -1 and call(valid=None) == -1 and call(w=None) == -1
    assert call(grad=None) == -1 and call(ws=None) == -1
    assert call(m=0) == -1 and call(spr=0) == -1 and call(rows=0) == -1 and call(rows=1 << 31) == -1
    assert call(n=-1) == -1 and call(meth=2) == -1
    assert call(dt=0.0) == -1 and call(dt=float("nan")) == -1
    assert call(nb=need - 1) == -4 and b"workspace too small" in lib.sb_last_error()
    bad = native._CLibrary(2, 6, 0, 0)
    assert call(lb=ctypes.byref(bad)) == -2
    assert call(lb=None) == -1
    assert lib.sb_rollout_score_grad_workspace_bytes(8, ctypes.byref(L), 0, 1, 3) == -1
    assert lib.sb_rollout_score_grad_workspace_bytes(1 << 40, ctypes.byref(L), 1 << 30, 1 << 20, 1 << 20) == -1


def test_batched_direction_is_the_step_s_own():
    """BatchedLBFGS.direction (the recursion BatchedLBFGS.step and refine_path share) on a random history, with
    per-problem history lengths and a rolled-over history, against the serial two-loop recursion of torch.optim.LBFGS
    on each problem."""
    import sweep
    g = torch.Generator().manual_seed(0)
    S, P, H = 4, 7, 5
    opt = sweep.BatchedLBFGS(torch.zeros(S, P, dtype=torch.float64), 1.0, history_size=H)
    for it in range(H + 2):                              # overflow the history to exercise the roll
        s = torch.randn(S, P, generator=g, dtype=torch.float64)
        y = s + 0.1 * torch.randn(S, P, generator=g, dtype=torch.float64)
        upd = torch.tensor([True, it % 2 == 0, it < 2, False])
        opt.push(y, s, upd, (y * s).sum(1))
    grad = torch.randn(S, P, generator=g, dtype=torch.float64)
    d = opt.direction(grad)
    for i in range(S):
        n = int(opt.hist[i])
        old_s, old_y = opt.old_s[i, :n], opt.old_y[i, :n]
        q = -grad[i].clone()
        al = [None] * n
        for j in range(n - 1, -1, -1):
            al[j] = float((old_s[j] * q).sum()) / float((old_y[j] * old_s[j]).sum())
            q -= al[j] * old_y[j]
        r = q * (opt.H_diag[i] if n else 1.0)
        for j in range(n):
            be = float((old_y[j] * r).sum()) / float((old_y[j] * old_s[j]).sum())
            r += (al[j] - be) * old_s[j]
        assert torch.allclose(d[i], r, rtol=1e-12, atol=1e-14), i
    assert int(opt.hist[3]) == 0 and torch.equal(d[3], -grad[3])
