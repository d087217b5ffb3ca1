"""Host-side checks of the coefficient standard errors (no GPU): the fp64 forward-mode reference against central
differences, the start elimination (Schur complement) against the dense inverse of the full normal matrix, the
constrained parameter map, argument validation before any device work, and the status codes and workspace arithmetic
of the new C entry points."""
import ctypes
import math

import pytest
import torch

from rollout_fp64_ref import step64
from rollout_gn_fp64_ref import gn64, jac64


def _states(x0, W, lib, dt, spr, n_rows, method):
    x, out = x0, []
    for _ in range(n_rows):
        for _ in range(spr):
            x = step64(x, W, lib, dt, method)
        out.append(x)
    return torch.stack(out)


@pytest.mark.parametrize("method", ["euler", "rk4"])
@pytest.mark.parametrize("horizon", [(1, 1), (7, 3)])
def test_reference_jacobian_matches_central_differences(method, horizon):
    n_rows, spr = horizon
    lib = (2, 2, False, False)
    g = torch.Generator().manual_seed(n_rows + spr)
    W = 0.2 * torch.randn(2, 6, generator=g, dtype=torch.float64)
    W[0, 1] -= 0.5
    x0 = torch.rand(4, 2, generator=g, dtype=torch.float64) - 0.5
    idx = torch.tensor([1, 8, -1, 3])
    dt, h = 0.02, 1e-6
    X, Jt, Jx = jac64(x0, W, idx, lib, dt, spr, n_rows, method)
    assert torch.allclose(X, _states(x0, W, lib, dt, spr, n_rows, method), rtol=0, atol=0)
    for p, q in enumerate(idx.tolist()):
        if q < 0:
            assert torch.all(Jt[..., p] == 0)
            continue
        Wp, Wq = W.clone().reshape(-1), W.clone().reshape(-1)
        Wp[q] += h
        Wq[q] -= h
        fd = (_states(x0, Wp.view(2, 6), lib, dt, spr, n_rows, method)
              - _states(x0, Wq.view(2, 6), lib, dt, spr, n_rows, method)) / (2 * h)
        assert torch.allclose(Jt[..., p], fd, rtol=1e-6, atol=1e-9)
    for j in range(2):
        xp, xq = x0.clone(), x0.clone()
        xp[:, j] += h
        xq[:, j] -= h
        fd = (_states(xp, W, lib, dt, spr, n_rows, method) - _states(xq, W, lib, dt, spr, n_rows, method)) / (2 * h)
        assert torch.allclose(Jx[..., j], fd, rtol=1e-6, atol=1e-9)
    # F and g from J, truncated per pair
    y = 0.3 * torch.randn(n_rows, 4, 2, generator=g, dtype=torch.float64)
    rows = torch.tensor([n_rows, 0, max(n_rows - 1, 0), 1])
    ref = gn64(x0, W, idx, lib, dt, spr, y, method, rows)
    keep = (torch.arange(n_rows)[:, None] < rows[None, :]).double()[..., None]
    e = (X - y) * keep
    assert torch.allclose(ref["jtj"], torch.einsum('rnip,rniq->pq', Jt * keep[..., None], Jt))
    assert torch.allclose(ref["jtr_x"], torch.einsum('rnij,rni->nj', Jx, e))
    assert torch.all(ref["jtj_px"][1] == 0) and torch.all(ref["jtj_xx"][1] == 0) and torch.all(ref["jtr_x"][1] == 0)


def test_schur_complement_is_the_block_of_the_dense_inverse():
    import sindy
    g = torch.Generator().manual_seed(5)
    U, N, P, d = 2, 4, 5, 3
    J = torch.randn(U, 40, P + N * d, generator=g, dtype=torch.float64)
    F = J.transpose(1, 2) @ J
    jtj = F[:, :P, :P]
    px = torch.stack([F[:, :P, P + n * d:P + (n + 1) * d] for n in range(N)], 1)          # (U, N, P, d)
    xx = torch.stack([F[:, P + n * d:P + (n + 1) * d, P + n * d:P + (n + 1) * d] for n in range(N)], 1)
    # the full normal matrix of coefficients and starts: no coupling between two starts, +I from the row-0 residual
    full = torch.zeros(U, P + N * d, P + N * d, dtype=torch.float64)
    full[:, :P, :P] = jtj
    for n in range(N):
        sl = slice(P + n * d, P + (n + 1) * d)
        full[:, :P, sl] = px[:, n]
        full[:, sl, :P] = px[:, n].transpose(1, 2)
        full[:, sl, sl] = xx[:, n] + torch.eye(d, dtype=torch.float64)
    S = sindy._schur_starts(jtj, px, xx)
    want = torch.linalg.inv(full)[:, :P, :P]
    assert torch.allclose(torch.linalg.inv(S), want, rtol=1e-10, atol=1e-12)
    cov, cond = sindy._gn_covariance(S[0], 2.0)
    assert torch.allclose(cov, 2.0 * want[0], rtol=1e-10, atol=1e-12)
    Dm = torch.diagonal(S[0]).rsqrt()
    assert cond == pytest.approx(float(torch.linalg.cond(Dm[:, None] * S[0] * Dm[None, :])), rel=1e-8)


def test_constrained_mapping_and_unidentifiable():
    import sindy
    g = torch.Generator().manual_seed(6)
    n, nq = 6, 3
    A = torch.randn(n, nq, generator=g, dtype=torch.float64)
    A = torch.cat([A, torch.zeros(n, 1, dtype=torch.float64)], 1)     # a parameter that reaches nothing is dropped
    J = torch.randn(30, n, generator=g, dtype=torch.float64)
    S = J.T @ J
    cov, cond = sindy._gn_covariance(S, 0.5, A)
    Aq = A[:, :nq]
    want = 0.5 * Aq @ torch.linalg.inv(Aq.T @ S @ Aq) @ Aq.T
    assert torch.allclose(cov, want, rtol=1e-10, atol=1e-13) and math.isfinite(cond)
    proj = torch.eye(n, dtype=torch.float64) - A @ torch.linalg.pinv(A)
    assert float((proj @ cov).abs().max()) < 1e-12 * float(cov.abs().max())
    # a coefficient the data do not determine: the factorisation fails
    S2 = S.clone()
    S2[:, 2] = S2[2, :] = 0
    assert sindy._gn_covariance(S2, 1.0) == (None, math.inf)
    Jc = torch.cat([J[:, :1], J[:, :1], J[:, 2:]], 1)                  # two identical columns
    assert sindy._gn_covariance(Jc.T @ Jc, 1.0)[0] is None


def _path(P=2, d=2, K=6, n_traj=4):
    return {"thresholds": torch.linspace(0.1, 0.3, P, dtype=torch.float64), "xi": torch.zeros(P, d, K),
            "mask": torch.ones(P, d, K, dtype=torch.bool), "x0": torch.zeros(P, n_traj, d)}


@pytest.mark.parametrize("kw", [dict(fit_ic=1), dict(window=3), dict(method="rk45"), dict(steps_per_row=0),
                                dict(blowup=-1.0), dict(dt=0.0)])
def test_coefficient_covariance_rejects_bad_arguments(kw):
    import sindy
    from sindy_b200.native import Library
    args = dict(dt=0.01)
    args.update(kw)
    with pytest.raises(ValueError):
        sindy.coefficient_covariance(Library(2, 2), _path(), torch.zeros(4, 10, 2), **args)


def test_coefficient_covariance_needs_the_starts():
    import sindy
    from sindy_b200.native import Library
    path = _path()
    del path["x0"]
    with pytest.raises(ValueError, match="x0"):
        sindy.coefficient_covariance(Library(2, 2), path, torch.zeros(4, 10, 2), 0.01, fit_ic=True)
    bad = _path(n_traj=3)
    with pytest.raises(ValueError, match="x0"):
        sindy.coefficient_covariance(Library(2, 2), bad, torch.zeros(4, 10, 2), 0.01, fit_ic=True)
    bad = _path()
    bad["x0"][0, 0, 0] = math.nan
    with pytest.raises(ValueError, match="x0"):
        sindy.coefficient_covariance(Library(2, 2), bad, torch.zeros(4, 10, 2), 0.01, fit_ic=True)
    with pytest.raises(ValueError):
        sindy.coefficient_covariance(Library(2, 2), _path(K=10), torch.zeros(4, 10, 2), 0.01)


def test_binding_checks_params():
    from sindy_b200 import native
    orig = native._require_cuda
    native._require_cuda = lambda t, name: None
    try:
        lib = native.Library(2, 2)
        ok = dict(x0=torch.zeros(4, 2), W=torch.zeros(2, 2, 6), lib=lib, dt=0.01, steps_per_row=1,
                  y_obs=torch.zeros(3, 4, 2))
        for bad in (torch.tensor([[0, 12]] * 2), torch.tensor([[-2, 0]] * 2), torch.zeros(3, 2, dtype=torch.long),
                    torch.zeros(2, 0, dtype=torch.long), torch.zeros(2, 2), torch.arange(12).repeat(15)[:177]):
            with pytest.raises(ValueError):
                native.rollout_score_gn(params=bad, **ok)
        with pytest.raises(ValueError):
            native.rollout_score_gn(params=torch.arange(12).repeat(15)[:175], x0_blocks=True, **ok)
        with pytest.raises(ValueError):
            native.rollout_score_gn(params=torch.zeros(2, 2, dtype=torch.long), x0_blocks=1, **ok)
    finally:
        native._require_cuda = orig


def _gn_bytes(N, d, K, M, P, x0b, spec):
    C = 4 if spec and K >= 32 else 8
    T = (P + (d if x0b else 0) + C - 1) // C
    G = max(1, 128 // T)
    blocks = min((N + G - 1) // G, 32)
    return M * blocks * (P * (P + 1) // 2 + P) * 8


def test_c_entry_points_validate_without_a_device():
    from sindy_b200 import native
    lib = native.load()
    L = native._CLibrary(2, 2, 0, 0)
    one = ctypes.c_void_p(16)
    for N, M, P, x0b in ((8, 2, 3, 0), (8, 2, 3, 1), (1000, 3, 12, 1), (4096, 1, 174, 1), (5, 2, 176, 0)):
        assert lib.sb_rollout_score_gn_workspace_bytes(N, ctypes.byref(L), M, P, x0b) == \
            _gn_bytes(N, 2, 6, M, P, x0b, True)
    L35 = native._CLibrary(3, 5, 0, 0)
    for N, P in ((4096, 168), (4096, 20), (7, 1)):
        assert lib.sb_rollout_score_gn_workspace_bytes(N, ctypes.byref(L35), 64, P, 1) == \
            _gn_bytes(N, 3, 56, 64, P, True, True)
    L4 = native._CLibrary(4, 2, 0, 0)
    assert lib.sb_rollout_score_gn_workspace_bytes(300, ctypes.byref(L4), 2, 9, 1) == \
        _gn_bytes(300, 4, 15, 2, 9, True, False)
    assert lib.sb_rollout_score_gn_workspace_bytes(8, ctypes.byref(L), 2, 0, 0) == -1
    assert lib.sb_rollout_score_gn_workspace_bytes(8, ctypes.byref(L), 2, 175, 1) == -2
    assert lib.sb_rollout_score_gn_workspace_bytes(-1, ctypes.byref(L), 2, 3, 0) == -1
    need = lib.sb_rollout_score_gn_workspace_bytes(8, ctypes.byref(L), 2, 3, 1)

    def gn(per=1, P=3, px=one, xx=one, rx=one, nb=need, x0=one, prm=one, jtj=one, method=1):
        return lib.sb_rollout_score_gn(x0, per, 8, ctypes.byref(L), one, 2, prm, P, 0.01, 1, 3, method, one, 0.0, one,
                                       one, jtj, one, px, xx, rx, one, nb, None)

    assert gn(per=2) == -1 and b"x0_per_model" in lib.sb_last_error()
    assert gn(px=None) == -1 and b"all be given" in lib.sb_last_error()
    assert gn(rx=None, xx=None) == -1
    assert gn(P=0) == -1 and b"n_params" in lib.sb_last_error()
    assert gn(P=175) == -2 and b"SB_GN_MAX_COLS" in lib.sb_last_error()
    assert gn(nb=need - 1) == -4 and b"workspace too small" in lib.sb_last_error()
    assert gn(x0=None) == -1 and b"x0 is NULL" in lib.sb_last_error()
    assert gn(prm=None) == -1 and b"params is NULL" in lib.sb_last_error()
    assert gn(jtj=None) == -1 and b"jtj is NULL" in lib.sb_last_error()
    assert gn(method=7) == -1
