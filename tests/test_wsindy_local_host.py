"""CPU checks of the compactly supported WSINDy test functions (WSINDyWrapper(test_func_family='poly')): the oracle's
definition recovers an analytic system exactly, the tables have the stated properties, the wrapper's host side (tables,
dense V, M, the pooled multi-trajectory solve) matches the oracle, and every out-of-range argument is refused. No compute
entry point is called."""
import math

import numpy as np
import pytest
import torch

from oracle import sindy_oracle as O
import wsindy_local_oracle as WL

DT, T = 0.002, 8000
# dx/dt = −0.1x − y, dy/dt = x − 0.1y over the poly-2 library [1, x, y, x², xy, y²]
XI_STAR = np.zeros((2, 6))
XI_STAR[0, 1], XI_STAR[0, 2], XI_STAR[1, 1], XI_STAR[1, 2] = -0.1, -1.0, 1.0, -0.1


def damped_oscillator(radius=1.3, phase=0.4, n=T, dt=DT):
    t = np.arange(n) * dt
    return radius * np.exp(-0.1 * t)[:, None] * np.stack([np.cos(t + phase), np.sin(t + phase)], 1)


def default_support(n, n_test):
    return min(n, 2 * (n // (n_test + 1)) + 1)


def fp64_fit(n_test, support, degree):
    x = damped_oscillator()
    V, Vd = WL.wsindy_local_test_functions(T, DT, n_test, support, degree, rounded=False)
    G, b = V @ O.theta(x, 2), -(Vd @ x)
    return V, G, b


# (n_test, support, degree): the defaults, one window, the whole trajectory as one window, non-overlapping windows
# (L = 151 < the start spacing 7849/49 ≈ 160), and the degrees 6 and 16
SHAPES = [(50, None, None), (1, None, 6), (1, T, 6), (50, 151, 6), (50, None, 16)]


@pytest.mark.parametrize("n_test,support,degree", SHAPES)
def test_oracle_definition_is_exact_on_an_analytic_system(n_test, support, degree):
    V, G, b = fp64_fit(n_test, support, degree)
    assert np.abs(b - G @ XI_STAR.T).max() <= 1e-10 * np.abs(b).max()
    if n_test >= G.shape[1]:        # one window is one equation per state: Ξ* is determined only with n_test ≥ K
        M = V @ V.T
        xi = np.linalg.solve(G.T @ M @ G, G.T @ M @ b).T
        assert np.abs(xi - XI_STAR).max() <= 1e-10


def test_oracle_definition_degree_one_is_first_order():
    """The window sum of d/dt(φ·x) is a rectangle rule whose error is set by φ's derivatives at the window ends; (4u(1−u))^p
    makes the first p−1 of them vanish there. At p = 1 φ' does not vanish, so the weak form holds to O(1/L) only: the
    relative residual is ≈ 3/L and halves when L doubles."""
    res = []
    for L in (313, 601):
        _, G, b = fp64_fit(20, L, 1)
        res.append(np.abs(b - G @ XI_STAR.T).max() / np.abs(b).max())
        assert 1.0 / L < res[-1] < 4.0 / L
    assert 0.4 < res[1] / res[0] < 0.6


@pytest.mark.parametrize("n_test,support,degree", SHAPES + [(500, 3, 1), (7, 1000, 32)])
def test_table_properties(n_test, support, degree):
    import sindy
    L, p, starts, phi, dphi = sindy._local_test_functions(T, DT, n_test, support, degree)
    assert L == (default_support(T, n_test) if support is None else support)
    assert p == (6 if degree is None else degree)
    assert starts[0] == 0 and starts[-1] == T - L and len(set(starts)) == n_test
    assert phi[0] == 0.0 and phi[-1] == 0.0
    V, Vd = WL.wsindy_local_test_functions(T, DT, n_test, support, degree, rounded=False)
    np.testing.assert_allclose((V * V).sum(1), DT, rtol=1e-12, atol=0)
    assert (V[:, 0] == 0).all() and (V[:, -1] == 0).all()


def test_default_support_formula():
    import sindy
    for n, n_test in ((8000, 50), (10 ** 6, 5000), (100, 1), (10, 4), (7, 2), (3, 1)):
        L = sindy._local_test_functions(n, DT, n_test)[0]
        assert L == min(n, 2 * (n // (n_test + 1)) + 1)


def _wrapper(n_test=50, support=None, degree=None, d=2, p=2, n=T, dt=DT):
    import sindy
    reg = sindy.SINDyRegression(d, p, False, False, threshold=0.05, device="cpu")
    t = torch.arange(n, dtype=torch.float32) * dt
    wr = sindy.WSINDyWrapper(reg, t, float(t[-1]), num_test_funcs=n_test, test_func_family="poly", device="cpu",
                             test_func_support=support, test_func_degree=degree)
    return reg, wr, float(t[1] - t[0])


@pytest.mark.parametrize("n_test,support,degree", [(50, None, None), (1, T, 6), (500, 3, 1), (200, 313, 16)])
def test_wrapper_tables_match_the_oracle(n_test, support, degree):
    _, wr, dt = _wrapper(n_test, support, degree)
    V, Vd = WL.wsindy_local_test_functions(T, dt, n_test, support, degree)
    for ours, ref in ((wr.V.numpy(), V), (wr.V_drv.numpy(), Vd)):
        assert ours.shape == ref.shape and ours.dtype == np.float32
        assert (ours == 0).sum() == (ref == 0).sum()
        ulp = np.spacing(np.abs(ref).astype(np.float32))
        assert (np.abs(ours.astype(np.float64) - ref) <= ulp).all()
    M = wr.V.double() @ wr.V.double().T
    assert wr.M.dtype == torch.float64 and torch.equal(wr.M, M)
    assert wr.test_func_support == (default_support(T, n_test) if support is None else support)


def _stlsq_fp64(A, rhs, w, thr, steps):
    """fp64 STLSQ on the summed normal equations: per equation, solve on the support, round to fp32 like the regressor's
    parameters, threshold."""
    d, K = rhs.shape[1], A.shape[0]
    mask = np.ones((d, K), bool)
    out = []
    for _ in range(steps):
        xi = np.zeros((d, K), np.float32)
        for i in range(d):
            m = mask[i]
            xi[i, m] = np.linalg.solve(A[np.ix_(m, m)] + w * np.eye(m.sum()), rhs[m, i]).astype(np.float32)
        mask = mask & (np.abs(xi) > thr)
        out.append((xi, mask.copy()))
    return out


def test_pooled_solve_matches_summed_normal_equations():
    rng = np.random.default_rng(7)
    xs = np.stack([damped_oscillator(r, ph) for r, ph in ((1.0, 0.0), (1.5, 0.7), (0.8, 2.1))]).astype(np.float32)
    xs = xs + 1e-3 * rng.standard_normal(xs.shape).astype(np.float32)   # noise, so that thresholding has work to do
    reg, wr, dt = _wrapper()
    Go, bo = WL.wsindy_local_integrals(xs, dt, 2, n_test=50)
    assert Go.shape == (3, 50, 6) and bo.shape == (3, 50, 2)
    wr.integrals = lambda x: (torch.from_numpy(Go), torch.from_numpy(bo))   # oracle instead of the kernel
    M = wr.M.numpy()
    A = sum(Go[r].T @ M @ Go[r] for r in range(3))
    rhs = sum(Go[r].T @ M @ bo[r] for r in range(3))
    w, thr = 1e-6, 0.05
    ref = _stlsq_fp64(A, rhs, w, thr, 4)
    for xi_ref, mask_ref in ref:
        wr.solve(torch.from_numpy(xs), w, thr)
        assert np.array_equal(reg.mask.numpy() > 0, mask_ref)
        np.testing.assert_allclose(reg.Xi.detach().numpy(), xi_ref, rtol=0, atol=1e-10)
    assert np.array_equal(ref[-1][1], XI_STAR != 0)


def test_single_trajectory_batch_equals_the_plain_solve():
    """(1, T, d) pools one trajectory: the same coefficients and residual as (T, d), for both families."""
    import sindy
    x = damped_oscillator().astype(np.float32)
    for family in ("trig", "poly"):
        res = []
        for xin in (x, x[None]):
            reg = sindy.SINDyRegression(2, 2, False, False, threshold=0.05, device="cpu")
            t = torch.arange(T, dtype=torch.float32) * DT
            wr = sindy.WSINDyWrapper(reg, t, float(t[-1]), test_func_family=family, device="cpu")
            dt = float(t[1] - t[0])
            if family == "poly":
                G, b = WL.wsindy_local_integrals(xin, dt, 2, n_test=50)
            else:
                G, b = O.wsindy_integrals(x, dt, float(t[-1]), 2)
                G, b = (G[None], b[None]) if xin.ndim == 3 else (G, b)
            wr.integrals = lambda _x, G=G, b=b: (torch.from_numpy(G), torch.from_numpy(b))
            r, _ = wr.solve(torch.from_numpy(xin), 1e-6, 0.05)
            res.append((r, reg.Xi.detach().numpy().astype(np.float64)))
        assert abs(res[0][0] - res[1][0]) <= 1e-12 * abs(res[0][0])
        np.testing.assert_allclose(res[1][1], res[0][1], rtol=1e-12, atol=0)


@pytest.mark.parametrize("kw", [
    dict(test_func_support=2), dict(test_func_support=T + 1), dict(test_func_support=0),
    dict(test_func_degree=0), dict(test_func_degree=33), dict(test_func_degree=2.5),
    dict(num_test_funcs=0), dict(num_test_funcs=T - 313 + 2, test_func_support=313),
    dict(num_test_funcs=2, test_func_support=T), dict(test_func_support=100.0),
])
def test_out_of_range_arguments_raise_value_error(kw):
    import sindy
    reg = sindy.SINDyRegression(2, 2, False, False, threshold=0.05, device="cpu")
    t = torch.arange(T, dtype=torch.float32) * DT
    with pytest.raises(ValueError):
        sindy.WSINDyWrapper(reg, t, float(t[-1]), test_func_family="poly", device="cpu", **kw)


def test_family_keywords():
    import sindy
    reg = sindy.SINDyRegression(2, 2, False, False, threshold=0.05, device="cpu")
    t = torch.arange(100, dtype=torch.float32) * DT
    for kw in (dict(test_func_support=11), dict(test_func_degree=4)):
        with pytest.raises(ValueError):
            sindy.WSINDyWrapper(reg, t, float(t[-1]), test_func_family="trig", device="cpu", **kw)
    with pytest.raises(NotImplementedError):
        sindy.WSINDyWrapper(reg, t, float(t[-1]), test_func_family="gauss", device="cpu")
    with pytest.raises(ValueError):   # a trajectory of the wrong length
        _, wr, _ = _wrapper(n=100)
        wr.solve(torch.zeros(2, 99, 2), 0.0, 0.05)
    assert math.isclose(float(sindy.WSINDyWrapper(reg, t, float(t[-1]), test_func_family="poly",
                                                  device="cpu").M.diagonal().mean()), DT, rel_tol=1e-6)
