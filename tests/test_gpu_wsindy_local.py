"""GPU checks of the compactly supported WSINDy integrals (sb_wsindy_local_integrals) and of WSINDyWrapper's 'poly'
family and pooled multi-trajectory solve: kernel against the fp64 oracle on ragged shapes, bitwise determinism across
batches and repeats, recovery of an analytic system, and the error paths."""
import numpy as np
import pytest
import torch

from oracle import sindy_oracle as O
import wsindy_local_oracle as WL

pytestmark = pytest.mark.gpu

DT = 0.002


@pytest.fixture(scope="module")
def nat():
    from sindy_b200 import native
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    native.load()
    return native


def tables(T, n_test, L, p, dt=DT):
    import sindy
    _, _, _, phi, dphi = sindy._local_test_functions(T, dt, n_test, L, p)
    return torch.from_numpy(phi).cuda(), torch.from_numpy(dphi).cuda()


# (d, p, sine, exp), n_traj, T, n_test, L, degree — every listed size occurs: n_traj 1/7/37/300, T = L / L+1 / 1000 /
# 8001, n_test 1/50/500, L 3/313/T, degree 1/6/16; L = 8001 walks the support in several 2048-sample blocks
CASES = [
    ((2, 2, 0, 0), 1, 8001, 50, 313, 6),
    ((2, 2, 0, 1), 7, 1000, 500, 3, 1),
    ((2, 3, 0, 0), 37, 1000, 500, 313, 16),
    ((2, 3, 0, 0), 300, 1000, 50, 313, 6),
    ((2, 3, 1, 0), 300, 314, 1, 313, 6),
    ((3, 3, 0, 0), 7, 8001, 1, 8001, 16),
    ((3, 5, 0, 0), 37, 8001, 50, 313, 1),
    ((3, 5, 0, 0), 1, 8001, 1, 8001, 6),
    ((1, 3, 1, 1), 300, 3, 1, 3, 6),
    ((8, 2, 1, 1), 7, 1000, 500, 313, 6),
    ((8, 2, 1, 1), 1, 8001, 1, 8001, 1),
]


@pytest.mark.parametrize("lib,n_traj,T,n_test,L,deg", CASES)
def test_kernel_matches_the_oracle(nat, lib, n_traj, T, n_test, L, deg):
    d, p, s, e = lib
    rng = np.random.default_rng(n_traj * 7 + T)
    x = (0.5 * rng.standard_normal((n_traj, T, d))).astype(np.float32)
    phi, dphi = tables(T, n_test, L, deg)
    G, b = nat.wsindy_local_integrals(torch.from_numpy(x).cuda(), nat.Library(d, p, bool(s), bool(e)), phi, dphi, n_test)
    Go, bo = WL.wsindy_local_integrals(x, DT, p, bool(s), bool(e), n_test=n_test, support=L, degree=deg)
    G, b = G.cpu().numpy(), b.cpu().numpy()
    assert G.shape == Go.shape and b.shape == bo.shape
    for r in range(n_traj):
        assert np.abs(G[r] - Go[r]).max() <= 1e-5 * np.abs(Go[r]).max(), r
        assert np.abs(b[r] - bo[r]).max() <= 1e-5 * np.abs(bo[r]).max(), r


def test_single_trajectory_shape(nat):
    x = torch.randn(1000, 2, device="cuda")
    phi, dphi = tables(1000, 50, 39, 6)
    lib = nat.Library(2, 3)
    G, b = nat.wsindy_local_integrals(x, lib, phi, dphi, 50)
    Gb, bb = nat.wsindy_local_integrals(x[None], lib, phi, dphi, 50)
    assert G.shape == (50, 10) and b.shape == (50, 2)
    assert torch.equal(G, Gb[0]) and torch.equal(b, bb[0])


@pytest.mark.parametrize("lib", [(2, 3, 0, 0), (3, 5, 0, 0), (2, 3, 1, 0)])
@pytest.mark.parametrize("T,L", [(1000, 313), (8001, 4500)])
def test_deterministic_across_batches_and_repeats(nat, lib, T, L):
    d, p, s, e = lib
    L_lib = nat.Library(d, p, bool(s), bool(e))
    x = torch.randn(37, T, d, device="cuda") * 0.5
    n_test = 50 if L < 4000 else 3
    phi, dphi = tables(T, n_test, L, 6)
    before = nat.kernel_launches()
    G, b = nat.wsindy_local_integrals(x, L_lib, phi, dphi, n_test)
    assert nat.kernel_launches() > before
    G2, b2 = nat.wsindy_local_integrals(x, L_lib, phi, dphi, n_test)
    assert torch.equal(G, G2) and torch.equal(b, b2)
    Gs, bs = nat.wsindy_local_integrals(x[5:12].clone(), L_lib, phi, dphi, n_test)
    assert torch.equal(G[5:12], Gs) and torch.equal(b[5:12], bs)
    for r in (0, 3, 36):
        G1, b1 = nat.wsindy_local_integrals(x[r].clone(), L_lib, phi, dphi, n_test)
        assert torch.equal(G[r], G1) and torch.equal(b[r], b1)


def oscillator(radius, phase, T=8000, dt=DT):
    t = np.arange(T) * dt
    return radius * np.exp(-0.1 * t)[:, None] * np.stack([np.cos(t + phase), np.sin(t + phase)], 1)


XI_STAR = np.zeros((2, 6))
XI_STAR[0, 1], XI_STAR[0, 2], XI_STAR[1, 1], XI_STAR[1, 2] = -0.1, -1.0, 1.0, -0.1


def fit(x, family="poly", iters=10):
    import sindy
    reg = sindy.SINDyRegression(2, 2, False, False, threshold=0.05, device="cuda")
    t = torch.arange(x.shape[-2], dtype=torch.float32) * DT
    wr = sindy.WSINDyWrapper(reg, t, float(t[-1]), test_func_family=family, device="cuda")
    for _ in range(iters):
        _, conv = wr.solve(x, 0.0, 0.05)
        if conv:
            break
    return reg, wr


@pytest.mark.parametrize("n_traj", [1, 16])
def test_recovery_through_the_wrapper(nat, n_traj):
    rng = np.random.default_rng(3)
    xs = [oscillator(0.5 + 1.5 * rng.random(), 2 * np.pi * rng.random()) for _ in range(n_traj)]
    x = torch.from_numpy(np.stack(xs).astype(np.float32)).cuda()
    reg, wr = fit(x[0] if n_traj == 1 else x)
    assert wr.test_func_support == 313
    assert np.array_equal(reg.mask.cpu().numpy() > 0, XI_STAR != 0)
    assert np.abs(reg.Xi.detach().cpu().numpy() - XI_STAR).max() <= 1e-4


def test_pooled_trig_solve_equals_summed_normal_equations(nat):
    import sindy
    rng = np.random.default_rng(5)
    x = torch.from_numpy(np.stack([oscillator(r, ph, T=2000) for r, ph in ((1.0, 0.0), (1.4, 1.0), (0.7, 2.0))])
                         .astype(np.float32) + 1e-3 * rng.standard_normal((3, 2000, 2)).astype(np.float32)).cuda()
    reg = sindy.SINDyRegression(2, 2, False, False, threshold=0.05, device="cuda")
    t = torch.arange(2000, dtype=torch.float32) * DT
    wr = sindy.WSINDyWrapper(reg, t, float(t[-1]), device="cuda")
    G, b = wr.integrals(x)
    wr.integrals = lambda _x: (G, b)
    M, Gn, bn = wr.M.cpu().numpy(), G.cpu().numpy(), b.cpu().numpy()
    A = sum(Gn[r].T @ M @ Gn[r] for r in range(3))
    rhs = sum(Gn[r].T @ M @ bn[r] for r in range(3))
    wr.solve(x, 1e-6, 0.0)                          # one full-support solve, no thresholding
    ref = np.linalg.solve(A + 1e-6 * np.eye(6), rhs).T
    xi = reg.Xi.detach().cpu().numpy().astype(np.float64)
    assert np.abs(xi - ref.astype(np.float32)).max() <= 1e-10 * max(1.0, np.abs(ref).max())

    # (1, T, d) pools one trajectory: the same as (T, d)
    out = []
    for xin in (x[0], x[:1]):
        reg1 = sindy.SINDyRegression(2, 2, False, False, threshold=0.05, device="cuda")
        wr1 = sindy.WSINDyWrapper(reg1, t, float(t[-1]), device="cuda")
        res, _ = wr1.solve(xin, 1e-6, 0.05)
        out.append((res, reg1.Xi.detach().cpu().numpy().astype(np.float64)))
    assert abs(out[0][0] - out[1][0]) <= 1e-12 * abs(out[0][0])
    np.testing.assert_allclose(out[1][1], out[0][1], rtol=1e-12, atol=0)


def test_errors(nat):
    phi, dphi = tables(1000, 50, 39, 6)
    lib = nat.Library(2, 3)
    with pytest.raises(RuntimeError):
        nat.wsindy_local_integrals(torch.zeros(1000, 2), lib, phi, dphi, 50)
    with pytest.raises(RuntimeError):
        nat.wsindy_local_integrals(torch.zeros(1000, 2, device="cuda"), lib, phi.cpu(), dphi.cpu(), 50)
    x = torch.zeros(2, 1000, 2, device="cuda")
    for bad_x, n_test in ((x, 1000 - 39 + 2), (x[:, :38], 1)):        # starts not distinct; support longer than T
        with pytest.raises(nat.SindyB200Error, match="status -1"):
            nat.wsindy_local_integrals(bad_x, lib, phi, dphi, n_test)
    with pytest.raises(nat.SindyB200Error, match="status -1"):         # support below 3
        nat.wsindy_local_integrals(x, lib, phi[:2], dphi[:2], 1)
    G, b = nat.wsindy_local_integrals(x[:0], lib, phi, dphi, 50)      # no trajectories: a no-op
    assert G.shape == (0, 50, 10) and b.shape == (0, 50, 2)
