"""CPU checks of the fp64 reference of the fused symmetry-regulariser kernels (`tests/symreg_fp64_ref.py`): its Θ is the
oracle's Θ, one Euler step is the oracle's h and J_h·v, and every gradient it returns — with respect to W, v and x,
the last through the jvp — agrees with central finite differences. Also the step limit of the fused backward is
refused at forward time. No compute entry point is called."""
import numpy as np
import pytest
import torch

from oracle import sindy_oracle as O
import symreg_fp64_ref as R

# the libraries of the fused kernels (SB_SYMREG_SHAPES in csrc/sb_symreg.cu) plus one sine library
SHAPES = [(2, 2, False, False), (2, 2, False, True), (2, 3, False, False), (3, 2, False, False), (3, 3, False, False),
          (2, 3, True, False)]
DT = 0.01


def inputs(lib, n, seed):
    d = lib[0]
    K = O.term_count(*lib)
    g = torch.Generator().manual_seed(seed)
    x = (torch.rand(n, d, generator=g) * 1.2 - 0.6).double()
    v = torch.randn(n, d, generator=g).double()
    W = (0.3 * torch.randn(d, K, generator=g)).double()
    a = torch.randn(n, d, generator=g).double()
    b = torch.randn(n, d, generator=g).double()
    return x, v, W, a, b


@pytest.mark.parametrize("lib", SHAPES)
def test_theta64_is_the_oracle_theta(lib):
    x = inputs(lib, 257, 1)[0]
    x[0] = 0.0                                                   # the monomials' corner cases
    ours = R.theta64(x, *lib).numpy()
    ref = O.theta(x.numpy(), lib[1], lib[2], lib[3])
    assert ours.shape == ref.shape
    assert np.abs(ours - ref).max() <= 1e-14 * np.abs(ref).max()


@pytest.mark.parametrize("lib", SHAPES)
def test_one_step_is_the_oracle_forward_and_jvp(lib):
    x, v, W = inputs(lib, 257, 2)[:3]
    fx, jv = R.flow64(x, v, W, lib, DT, 1)
    xn, vn, Wn = x.numpy(), v.numpy(), W.numpy()
    want_fx = xn + DT * (O.theta(xn, lib[1], lib[2], lib[3]) @ Wn.T)
    want_jv = vn + DT * O.jvp(xn, vn, Wn, lib[1], lib[2], lib[3])
    assert np.abs(fx.numpy() - want_fx).max() <= 1e-14 * np.abs(want_fx).max()
    assert np.abs(jv.numpy() - want_jv).max() <= 1e-14 * np.abs(want_jv).max()
    fx0, jv0 = R.flow64(x, v, W, lib, DT, 0)
    assert torch.equal(fx0, x) and torch.equal(jv0, v)


def per_sample_loss(x, v, W, a, b, lib, n_steps):
    fx, jv = R.flow64(x, v, W, lib, DT, n_steps)
    return (a * fx).sum(1) + (b * jv).sum(1)


def fd_error(lib, n_steps, n=6, eps=1e-5):
    """max |autograd − central difference| / max |central difference| over gW, gv and gx of Σ a·fx + Σ b·jv. Samples
    are independent, so perturbing one coordinate of every sample at once gives each sample's derivative."""
    x, v, W, a, b = inputs(lib, n, 3 + n_steps)
    fx, jv, [(gW, gv, gx)] = R.flow64_grads(x, v, W, lib, DT, n_steps, [(a, b)])
    err = {}
    fd_W = torch.zeros_like(W)
    for i in range(W.shape[0]):
        for k in range(W.shape[1]):
            dW = torch.zeros_like(W)
            dW[i, k] = eps
            fd_W[i, k] = (per_sample_loss(x, v, W + dW, a, b, lib, n_steps).sum()
                          - per_sample_loss(x, v, W - dW, a, b, lib, n_steps).sum()) / (2 * eps)
    err["gW"] = ((gW - fd_W).abs().max() / fd_W.abs().max()).item() if n_steps else gW.abs().max().item()
    for name, g, which in (("gv", gv, 1), ("gx", gx, 0)):
        fd = torch.zeros_like(x)
        for q in range(x.shape[1]):
            e = torch.zeros_like(x)
            e[:, q] = eps
            args_p, args_m = [x, v], [x, v]
            args_p[which], args_m[which] = args_p[which] + e, args_m[which] - e
            fd[:, q] = (per_sample_loss(*args_p, W, a, b, lib, n_steps)
                        - per_sample_loss(*args_m, W, a, b, lib, n_steps)) / (2 * eps)
        err[name] = ((g - fd).abs().max() / fd.abs().max()).item()
    return err


@pytest.mark.parametrize("n_steps", [0, 1, 10, 40])
@pytest.mark.parametrize("lib", [(2, 2, False, True), (3, 2, False, False), (2, 3, True, False)])
def test_gradients_agree_with_central_differences(lib, n_steps):
    err = fd_error(lib, n_steps)
    print(f"fp64 reference vs central differences {lib} steps={n_steps}: {err}")
    if n_steps == 0:
        assert err["gW"] == 0.0                                   # W is unused: the gradient is exactly zero
    assert max(err.values()) < 1e-7, err


def test_chunked_evaluation_matches_one_chunk():
    lib = (2, 2, False, True)
    x, v, W, a, b = inputs(lib, 1001, 4)
    one = R.flow64_grads(x, v, W, lib, DT, 7, [(a, None), (None, b)])
    many = R.flow64_grads(x, v, W, lib, DT, 7, [(a, None), (None, b)], chunk=300)
    assert torch.equal(one[0], many[0]) and torch.equal(one[1], many[1])
    for g1, g2 in zip(one[2], many[2]):
        assert torch.allclose(g1[0], g2[0], rtol=1e-13, atol=0)
        assert torch.equal(g1[1], g2[1]) and torch.equal(g1[2], g2[2])
    gx = x + 0.05 * torch.randn(x.shape, dtype=torch.float64)
    J = torch.eye(2, dtype=torch.float64) + 0.1 * torch.randn(1001, 2, 2, dtype=torch.float64)
    s1, gW1 = R.symreg_r64_grads(x, gx, J, W, lib)
    s2, gW2 = R.symreg_r64_grads(x, gx, J, W, lib, chunk=300)
    want = O.symmreg_r_precomputed(x.numpy(), [gx.numpy()], [J.numpy()], W.numpy(), 2, False, True)
    assert abs(float(s1) / (1001 * 2) - want) <= 1e-6 * want      # the oracle forms Θ in fp32
    assert abs(float(s1 - s2)) <= 1e-13 * float(s1) and torch.allclose(gW1, gW2, rtol=1e-13, atol=1e-15)


def test_a_differentiable_flow_longer_than_the_fused_backward_is_refused_at_forward_time():
    """The fused backward keeps at most EULER_FLOW_MAX_STEPS states per sample: ops.euler_flow refuses a longer flow
    that will need a gradient before any device work (here on CPU tensors, so no kernel could have run)."""
    from sindy_b200 import native, ops
    lib = native.Library(2, 2)
    x = torch.zeros(4, 2, requires_grad=True)
    w = torch.zeros(2, 6)
    limit = native.EULER_FLOW_MAX_STEPS
    assert limit == 32
    for v in (None, torch.zeros(4, 2)):
        with pytest.raises(ValueError, match="at most 32 steps"):
            ops.euler_flow(x, v, w, lib, 0.01, limit + 1)
        with pytest.raises(ValueError):
            ops.euler_flow(x.detach(), v, w.requires_grad_(True), lib, 0.01, 100)
        w.requires_grad_(False)
