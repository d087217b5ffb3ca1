"""The fused symmetry-regulariser kernels of csrc/sb_symreg.cu against an independent fp64 autograd reference
(`tests/symreg_fp64_ref.py`): the Euler flow map and its JVP (`euler_flow_fwd_kernel`), the adjoint sweep with the
Hessian-vector term (`euler_flow_bwd_kernel`) and the reversed regulariser (`symreg_r_kernel`), at step counts up to the
backward's limit, at sizes past one full grid (1184 blocks × 128 threads = 151 552 samples: grid-stride loop, ordered
fp64 reduction over every block), for every cotangent combination, through autograd, and end to end through
`EulerFlowMap` and `train_SIGED_lbfgs` with flows longer than the fused backward handles.

Errors are rel() = max |kernel − reference| / max |reference| over the tensor; each case prints what it achieved (-s).
"""
import math

import numpy as np
import pytest
import torch

import symreg_fp64_ref as R

pytestmark = pytest.mark.gpu

# the libraries with fused kernels (SB_SYMREG_SHAPES): (d, poly_order, sine, exp)
SHAPES = [(2, 2, False, False), (2, 2, False, True), (2, 3, False, False), (3, 2, False, False), (3, 3, False, False)]
DT = 0.01
DT32 = float(np.float32(DT))          # the step the kernels and the fp32 compositions actually take
FULL_GRID = 148 * 8 * 128

# Bounds: about 4x the worst error measured on one B200 (1000 W) over the cases that use each bound.
VALUE_TOL = 3e-6          # measured 8.0e-7 (euler_flow), 6.0e-7 (ops.euler_flow), 3.4e-7 (EulerFlowMap, <= 32 steps)
GRAD_TOL = 4e-6           # measured 8.8e-7 (euler_flow_backward), 3.5e-7 (ops.euler_flow), 1.9e-7 (EulerFlowMap)
SYMREG_R_TOL = 5e-7       # measured 1.2e-7 for n >= 129
# One sample: the sum is a single fp32 residual J h(x) − h(g x) of two nearly equal terms, so its relative error is
# that of a cancelling difference. Measured 4.4e-6 on the value, 1.5e-6 on the gradient.
SYMREG_R_ONE_SAMPLE_TOL = 2e-5
LONG_VALUE_TOL = 3e-6     # 50 and 100 steps on the composed path: measured 7.9e-7 (100-step forward kernel: 5.7e-7)
LONG_GRAD_TOL = 1e-5      # measured 2.1e-6


@pytest.fixture(scope="module")
def nat():
    from sindy_b200 import native
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    native.load()
    return native


def rel(a, b):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.detach().cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    a, b = a.astype(np.float64), b.astype(np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def inputs(nat, lib, n, seed):
    """x ∈ [−0.6, 0.6], W = 0.3·randn, tangent and cotangents randn: flows of dt = 0.01 stay bounded."""
    d, K = lib[0], nat.Library(*lib).K
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.rand(n, d, device="cuda", generator=g) * 1.2 - 0.6
    v = torch.randn(n, d, device="cuda", generator=g)
    W = 0.3 * torch.randn(d, K, device="cuda", generator=g)
    a = torch.randn(n, d, device="cuda", generator=g)
    b = torch.randn(n, d, device="cuda", generator=g)
    return x, v, W, a, b


def report(tag, errs):
    print(f"{tag}: " + " ".join(f"{k} {v:.2e}" for k, v in errs.items()))
    return errs


def seed_of(lib, n, n_steps):
    d, p, s, e = lib
    return (n * 131 + n_steps * 17 + d * 1000 + p * 100 + s * 10 + e) % (2 ** 31)


# ---------------------------------------------------------------------------------------------------------
# euler_flow / euler_flow_backward through the binding
# ---------------------------------------------------------------------------------------------------------
CASES = [(3001, s) for s in (0, 1, 2, 10, 31, 32)] + \
        [(n, s) for n in (1, 127, 129, FULL_GRID + 1, 1_000_003) for s in (10, 32)]


@pytest.mark.parametrize("n,n_steps", CASES)
@pytest.mark.parametrize("lib", SHAPES)
def test_euler_flow_forward_and_backward_vs_fp64(nat, lib, n, n_steps):
    L = nat.Library(*lib)
    x, v, W, a, b = inputs(nat, lib, n, seed_of(lib, n, n_steps))
    fx_r, jv_r, [(gW_a, gv_a, gx_a), (gW_b, gv_b, gx_b)] = R.flow64_grads(x, v, W, lib, DT32, n_steps,
                                                                          [(a, None), (None, b)])
    fx, jv = nat.euler_flow(x, v, W, L, DT, n_steps)
    fx1, none = nat.euler_flow(x, None, W, L, DT, n_steps)
    assert none is None
    val = {"fx": rel(fx, fx_r), "jv": rel(jv, jv_r), "fx(v=None)": rel(fx1, fx_r)}
    # gradients are linear in the cotangents: the reference of the case with both is the sum of the single ones
    cases = {"g_fx": (a, None, gW_a, gv_a, gx_a), "g_jv": (None, b, gW_b, gv_b, gx_b),
             "both": (a, b, gW_a + gW_b, gv_a + gv_b, gx_a + gx_b)}
    grad = {}
    for name, (ga, gb, gW_r, gv_r, gx_r) in cases.items():
        gW, gv, gx = nat.euler_flow_backward(x, v, ga, gb, W, L, DT, n_steps, need_gv=True, need_gx=True)
        grad.update({f"{name}:gW": rel(gW, gW_r), f"{name}:gv": rel(gv, gv_r), f"{name}:gx": rel(gx, gx_r)})
        if n_steps == 0:            # the identity flow: exact
            assert torch.equal(gW, torch.zeros_like(gW))
            assert torch.equal(gv, gb if gb is not None else torch.zeros_like(v))
            assert torch.equal(gx, ga if ga is not None else torch.zeros_like(x))
    # v = None with dL/dx: the path `symmreg_f` takes (f evaluated at g(x), which carries a gradient)
    gW, gv, gx = nat.euler_flow_backward(x, None, a, None, W, L, DT, n_steps, need_gv=False, need_gx=True)
    assert gv is None
    grad.update({"v=None:gW": rel(gW, gW_a), "v=None:gx": rel(gx, gx_a)})
    report(f"euler_flow {lib} n={n} steps={n_steps}", {**val, **grad})
    if n_steps == 0:
        assert torch.equal(fx, x) and torch.equal(jv, v) and torch.equal(fx1, x)
    assert max(val.values()) < VALUE_TOL, val
    assert max(grad.values()) < GRAD_TOL, grad


def test_backward_step_limit_and_long_forward(nat):
    """The backward kernel keeps at most kMaxSteps = native.EULER_FLOW_MAX_STEPS states per sample: 32 steps run, 33 are
    refused by the C entry point, and ops.euler_flow refuses them at forward time when a gradient will be needed. The
    forward has no limit: a 100-step flow without gradient runs and matches the reference."""
    from sindy_b200 import ops
    lib = (2, 2, False, True)
    L = nat.Library(*lib)
    x, v, W, a, b = inputs(nat, lib, 4099, 1)
    assert nat.EULER_FLOW_MAX_STEPS == 32
    nat.euler_flow_backward(x, v, a, b, W, L, DT, 32, need_gx=True)
    with pytest.raises(nat.SindyB200Error, match="n_steps=33"):
        nat.euler_flow_backward(x, v, a, b, W, L, DT, 33, need_gx=True)
    with pytest.raises(ValueError, match="at most 32 steps"):
        ops.euler_flow(x, v, W.clone().requires_grad_(True), L, DT, 33)
    fx_r, jv_r, _ = R.flow64_grads(x, v, W, lib, DT32, 100, [], need_gx=False)
    fx, jv = ops.euler_flow(x, v, W, L, DT, 100)
    with torch.no_grad():
        fx2, jv2 = ops.euler_flow(x, v, W.clone().requires_grad_(True), L, DT, 100)
    errs = report("euler_flow forward, 100 steps", {"fx": rel(fx, fx_r), "jv": rel(jv, jv_r)})
    assert torch.equal(fx, fx2) and torch.equal(jv, jv2)
    assert max(errs.values()) < LONG_VALUE_TOL, errs


# ---------------------------------------------------------------------------------------------------------
# ops.euler_flow through autograd: the layouts and dtypes callers hand in
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lib", SHAPES)
def test_euler_flow_through_autograd_vs_fp64(nat, lib):
    from sindy_b200 import ops
    L = nat.Library(*lib)
    n, n_steps = 4098, 32
    x, v, W, a, b = inputs(nat, lib, n, seed_of(lib, n, n_steps))
    ones = torch.ones_like(x)
    fx_r, jv_r, refs = R.flow64_grads(x, v, W, lib, DT32, n_steps, [(a, None), (None, b), (ones, None), (None, ones)])
    (gW_a, _, gx_a), (gW_b, gv_b, gx_b), (gW_1, _, gx_1), (gW_j1, gv_j1, gx_j1) = refs
    gW_r, gv_r, gx_r = gW_a + gW_b, gv_b, gx_a + gx_b
    errs = {}

    def check(tag, got, want):
        for k, (g, w) in zip(("fx", "jv", "gW", "gv", "gx"), zip(got, want)):
            if g is not None:
                errs[f"{tag}:{k}"] = rel(g, w)

    # x as the non-contiguous view x_fx[:, 0] that symmreg_i passes (x_fx requires grad through its other half)
    x_fx = torch.stack([x, torch.zeros_like(x)], dim=1).requires_grad_(True)
    Wq, vq = W.clone().requires_grad_(True), v.clone().requires_grad_(True)
    xv = x_fx[:, 0]
    assert not xv.is_contiguous()
    fx, jv = ops.euler_flow(xv, vq, Wq, L, DT, n_steps)
    gW, gv, gxf = torch.autograd.grad((fx * a).sum() + (jv * b).sum(), (Wq, vq, x_fx))
    assert torch.equal(gxf[:, 1], torch.zeros_like(x))
    check("view", (fx, jv, gW, gv, gxf[:, 0]), (fx_r, jv_r, gW_r, gv_r, gx_r))
    # (B, 2, d): the stacked [x, f(x)] layout
    B = n // 2
    x3 = x.view(B, 2, -1).clone().requires_grad_(True)
    v3 = v.view(B, 2, -1).clone().requires_grad_(True)
    Wq = W.clone().requires_grad_(True)
    fx, jv = ops.euler_flow(x3, v3, Wq, L, DT, n_steps)
    assert fx.shape == x3.shape and jv.shape == x3.shape
    gW, gv, gx = torch.autograd.grad((fx * a.view_as(fx)).sum() + (jv * b.view_as(jv)).sum(), (Wq, v3, x3))
    assert gv.shape == x3.shape and gx.shape == x3.shape
    check("B2d", (fx.reshape(n, -1), jv.reshape(n, -1), gW, gv.reshape(n, -1), gx.reshape(n, -1)),
          (fx_r, jv_r, gW_r, gv_r, gx_r))
    # float64 inputs (holding the same fp32 values): gradients come back in float64
    x64, v64, W64 = (t.double().requires_grad_(True) for t in (x, v, W))
    fx, jv = ops.euler_flow(x64, v64, W64, L, DT, n_steps)
    gW, gv, gx = torch.autograd.grad((fx * a).sum() + (jv * b).sum(), (W64, v64, x64))
    assert gW.dtype == gv.dtype == gx.dtype == torch.float64
    check("fp64-in", (fx, jv, gW, gv, gx), (fx_r, jv_r, gW_r, gv_r, gx_r))
    # loss = fx.sum() + jv.sum(): the cotangents arrive as expanded ones with zero strides
    xq, vq, Wq = (t.clone().requires_grad_(True) for t in (x, v, W))
    fx, jv = ops.euler_flow(xq, vq, Wq, L, DT, n_steps)
    gW, gv, gx = torch.autograd.grad(fx.sum() + jv.sum(), (Wq, vq, xq))
    check("sum", (gW, gv, gx), (gW_1 + gW_j1, gv_j1, gx_1 + gx_j1))
    # the value alone (v = None) with dL/dW and dL/dx
    xq, Wq = x.clone().requires_grad_(True), W.clone().requires_grad_(True)
    fx, none = ops.euler_flow(xq, None, Wq, L, DT, n_steps)
    assert none is None
    gW, gx = torch.autograd.grad((fx * a).sum(), (Wq, xq))
    check("value", (fx, None, gW, None, gx), (fx_r, None, gW_a, None, gx_a))
    report(f"ops.euler_flow {lib} n={n} steps={n_steps}", errs)
    vals = {k: e for k, e in errs.items() if k.endswith((":fx", ":jv"))}
    grads = {k: e for k, e in errs.items() if k not in vals}
    assert max(vals.values()) < VALUE_TOL, vals
    assert max(grads.values()) < GRAD_TOL, grads


# ---------------------------------------------------------------------------------------------------------
# reversed regulariser
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 129, FULL_GRID + 1, 1_000_003])
@pytest.mark.parametrize("lib", SHAPES)
def test_symreg_r_loss_and_gradient_vs_fp64(nat, lib, n):
    from sindy_b200 import ops
    L = nat.Library(*lib)
    d, K = lib[0], L.K
    x, _, W, _, _ = inputs(nat, lib, n, seed_of(lib, n, -1))
    g = torch.Generator(device="cuda").manual_seed(n + d)
    gx = x + 0.05 * torch.randn(n, d, device="cuda", generator=g)
    J = torch.eye(d, device="cuda") + 0.1 * torch.randn(n, d, d, device="cuda", generator=g)
    total_r, gW_r = R.symreg_r64_grads(x, gx, J, W, lib)
    out = nat.symreg_r(x, gx, J, W, L)
    Wq = W.clone().requires_grad_(True)
    loss = ops.symreg_r_loss(x, gx, J, Wq, L)
    (gW,) = torch.autograd.grad(loss, (Wq,))
    errs = report(f"symreg_r {lib} n={n}", {
        "sum": abs(float(out[d * K]) - float(total_r)) / float(total_r),
        "sums_gW": rel(out[:d * K].view(d, K), gW_r / 2),        # the kernel's sums are ½ dΣr²/dW
        "loss": abs(float(loss) - float(total_r) / (n * d)) / (float(total_r) / (n * d)),
        "gW": rel(gW, gW_r / (n * d)),
    })
    assert max(errs.values()) < (SYMREG_R_TOL if n > 1 else SYMREG_R_ONE_SAMPLE_TOL), errs


def test_reductions_are_deterministic(nat):
    """The d×K sums are reduced in a fixed order (per-block partials, then the last block adds them in block order): a
    repeat call returns the same bits, at a size where every block of the full grid loops several times."""
    n = 1_000_003
    for lib in ((2, 2, False, True), (3, 3, False, False)):
        L = nat.Library(*lib)
        x, v, W, a, b = inputs(nat, lib, n, 5)
        first = nat.euler_flow_backward(x, v, a, b, W, L, DT, 32, need_gx=True)
        J = torch.eye(lib[0], device="cuda").expand(n, -1, -1).contiguous()
        r_first = nat.symreg_r(x, x + 0.01 * a, J, W, L)
        for _ in range(2):
            again = nat.euler_flow_backward(x, v, a, b, W, L, DT, 32, need_gx=True)
            assert all(torch.equal(p, q) for p, q in zip(first, again)), lib
            assert torch.equal(nat.symreg_r(x, x + 0.01 * a, J, W, L), r_first), lib


# ---------------------------------------------------------------------------------------------------------
# EulerFlowMap end to end: fused flows, flows longer than the fused backward, libraries without a fused kernel
# ---------------------------------------------------------------------------------------------------------
def flow_map_tol(n_steps):
    return (VALUE_TOL, GRAD_TOL) if n_steps <= 32 else (LONG_VALUE_TOL, LONG_GRAD_TOL)


@pytest.mark.parametrize("t", [0.1, 0.5, 1.0])
@pytest.mark.parametrize("lib", [(2, 2, False, True), (2, 2, True, False), (2, 3, False, True)])
def test_euler_flow_map_vs_fp64(nat, lib, t):
    import model_utils
    import sindy
    n = 2001
    x, v, W, a, b = inputs(nat, lib, n, seed_of(lib, n, int(100 * t)))
    reg = sindy.SINDyRegression(lib[0], lib[1], lib[2], lib[3], threshold=0.05, device="cuda")
    reg.Xi.data = W.clone()
    flow = model_utils.EulerFlowMap(reg, t, DT)
    n_steps = flow.n_steps
    assert n_steps == round(t / DT)
    fx_r, jv_r, [(gW_a, _, gx_a), (gW_b, gv_b, gx_b)] = R.flow64_grads(x, v, W, lib, DT32, n_steps,
                                                                       [(a, None), (None, b)])
    xq = x.clone().requires_grad_(True)
    y = flow(xq)
    gXi, gx = torch.autograd.grad((y * a).sum(), (reg.Xi, xq))
    val = {"call:fx": rel(y, fx_r)}
    grad = {"call:gW": rel(gXi, gW_a), "call:gx": rel(gx, gx_a)}
    xq, vq = x.clone().requires_grad_(True), v.clone().requires_grad_(True)
    fx, jv = flow.jvp(xq, vq, require_grad=True)
    gXi, gv, gx = torch.autograd.grad((fx * a).sum() + (jv * b).sum(), (reg.Xi, vq, xq))
    val.update({"jvp:fx": rel(fx, fx_r), "jvp:jv": rel(jv, jv_r)})
    grad.update({"jvp:gW": rel(gXi, gW_a + gW_b), "jvp:gv": rel(gv, gv_b), "jvp:gx": rel(gx, gx_a + gx_b)})
    fused = nat.symreg_supported(reg.library)
    assert flow._fused(x) == (fused and n_steps <= nat.EULER_FLOW_MAX_STEPS)
    kind = ("fused" if n_steps <= nat.EULER_FLOW_MAX_STEPS else "long") if fused else "fallback"
    report(f"EulerFlowMap {lib} {kind} steps={n_steps}", {**val, **grad})
    vt, gt = flow_map_tol(n_steps)
    assert max(val.values()) < vt, val
    assert max(grad.values()) < gt, grad


def test_lbfgs_fit_with_symmreg_i_over_a_50_step_flow(nat, golden, capsys):
    """train_SIGED_lbfgs with sym_reg_type 'i' and int_t / int_dt = 0.5 / 0.01: 50 Euler steps, more than the fused
    backward handles. The flow map takes the composed path and the fit runs with finite losses."""
    import sindy
    import standins
    import train
    g = golden("lbfgs")
    x = torch.as_tensor(g["x"], dtype=torch.float32).cuda()
    dx = torch.as_tensor(g["dx"], dtype=torch.float32).cuda()
    loader = [(x, dx)]
    ae, gen = standins.make_standins(seed=0, input_dim=2, n_comps=2, hidden=32, device="cuda")
    reg = sindy.SINDyRegression(2, 2, False, False, threshold=0.05, device="cuda", constrain_constant=True)
    reg.Xi.data = torch.as_tensor(g["sindy_init_Xi"], dtype=torch.float32).cuda()
    train.train_SIGED_lbfgs(
        train_loader=loader, test_loader=loader, num_epochs=2, device="cuda", log_interval=1,
        save_interval=100000, save_dir=None, autoencoder=ae, generator=gen, regressor=reg, regressor_dst=None,
        use_latent=False, distill_latent=False, lr_sindy=0.1, w_sindy_z=0.0, w_sindy_x=1.0, sindy_reg_type='l1',
        w_sindy_reg=0.0, sym_reg_type='i', w_sym_reg=0.05, st_freq=50, threshold=0.05, int_t=0.5, int_dt=0.01,
        print_eq=False)
    out = capsys.readouterr().out
    logged = [dict(kv.split(": ") for kv in line.split(", ")[1:]) for line in out.splitlines()
              if line.startswith("Epoch ") and "loss_sym_reg" in line]
    assert len(logged) == 2, out
    for m in logged:
        assert all(math.isfinite(float(val)) for val in m.values()), m
    assert torch.isfinite(reg.Xi).all()
