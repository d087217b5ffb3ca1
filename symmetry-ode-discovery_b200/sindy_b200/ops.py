"""Differentiable operators over the C ABI.

`h(x) = Θ(x)·Wᵀ` and everything autograd can ask of it form a closed family of six operators, each a
`torch.autograd.Function` whose backward is written with the others, so first-order training
(`train.py:689`), the double-vjp JVP trick of `torch.autograd.functional.jvp(..., create_graph=True)` used by
the symmetry regularisers (`model_utils.py:32,53,56`) and the outer `loss.backward()` through those JVPs all
run on the CUDA kernels:

    F (x, W)      = Θ(x) Wᵀ                       sb_forward
    Bx(x, W, g)   = J_h(x)ᵀ g                     sb_backward  (gx)
    Bw(x, g)      = gᵀ Θ(x)               (d×K)   sb_backward  (gw)
    T (x, u, W)   = J_h(x) u                      sb_jvp
    Tw(x, u, g)   = gᵀ (J_Θ(x) u)         (d×K)   sb_jvp_backward (gw)
    Hx(x, u, W, g)= ∂/∂x [gᵀ J_h(x) u]            sb_jvp_backward (gx)   (terminal: third order not provided)

`fused_mse` is the one-pass train step: loss and dL/dW from a single sweep over (x, dx) (sb_train_step).
"""
from __future__ import annotations

import torch
from torch.autograd import Function

from . import native
from .native import Library


def _rg(ctx, i):
    return ctx.needs_input_grad[i]


class _F(Function):
    @staticmethod
    def forward(ctx, x, w, lib: Library):
        ctx.lib = lib
        ctx.save_for_backward(x, w)
        return native.forward(x, w, lib)

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        lib = ctx.lib
        gx = _Bx.apply(x, w, gy, lib) if _rg(ctx, 0) else None
        gw = _Bw.apply(x, gy, lib).to(w.dtype) if _rg(ctx, 1) else None
        return gx, gw, None


class _Bx(Function):
    @staticmethod
    def forward(ctx, x, w, g, lib: Library):
        ctx.lib = lib
        ctx.save_for_backward(x, w, g)
        _, gx = native.backward(x, g, w, lib, need_gw=False, need_gx=True)
        return gx

    @staticmethod
    def backward(ctx, c):
        x, w, g = ctx.saved_tensors
        lib = ctx.lib
        gx = _Hx.apply(x, c, w, g, lib) if _rg(ctx, 0) else None
        gw = _Tw.apply(x, c, g, lib).to(w.dtype) if _rg(ctx, 1) else None
        gg = _T.apply(x, c, w, lib) if _rg(ctx, 2) else None
        return gx, gw, gg, None


class _Bw(Function):
    @staticmethod
    def forward(ctx, x, g, lib: Library):
        ctx.lib = lib
        ctx.save_for_backward(x, g)
        gw, _ = native.backward(x, g, torch.empty(0, device=x.device), lib, need_gw=True, need_gx=False)
        return gw.to(torch.float32)

    @staticmethod
    def backward(ctx, C):
        x, g = ctx.saved_tensors
        lib = ctx.lib
        C = C.to(torch.float32)
        gx = _Bx.apply(x, C, g, lib) if _rg(ctx, 0) else None
        gg = _F.apply(x, C, lib) if _rg(ctx, 1) else None
        return gx, gg, None


class _T(Function):
    @staticmethod
    def forward(ctx, x, u, w, lib: Library):
        ctx.lib = lib
        ctx.save_for_backward(x, u, w)
        return native.jvp(x, u, w, lib)

    @staticmethod
    def backward(ctx, g):
        x, u, w = ctx.saved_tensors
        lib = ctx.lib
        gx = _Hx.apply(x, u, w, g, lib) if _rg(ctx, 0) else None
        gu = _Bx.apply(x, w, g, lib) if _rg(ctx, 1) else None
        gw = _Tw.apply(x, u, g, lib).to(w.dtype) if _rg(ctx, 2) else None
        return gx, gu, gw, None


class _Tw(Function):
    @staticmethod
    def forward(ctx, x, u, g, lib: Library):
        ctx.lib = lib
        ctx.save_for_backward(x, u, g)
        gw, _, _ = native.jvp_backward(x, u, g, torch.empty(0, device=x.device), lib, need_gw=True,
                                       need_gx=False, need_gu=False)
        return gw.to(torch.float32)

    @staticmethod
    def backward(ctx, C):
        x, u, g = ctx.saved_tensors
        lib = ctx.lib
        C = C.to(torch.float32)
        gx = _Hx.apply(x, u, C, g, lib) if _rg(ctx, 0) else None
        gu = _Bx.apply(x, C, g, lib) if _rg(ctx, 1) else None
        gg = _T.apply(x, u, C, lib) if _rg(ctx, 2) else None
        return gx, gu, gg, None


class _Hx(Function):
    @staticmethod
    def forward(ctx, x, u, w, g, lib: Library):
        _, gx, _ = native.jvp_backward(x, u, g, w, lib, need_gw=False, need_gx=True, need_gu=False)
        return gx

    @staticmethod
    def backward(ctx, c):
        raise NotImplementedError(
            "sindy_b200: third-order derivatives of the SINDy library are not provided (no reference path needs them)")


def sindy_forward(x: torch.Tensor, w: torch.Tensor, lib: Library) -> torch.Tensor:
    """Differentiable h(x) = Θ(x)·Wᵀ (any order the reference's losses need)."""
    return _F.apply(x, w, lib)


def sindy_jvp(x: torch.Tensor, u: torch.Tensor, w: torch.Tensor, lib: Library) -> torch.Tensor:
    """Differentiable J_h(x)·u (closed form of `jvp(regressor, x, u)[1]`, `train.py:503-507`)."""
    return _T.apply(x, u, w, lib)


class _FusedMSE(Function):
    """loss = mean((Θ(x)Wᵀ − dx)²) with dL/dW from the same pass (`train.py:663-664,689`)."""

    @staticmethod
    def forward(ctx, x, dx, w, lib: Library):
        flags = native.SB_STEP_LOSS | native.SB_STEP_GRAD
        out = native.train_step(x, dx, w, lib, flags)
        n = x.numel() // lib.dim
        denom = float(max(n, 1) * lib.dim)
        ctx.save_for_backward(out)
        ctx.meta = (lib, denom, w.dtype)
        return (out[0] / denom).to(torch.float32)

    @staticmethod
    def backward(ctx, gl):
        (out,) = ctx.saved_tensors
        lib, denom, wdtype = ctx.meta
        gw = None
        if ctx.needs_input_grad[2]:
            gw = (out[2:2 + lib.dim * lib.K].view(lib.dim, lib.K) * (2.0 / denom) * gl.double()).to(wdtype)
        return None, None, gw, None


def fused_mse(x: torch.Tensor, dx: torch.Tensor, w: torch.Tensor, lib: Library) -> torch.Tensor:
    """One-pass MSE loss whose backward (w.r.t. W only) costs nothing extra. The fused pass differentiates with respect
    to the PARAMETERS only: if x or dx carry a gradient (a latent z / dz from an encoder being trained) the loss is
    composed from the differentiable forward operator instead, so that no gradient is silently dropped."""
    if torch.is_grad_enabled() and (x.requires_grad or dx.requires_grad):
        return torch.nn.functional.mse_loss(sindy_forward(x, w, lib), dx)
    return _FusedMSE.apply(x, dx, w, lib)


class _EulerFlow(Function):
    """(fx, jv) = (f(x), J_f(x)·v) for the flow map f of n explicit-Euler steps of h (`model_utils.py:236-240, 55-56`):
    one launch forward, one launch backward (gradients w.r.t. v, W and — if asked — x). Once differentiable: the
    reference needs second order only because it builds the JVP itself by a double vjp."""

    @staticmethod
    def forward(ctx, x, v, w, lib: Library, dt: float, n_steps: int):
        ctx.meta = (lib, float(dt), int(n_steps))
        ctx.save_for_backward(x, v, w)
        fx, jv = native.euler_flow(x, v, w, lib, dt, n_steps)
        return fx, jv

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_fx, g_jv):
        x, v, w = ctx.saved_tensors
        lib, dt, n_steps = ctx.meta
        gw, gv, gx = native.euler_flow_backward(x, v, g_fx, g_jv, w, lib, dt, n_steps, need_gv=_rg(ctx, 1),
                                                need_gx=_rg(ctx, 0))
        return gx, gv, (gw.to(w.dtype) if _rg(ctx, 2) else None), None, None, None


class _EulerFlowValue(Function):
    """fx = f(x) alone (no tangent)."""

    @staticmethod
    def forward(ctx, x, w, lib: Library, dt: float, n_steps: int):
        ctx.meta = (lib, float(dt), int(n_steps))
        ctx.save_for_backward(x, w)
        return native.euler_flow(x, None, w, lib, dt, n_steps)[0]

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_fx):
        x, w = ctx.saved_tensors
        lib, dt, n_steps = ctx.meta
        gw, _, gx = native.euler_flow_backward(x, None, g_fx, None, w, lib, dt, n_steps, need_gv=False,
                                               need_gx=_rg(ctx, 0))
        return gx, (gw.to(w.dtype) if _rg(ctx, 1) else None), None, None, None


def euler_flow(x, v, w, lib: Library, dt: float, n_steps: int):
    """Differentiable (f(x), J_f(x)·v) — v may be None: (f(x), None). The backward handles at most
    native.EULER_FLOW_MAX_STEPS steps: a longer flow that will need a gradient is refused here, at forward time."""
    if (n_steps > native.EULER_FLOW_MAX_STEPS and torch.is_grad_enabled()
            and any(t is not None and t.requires_grad for t in (x, v, w))):
        raise ValueError(f"euler_flow: the fused backward handles at most {native.EULER_FLOW_MAX_STEPS} steps, got "
                         f"{n_steps}; differentiate a longer flow by composing its steps (model_utils.odeint)")
    if v is None:
        return _EulerFlowValue.apply(x, w, lib, dt, n_steps), None
    return _EulerFlow.apply(x, v, w, lib, dt, n_steps)


class _SymregR(Function):
    """mean((J_g(x)h(x) − h(g(x)))²) for one group element with precomputed g(x), J_g(x): value and dL/dW from ONE
    streaming pass (`model_utils.py:126-170`)."""

    @staticmethod
    def forward(ctx, x, gx, jgx, w, lib: Library):
        out = native.symreg_r(x, gx, jgx, w, lib)
        n = x.numel() // lib.dim
        denom = float(max(n, 1) * lib.dim)
        ctx.save_for_backward(out)
        ctx.meta = (lib, denom, w.dtype)
        return (out[lib.dim * lib.K] / denom).to(torch.float32)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gl):
        (out,) = ctx.saved_tensors
        lib, denom, wdtype = ctx.meta
        gw = None
        if ctx.needs_input_grad[3]:
            gw = (out[:lib.dim * lib.K].view(lib.dim, lib.K) * (2.0 / denom) * gl.double()).to(wdtype)
        return None, None, None, gw, None


def symreg_r_loss(x, gx, jgx, w, lib: Library) -> torch.Tensor:
    return _SymregR.apply(x, gx, jgx, w, lib)
