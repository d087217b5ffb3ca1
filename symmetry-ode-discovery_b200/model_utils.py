"""Drop-in replacement for the reference's `model_utils.py`: symmetry-regularisation losses and `odeint`.

The losses keep the reference's signatures and values (`model_utils.py:8-221`). The autoencoder / generator are
frozen inputs and stay ordinary PyTorch modules; everything that touches the SINDy library — h(x), J_h(x)·u and
their derivatives — goes through the CUDA operators of `sindy_b200.ops`, which are closed under the
differentiation the double-vjp `jvp(..., create_graph=True)` trick performs.

`odeint` (`model_utils.py:223-255`) dispatches to the batched rollout kernel whenever no gradient is needed and
`f` is a SINDyRegression on a CUDA device; otherwise it steps `f` in Python (differentiable, same formulas).
"""
from __future__ import annotations

from functools import partial

import torch
from torch.autograd.functional import jvp

import os

from sindy_b200 import mlp as _mlp
from sindy_b200 import native, ops

__all__ = [
    "symmreg_i", "symmreg_f", "symmreg_r", "symmreg_r_precomputed", "precompute_symmreg_r", "odeint", "EulerFlowMap",
    "group_action_and_jacobian", "encode_constant_component",
    "make_symmreg", "make_symmreg_pttrain", "make_symmreg_np", "make_fsymmreg", "make_fsymmreg_pttrain",
    "make_fsymmreg_np", "make_rsymmreg", "make_rsymmreg_pttrain",
]


def _jvp_fn(require_grad):
    return partial(jvp, create_graph=True, strict=True) if require_grad else jvp


def _is_regressor(f):
    return hasattr(f, 'library') and hasattr(f, 'mask') and hasattr(f, '_current_Xi')


class EulerFlowMap:
    """f(x) = odeint(regressor, x, t, dt) with method 'euler' — the flow map `train.py:669-673` builds as a local
    closure — as an object that ALSO knows its Jacobian-vector product: `jvp(x, v)` returns (f(x), J_f(x)·v) from ONE
    kernel launch (sb_euler_flow) with a one-launch backward, where the reference runs two reverse passes through
    n Python Euler steps with create_graph=True (`model_utils.py:55-56`). `symmreg_i` uses it when it is handed one;
    any other callable takes the reference's double-vjp path. Falls back to the operator-by-operator composition for
    libraries without a fused kernel, off the GPU, and for flows longer than the fused backward handles
    (native.EULER_FLOW_MAX_STEPS)."""

    def __init__(self, regressor, t, dt):
        self.regressor, self.t, self.dt = regressor, t, dt
        self.n_steps = int(t / dt)

    def _fused(self, x):
        return (_is_regressor(self.regressor) and torch.is_tensor(x) and x.is_cuda
                and self.n_steps <= native.EULER_FLOW_MAX_STEPS and native.symreg_supported(self.regressor.library))

    def _w(self):
        reg = self.regressor
        reg.Xi = reg._current_Xi()
        return reg.Xi * reg.mask

    def __call__(self, x):
        # first-order differentiable in x and Ξ (one launch forward, one backward); a caller that differentiates THROUGH
        # the backward (torch.autograd.functional.jvp's double vjp) must use `.jvp` or a plain closure over `odeint`
        if self._fused(x):
            return ops.euler_flow(x, None, self._w(), self.regressor.library, self.dt, self.n_steps)[0]
        return odeint(self.regressor, x, self.t, self.dt)

    def jvp(self, x, v, require_grad=True):
        # first-order differentiable in x, v and Ξ (sb_euler_flow_backward carries the second derivatives of the library
        # that dL/dx needs). `symmreg_i` hands in x = x_fx[:, 0], a view of a tensor that requires grad because its OTHER
        # half is f(x): the fused launch must not be lost to that flag.
        if self._fused(x):
            return ops.euler_flow(x, v, self._w(), self.regressor.library, self.dt, self.n_steps)
        return _jvp_fn(require_grad)(lambda q: odeint(self.regressor, q, self.t, self.dt), x, v)


def _fast_ae(autoencoder, x):
    """(encoder, decoder) on the tensor cores (`sindy_b200.mlp.FrozenMLP`) when the autoencoder is the reference's MLP,
    frozen, in eval mode and x lives on the GPU; None keeps the PyTorch modules. SINDY_B200_AE_MLP=0 switches it off,
    =require raises instead of falling back."""
    mode = os.environ.get("SINDY_B200_AE_MLP", "1")
    if not (torch.is_tensor(x) and x.is_cuda) or mode == "0":
        return None
    if torch._C._functorch.maybe_current_level() is not None:
        return None       # inside vmap / jacfwd (`precompute_symmreg_r`, `model_utils.py:172-211`): PyTorch modules only
    pair = _mlp.accelerate(autoencoder)
    if pair is None and mode == "require":          # tests: prove that the tensor-core path is the one that ran
        raise RuntimeError("SINDY_B200_AE_MLP=require: this autoencoder is not served by sindy_b200.mlp.FrozenMLP")
    return pair


def _encode(autoencoder, x, fast_ok=True):
    fast = _fast_ae(autoencoder, x) if fast_ok else None
    return fast[0].value(x) if fast is not None else autoencoder.encode(x)


def _decode(autoencoder, z, fast_ok=True):
    fast = _fast_ae(autoencoder, z) if fast_ok else None
    return fast[1].value(z) if fast is not None else autoencoder.decode(z)


def _decoder_tangent(autoencoder, z, v, require_grad):
    """J_decoder(z)·v (`jvp(autoencoder.decoder, z, v)[1]`, `model_utils.py:32`)."""
    fast = _fast_ae(autoencoder, z)
    if fast is not None:
        return fast[1].value_and_jvp(z, v)[1]
    return _jvp_fn(require_grad)(autoencoder.decoder, z, v=v)[1]


def encode_constant_component(autoencoder, x):
    """Encoder output of the DATA half of x_fx = [x, f(x)] (`train.py:669-673`), (B × latent), for `symmreg_i(..., z_x=)`:
    x does not change during a fit, the encoder is row-wise (Linear + eval-mode BatchNorm + ReLU), so its value on the x
    rows is computed once per fit instead of in every closure — and needs no backward. Only with the tensor-core MLP
    (None otherwise: the PyTorch module's reshapes pair the rows of a batch)."""
    fast = _fast_ae(autoencoder, x)
    if fast is None:
        return None
    with torch.no_grad():
        return fast[0].value_rows(x)


def _centred_latent(autoencoder, x, normalize, z_mean, fast_ok=True, z_first=None):
    """z = encode(x) − centre, centre = batch mean ('in_batch') or z_mean / last BatchNorm bias ('global').
    z_first: precomputed encoder output of x[:, 0] (`encode_constant_component`)."""
    fast = _fast_ae(autoencoder, x) if (z_first is not None and fast_ok) else None
    if fast is not None and x.dim() == 3 and x.shape[1] == 2 and z_first.shape[0] == x.shape[0]:
        z = torch.stack([z_first, fast[0].value_rows(x[:, 1])], dim=1)
    else:
        z = _encode(autoencoder, x, fast_ok)
    if normalize == 'in_batch':
        z = z - z.mean(dim=0, keepdim=True)
    elif normalize == 'global':
        if z_mean is None:
            z_mean = autoencoder.encoder[-2].bias
        z = z - z_mean
    return z, z_mean


def _act_on_latent(mat, z):
    """Apply an (n_dims × n_dims) matrix to the flattened latent of every sample, keep z's shape."""
    flat = z.reshape(z.shape[0], -1)
    return torch.einsum('jk,...k->...j', mat, flat).reshape(z.shape)


def symmreg_i(x_fx, autoencoder, generator, f=None, dfdx=None, normalize='global', z_mean=None, relative=True,
              require_grad=False, numpy=False, z_x=None):
    '''
    Infinitesimal (Lie-derivative) symmetry loss: for every generator v,
        mean((J_f(x)·v_x − v_fx)²) [/ mean((J_f(x)·v_x)²) if relative],
    with (v_x, v_fx) = J_decoder(z)·(v z), z = encode([x, f(x)]) − centre.
    x_fx: (batch, 2, input_dim) input and predicted output; f: map to be symmetrised (or dfdx: its Jacobian).
    z_x (extension): `encode_constant_component(autoencoder, x_fx[:, 0])`, computed once per fit.
    '''
    if numpy:
        x_fx = torch.from_numpy(x_fx).float().to(autoencoder.device)
        if z_mean is not None:
            z_mean = torch.from_numpy(z_mean).float().to(autoencoder.device)
        if require_grad:
            raise ValueError('Cannot require grad when numpy=True.')
    if f is None and dfdx is None:
        raise ValueError('Either f or dfdx must be specified.')
    if f is not None and dfdx is not None:
        raise ValueError('Only one of f and dfdx can be specified.')
    jvp_fn = _jvp_fn(require_grad)
    autoencoder.eval()
    generator.eval()

    with torch.set_grad_enabled(require_grad):
        z, _ = _centred_latent(autoencoder, x_fx, normalize, z_mean, z_first=z_x)
        x = x_fx[:, 0]
        loss = 0.0
        for v in generator.get_full_basis_list():
            tangent = _decoder_tangent(autoencoder, z, _act_on_latent(v, z), require_grad)
            v_x, v_fx = tangent[:, 0], tangent[:, 1]
            if isinstance(f, EulerFlowMap):
                pushed = f.jvp(x, v_x, require_grad)[1]          # one fused launch instead of a double vjp
            elif f is not None:
                pushed = jvp_fn(f, x, v_x)[1]
            else:
                pushed = torch.einsum('bjk,bk->bj', dfdx, v_x)
            defect = torch.mean((pushed - v_fx) ** 2)
            loss += defect / torch.mean(pushed ** 2) if relative else defect

    return loss.cpu().numpy() if numpy else loss


def symmreg_f(x_fx, autoencoder, generator, f, normalize='global', z_mean=None, relative=True, require_grad=False,
              numpy=False):
    '''Finite-group symmetry loss mean((f(g·x) − g·f(x))²) [/ mean((f(g·x) − f(x))²)] over the deterministic
    group elements of the generator, transported through the autoencoder (reference `model_utils.py:69-124`).'''
    autoencoder.eval()
    generator.eval()
    if numpy:
        dev = generator.Li[0].device
        x_fx = torch.from_numpy(x_fx).float().to(dev)
        if z_mean is not None:
            z_mean = torch.from_numpy(z_mean).float().to(dev)
        if require_grad:
            raise ValueError('Cannot require grad when numpy=True.')

    with torch.set_grad_enabled(require_grad):
        z, z_mean = _centred_latent(autoencoder, x_fx, normalize, z_mean)
        fx = x_fx[:, 1]
        loss = 0.0
        for g in generator.get_deterministic_group_elems():
            moved = _decode(autoencoder, _act_on_latent(g, z) + z_mean)
            g_x, g_fx = moved[:, 0], moved[:, 1]
            if numpy:
                f_g_x = torch.from_numpy(f(g_x.cpu().numpy())).float().to(generator.Li[0].device)
            else:
                f_g_x = f(g_x)
            defect = torch.mean((f_g_x - g_fx) ** 2)
            loss += defect / torch.mean((f_g_x - fx) ** 2) if relative else defect

    return loss.cpu().numpy() if numpy else loss


def _group_transform(autoencoder, g, x, normalize='global', z_mean=None, fast_ok=True):
    """x -> decode(g·(encode(x) − centre) + centre), first component (reference `model_utils.py:145-158`)."""
    z, z_mean = _centred_latent(autoencoder, torch.stack([x, x], dim=1), normalize, z_mean, fast_ok)
    return _decode(autoencoder, _act_on_latent(g, z) + z_mean, fast_ok)[:, 0]


def _group_transform_jvp(autoencoder, g, x, v, normalize, z_mean, require_grad):
    """(g(x), J_g(x)·v) for the map of `_group_transform` (`model_utils.py:145-163`). With the tensor-core MLPs the
    tangent is pushed through encoder, latent action and decoder in forward mode; otherwise the reference's double vjp."""
    fast = _fast_ae(autoencoder, x)
    if fast is None or normalize != 'global':         # 'in_batch': the batch mean couples the rows, keep autograd's graph
        # the double vjp differentiates its function twice: PyTorch modules only (the tensor-core operators are
        # first-order)
        move = partial(_group_transform, autoencoder, g, normalize=normalize, z_mean=z_mean, fast_ok=False)
        return move(x), _jvp_fn(require_grad)(move, x, v=v)[1]
    enc, dec = fast
    z, dz = enc.value_and_jvp(torch.stack([x, x], dim=1), torch.stack([v, v], dim=1))
    if z_mean is None:
        z_mean = autoencoder.encoder[-2].bias
    moved, dmoved = dec.value_and_jvp(_act_on_latent(g, z - z_mean) + z_mean, _act_on_latent(g, dz))
    return moved[:, 0], dmoved[:, 0]


def symmreg_r(x, autoencoder, generator, h, normalize='global', z_mean=None, require_grad=False, scale=0.01):
    '''Reversed symmetry loss sum_g mean((J_g(x)·h(x) − h(g(x)))²) (reference `model_utils.py:126-170`).'''
    jvp_fn = _jvp_fn(require_grad)
    autoencoder.eval()
    generator.eval()
    with torch.set_grad_enabled(require_grad):
        loss = 0.0
        for g in generator.get_deterministic_group_elems(scale=scale):
            gx, pushed = _group_transform_jvp(autoencoder, g, x, h(x), normalize, z_mean, require_grad)
            loss += torch.mean((pushed - h(gx)) ** 2)
    return loss


def symmreg_r_precomputed(x, gx_list, Jgx_list, h):
    '''symmreg_r with g(x) and J_g(x) precomputed (they do not depend on Ξ): a pure streaming loss — two library
    evaluations and one d×d mat-vec per sample and group element. When `h` is a SINDyRegression on the GPU with a fused
    kernel (sb_symreg_r) value AND dL/dΞ come from ONE launch per group element; otherwise composed from h(x), h(g(x)).'''
    loss = 0.0
    fused = (_is_regressor(h) and x.is_cuda and native.symreg_supported(h.library)
             and not (torch.is_grad_enabled() and x.requires_grad))
    if fused:
        h.Xi = h._current_Xi()
        w = h.Xi * h.mask
    for gx, Jgx in zip(gx_list, Jgx_list):
        d = x.shape[-1]
        if fused:
            loss = loss + ops.symreg_r_loss(x, gx, Jgx.reshape(-1, d, d), w, h.library)
            continue
        pushed = torch.einsum('bij,bj->bi', Jgx.reshape(-1, d, d), h(x))  # the reference's Jgx is (B, 1, d, d)
        loss = loss + torch.mean((pushed - h(gx)) ** 2)
    return loss


def group_action_and_jacobian(x, autoencoder, generator, z_mean=None, scale=0.01, normalize='global'):
    '''g(x) and the TRUE Jacobian J_g(x) (B, d, d) of every deterministic group element, as `symmreg_r` uses them
    (`model_utils.py:145-163`: `jvp(group_transform, x, v=h(x))`): column j of J_g is the JVP with the j-th unit vector.
    They do not depend on Ξ, so a fit computes them ONCE and evaluates `symmreg_r_precomputed` in every closure — the
    autoencoder leaves the closure entirely. (`precompute_symmreg_r` keeps the reference's own `vmap(jacfwd)` result,
    which stacks on the wrong axis; this is the quantity the loss `symmreg_r` actually contracts with.)'''
    autoencoder.eval()
    generator.eval()
    gx_list, Jgx_list = [], []
    d = x.shape[-1]
    with torch.no_grad():
        for g in generator.get_deterministic_group_elems(scale=scale):
            gx_list.append(_group_transform(autoencoder, g, x, normalize=normalize, z_mean=z_mean))
            cols = []
            for j in range(d):
                e = torch.zeros_like(x)
                e[:, j] = 1.0
                with torch.enable_grad():
                    cols.append(_group_transform_jvp(autoencoder, g, x, e, normalize, z_mean, False)[1].detach())
            Jgx_list.append(torch.stack(cols, dim=-1))            # [b, a, j] = d g_a / d x_j
    return gx_list, Jgx_list


def precompute_symmreg_r(x, autoencoder, generator, z_mean=None, scale=0.01):
    '''g(x) and its Jacobian J_g(x) for every deterministic group element (reference `model_utils.py:172-211`).'''
    from torch.func import jacfwd, vmap

    autoencoder.eval()
    generator.eval()
    gx_list, Jgx_list = [], []
    with torch.no_grad():
        for g in generator.get_deterministic_group_elems(scale=scale):
            move = partial(_group_transform, autoencoder, g, normalize='global', z_mean=z_mean)
            gx_list.append(move(x))
            Jgx_list.append(vmap(jacfwd(move))(x))
    return gx_list, Jgx_list


def make_symmreg(autoencoder, generator):
    return partial(symmreg_i, autoencoder=autoencoder, generator=generator)


def make_symmreg_pttrain(autoencoder, generator):
    return partial(symmreg_i, autoencoder=autoencoder, generator=generator, require_grad=True)


def make_symmreg_np(autoencoder, generator):
    return partial(symmreg_i, autoencoder=autoencoder, generator=generator, numpy=True)


def make_fsymmreg(autoencoder, generator):
    return partial(symmreg_f, autoencoder=autoencoder, generator=generator)


def make_fsymmreg_pttrain(autoencoder, generator):
    return partial(symmreg_f, autoencoder=autoencoder, generator=generator, require_grad=True)


def make_fsymmreg_np(autoencoder, generator):
    return partial(symmreg_f, autoencoder=autoencoder, generator=generator, numpy=True)


def make_rsymmreg(autoencoder, generator):
    return partial(symmreg_r, autoencoder=autoencoder, generator=generator)


def make_rsymmreg_pttrain(autoencoder, generator):
    return partial(symmreg_r, autoencoder=autoencoder, generator=generator, require_grad=True)


def _kernel_rollout_ok(f, x0):
    """The fused rollout applies when f is a SINDyRegression-like module on CUDA and nothing needs a gradient."""
    if not (hasattr(f, 'library') and hasattr(f, 'mask') and hasattr(f, '_current_Xi')):
        return False
    if not (torch.is_tensor(x0) and x0.is_cuda):
        return False
    if torch.is_grad_enabled() and (x0.requires_grad or any(p.requires_grad for p in f.parameters())):
        return False
    return True


def odeint(f, x0, t, dt, method='euler', full_traj=False):
    '''
    Integrate dx/dt = f(x) over [0, t] with fixed step dt ('euler' or 'rk4'). n_steps = int(t / dt) as the
    reference. full_traj: return the (n_steps, ...) stack of states after each step (x0 excluded), else the
    final state.
    '''
    n_steps = int(t / dt)
    if method not in ('euler', 'rk4'):
        raise ValueError('Unrecognized ODEInt method.')

    if _kernel_rollout_ok(f, x0):
        with torch.no_grad():
            w = (f._current_Xi() * f.mask).detach()
            traj, _, last = native.rollout(x0, w, f.library, dt, n_steps, stride=1, method=method,
                                           record_dx=False, want_traj=full_traj, want_last=not full_traj)
        if full_traj:
            return traj.view(n_steps, *x0.shape)
        return last.view(x0.shape)

    def step(x):
        if method == 'euler':
            return x + dt * f(x)
        k1 = f(x)
        k2 = f(x + dt / 2 * k1)
        k3 = f(x + dt / 2 * k2)
        k4 = f(x + dt * k3)
        return x + dt / 6 * (k1 + 2 * k2 + 2 * k3 + k4)

    traj = []
    for _ in range(n_steps):
        x0 = step(x0)
        if full_traj:
            traj.append(x0)
    return torch.stack(traj, dim=0) if full_traj else x0
