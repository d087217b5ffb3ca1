"""fp64 autograd reference of the fused symmetry-regulariser kernels (csrc/sb_symreg.cu) — TEST INFRASTRUCTURE ONLY.

Plain PyTorch in float64, written from the definitions and independent of the product: nothing here imports
`sindy_b200`, `ops`, `model_utils` or `sindy`. The library Θ takes its column order from `oracle.sindy_oracle`.

  * flow64: f(x) = n explicit-Euler steps q ← q + dt·Θ(q)Wᵀ (the reference's `model_utils.py:236-240`) and J_f(x)·v
    from `torch.func.jvp`;
  * symreg_r64: the reversed regulariser mean((J h(x) − h(g x))²) (the reference's `model_utils.py:126-170`).

Gradients come from `torch.autograd.grad`; the one with respect to x differentiates through the jvp, so it exercises the
second derivatives of Θ that the backward kernel carries in its Hessian-vector term. Callers hand in the fp32 tensors
the kernel sees; they are cast exactly to fp64, so a comparison measures only the kernel's own rounding. The functions
`flow64_grads` and `symreg_r64_grads` evaluate in sample chunks and add the d×K gradient sums in fp64, so memory stays
bounded at 10⁶ samples.
"""
import torch

from oracle import sindy_oracle as O

CHUNK = 250_000


def theta64(x, d, p, sine=False, exp=False):
    """Θ(x): (..., d) -> (..., K). Monomials as left-to-right products of coordinates — not `x ** E` with an exponent
    tensor, whose second derivative is NaN at x = 0 through pow's backward — then sin and exp columns."""
    assert x.shape[-1] == d
    cols = []
    for c in O.poly_tuples(d, p):
        if not c:
            cols.append(torch.ones_like(x[..., 0]))
            continue
        v = x[..., c[0]]
        for j in c[1:]:
            v = v * x[..., j]
        cols.append(v)
    if sine:
        cols += [torch.sin(x[..., j]) for j in range(d)]
    if exp:
        cols += [torch.exp(x[..., j]) for j in range(d)]
    return torch.stack(cols, dim=-1)


def euler64(x, W, lib, dt, n_steps):
    """n_steps explicit-Euler steps of h(q) = Θ(q)Wᵀ; lib = (d, p, sine, exp)."""
    q = x
    for _ in range(n_steps):
        q = q + dt * (theta64(q, *lib) @ W.T)
    return q


def flow64(x, v, W, lib, dt, n_steps):
    """(f(x), J_f(x)·v); (f(x), None) without v. At n_steps = 0 the flow is the identity: (x, v)."""
    if n_steps == 0:
        return x, v
    if v is None:
        return euler64(x, W, lib, dt, n_steps), None
    return torch.func.jvp(lambda q: euler64(q, W, lib, dt, n_steps), (x,), (v,))


def _grads(loss, inputs, retain_graph):
    if not loss.requires_grad:                           # nothing in the graph depends on an input (n_steps = 0)
        return [torch.zeros_like(t) for t in inputs]
    return torch.autograd.grad(loss, inputs, retain_graph=retain_graph, allow_unused=True, materialize_grads=True)


def flow64_grads(x, v, W, lib, dt, n_steps, cotangents, need_gx=True, chunk=CHUNK):
    """fp64 fx, jv (None without v) and, for every (g_fx, g_jv) in `cotangents` (either may be None), the gradients
    (gW, gv, gx) of Σ g_fx·fx + Σ g_jv·jv; gv is None without v, gx None unless need_gx. x, v, g_*: (n, d)."""
    n, d = x.shape
    W64 = W.detach().to(torch.float64).requires_grad_(True)
    fx = torch.empty(n, d, dtype=torch.float64, device=x.device)
    jv = torch.empty_like(fx) if v is not None else None
    out = [[torch.zeros_like(W64, requires_grad=False),
            torch.empty_like(fx) if v is not None else None,
            torch.empty_like(fx) if need_gx else None] for _ in cotangents]
    for i in range(0, n, chunk):
        j = min(n, i + chunk)
        xc = x[i:j].detach().to(torch.float64).requires_grad_(need_gx)
        vc = v[i:j].detach().to(torch.float64).requires_grad_(True) if v is not None else None
        f, t = flow64(xc, vc, W64, lib, dt, n_steps)
        fx[i:j] = f.detach()
        if v is not None:
            jv[i:j] = t.detach()
        inputs = [W64] + ([vc] if v is not None else []) + ([xc] if need_gx else [])
        for c, (g_fx, g_jv) in enumerate(cotangents):
            loss = torch.zeros((), dtype=torch.float64, device=x.device)
            if g_fx is not None:
                loss = loss + (f * g_fx[i:j].to(torch.float64)).sum()
            if g_jv is not None and v is not None:
                loss = loss + (t * g_jv[i:j].to(torch.float64)).sum()
            g = list(_grads(loss, inputs, retain_graph=c + 1 < len(cotangents)))
            out[c][0] += g.pop(0)
            if v is not None:
                out[c][1][i:j] = g.pop(0)
            if need_gx:
                out[c][2][i:j] = g.pop(0)
    return fx, jv, [tuple(o) for o in out]


def symreg_r64(x, gx, J, W, lib):
    """mean((J h(x) − h(gx))²) over all n·d entries, h(q) = Θ(q)Wᵀ; J: (n, d, d)."""
    h = theta64(x, *lib) @ W.T
    pushed = torch.einsum('bij,bj->bi', J, h)
    return torch.mean((pushed - theta64(gx, *lib) @ W.T) ** 2)


def symreg_r64_grads(x, gx, J, W, lib, chunk=CHUNK):
    """(Σ‖J h(x) − h(gx)‖², its gradient with respect to W), both fp64, summed over sample chunks."""
    n, d = x.shape
    W64 = W.detach().to(torch.float64).requires_grad_(True)
    total = torch.zeros((), dtype=torch.float64, device=x.device)
    gW = torch.zeros_like(W64, requires_grad=False)
    for i in range(0, n, chunk):
        j = min(n, i + chunk)
        s = symreg_r64(x[i:j].to(torch.float64), gx[i:j].to(torch.float64), J[i:j].to(torch.float64), W64, lib) \
            * ((j - i) * d)
        (g,) = torch.autograd.grad(s, (W64,))
        total += s.detach()
        gW += g
    return total, gW
