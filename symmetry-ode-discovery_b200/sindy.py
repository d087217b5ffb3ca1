"""Drop-in replacement for the reference's `sindy.py` (SINDyRegression, solve_SINDy*, WSINDyWrapper).

Put this directory in front of the reference on PYTHONPATH: `from sindy import *` then resolves here and
the reference's `train.py` / `main.py` / `run_configs/*.cfg` work unchanged on a CUDA device. The public
surface (constructor kwargs, attributes, method names, return values, printed equation format, RNG draw
order) follows the reference; the tensor arithmetic runs in libsindy_b200.so:

  * Θ(x), h(x)=Θ(x)(Ξ⊙mask)ᵀ and all derivatives autograd asks for -> sindy_b200.ops (reference `sindy.py:79-82,201-203`)
  * STLSQ (`sindy.py:250-324`): one fused Gram pass (ΘᵀΘ, ΘᵀẊ in fp64) + K×K normal-equation solves instead of
    a QR of the (N+K)·d × d·K block-diagonal matrix
  * WSINDy (`sindy.py:332-395`): weak-form integrals VΘ(x), V'x generated on the fly + n_test×K normal equations
  * the equivariance constraint basis Q (`sindy.py:85-144`) is host-side setup; the symbolic map M is built
    from exponent arithmetic instead of SymPy.

There is no CPU fallback: calling the model on CPU tensors raises.
"""
from __future__ import annotations

import itertools
import math
import os

import numpy as np
import torch
import torch.nn as nn

from sindy_b200 import native, ops
from sindy_b200.native import Library

__all__ = ["SINDyRegression", "solve_SINDy_one_step", "solve_SINDy", "WSINDyWrapper", "stlsq_statistics",
           "allreduce_statistics", "stlsq_path", "score_path", "refine_path", "information_criteria", "apply_candidate", "SINDyConst", "SINDyPoly1", "SINDyPoly2", "SINDyPoly3", "SINDySine", "SINDyExp"]


# ---- the reference's per-block library functions (`sindy.py:7-30`) --------------------------------------------------
# In the reference Θ is the concatenation of these six callables' outputs; here the columns are produced inside the
# kernels and nothing in this package calls them. They exist for `from sindy import *` users: each evaluates Θ of the
# smallest library containing its block with `sb_theta` and returns that block — the same column order and the same
# left-to-right products (monomials bit-exact, sin / exp within 2 ulp of torch's). Values only: a tensor that carries a
# gradient is refused instead of silently losing it (differentiate through `SINDyRegression.forward`). CUDA tensors
# only, like everything else here.
def _library_block(x, poly_order, sine, exp, lo, hi):
    if not torch.is_tensor(x) or x.dim() < 1:
        raise TypeError("expected a tensor (..., d)")
    if torch.is_grad_enabled() and x.requires_grad:
        raise NotImplementedError("the per-block library functions return values only; differentiate through "
                                  "SINDyRegression.forward / ops.sindy_forward")
    d = int(x.shape[-1])
    theta = native.theta(x, Library(d, poly_order, sine, exp))
    lo, hi = lo(d), hi(d)
    return theta[..., lo:hi].contiguous()


def _n_upto(d, n):
    """Number of monomials of degree <= n in d variables (the polynomial block ends there)."""
    return math.comb(d + n, n)


def SINDyConst(x):
    return _library_block(x, 1, False, False, lambda d: 0, lambda d: 1)


def SINDyPoly1(x):
    return _library_block(x, 1, False, False, lambda d: 1, lambda d: _n_upto(d, 1))


def SINDyPoly2(x):
    return _library_block(x, 2, False, False, lambda d: _n_upto(d, 1), lambda d: _n_upto(d, 2))


def SINDyPoly3(x):
    return _library_block(x, 3, False, False, lambda d: _n_upto(d, 2), lambda d: _n_upto(d, 3))


def SINDySine(x):
    return _library_block(x, 1, True, False, lambda d: _n_upto(d, 1), lambda d: _n_upto(d, 1) + d)


def SINDyExp(x):
    return _library_block(x, 1, False, True, lambda d: _n_upto(d, 1), lambda d: _n_upto(d, 1) + d)


def _poly_index_tuples(dim: int, order: int):
    """Index tuples of the polynomial columns: () ; (i) ; (i<=j) ; ... in the reference's column order."""
    cols = [()]
    for n in range(1, order + 1):
        cols.extend(itertools.combinations_with_replacement(range(dim), n))
    return cols


def _lie_derivative_matrix(dim: int, order: int, L: torch.Tensor) -> torch.Tensor:
    """M with J_Θ(z)·L·z = M·Θ(z) for the polynomial library (reference `sindy.py:123-144`, there via SymPy).

    d/dz_j z^a = a_j z^(a-e_j) and (Lz)_j = sum_l L[j,l] z_l, so row a gets a_j·L[j,l] at column a-e_j+e_l.
    """
    cols = _poly_index_tuples(dim, order)
    where = {c: k for k, c in enumerate(cols)}
    Lm = np.asarray(L, dtype=np.float64)
    M = np.zeros((len(cols), len(cols)))
    for k, c in enumerate(cols):
        for pos, j in enumerate(c):  # one factor z_j of the monomial at a time (multiplicity = a_j)
            rest = c[:pos] + c[pos + 1:]
            for l in range(dim):
                if Lm[j, l] != 0.0:
                    M[k, where[tuple(sorted(rest + (l,)))]] += Lm[j, l]
    return torch.tensor(M, dtype=torch.float32)


class SINDyRegression(nn.Module):
    """Sparse regression dz/dt = Θ(z)·(Ξ⊙mask)ᵀ, optionally with Ξ constrained to be equivariant.

    Arguments (as the reference): latent_dim, poly_order (reference: ≤3; here up to 5), include_sine,
    include_exp, L_list (Lie algebra generators; non-empty => equivariance-constrained Ξ = reshape(Q·β)),
    kwargs["threshold"], kwargs["device"], kwargs["constrain_constant"].

    Initial parameters are drawn with `torch.randn(..., device=device)` exactly like the reference (`sindy.py:57-64`), so
    a run on a CUDA device consumes the CUDA generator and starts where the reference ON THE SAME DEVICE starts. To
    reproduce a run of the reference on the CPU seed for seed (the goldens of tests/golden/configs.npz), pass
    `init_rng='cpu'` or set SINDY_B200_INIT_RNG=cpu: the same shapes are then drawn from the CPU generator and moved.
    """

    def __init__(self, latent_dim, poly_order, include_sine, include_exp, L_list=[], **kwargs):
        super().__init__()
        device = kwargs["device"]
        self.latent_dim = latent_dim
        self.poly_order = poly_order
        self.L_list = L_list
        self.constraint = len(L_list) != 0
        # trigonometric / exponential columns are dropped under the constraint (reference `sindy.py:47-48`)
        self.include_sine = bool(include_sine) and not self.constraint
        self.include_exp = bool(include_exp) and not self.constraint
        self.threshold = kwargs["threshold"]
        self.library = Library(int(latent_dim), int(poly_order), self.include_sine, self.include_exp)
        init_rng = kwargs.get('init_rng') or os.environ.get('SINDY_B200_INIT_RNG', 'device')
        if init_rng not in ('device', 'cpu'):
            raise ValueError(f"init_rng must be 'device' or 'cpu', got {init_rng!r}")

        def randn(*shape):
            return torch.randn(*shape, device=device) if init_rng == 'device' else torch.randn(*shape).to(device)

        if self.constraint:
            print('Computing equivariance constraint...')
            self.Q = self.get_Q().to(device)
            self.beta = nn.Parameter(randn(self.Q.shape[1]))
            self.const = nn.Parameter(randn(latent_dim, 1))
            self.allow_constant = not kwargs['constrain_constant']
            self.Xi = self.get_Xi()
        else:
            self.Xi = nn.Parameter(randn(latent_dim, self.get_term_num()))
        self.mask = torch.ones_like(self.Xi, device=device)
        # kept for API compatibility: names of the column groups
        self.terms = ['const', 'poly1'] + [f'poly{n}' for n in range(2, poly_order + 1)]
        if self.include_sine:
            self.terms.append('sine')
        if self.include_exp:
            self.terms.append('exp')

    # ---- library / model -------------------------------------------------------------------------
    def get_term_num(self):
        return sum(math.comb(self.latent_dim + n - 1, n) for n in range(self.poly_order + 1)) \
            + self.latent_dim * (int(self.include_sine) + int(self.include_exp))

    def _current_Xi(self):
        return self.get_Xi() if self.constraint else self.Xi

    def forward(self, x):
        self.Xi = self._current_Xi()
        return ops.sindy_forward(x, self.Xi * self.mask, self.library)

    def eval_Theta_at(self, x):
        return native.theta(x, self.library)

    def mse_loss(self, x, dx):
        """mean((forward(x) − dx)²) and its gradient w.r.t. the parameters from ONE pass over the data
        (the fused train step; same value as `MSELoss()(self(x), dx)`, `train.py:663-664`)."""
        self.Xi = self._current_Xi()
        return ops.fused_mse(x, dx, self.Xi * self.mask, self.library)

    def sufficient_statistics(self, x, dx):
        """One pass over (x, dx): everything the MSE objective needs, as fp64 tensors (G = ΘᵀΘ, b = ΘᵀẊ, Σẋ², n).
        The MSE (and the linear Lie-derivative regulariser) are exact quadratics in Ξ given these (SURVEY §8f-1)."""
        lib = self.library
        flags = native.SB_STEP_GRAM | native.SB_STEP_B
        with torch.no_grad():
            parts = native.unpack_step(native.train_step(x, dx, None, lib, flags), lib, flags)
            yy = _column_sums_of_squares(dx, lib.dim).sum()
        return {"G": parts["gram"], "b": parts["b"], "yy": yy, "n": float(parts["n"])}

    def mse_loss_from_statistics(self, stats):
        """mean((Θ(x)(Ξ⊙mask)ᵀ − dx)²) = (tr(W G Wᵀ) − 2 tr(W b) + Σẋ²)/(n·d) with NO pass over the data; differentiable
        w.r.t. the parameters (fp64 algebra on K×K, result cast to the parameter dtype). One data pass per FIT instead
        of one per closure evaluation (`train.py:693-695` makes up to 20 per epoch)."""
        self.Xi = self._current_Xi()
        W = (self.Xi * self.mask).double()
        quad = ((W @ stats["G"]) * W).sum() - 2.0 * (W * stats["b"].T).sum() + stats["yy"]
        return (quad / (stats["n"] * self.latent_dim)).to(self.Xi.dtype)

    def lie_reg_loss(self, z, generators, method='auto'):
        """Linear Lie-derivative regulariser Σ_v Σ_n ‖J_h(z_n)(v z_n) − v h(z_n)‖² (the intended formula of the
        reference's `train.py:503-507`), differentiable w.r.t. the parameters. 'gram': one moment pass + K×K
        algebra (polynomial libraries); 'jvp': per-sample CUDA JVPs (any library); 'auto' picks."""
        from sindy_b200 import symreg
        self.Xi = self._current_Xi()
        W = self.Xi * self.mask
        poly = not (self.include_sine or self.include_exp)
        needs_z_grad = torch.is_grad_enabled() and torch.is_tensor(z) and z.requires_grad
        if method == 'auto':
            method = 'gram' if (poly and not needs_z_grad) else 'jvp'
        if method == 'gram' and needs_z_grad:
            raise ValueError("lie_reg_loss(method='gram') differentiates with respect to the parameters only (the Gram "
                             "matrix of z is formed without a graph); use method='jvp' when z carries a gradient")
        if method == 'gram':
            key = tuple(float(q) for v in generators for q in torch.as_tensor(v).flatten().tolist())
            if getattr(self, '_lie_key', None) != key:
                self._lie_Ms = [symreg.lie_matrix(self.library, v) for v in generators]
                self._lie_key = key
            with torch.no_grad():
                G = symreg.gram(z.reshape(-1, self.latent_dim), self.library)
            return symreg.lie_loss_from_gram(G, W, generators, self._lie_Ms).to(W.dtype)
        return symreg.lie_loss_per_sample(z.reshape(-1, self.latent_dim), W, generators, self.library)

    # ---- equivariance constraint (host-side setup) -------------------------------------------------
    def get_M_list(self):
        return [_lie_derivative_matrix(self.latent_dim, self.poly_order, Li) for Li in self.L_list]

    def get_Theta(self):
        """The polynomial library as a SymPy column matrix in the symbols z0..z{d-1} (reference `sindy.py:147-166`, where
        it feeds `get_M_list`; here M comes from exponent arithmetic and this method only serves callers that want the
        symbolic library — any poly_order, same column order as the kernels)."""
        import sympy as sp
        z = [sp.Symbol(f"z{i}") for i in range(self.latent_dim)]
        return sp.Matrix([sp.Mul(*[z[i] for i in idx]) if idx else sp.Integer(1)
                          for idx in _poly_index_tuples(self.latent_dim, self.poly_order)])

    def get_Q(self):
        """Null-space basis of the stacked constraint matrices (reference `sindy.py:85-115`)."""
        blocks = []
        for M, L in zip(self.get_M_list(), self.L_list):
            L = torch.as_tensor(L, dtype=torch.float32)
            if torch.det(L) < 1e-5:  # singular generator: Sylvester form, Ξ stored term-major
                self.use_kron_product = False
                Mt = M.transpose(0, 1).contiguous()
                C = torch.kron(-Mt, torch.eye(L.shape[0])) + torch.kron(torch.eye(Mt.shape[0]), L)
            else:  # invertible generator: Ξ stored equation-major
                self.use_kron_product = True
                C = torch.kron(L.inverse(), M.T)
                C = C - torch.eye(C.shape[0])
            blocks.append(C)
        _, sigma, V = torch.svd(torch.cat(blocks, dim=0))
        # count trailing singular values below 5e-3; r == 0 keeps the reference's `V[:, -0:]` (= all of V)
        r = 0
        for r in range(len(sigma)):
            if abs(sigma[-1 - r]) > 5e-3:
                break
        return V[:, -r:]

    def update_Q(self, new_Li):
        self.L_list = new_Li
        self.Q = self.get_Q().to(self.Xi.device)
        self.beta = nn.Parameter(torch.randn(self.Q.shape[1], device=self.Xi.device))

    def get_Xi(self):
        flat = self.Q @ self.beta
        if self.use_kron_product:
            Xi = flat.view(self.latent_dim, -1)
        else:
            Xi = flat.view(-1, self.latent_dim).transpose(0, 1)
        if self.allow_constant:
            pad = torch.zeros((Xi.shape[0], Xi.shape[1] - 1), device=Xi.device)
            Xi += torch.cat([self.const, pad], dim=1)
        return Xi

    # ---- sparsity mask -----------------------------------------------------------------------------
    def set_threshold(self, threshold):
        self.Xi = self._current_Xi()
        keep = torch.logical_and(torch.abs(self.Xi) > threshold, self.mask)
        self.mask.data = keep.float()

    def reset_mask(self):
        self.mask.data = torch.ones_like(self.Xi, device=self.Xi.device)

    # ---- pretty printer ----------------------------------------------------------------------------
    def term_names(self):
        names = ['']
        for c in _poly_index_tuples(self.latent_dim, self.poly_order)[1:]:
            names.append('*' + '*'.join(f'z{j}' for j in c))
        if self.include_sine:
            names += [f'*sin(z{j})' for j in range(self.latent_dim)]
        if self.include_exp:
            names += [f'*exp(z{j})' for j in range(self.latent_dim)]
        return names

    def print(self):
        Xi = self._current_Xi()
        names = self.term_names()
        for i in range(self.latent_dim):
            line = f'dz{i} ='
            for k, suffix in enumerate(names):
                if self.mask[i, k]:
                    line += f' {Xi[i, k]:.3f}{suffix} +'
            print(line)


# --------------------------------------------------------------------------------------------------------
# sequentially thresholded least squares on the Gram matrix
# --------------------------------------------------------------------------------------------------------
def _lstsq_driver(kwargs=None):
    """Which LAPACK driver of the reference's `torch.linalg.lstsq` (`sindy.py:288,386`) the normal-equation solves
    follow. 'gels' (default) is what the reference gets ON A CUDA DEVICE — the only device this package runs on: plain
    QR, no rank decision. 'gelsy' is what it gets on the CPU: rank-revealing, directions under rcond = eps32·max(M, N)
    dropped, minimum-norm solution — needed to reproduce CPU runs of rank-deficient fits (WSINDy on Sel'kov with w = 0),
    and wrong for large or badly scaled problems: at 2·10^4 rows the cut is 2.4e-3 in relative singular value, so a
    library with cond(Θ) > 400 (raw-unit Lorenz data, cubic library) silently loses its small directions.
    Selected by the keyword `lstsq_driver` of solve_SINDy* / WSINDyWrapper, else $SINDY_B200_LSTSQ."""
    driver = (kwargs or {}).get('lstsq_driver') or os.environ.get('SINDY_B200_LSTSQ', 'gels')
    if driver not in ('gels', 'gelsy'):
        raise ValueError(f"lstsq driver must be 'gels' or 'gelsy', got {driver!r}")
    return driver


def _min_norm_solve(H: torch.Tensor, rhs: torch.Tensor, rcond: float) -> torch.Tensor:
    """Solution of the symmetric PSD system H·s = rhs (fp64).

    rcond > 0 ('gelsy'): minimum-norm solution, dropping directions whose singular value in the original least-squares
    matrix would fall under rcond·σ_max (eigenvalue of H < rcond²·λ_max) — LAPACK gelsy's rank rule.
    rcond == 0 ('gels'): full-rank solve. H is equilibrated first (D^-1/2 H D^-1/2 with D = diag H, i.e. the columns
    of the least-squares matrix scaled to unit length — removes the spread between x and x^5 or between raw-unit
    coordinates), decomposed by eigh, and only directions at the fp64 round-off level (λ < K·eps64·λ_max) are left out,
    so an exactly singular system still returns its minimum-norm solution instead of Inf."""
    if H.numel() == 0:
        return rhs.new_zeros(rhs.shape)
    if rcond > 0.0:
        lam, U = torch.linalg.eigh(H)
        keep = lam > (rcond * rcond) * lam.max().clamp_min(0)
        inv = torch.where(keep, 1.0 / lam.clamp_min(torch.finfo(lam.dtype).tiny), torch.zeros_like(lam))
        return U @ (inv.unsqueeze(-1) * (U.T @ rhs)) if rhs.dim() == 2 else U @ (inv * (U.T @ rhs))
    diag = torch.diagonal(H)
    scale = torch.where(diag > 0, diag.clamp_min(torch.finfo(H.dtype).tiny).rsqrt(), torch.zeros_like(diag))
    Hs = H * scale.unsqueeze(0) * scale.unsqueeze(1)
    lam, U = torch.linalg.eigh(Hs)
    keep = lam > H.shape[0] * torch.finfo(H.dtype).eps * lam.max().clamp_min(0)
    inv = torch.where(keep, 1.0 / lam.clamp_min(torch.finfo(lam.dtype).tiny), torch.zeros_like(lam))
    if rhs.dim() == 2:
        return scale.unsqueeze(-1) * (U @ (inv.unsqueeze(-1) * (U.T @ (scale.unsqueeze(-1) * rhs))))
    return scale * (U @ (inv * (U.T @ (scale * rhs))))


def _masked_solve_batched(H, b, mask, rcond):
    """The solves of `_min_norm_solve` for the d equations at once: equation i solves H[m_i, m_i]·ξ = b[m_i, i] on its
    support m_i = mask[i]. Same equilibration, same rank rule (threshold relative to the largest eigenvalue over ALL
    equations, dimension = number of live coefficients — K when every coefficient is live, as the reference then solves
    one K×K system with d right-hand sides). Returns Ξ (d × K, fp64), zero off the support."""
    return _masked_solve_path(H, b, mask.unsqueeze(0), rcond)[0]


def _masked_solve_path(H, b, masks, rcond):
    """`_masked_solve_batched` for P supports at once (masks P × d × K -> Ξ P × d × K, fp64). Every decision that
    function takes over its d equations — the Cholesky fast path, the rank threshold and the largest eigenvalue it is
    relative to — is taken here per candidate p, so a rank-deficient candidate leaves the others' numerics alone."""
    P, d, K = masks.shape
    M = masks.to(H.dtype)
    if rcond > 0.0:
        scale = torch.ones(K, dtype=H.dtype, device=H.device)
    else:
        diag = torch.diagonal(H)
        scale = torch.where(diag > 0, diag.clamp_min(torch.finfo(H.dtype).tiny).rsqrt(), torch.zeros_like(diag))
    Hs = H * scale.unsqueeze(0) * scale.unsqueeze(1)
    Hb = M.unsqueeze(-1) * Hs * M.unsqueeze(-2)                           # P × d × K × K
    rhs = (scale.unsqueeze(1) * b).T * M                                   # P × d × K
    sol = None
    if rcond > 0.0:
        cut = torch.full((P,), rcond * rcond, dtype=H.dtype, device=H.device)
    else:
        n_live = M.sum(dim=(1, 2))
        cut = torch.where(n_live == d * K, torch.full_like(n_live, float(K)), n_live) * torch.finfo(H.dtype).eps
        # Fast path for the full-rank case, which is every well-posed fit: Cholesky of the equilibrated blocks (dead
        # coordinates padded with ones). λ_min ≥ 1/‖L⁻¹‖_F² and λ_max ≤ K (unit diagonal), so when the bound clears the
        # rank rule's threshold no direction would have been dropped and the Cholesky solution IS the min-norm solution;
        # a 56 × 56 fp64 syevd costs ~0.6 ms on the device, nine of them per `solve_SINDy`, the batched Cholesky ~0.1.
        L, info = torch.linalg.cholesky_ex(Hb + torch.diag_embed(1.0 - M))
        Linv = torch.linalg.solve_triangular(L, torch.eye(K, dtype=H.dtype, device=H.device).expand(P, d, K, K),
                                             upper=False)
        lam_min_bound = 1.0 / (Linv * Linv).sum(dim=(-1, -2)).clamp_min(torch.finfo(H.dtype).tiny)
        full_rank = ((info == 0).all(1) & (lam_min_bound.amin(1) > cut * K)
                     & torch.isfinite(Linv).flatten(1).all(1))
        n_full = int(full_rank.sum())                                      # one host sync (the loop has one per step anyway)
        if n_full:
            # two triangular solves (cuBLAS trsm); `torch.cholesky_solve` costs ~1 s of solver-library start-up on its
            # first call, a third of a whole `main_wsindy.py` run on the test fixture
            y = torch.linalg.solve_triangular(L, rhs.unsqueeze(-1), upper=False)
            sol = torch.linalg.solve_triangular(L.transpose(-1, -2), y, upper=True).squeeze(-1)
            if n_full == P:
                return sol * scale * M
    lam, U = torch.linalg.eigh(Hb)
    keep = lam > cut.view(P, 1, 1) * lam.amax(dim=(1, 2), keepdim=True).clamp_min(0)
    inv = torch.where(keep, 1.0 / lam.clamp_min(torch.finfo(lam.dtype).tiny), torch.zeros_like(lam))
    proj = torch.matmul(U.transpose(-1, -2), rhs.unsqueeze(-1)).squeeze(-1)
    eig = torch.matmul(U, (inv * proj).unsqueeze(-1)).squeeze(-1)
    if sol is not None:
        eig = torch.where(full_rank.view(P, 1, 1), sol, eig)
    return eig * scale * M


def _stlsq_update(regressor, G, b, ridge, n_rows, st_threshold, driver='gels'):
    """Shared tail of solve_SINDy_one_step / WSINDyWrapper.solve: solve on the current support, write the
    parameters back, threshold, report convergence. G (K×K) and b (K×d) are fp64 normal-equation blocks;
    `ridge` is what is added to G's diagonal; n_rows is the row count of the reference's least-squares matrix
    (only used for gelsy's rank tolerance); `driver`: see _lstsq_driver."""
    d, K = regressor.latent_dim, G.shape[0]
    dev = G.device
    H = G + ridge * torch.eye(K, dtype=G.dtype, device=dev)
    mask = regressor.mask > 0.0
    # 'gelsy': LAPACK's default rank tolerance eps·max(rows, cols) in the reference's fp32. It stops being a rank test
    # when the row count grows (0.48 at 4e6 rows, 11.9 at 1e8: every direction would be dropped), so it is held at its
    # value for 2^14 rows (2e-3) beyond that. 'gels': no rank decision (0).
    rcond = float(torch.finfo(torch.float32).eps) * min(max(n_rows, K), 1 << 14) if driver == 'gelsy' else 0.0
    prev_mask = regressor.mask.clone()

    if not regressor.constraint:
        # d independent systems on the supports of the d equations, solved as ONE batch of K×K problems with the
        # masked-out rows and columns zeroed (their eigenvalues are zero and are dropped by the rank rule): no index
        # lists, no host synchronisation, and 3 eigenproblems of size K instead of one of size d·K
        regressor.Xi.data = _masked_solve_batched(H, b, mask, rcond).to(torch.float32).contiguous()
    else:
        flat_mask = mask.flatten()                               # equation-major: i*K + k
        idx = torch.nonzero(flat_mask, as_tuple=False).flatten()
        eq, col = idx // K, idx % K
        # (I_d ⊗ H)[m, m]: zero between different equations
        Hm = H[col][:, col] * (eq.unsqueeze(1) == eq.unsqueeze(0)).to(H.dtype)
        rhs = b.T.reshape(-1)[idx]
        Q = regressor.Q.to(torch.float64)
        if regressor.allow_constant:
            extra = torch.zeros((Q.shape[0], d), dtype=Q.dtype, device=dev)
            for i in range(d):
                extra[i * Q.shape[0] // d, i] = 1.0
            Q = torch.cat([Q, extra], dim=1)
        Qm = Q[idx]
        effective = torch.any(Qm != 0.0, dim=0)              # drop parameters that touch no live column
        Qe = Qm[:, effective]
        sol = _min_norm_solve(Qe.T @ Hm @ Qe, Qe.T @ rhs, rcond)
        full = torch.zeros(Q.shape[1], dtype=torch.float64, device=dev)
        full[effective] = sol
        full = full.to(torch.float32)
        if regressor.allow_constant:
            regressor.beta.data = full[:-d].contiguous()
            regressor.const.data = full[-d:].view(-1, 1).contiguous()
        else:
            regressor.beta.data = full
    regressor.set_threshold(st_threshold)
    return torch.allclose(prev_mask, regressor.mask)


def _column_sums_of_squares(y, d):
    """Σ_n y[n,i]² per equation as fp64 (d,), in ONE pass without an fp64 copy of y (2.4 GB at N = 1e8)."""
    return torch.linalg.vector_norm(y.reshape(-1, d), dim=0, dtype=torch.float64) ** 2


def allreduce_statistics(stats, group=None):
    """Sum the sufficient statistics of sample shards over the ranks of `group` (one all-reduce of K² + K·d + d + 1
    doubles): afterwards every rank holds the statistics of the WHOLE data set and solves the identical K×K systems,
    so masks and coefficients stay replicated without further communication (SURVEY §8e). No-op without
    torch.distributed."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return stats
    G, b, yy = stats["G"], stats["b"], stats["yy"]
    flat = torch.cat([G.reshape(-1), b.reshape(-1), yy.reshape(-1),
                      torch.tensor([float(stats["n"])], dtype=G.dtype, device=G.device)])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    k2, kd = G.numel(), b.numel()
    return {"G": flat[:k2].view_as(G), "b": flat[k2:k2 + kd].view_as(b), "yy": flat[k2 + kd:k2 + kd + yy.numel()].view_as(yy),
            "n": int(round(float(flat[-1])))}


def stlsq_statistics(regressor, x, y, group=None):
    """The data-dependent part of an STLSQ solve — G = ΘᵀΘ, b = ΘᵀY, Σy² per equation, n — from one pass over (x, y).
    They do not depend on the mask: `solve_SINDy` forms them once for all its thresholding iterations (the reference
    rebuilds Θ and re-runs LAPACK on the N-row matrix every iteration, `sindy.py:260-288,319-323`). With
    torch.distributed initialised and samples sharded over the ranks, pass `group` (or rely on the default group via
    `solve_SINDy(..., sharded=True)`) to all-reduce them."""
    lib = regressor.library
    flags = native.SB_STEP_GRAM | native.SB_STEP_B
    with torch.no_grad():
        parts = native.unpack_step(native.train_step(x, y, None, lib, flags), lib, flags)
        stats = {"G": parts["gram"], "b": parts["b"], "yy": _column_sums_of_squares(y, lib.dim),
                 "n": x.reshape(-1, lib.dim).shape[0]}
    return stats


def solve_SINDy_one_step(regressor, x, y, w_sindy_reg, st_threshold, **kwargs):
    '''
    One STLSQ step: argmin_w ||y - Θ(x) w||² + w_sindy_reg²·||w||² on the current support (the reference stacks
    w_sindy_reg·I under Θ, `sindy.py:262`, hence the square), then threshold.

    x & y: (n_samples, dim). Returns (mean squared residual / n_samples, converged) like the reference's
    `residuals.mean() / x.shape[0]`; the residual is computed from the normal equations (the reference's LAPACK
    driver returns an empty `residuals`, i.e. NaN, for this shape).
    '''
    lib = regressor.library
    stats = kwargs.get('stats')
    if stats is None:
        stats = stlsq_statistics(regressor, x, y)
        if kwargs.get('sharded'):
            stats = allreduce_statistics(stats, kwargs.get('group'))
    with torch.no_grad():
        G, b, yy, n = stats["G"], stats["b"], stats["yy"], stats["n"]
        converged = _stlsq_update(regressor, G, b, float(w_sindy_reg) ** 2, n + lib.K, st_threshold,
                                  _lstsq_driver(kwargs))
        # residual of the augmented system with the parameters just written (before masking by the new mask)
        Xi = regressor._current_Xi().to(torch.float64)
        quad = torch.einsum('ik,kl,il->i', Xi, G, Xi) - 2.0 * torch.einsum('ik,ki->i', Xi, b) + yy
        quad = quad + float(w_sindy_reg) ** 2 * (Xi ** 2).sum(1)
        residual = (quad.mean() / n).to(torch.float32)
    return residual, converged


def solve_SINDy(regressor, x, y, w_sindy_reg, st_threshold, max_iter=5, **kwargs):
    regressor.reset_mask()
    residual = None
    stats = stlsq_statistics(regressor, x, y)   # one data pass for all thresholding iterations
    if kwargs.get('sharded'):                   # x, y are this rank's shard: one all-reduce, identical solves everywhere
        stats = allreduce_statistics(stats, kwargs.get('group'))
    for _ in range(max_iter):
        residual, converged = solve_SINDy_one_step(regressor, x, y, w_sindy_reg, st_threshold, stats=stats,
                                                   lstsq_driver=kwargs.get('lstsq_driver'))
        if converged:
            break
    return residual


# --------------------------------------------------------------------------------------------------------
# model selection along the threshold path (Mangan et al., Model selection for dynamical systems via sparse regression
# and information criteria, Proc. R. Soc. A 2017): sweep the threshold, keep each candidate model, simulate every
# candidate on held-out trajectories and rank them by an information criterion of the simulation error
# --------------------------------------------------------------------------------------------------------
def _path_thresholds(thresholds):
    thr = np.asarray(thresholds, dtype=np.float64)
    if thr.ndim != 1 or thr.size == 0:
        raise ValueError(f"thresholds must be a non-empty 1-D sequence, got shape {thr.shape}")
    if not np.all(np.isfinite(thr)) or np.any(thr < 0):
        raise ValueError("thresholds must be finite and non-negative")
    return thr


def _path_max_iter(max_iter):
    if isinstance(max_iter, bool) or not isinstance(max_iter, (int, np.integer)) or max_iter < 1:
        raise ValueError(f"max_iter must be a positive integer, got {max_iter!r}")
    return int(max_iter)


def _stlsq_path_solve(regressor, A, rhs, bb, ridge, n_rows, thr, max_iter, driver, step):
    """Candidate p = what `reset_mask()` and up to max_iter STLSQ updates with threshold thr[p] on the normal equations
    (A + ridge·I) ξ = rhs leave, stopping at the first converged update. Returns the path dict with Ξ (fp32, masked),
    the masks, convergence flags and the quadratic residual Σ-per-equation q_i = ξᵢᵀAξᵢ − 2ξᵢᵀrhsᵢ + bbᵢ + ridge·‖ξᵢ‖²
    of each candidate's last solve (fp64, P × d). Unconstrained: the P·d masked solves of each iteration are one batch
    (`_masked_solve_path`). Constrained: `step()` (one update of the regressor itself) in a loop; the regressor's
    parameters and mask are restored afterwards."""
    d, K = regressor.latent_dim, A.shape[0]
    dev = A.device
    P = thr.shape[0]
    out = {"thresholds": torch.from_numpy(thr.copy())}
    if not regressor.constraint:
        H = A + ridge * torch.eye(K, dtype=A.dtype, device=dev)
        rcond = float(torch.finfo(torch.float32).eps) * min(max(n_rows, K), 1 << 14) if driver == 'gelsy' else 0.0
        thr32 = torch.as_tensor(thr, dtype=torch.float64, device=dev).to(torch.float32).view(P, 1, 1)
        masks = torch.ones(P, d, K, dtype=torch.bool, device=dev)
        xi = torch.zeros(P, d, K, dtype=torch.float32, device=dev)
        converged = torch.zeros(P, dtype=torch.bool, device=dev)
        active = torch.arange(P, device=dev)
        for _ in range(max_iter):
            sol = _masked_solve_path(H, rhs, masks[active], rcond).to(torch.float32)
            keep = (sol.abs() > thr32[active]) & masks[active]     # set_threshold: |Ξ| > threshold in fp32
            conv = (keep == masks[active]).flatten(1).all(1)
            xi[active], masks[active], converged[active] = sol, keep, conv
            active = active[~conv]
            if active.numel() == 0:
                break
        out.update(xi=xi * masks, mask=masks, converged=converged)
    else:
        saved = ({n: p.data for n, p in regressor.named_parameters()}, regressor.mask.data, regressor.Xi)
        xis, betas, consts, masks, converged = [], [], [], [], []
        try:
            for t in thr.tolist():
                regressor.reset_mask()
                for _ in range(max_iter):
                    conv = step(float(t))
                    if conv:
                        break
                xi = regressor._current_Xi().detach()
                xis.append(xi.to(torch.float32))
                betas.append(regressor.beta.data.clone())
                consts.append(regressor.const.data.clone())
                masks.append(regressor.mask > 0)
                converged.append(bool(conv))
        finally:
            params, regressor.mask.data, regressor.Xi = saved
            for n, p in regressor.named_parameters():
                p.data = params[n]
        xi, masks = torch.stack(xis), torch.stack(masks)
        out.update(xi=xi, beta=torch.stack(betas), const=torch.stack(consts), mask=masks,
                   converged=torch.tensor(converged, device=dev))
        out["xi"] = xi * masks
    # residual from the last solve's parameters (zero off the previous support, not yet masked by the new one) — for
    # live coefficients equal to out["xi"], for thresholded ones the values just cut
    raw = xi.to(torch.float64)
    quad = torch.einsum('pik,kl,pil->pi', raw, A, raw) - 2.0 * torch.einsum('pik,ki->pi', raw, rhs) + bb
    out["quad"] = quad + ridge * (raw ** 2).sum(-1)
    out["n_terms"] = out["mask"].flatten(1).sum(1)
    return out


def stlsq_path(regressor, x, y, thresholds, w_sindy_reg=0.0, max_iter=5, **kwargs):
    """The STLSQ threshold path from ONE statistics pass: candidate p is what
    `solve_SINDy(regressor, x, y, w_sindy_reg, thresholds[p], max_iter)` leaves in the regressor. Takes `sharded` /
    `group` / `lstsq_driver` as solve_SINDy does. Returns a dict of
      thresholds (P,) fp64 (host), xi (P, d, K) fp32 = Ξ⊙mask, mask (P, d, K) bool, residual (P,) fp32 (solve_SINDy's
      return value), n_terms (P,), converged (P,) bool,
    and, for an equivariance-constrained regressor, the raw beta (P, ·) / const (P, d, 1). The regressor's parameters
    and mask are left as they were; `apply_candidate` writes one candidate into it."""
    thr = _path_thresholds(thresholds)
    max_iter = _path_max_iter(max_iter)
    lib = regressor.library
    stats = stlsq_statistics(regressor, x, y)
    if kwargs.get('sharded'):
        stats = allreduce_statistics(stats, kwargs.get('group'))
    driver = _lstsq_driver(kwargs)
    G, b, yy, n = stats["G"], stats["b"], stats["yy"], stats["n"]
    ridge = float(w_sindy_reg) ** 2

    def step(t):
        return _stlsq_update(regressor, G, b, ridge, n + lib.K, t, driver)

    with torch.no_grad():
        out = _stlsq_path_solve(regressor, G, b, yy, ridge, n + lib.K, thr, max_iter, driver, step)
        out["residual"] = (out.pop("quad").mean(-1) / n).to(torch.float32)
    return out


def score_path(library, path, x_val, dt, steps_per_row=1, method='rk4', blowup=None, criterion='aicc', fit_ic=False,
               window=None, ic_iter=20):
    """Scores the candidates of `stlsq_path` / `WSINDyWrapper.solve_path` by simulation on held-out trajectories.

    x_val (n_traj, T, d): trajectories with rows dt·steps_per_row apart. Every distinct candidate model is integrated
    once (`native.rollout_score`, one launch for all of them) from x_val[:, 0] with step dt and compared with rows
    1..T−1. Per candidate: sse (fp64), diverged (some IC hit a non-finite state or |x| > blowup), k = live
    coefficients, and, with n = n_obs = n_traj·(T−1)·d,
      AIC = n·ln(SSE/n) + 2k,  AICc = AIC + 2k(k+1)/(n−k−1),  BIC = n·ln(SSE/n) + k·ln n
    (+inf for a diverged candidate; AICc also when n−k−1 ≤ 0). `chosen` is the argmin of `criterion` ('aic', 'aicc' or
    'bic'); ties go to the smaller k, then the larger threshold; None if every candidate scores +inf. `library` is a
    `native.Library` or a SINDyRegression.

    window=R (an integer ≥ 2 dividing T) splits every trajectory into T/R consecutive windows of R rows, each scored as
    a trajectory of its own (n_starts = n_traj·T/R starts); None is R = T.

    fit_ic=True estimates every start: with the candidate's W fixed, each (candidate, start) pair's x̂0 minimises
    ‖rollout from x̂0 − rows 1..R−1‖² + ‖x̂0 − row 0‖², an independent d-dimensional problem. All pairs of all
    candidates run as one batch of `ic_iter` lock-step L-BFGS iterations (gradients from the start-only variant of
    `native.rollout_score_grad`, trial points from one per-model-start `native.rollout_score` launch; a trial that
    diverges counts as +inf, so `diverged` can only shrink). x̂0 starts at row 0 and each pair keeps its best iterate, so
    every candidate's sse (which now includes the row-0 residuals) is at most its fixed-start sse. The criteria use
    n = n_starts·R·d and k_eff = k + k_ic, k_ic = n_starts·d; `k` stays the live-coefficient count. Adds k_ic and x0
    (P, n_starts, d) fp32."""
    lib = getattr(library, 'library', library)
    if not isinstance(lib, Library):
        raise ValueError(f"library must be a native.Library or a SINDyRegression, got {type(library).__name__}")
    if criterion not in ('aic', 'aicc', 'bic'):
        raise ValueError(f"criterion must be 'aic', 'aicc' or 'bic', got {criterion!r}")
    x_val, dt = _check_rollout_args(lib, x_val, "x_val", dt, steps_per_row, method, blowup, fit_ic, window, ic_iter)
    n_traj, T, d = x_val.shape
    W, masks = path["xi"], path["mask"]
    if W.dim() != 3 or W.shape[1:] != (d, lib.K) or masks.shape != W.shape:
        raise ValueError(f"path['xi'] / path['mask'] must be (P, {d}, {lib.K}), got {tuple(W.shape)} / "
                         f"{tuple(masks.shape)}")
    thr = torch.as_tensor(path["thresholds"], dtype=torch.float64).cpu()
    P = W.shape[0]
    dev = W.device
    xv = x_val.to(device=dev, dtype=torch.float32)
    models, inverse = torch.unique(W.reshape(P, -1), dim=0, return_inverse=True)
    x0, y = xv[:, 0].contiguous(), xv[:, 1:].transpose(0, 1).contiguous()
    with torch.no_grad():
        sse, valid = native.rollout_score(x0, models.view(-1, d, lib.K), lib, dt, int(steps_per_row), y, method, blowup)
        if fit_ic:
            sse, valid, x0_hat = _fit_starts(lib, models.view(-1, d, lib.K), x0, y, dt, int(steps_per_row), method,
                                             blowup, sse, valid, int(ic_iter))
    sse = sse.sum(1).cpu()[inverse.cpu()]
    diverged = (valid < T - 1).any(1).cpu()[inverse.cpu()]
    k = masks.flatten(1).sum(1).cpu().to(torch.float64)
    n, k_ic = _obs_counts(n_traj, T, d, fit_ic)
    crit = information_criteria(sse, n, k + k_ic)
    for c in crit.values():
        c[diverged] = math.inf
    out = {"sse": sse, "diverged": diverged, "n_obs": n, "k": k.to(torch.int64), **crit, "criterion": criterion}
    if fit_ic:
        out["k_ic"] = k_ic
        out["x0"] = x0_hat[inverse.to(dev)]
    c = crit[criterion].numpy()
    order = np.lexsort((-thr.numpy(), k.numpy(), c))                      # last key sorts first
    out["chosen"] = int(order[0]) if c[order[0]] < math.inf else None
    return out


def _obs_counts(n_starts, R, d, fit_ic):
    """(n_obs, k_ic) of n_starts trajectories of R rows: rows 1..R−1 are compared, and with start estimation row 0 is
    one more residual and every start adds d parameters."""
    return (n_starts * R * d, n_starts * d) if fit_ic else (n_starts * (R - 1) * d, 0)


def _fit_starts(lib, W, x0, y, dt, spr, method, blowup, sse0, valid0, max_iter):
    """score_path(fit_ic=True): per (model, start) pair, x̂0 minimising (pair SSE from x̂0 + ‖x̂0 − x0‖²) / (R·d) with W
    fixed, all pairs through `_lockstep_lbfgs` at once. Returns the pair totals (sse + start residual, M × N fp64), the
    valid rows at x̂0 and x̂0 (M × N × d fp32). sse0 / valid0 are the fixed-start scores: a pair that diverged there
    keeps x0."""
    M, (N, d), R = W.shape[0], x0.shape, y.shape[0] + 1
    nrm = R * d
    x0d = x0.to(torch.float64).expand(M, N, d).reshape(M * N, d)

    def loss_grad(q):
        sse, valid, _, gx = native.rollout_score_grad(q.view(M, N, d).float(), W, lib, dt, spr, y, method, blowup,
                                                       x0_grad=True, w_grad=False)
        r = q - x0d
        f = (sse.reshape(-1) + (r * r).sum(1)) / nrm
        f = torch.where(valid.reshape(-1) < R - 1, torch.full_like(f, math.inf), f)
        return f, (gx.reshape(-1, d) + 2 * r) / nrm

    def loss(q, rows):
        full = x0d.clone()                       # the pairs outside `rows` are evaluated at x0 and discarded
        full[rows] = q
        sse, valid = native.rollout_score(full.view(M, N, d).float(), W, lib, dt, spr, y, method, blowup)
        r = q - x0d[rows]
        f = (sse.reshape(-1)[rows] + (r * r).sum(1)) / nrm
        return torch.where(valid.reshape(-1)[rows] < R - 1, torch.full_like(f, math.inf), f)

    q, _, _, iters = _lockstep_lbfgs(x0d.clone(), loss_grad, loss, max_iter, 1e-7)
    x0_hat = q.view(M, N, d).float()
    sse, valid = native.rollout_score(x0_hat, W, lib, dt, spr, y, method, blowup)
    r = q.view(M, N, d) - x0d.view(M, N, d)
    moved = (iters > 0).view(M, N)
    # a pair that never accepted a step is exactly at x0 (start residual 0, the fixed-start scores); a pair that did
    # has a strictly lower objective
    tot = torch.where(moved, sse + (r * r).sum(2), sse0)
    return tot, torch.where(moved, valid, valid0), x0_hat


def _check_rollout_args(lib, x, name, dt, steps_per_row, method, blowup, fit_ic=False, window=None, ic_iter=1):
    """The checks score_path and refine_path share; returns (x as a tensor, dt). With window=R the returned x holds
    the n_traj·T/R windows of R consecutive rows as trajectories."""
    if method not in ('euler', 'rk4'):
        raise ValueError(f"method must be 'euler' or 'rk4', got {method!r}")
    if isinstance(steps_per_row, bool) or not isinstance(steps_per_row, (int, np.integer)) or steps_per_row < 1:
        raise ValueError(f"steps_per_row must be a positive integer, got {steps_per_row!r}")
    dt = float(dt)
    if not (math.isfinite(dt) and dt > 0):
        raise ValueError(f"dt must be positive, got {dt}")
    if blowup is not None and not (math.isfinite(float(blowup)) and float(blowup) > 0):
        raise ValueError(f"blowup must be a positive number or None, got {blowup!r}")
    if not isinstance(fit_ic, (bool, np.bool_)):
        raise ValueError(f"fit_ic must be True or False, got {fit_ic!r}")
    if isinstance(ic_iter, bool) or not isinstance(ic_iter, (int, np.integer)) or ic_iter < 1:
        raise ValueError(f"ic_iter must be a positive integer, got {ic_iter!r}")
    x = torch.as_tensor(x)
    if x.dim() != 3 or x.shape[-1] != lib.dim:
        raise ValueError(f"{name} must be (n_traj, T, {lib.dim}), got {tuple(x.shape)}")
    if x.shape[1] < 2 or x.shape[0] < 1:
        raise ValueError(f"{name} needs at least one trajectory of T >= 2 rows, got {tuple(x.shape)}")
    if window is not None:
        T = x.shape[1]
        if isinstance(window, bool) or not isinstance(window, (int, np.integer)) or window < 2 or T % window:
            raise ValueError(f"window must be an integer >= 2 that divides T = {T}, got {window!r}")
        x = x.reshape(x.shape[0] * (T // int(window)), int(window), x.shape[2])
    if not bool(torch.isfinite(x).all()):
        raise ValueError(f"{name} has non-finite values")
    return x, dt


def _lockstep_lbfgs(p, loss_grad, loss, max_iter, tol, dir_mask=None):
    """Minimises U independent problems in lock-step: p (U, n) fp64 starting parameters; loss_grad(q) gives the losses
    (U,) and gradients (U, n) of all problems in one batch, loss(q, rows) the losses of the problems `rows` at q (one row
    each); +inf marks a diverged point. Per iteration: the L-BFGS direction (`sweep.BatchedLBFGS.direction`, times
    dir_mask when given), steepest descent where that is not a descent direction, then a backtracking (Armijo) line
    search whose trial points of every problem still searching are evaluated by one `loss` call. A problem stops after
    max_iter iterations, when its loss falls by less than tol·loss, or when no step length decreases it; its best
    iterate is kept. Returns (p, loss, loss at the start, accepted iterations), the last three per problem."""
    import sweep
    U = p.shape[0]
    f, g = loss_grad(p)
    f_before = f.clone()
    opt = sweep.BatchedLBFGS(p, 1.0, history_size=10)
    iters = torch.zeros(U, dtype=torch.long, device=p.device)
    active = torch.isfinite(f) & (g.abs().amax(1) > 0)
    c1, max_ls = 1e-4, 30
    for _ in range(max_iter):
        if not bool(active.any()):
            break
        dirn = opt.direction(g)
        if dir_mask is not None:
            dirn = dirn * dir_mask
        gtd = (g * dirn).sum(1)
        restart = gtd >= 0                                       # not a descent direction: steepest descent
        dirn = torch.where(restart.unsqueeze(1), -g, dirn)
        gtd = torch.where(restart, -(g * g).sum(1), gtd)
        t = torch.where(opt.hist == 0, torch.clamp(1.0 / g.abs().sum(1), max=1.0), torch.ones_like(f))
        searching, accepted = active.clone(), torch.zeros_like(active)
        for _ls in range(max_ls):
            idx = torch.nonzero(searching).flatten()
            if idx.numel() == 0:
                break
            trial = p[idx] + t[idx].unsqueeze(1) * dirn[idx]
            ft = loss(trial, idx)
            ok = ft <= f[idx] + c1 * t[idx] * gtd[idx]
            accepted[idx[ok]] = True
            searching[idx[ok]] = False
            t[idx[~ok]] *= 0.5
        active &= accepted                                        # no step length decreased the loss: done
        p_new = torch.where(active.unsqueeze(1), p + t.unsqueeze(1) * dirn, p)
        f_new, g_new = loss_grad(p_new)
        f_new = torch.where(active, f_new, f)
        g_new = torch.where(active.unsqueeze(1), g_new, g)
        sv, yv = p_new - p, g_new - g
        ys = (sv * yv).sum(1)
        opt.push(yv, sv, active & (ys > 1e-10), ys)
        iters += active.long()
        small = (f - f_new) <= tol * f.abs()
        p, f, g = p_new, f_new, g_new
        active &= ~small & (g.abs().amax(1) > 0)
    return p, f, f_before, iters


def refine_path(regressor, path, x_fit, dt, steps_per_row=1, method='rk4', blowup=None, max_iter=50, tol=1e-7,
                fit_ic=False, window=None):
    """Trajectory refit of the candidates of `stlsq_path` / `WSINDyWrapper.solve_path`: every distinct candidate's
    coefficients are refit on its own support by minimising the simulation error on the fitting trajectories,
      loss = SSE / n_obs of the rollouts from x_fit[:, 0] (step dt) against rows 1..T−1, n_obs = n_traj·(T−1)·d,
    the objective `score_path` ranks by. Derivative regression leaves a bias that grows with the noise of the smoothed
    derivatives; this refit judges a support by its best coefficients rather than by the ones regression gave it.

    All candidates advance together (`_lockstep_lbfgs`): one `native.rollout_score_grad` launch gives every loss and
    gradient (discrete adjoint of the fp32 rollout), the L-BFGS direction is `sweep.BatchedLBFGS.direction` over the
    candidate axis, and a per-candidate backtracking (Armijo) line search evaluates the trial points of every candidate
    still searching in one `native.rollout_score` launch; a trial that diverges (fewer rows than T−1 compared) counts as
    +inf. A candidate stops after max_iter iterations, when its loss falls by less than tol·loss, or when no step length
    decreases it; its best iterate is kept, so sse_after <= sse_before. Masks are fixed: dead coefficients stay exactly
    0. An equivariance-constrained regressor is refit in its parameters (β, const), vec(Ξ) = A·[β, const], A from
    `sweep.param_map`, and the returned path carries the new beta / const for `apply_candidate`.

    window=R (an integer ≥ 2 dividing T) fits on the n_traj·T/R consecutive windows of R rows as trajectories of their
    own (n_starts of them; None is R = T): over a long horizon the single-shooting SSE is dominated by phase drift.

    fit_ic=True also estimates every start, since row 0 is an observation with the noise of the others: each
    candidate's parameters become [coefficients (or β, const), x̂0 of every start] and the loss
      (Σ SSE of the rollouts from x̂0 against rows 1..R−1 + Σ ‖x̂0 − row 0‖²) / n_obs,  n_obs = n_starts·R·d,
    with ∂/∂x̂0 from `native.rollout_score_grad(x0_grad=True)` (per-model starts) plus 2(x̂0 − row 0). x̂0 starts at
    row 0, so sse_before is the fixed-start value; the starts are unconstrained (also for a constrained regressor),
    and one step length moves coefficients and starts together. Adds x0 (P, n_starts, d) fp32.

    Returns a copy of `path` with xi refit and sse_before, sse_after (P,) fp64 and iterations (P,) added; a candidate that
    diverges from the start keeps its coefficients (sse_before = sse_after = +inf)."""
    import sweep
    lib = getattr(regressor, 'library', regressor)
    if not isinstance(lib, Library):
        raise ValueError(f"regressor must be a SINDyRegression or a native.Library, got {type(regressor).__name__}")
    constrained = bool(getattr(regressor, 'constraint', False))
    x_fit, dt = _check_rollout_args(lib, x_fit, "x_fit", dt, steps_per_row, method, blowup, fit_ic, window)
    if isinstance(max_iter, bool) or not isinstance(max_iter, (int, np.integer)) or max_iter < 1:
        raise ValueError(f"max_iter must be a positive integer, got {max_iter!r}")
    if not (math.isfinite(float(tol)) and float(tol) >= 0):
        raise ValueError(f"tol must be a non-negative number, got {tol!r}")
    n_traj, T, d = x_fit.shape
    W0, masks = path["xi"], path["mask"]
    if W0.dim() != 3 or W0.shape[1:] != (d, lib.K) or masks.shape != W0.shape:
        raise ValueError(f"path['xi'] / path['mask'] must be (P, {d}, {lib.K}), got {tuple(W0.shape)} / "
                         f"{tuple(masks.shape)}")
    if constrained and ("beta" not in path or "const" not in path):
        raise ValueError("an equivariance-constrained regressor needs path['beta'] and path['const']")
    P, dK = W0.shape[0], d * lib.K
    dev = W0.device
    xf = x_fit.to(device=dev, dtype=torch.float32)
    x0, y = xf[:, 0].contiguous(), xf[:, 1:].transpose(0, 1).contiguous()
    n_obs = n_traj * (T - 1) * d
    # distinct candidates (coefficients and mask), each refit once
    key = torch.cat([W0.reshape(P, -1), masks.reshape(P, -1).to(W0.dtype)], 1)
    _, inverse = torch.unique(key, dim=0, return_inverse=True)
    U = int(inverse.max()) + 1
    first = torch.full((U,), P, dtype=torch.long, device=dev).scatter_reduce(0, inverse.to(dev),
                                                                            torch.arange(P, device=dev), 'amin')
    mk = masks[first].reshape(U, dK).to(torch.float64)
    if constrained:
        A, _ = sweep.param_map(regressor)
        A = A.to(dev)
        p = torch.cat([path["beta"][first].reshape(U, -1), path["const"][first].reshape(U, -1)], 1).to(dev, torch.float64)
    else:
        A = None
        p = W0[first].reshape(U, dK).to(torch.float64)

    def W_of(q, m):
        v = q if A is None else q @ A.T
        return (v * m).to(torch.float32).view(-1, d, lib.K)

    def diverged(f, valid):
        return torch.where((valid < T - 1).any(1), torch.full_like(f, math.inf), f)

    with torch.no_grad():
        if not fit_ic:
            def loss_grad(q):
                sse, valid, g = native.rollout_score_grad(x0, W_of(q, mk), lib, dt, int(steps_per_row), y, method,
                                                          blowup)
                g = g.reshape(-1, dK) * mk / n_obs
                return diverged(sse.sum(1) / n_obs, valid), (g if A is None else g @ A)

            def loss(q, rows):
                sse, valid = native.rollout_score(x0, W_of(q, mk[rows]), lib, dt, int(steps_per_row), y, method,
                                                  blowup)
                return diverged(sse.sum(1) / n_obs, valid)

            p, f, f_before, iters = _lockstep_lbfgs(p, loss_grad, loss, max_iter, tol, mk if A is None else None)
            sse_before, sse_after = f_before * n_obs, f * n_obs
        else:
            nc, n_ic = p.shape[1], _obs_counts(n_traj, T, d, True)[0]
            x0d = x0.to(torch.float64).reshape(1, -1)
            first_sse = []

            def split(q):
                return q[:, :nc], q[:, nc:]

            def objective(q_ic, sse, valid):
                r = q_ic - x0d
                return diverged((sse.sum(1) + (r * r).sum(1)) / n_ic, valid), r

            def loss_grad(q):
                c, s = split(q)
                sse, valid, g, gx = native.rollout_score_grad(s.view(-1, n_traj, d).float(), W_of(c, mk), lib, dt,
                                                              int(steps_per_row), y, method, blowup, x0_grad=True)
                if not first_sse:
                    first_sse.append(diverged(sse.sum(1) / n_obs, valid) * n_obs)   # the fixed-start sse_before
                f, r = objective(s, sse, valid)
                g = g.reshape(-1, dK) * mk / n_ic
                return f, torch.cat([g if A is None else g @ A, (gx.reshape(-1, n_traj * d) + 2 * r) / n_ic], 1)

            def loss(q, rows):
                c, s = split(q)
                sse, valid = native.rollout_score(s.view(-1, n_traj, d).float(), W_of(c, mk[rows]), lib, dt,
                                                  int(steps_per_row), y, method, blowup)
                return objective(s, sse, valid)[0]

            q0 = torch.cat([p, x0d.expand(U, -1)], 1)
            dmask = torch.cat([mk, torch.ones_like(q0[:, nc:])], 1) if A is None else None
            q, f, _, iters = _lockstep_lbfgs(q0, loss_grad, loss, max_iter, tol, dmask)
            p, x0_hat = split(q)
            sse_before = first_sse[0]
            # a candidate that accepted no step is where it started: its sse is sse_before
            sse_after = torch.where(iters > 0, f * n_ic, sse_before)
        out = dict(path)
        inv = inverse.to(dev)
        out["xi"] = (W_of(p, mk)[inv] * masks).to(W0.dtype)
        if constrained:
            nb = path["beta"].shape[1]
            out["beta"] = p[inv, :nb].to(path["beta"].dtype)
            out["const"] = p[inv, nb:].reshape(P, d, 1).to(path["const"].dtype)
        out["sse_before"] = sse_before[inv].cpu()
        out["sse_after"] = sse_after[inv].cpu()
        out["iterations"] = iters[inv].cpu()
        if fit_ic:
            out["x0"] = x0_hat[inv].reshape(P, n_traj, d).to(torch.float32)
    return out


def _schur_starts(jtj, jtj_px, jtj_xx):
    """S = F_θθ − Σ_n F_θx,n (F_xx,n + I)⁻¹ F_θx,nᵀ: the information of θ with every start x_n eliminated, the +I from
    the row-0 residual x_n − row 0. jtj (U, P, P), jtj_px (U, N, P, d), jtj_xx (U, N, d, d), fp64."""
    eye = torch.eye(jtj_xx.shape[-1], dtype=jtj_xx.dtype, device=jtj_xx.device)
    Z = torch.linalg.solve(jtj_xx + eye, jtj_px.transpose(-1, -2))              # (U, N, d, P)
    return jtj - torch.einsum('unpd,undq->upq', jtj_px, Z)


def _gn_covariance(S, sigma2, A=None):
    """σ²·A (AᵀSA)⁻¹ Aᵀ (A = None: σ²·S⁻¹) from a Cholesky factorisation of the equilibrated D·AᵀSA·D, D = diag^(−1/2);
    columns of A that are zero are dropped first. Returns (covariance, condition number of the equilibrated matrix), or
    (None, inf) when it is not positive definite."""
    if A is not None:
        A = A[:, A.abs().sum(0) > 0]                        # parameters that reach no listed coefficient
        S = A.T @ S @ A
    dg = torch.diagonal(S)
    if S.shape[0] == 0 or not bool(torch.isfinite(S).all()) or not bool((dg > 0).all()):
        return None, math.inf
    Dm = dg.rsqrt()
    Se = Dm[:, None] * S * Dm[None, :]
    L, info = torch.linalg.cholesky_ex(Se)
    if int(info) != 0:
        return None, math.inf
    ev = torch.linalg.eigvalsh(Se)
    cond = float(ev[-1] / ev[0]) if float(ev[0]) > 0 else math.inf
    cov = sigma2 * (Dm[:, None] * torch.cholesky_inverse(L) * Dm[None, :])
    return (cov if A is None else A @ cov @ A.T), cond


def coefficient_covariance(regressor, path, x, dt, steps_per_row=1, method='rk4', blowup=None, fit_ic=False,
                           window=None):
    """Gauss–Newton covariance of the coefficients of a `refine_path` result (with its arguments: the same
    trajectories, step, method, fit_ic and window; with fit_ic=True, path['x0'] holds the fitted starts).

    The refit minimises the simulation SSE with iid Gaussian residuals on every compared row (and on row 0 for the
    starts), so Cov(θ) ≈ σ̂²·S⁻¹ with S = JᵀJ, J the Jacobian of every compared state with respect to the parameters.
    Every distinct candidate (coefficients and mask, and starts with fit_ic) is evaluated once, all of them in one
    `native.rollout_score_gn` launch (tangent-linear rollouts of the fp32 recurrence that was scored), which gives
    F_θθ = Σ JθᵀJθ over the live coefficients and, with fit_ic, the per-start blocks F_θx,n and F_xx,n. The starts are
    eliminated by the Schur complement S = F_θθ − Σ_n F_θx,n (F_xx,n + I)⁻¹ F_θx,nᵀ (the +I is the row-0 residual);
    without fit_ic S = F_θθ and the starts count as exact. σ̂² = SSE / (n_obs − k_eff), n_obs and k_eff = live
    coefficients (+ n_starts·d) as `score_path` counts them. S⁻¹ comes from a Cholesky factorisation of D·S·D,
    D = diag(S)^(−1/2), in fp64. An equivariance-constrained regressor is parametrised by (β, const): vec(Ξ) = A·q with A
    from `sweep.param_map` restricted to the live rows (and to the columns that reach them), S_q = AᵀSA and
    Cov(vec Ξ) = A·Cov_q·Aᵀ.

    Returns, per path entry: sse (P,) fp64 (rows compared, plus the row-0 residuals with fit_ic), sigma2 (P,), cov
    (P, d·K, d·K) fp64 over vec(Ξ) (equation-major), zero off the mask; stderr (P, d, K), the square root of its
    diagonal, zero off the mask; tstat = Ξ / stderr on the mask; cond (P,), the condition number of D·S·D;
    identifiable (P,) bool, False when the factorisation fails (stderr is then +inf and cov NaN on the mask); diverged
    (P,) bool as in `score_path` (stderr and cov are then NaN on the mask); n_obs. All on the host."""
    import sweep
    lib = getattr(regressor, 'library', regressor)
    if not isinstance(lib, Library):
        raise ValueError(f"regressor must be a SINDyRegression or a native.Library, got {type(regressor).__name__}")
    constrained = bool(getattr(regressor, 'constraint', False))
    x, dt = _check_rollout_args(lib, x, "x", dt, steps_per_row, method, blowup, fit_ic, window)
    n_traj, T, d = x.shape
    K, dK = lib.K, d * lib.K
    W0, masks = path["xi"], path["mask"]
    if W0.dim() != 3 or W0.shape[1:] != (d, K) or masks.shape != W0.shape:
        raise ValueError(f"path['xi'] / path['mask'] must be (P, {d}, {K}), got {tuple(W0.shape)} / "
                         f"{tuple(masks.shape)}")
    P = W0.shape[0]
    dev = W0.device
    if fit_ic:
        if "x0" not in path:
            raise ValueError("fit_ic=True needs the fitted starts path['x0'] (refine_path(fit_ic=True) adds them)")
        x0p = torch.as_tensor(path["x0"])
        if x0p.shape != (P, n_traj, d):
            raise ValueError(f"path['x0'] must be ({P}, {n_traj}, {d}), got {tuple(x0p.shape)}")
        if not bool(torch.isfinite(x0p).all()):
            raise ValueError("path['x0'] has non-finite values")
        x0p = x0p.to(device=dev, dtype=torch.float32)
    n_live_max = int(masks.flatten(1).sum(1).max()) if P else 0
    if n_live_max + (d if fit_ic else 0) > native.GN_MAX_COLS:
        raise ValueError(f"{n_live_max} live coefficients{' and ' + str(d) + ' start columns' if fit_ic else ''} "
                         f"exceed the {native.GN_MAX_COLS} tangent columns of native.rollout_score_gn")
    xf = x.to(device=dev, dtype=torch.float32)
    x0, y = xf[:, 0].contiguous(), xf[:, 1:].transpose(0, 1).contiguous()
    n_obs, k_ic = _obs_counts(n_traj, T, d, fit_ic)
    # distinct candidates (coefficients, mask and starts), each evaluated once
    key = [W0.reshape(P, -1), masks.reshape(P, -1).to(W0.dtype)] + ([x0p.reshape(P, -1).to(W0.dtype)] if fit_ic else [])
    _, inverse = torch.unique(torch.cat(key, 1), dim=0, return_inverse=True)
    U = int(inverse.max()) + 1
    first = torch.full((U,), P, dtype=torch.long, device=dev).scatter_reduce(0, inverse.to(dev),
                                                                            torch.arange(P, device=dev), 'amin')
    mk = masks[first].reshape(U, dK)
    live = [torch.nonzero(mk[u]).flatten() for u in range(U)]
    n_par = max(1, max(int(v.numel()) for v in live))
    params = torch.full((U, n_par), -1, dtype=torch.int32, device=dev)
    for u, v in enumerate(live):
        params[u, :v.numel()] = v.to(torch.int32)
    Wu = (W0[first].reshape(U, dK) * mk).to(torch.float32).view(U, d, K)
    with torch.no_grad():
        gn = native.rollout_score_gn(x0p[first] if fit_ic else x0, Wu, params, lib, dt, int(steps_per_row), y, method,
                                     blowup, x0_blocks=fit_ic)
        sse = gn["sse"].sum(1)
        S = gn["jtj"]
        if fit_ic:
            r = x0p[first].to(torch.float64) - x0.to(torch.float64)
            sse = sse + (r * r).sum((1, 2))
            S = _schur_starts(S, gn["jtj_px"], gn["jtj_xx"])
        diverged = (gn["valid_rows"] < T - 1).any(1)
        A = sweep.param_map(regressor)[0].to(dev) if constrained else None
        k_eff = mk.sum(1).to(torch.float64) + k_ic
        den = n_obs - k_eff
        sigma2 = torch.where(den > 0, sse / den.clamp_min(1.0), torch.full_like(sse, math.nan))
        cov = torch.zeros(U, dK, dK, dtype=torch.float64)
        cond = torch.full((U,), math.inf, dtype=torch.float64)
        ident = torch.zeros(U, dtype=torch.bool)
        S, sigma2_h, div_h = S.cpu(), sigma2.cpu(), diverged.cpu()
        for u, v in enumerate(live):
            n, vc = int(v.numel()), v.cpu()
            if n == 0:
                ident[u] = True
                cond[u] = 1.0
                continue
            blk = torch.full((n, n), math.nan, dtype=torch.float64)
            if not bool(div_h[u]):
                c, cond[u] = _gn_covariance(S[u, :n, :n], float(sigma2_h[u]), None if A is None else A.cpu()[vc])
                if c is not None:
                    blk, ident[u] = c, True
            cov[u][vc[:, None], vc[None, :]] = blk
        inv = inverse.cpu()
        cov = cov[inv]
        mflat = masks.reshape(P, dK).cpu()
        var = torch.diagonal(cov, dim1=1, dim2=2)
        se = torch.where(mflat, var.sqrt(), torch.zeros_like(var))
        ident, div_p = ident[inv], div_h[inv]
        bad = (~ident & ~div_p)[:, None] & mflat
        se = torch.where(bad, torch.full_like(se, math.inf), se)
        se = se.view(P, d, K)
        xi = (W0.reshape(P, dK).cpu().to(torch.float64) * mflat).view(P, d, K)
        tstat = torch.where(masks.cpu(), xi / se, torch.zeros_like(xi))
    return {"sse": sse.cpu()[inv], "sigma2": sigma2_h[inv], "cov": cov, "stderr": se, "tstat": tstat,
            "cond": cond[inv], "identifiable": ident, "diverged": div_p, "n_obs": n_obs}


def information_criteria(sse, n, k):
    """AIC, AICc and BIC of Gaussian residuals with sum of squares `sse` over n observations and k parameters (fp64
    tensors of one shape, or scalars): n·ln(SSE/n) + 2k, that + 2k(k+1)/(n−k−1) (+inf when n−k−1 ≤ 0), and
    n·ln(SSE/n) + k·ln n."""
    sse = torch.as_tensor(sse, dtype=torch.float64)
    k = torch.as_tensor(k, dtype=torch.float64)
    fit = n * torch.log(sse / n)
    aic = fit + 2.0 * k
    den = n - k - 1.0
    aicc = torch.where(den > 0, aic + 2.0 * k * (k + 1.0) / den.clamp_min(1.0), torch.full_like(aic, math.inf))
    bic = fit + k * math.log(n)
    return {"aic": aic, "aicc": aicc, "bic": bic}


def apply_candidate(regressor, path, i):
    """Writes candidate i of a threshold path into the regressor: Ξ (or β / const) and the mask."""
    i = int(i)
    with torch.no_grad():
        mask = path["mask"][i].to(device=regressor.mask.device, dtype=regressor.mask.dtype)
        if regressor.constraint:
            regressor.beta.data = path["beta"][i].to(regressor.beta.device).clone()
            regressor.const.data = path["const"][i].to(regressor.const.device).clone()
            regressor.Xi = regressor.get_Xi()
        else:
            regressor.Xi.data = path["xi"][i].to(regressor.Xi.device).clone()
        regressor.mask.data = mask.clone()
    return regressor


def _local_test_functions(T, dt, n_test, support=None, degree=None):
    """The compactly supported piecewise-polynomial family of WSINDyWrapper(test_func_family='poly') (Messenger &
    Bortz, Weak SINDy for ODEs, 2021): every row is the same window of L samples at its own start
      φ_q = (4u(1−u))^p,  φ'_q = p·(4u(1−u))^(p−1)·4(1−2u)/((L−1)·dt),  u = q/(L−1),  q = 0..L−1,
      phi = fp32(dt·c·φ),  dphi = fp32(dt·c·φ'),  c = 1/sqrt(dt·Σφ²)   (Σ_t V[j,t]² = dt, the scale of the trig rows),
      s_j = ⌊j·(T−L)/(n_test−1)⌋  (s_0 = 0 when n_test = 1).
    Defaults: L = min(T, 2·⌊T/(n_test+1)⌋ + 1) (about two-fold overlap), p = 6. Returns (L, p, starts, phi, dphi) with
    numpy fp32 tables; raises ValueError unless 3 ≤ L ≤ T, 1 ≤ p ≤ 32 and 1 ≤ n_test ≤ T − L + 1."""
    def integer(v, name):
        if isinstance(v, bool) or not isinstance(v, (int, np.integer)):
            raise ValueError(f"{name} must be an integer, got {v!r}")
        return int(v)
    T, n_test = integer(T, "the number of time samples"), integer(n_test, "num_test_funcs")
    if n_test < 1:
        raise ValueError(f"num_test_funcs must be at least 1, got {n_test}")
    L = min(T, 2 * (T // (n_test + 1)) + 1) if support is None else integer(support, "test_func_support")
    p = 6 if degree is None else integer(degree, "test_func_degree")
    if not 3 <= L <= T:
        raise ValueError(f"test_func_support must lie in [3, T = {T}], got {L}")
    if not 1 <= p <= 32:
        raise ValueError(f"test_func_degree must lie in [1, 32], got {p}")
    if n_test > T - L + 1:
        raise ValueError(f"num_test_funcs = {n_test} exceeds T − L + 1 = {T - L + 1}: the windows would not have "
                         f"distinct starts")
    if not (math.isfinite(dt) and dt > 0):
        raise ValueError(f"the time step must be positive, got {dt}")
    u = np.arange(L, dtype=np.float64) / (L - 1)
    s = 4.0 * u * (1.0 - u)
    phi = s ** p
    dphi = p * s ** (p - 1) * 4.0 * (1.0 - 2.0 * u) / ((L - 1) * dt)
    c = 1.0 / math.sqrt(dt * float(np.sum(phi * phi)))
    starts = [0] if n_test == 1 else [j * (T - L) // (n_test - 1) for j in range(n_test)]
    return L, p, starts, (dt * c * phi).astype(np.float32), (dt * c * dphi).astype(np.float32)


class WSINDyWrapper():
    """Weak SINDy as a regularised least-squares problem (reference `sindy.py:327-395`).

    test_func_family='trig' (the reference's): g_k(t) = sqrt(2/T)·sin(kπt/T), k = 1..num_test_funcs, each spanning the
    whole window. test_func_family='poly': compactly supported piecewise polynomials (`_local_test_functions`) of
    test_func_support samples (default about 2·T/num_test_funcs) and degree test_func_degree (default 6); a sample then
    costs only the few windows that cover it, so hundreds or thousands of test functions can be placed along a long
    trajectory. `t` must be the uniform grid t_i = i·dt starting at 0 that `main_wsindy.py:41` builds.
    """

    def __init__(self, regressor, t, t_max, num_test_funcs=50, test_func_family='trig', device='cuda',
                 test_func_support=None, test_func_degree=None, **kwargs):
        if test_func_family not in ('trig', 'poly'):
            raise NotImplementedError(f'test_func_family={test_func_family} not implemented')
        if test_func_family == 'trig' and (test_func_support is not None or test_func_degree is not None):
            raise ValueError("test_func_support / test_func_degree apply to test_func_family='poly' only")
        if test_func_family == 'poly':
            layout = _local_test_functions(int(t.shape[0]), float(t[1] - t[0]), num_test_funcs, test_func_support,
                                           test_func_degree)
        self.test_func_family = test_func_family
        self.t = t.to(device)
        self.dt = self.t[1] - self.t[0]
        self.t_max = float(t_max)
        self.num_test_funcs = int(num_test_funcs)
        self.regressor = regressor
        self.kwargs = {'lstsq_driver': kwargs.get('lstsq_driver')}
        if test_func_family == 'poly':
            L, p, starts, phi, dphi = layout
            self.test_func_support, self.test_func_degree = L, p
            self.phi = torch.from_numpy(phi).to(device)
            self.dphi = torch.from_numpy(dphi).to(device)
            # dense V, V' (n_test × T) for attribute parity with the trig family and for M = V·Vᵀ; the kernel reads
            # only the L-sample tables
            T = self.t.shape[0]
            cols = (torch.tensor(starts, dtype=torch.int64).view(-1, 1) + torch.arange(L).view(1, -1)).to(device)
            self.V = torch.zeros(self.num_test_funcs, T, dtype=torch.float32, device=device)
            self.V_drv = torch.zeros_like(self.V)
            self.V.scatter_(1, cols, self.phi.expand(self.num_test_funcs, L).contiguous())
            self.V_drv.scatter_(1, cols, self.dphi.expand(self.num_test_funcs, L).contiguous())
            self.M = self.V.double() @ self.V.double().T
            return
        # dense V only to form the n_test×n_test weight M = V·Vᵀ once (the reference multiplies by Vᵀ on the
        # left of both sides, `sindy.py:369-370`); the data-dependent integrals never read V.
        k = torch.arange(1, num_test_funcs + 1, dtype=torch.float32, device=device).view(-1, 1)
        phase = k * torch.pi * self.t / t_max
        amp = math.sqrt(2 / t_max)
        self.V = self.dt * (amp * torch.sin(phase))
        self.V_drv = self.dt * (amp * k * np.pi / t_max * torch.cos(phase))
        self.M = self.V.double() @ self.V.double().T

    def integrals(self, x):
        """G = V·Θ(x) (n_test×K) and b = −V'·x (n_test×d), fp64, from the fused kernel; x of shape (T, d), or
        (n_traj, T, d) for per-trajectory (n_traj×n_test×K, n_traj×n_test×d)."""
        if self.test_func_family == 'poly':
            return native.wsindy_local_integrals(x, self.regressor.library, self.phi, self.dphi, self.num_test_funcs)
        return native.wsindy_integrals(x, self.regressor.library, float(self.dt), self.t_max, self.num_test_funcs)

    def _normal_equations(self, x):
        """(GᵀMG, GᵀMb, bᵀMb per equation, row count of the reference's least-squares matrix) for (T, d) or pooled
        (n_traj, T, d) input."""
        if x.shape[-2] != self.t.shape[0] or x.dim() not in (2, 3):
            raise ValueError(f'x has {x.shape[-2]} time samples, the wrapper was built for {self.t.shape[0]}')
        Gw, bw = self.integrals(x)
        if x.dim() == 2:
            MG = self.M @ Gw
            A = Gw.T @ MG                                    # K×K
            rhs = MG.T @ bw                                  # K×d
            bb = torch.einsum('ji,jl,li->i', bw, self.M, bw)
            n_rows = x.shape[0]
        else:
            MG = self.M @ Gw                                 # n_traj × n_test × K
            A = (Gw.transpose(1, 2) @ MG).sum(0)
            rhs = (MG.transpose(1, 2) @ bw).sum(0)
            bb = torch.einsum('rji,jl,rli->i', bw, self.M, bw)
            n_rows = x.shape[0] * x.shape[1]
        return A, rhs, bb, n_rows

    def solve(self, x, w_sindy_reg, st_threshold, **kwargs):
        '''
        x: (seq_len, dim) on the wrapper's uniform grid. Solves [VᵀG; sqrt(w)·I] ξ = [Vᵀb; 0] on the current
        support through its normal equations (GᵀMG + w·I) ξ = GᵀM b, then thresholds.
        x: (n_traj, seq_len, dim): one equation from all trajectories, pooled through the summed normal equations
        (Σ_r G_rᵀMG_r + w·I) ξ = Σ_r G_rᵀMb_r.
        Returns (mean squared residual of that system, converged).
        '''
        with torch.no_grad():
            A, rhs, bb, n_rows = self._normal_equations(x)
            K = A.shape[0]
            converged = _stlsq_update(self.regressor, A, rhs, float(w_sindy_reg), n_rows + K, st_threshold,
                                      _lstsq_driver(kwargs if kwargs.get('lstsq_driver') else self.kwargs))
            Xi = self.regressor._current_Xi().to(torch.float64)
            quad = torch.einsum('ik,kl,il->i', Xi, A, Xi) - 2.0 * torch.einsum('ik,ki->i', Xi, rhs) + bb
            quad = quad + float(w_sindy_reg) * (Xi ** 2).sum(1)
        return quad.mean().item(), converged

    def solve_path(self, x, w_sindy_reg, thresholds, max_iter=5, **kwargs):
        """The threshold path of `solve` from one evaluation of the integrals (x of shape (T, d) or (n_traj, T, d)):
        candidate p is what `reset_mask()` followed by up to max_iter calls of `solve(x, w_sindy_reg, thresholds[p])`,
        stopping at the first converged call, leaves in the regressor. Returns the dict of `stlsq_path` with `residual`
        (P,) fp64 = the value the last `solve` returns; the regressor is left as it was."""
        thr = _path_thresholds(thresholds)
        max_iter = _path_max_iter(max_iter)
        driver = _lstsq_driver(kwargs if kwargs.get('lstsq_driver') else self.kwargs)
        with torch.no_grad():
            A, rhs, bb, n_rows = self._normal_equations(x)
            K = A.shape[0]
            ridge = float(w_sindy_reg)

            def step(t):
                return _stlsq_update(self.regressor, A, rhs, ridge, n_rows + K, t, driver)

            out = _stlsq_path_solve(self.regressor, A, rhs, bb, ridge, n_rows + K, thr, max_iter, driver, step)
            out["residual"] = out.pop("quad").mean(-1)
        return out
