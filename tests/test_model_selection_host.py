"""Host-side checks of model selection along the STLSQ threshold path (no GPU): argument validation before any device
work, the information criteria on hand-computed values, the batched path against the per-threshold STLSQ loop with the
Gram sums supplied by the oracle, and the C entry point's argument checks."""
import copy
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle import sindy_oracle as O


def _stats(x, y, p):
    s = O.train_step_sums(x, y, np.zeros((y.shape[1], O.term_count(x.shape[1], p))), p)
    return (torch.from_numpy(s["gram"]), torch.from_numpy(s["b"]),
            torch.from_numpy((y.astype(np.float64) ** 2).sum(0)), x.shape[0])


def _reg(d=2, p=2):
    import sindy
    return sindy.SINDyRegression(d, p, False, False, threshold=0.05, device="cpu", constrain_constant=True)


def test_information_criteria_hand_computed():
    import sindy
    c = sindy.information_criteria(torch.tensor([2.0, 8.0]), 100, torch.tensor([3.0, 97.0]))
    fit = 100 * math.log(0.02)
    assert c["aic"][0].item() == pytest.approx(fit + 6)
    assert c["aicc"][0].item() == pytest.approx(fit + 6 + 2 * 3 * 4 / 96)
    assert c["bic"][0].item() == pytest.approx(fit + 3 * math.log(100))
    assert c["aicc"][1].item() == pytest.approx(100 * math.log(0.08) + 194 + 2 * 97 * 98 / 2)
    # n − k − 1 ≤ 0: AICc is undefined, reported as +inf
    c = sindy.information_criteria(torch.tensor([1.0]), 10, torch.tensor([9.0]))
    assert math.isinf(c["aicc"][0].item()) and math.isfinite(c["aic"][0].item())


@pytest.mark.parametrize("bad", [[], [[0.1]], [-0.1, 0.2], [0.1, float("nan")], [float("inf")]])
def test_bad_thresholds_raise_before_any_device_work(bad):
    import sindy
    reg = _reg()
    x = torch.zeros(10, 2)
    with pytest.raises(ValueError):
        sindy.stlsq_path(reg, x, x, bad)
    t = torch.arange(40, dtype=torch.float32) * 0.1
    with pytest.raises(ValueError):
        sindy.WSINDyWrapper(reg, t, 4.0, num_test_funcs=5, device="cpu").solve_path(torch.zeros(40, 2), 0.0, bad)


def _path(P=3, d=2, K=6):
    return {"thresholds": torch.linspace(0.1, 0.3, P, dtype=torch.float64), "xi": torch.zeros(P, d, K),
            "mask": torch.ones(P, d, K, dtype=torch.bool)}


@pytest.mark.parametrize("kw", [
    dict(x_val=torch.zeros(4, 10)),                 # not (n_traj, T, d)
    dict(x_val=torch.zeros(4, 10, 3)),              # d mismatch
    dict(x_val=torch.zeros(4, 1, 2)),               # T < 2
    dict(steps_per_row=0),
    dict(steps_per_row=1.5),
    dict(dt=0.0),
    dict(method="midpoint"),
    dict(criterion="hqc"),
    dict(blowup=-1.0),
    dict(x_val=torch.full((4, 10, 2), float("nan"))),
    dict(path={**_path(), "xi": torch.zeros(3, 2, 5)}),
])
def test_score_path_argument_errors(kw):
    import sindy
    from sindy_b200.native import Library
    args = dict(library=Library(2, 2), path=_path(), x_val=torch.zeros(4, 10, 2), dt=0.01)
    args.update(kw)
    with pytest.raises(ValueError):
        sindy.score_path(**args)


def _loop(reg, G, b, ridge, n, thr, max_iter=5):
    import sindy
    masks, xis = [], []
    for t in thr:
        r = copy.deepcopy(reg)
        r.reset_mask()
        for _ in range(max_iter):
            if sindy._stlsq_update(r, G, b, ridge, n, float(t)):
                break
        masks.append(r.mask > 0)
        xis.append((r.Xi * r.mask).detach())
    return torch.stack(masks), torch.stack(xis)


@pytest.mark.parametrize("case", ["selkov", "dosc", "growth", "lorenz", "rank_deficient"])
def test_batched_path_equals_the_per_threshold_loop(golden, case):
    """The batched solves of _stlsq_path_solve against the loop of _stlsq_update, on the oracle's Gram sums. In the
    rank-deficient case (x1 = 2·x0) the full-library solves take the eigh path while small supports are full rank:
    the Cholesky / eigh choice is made per threshold."""
    import sindy
    g = golden("stlsq")
    if case == "rank_deficient":
        t = np.linspace(-1, 1, 400)
        x = np.stack([t, 2 * t], 1)
        y = np.stack([-0.5 * t + 0.3 * t * t, 0.1 + t], 1)
        d, p = 2, 2
    else:
        x, y = g[case + "_x"], g[case + "_y"]
        d, p = x.shape[1], (3 if case in ("selkov", "lorenz") else 2)
    G, b, yy, n = _stats(x, y, p)
    reg = _reg(d, p)
    before = reg.Xi.detach().clone()
    thr = np.concatenate([[0.0], np.logspace(-4, 0.5, 20)])
    for ridge in (0.0, 0.09):
        path = sindy._stlsq_path_solve(reg, G, b, yy, ridge, n + G.shape[0], thr, 5, "gels", None)
        masks, xis = _loop(reg, G, b, ridge, n + G.shape[0], thr)
        assert torch.equal(path["mask"], masks)
        scale = xis.abs().amax(dim=(1, 2), keepdim=True)
        assert torch.all((path["xi"] - xis).abs() <= 1e-6 * scale)
    assert torch.equal(reg.Xi.detach(), before) and torch.all(reg.mask == 1)


def test_per_threshold_rank_decision():
    """One singular candidate in the batch must not move a full-rank candidate off its Cholesky solution."""
    import sindy
    t = torch.linspace(-1, 1, 300, dtype=torch.float64)
    Th = torch.stack([torch.ones_like(t), t, 2 * t], 1)        # columns 1 and 2 collinear
    H = Th.T @ Th
    b = Th.T @ torch.stack([0.3 + t, 1 - t], 1)
    full = torch.ones(2, 3, dtype=torch.bool)
    small = torch.tensor([[1, 1, 0], [1, 0, 1]], dtype=torch.bool)
    both = sindy._masked_solve_path(H, b, torch.stack([full, small]), 0.0)
    assert torch.equal(both[1], sindy._masked_solve_batched(H, b, small, 0.0))
    assert torch.allclose(both[0], sindy._masked_solve_batched(H, b, full, 0.0), rtol=0, atol=1e-12)


def test_c_entry_point_validates_without_a_device():
    from sindy_b200 import native
    lib = native.load()
    L = native._CLibrary(2, 2, 0, 0)
    one = ctypes.c_void_p(16)

    def call(x0=one, n=8, lb=ctypes.byref(L), w=one, m=2, dt=0.01, spr=1, rows=3, meth=1, y=one, sse=one, valid=one):
        return lib.sb_rollout_score(x0, n, lb, w, m, dt, spr, rows, meth, y, 0.0, sse, valid, None)

    assert call(x0=None) == -1 and b"x0 is NULL" in lib.sb_last_error()
    assert call(y=None) == -1 and call(sse=None) == -1 and call(valid=None) == -1 and call(w=None) == -1
    assert call(m=0) == -1 and call(spr=0) == -1 and call(rows=0) == -1 and call(rows=1 << 31) == -1
    assert call(n=-1) == -1 and call(meth=2) == -1
    assert call(dt=0.0) == -1 and call(dt=float("nan")) == -1
    bad = native._CLibrary(2, 6, 0, 0)
    assert call(lb=ctypes.byref(bad)) == -2
    assert call(lb=None) == -1
    assert call(n=0) == 0                                       # nothing to do
