"""CPU-only checks: the C-ABI library loads and exports every symbol include/sindy_b200.h declares, the host-side
library enumeration matches the oracle, and the host logic of the drop-in modules (constraint basis, STLSQ update
on normal equations, thresholding) reproduces the reference goldens when fed oracle-computed sums.
No compute entry point is called (no GPU here)."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from oracle import sindy_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from sindy_b200 import native
    header = open(os.path.join(ROOT, "include", "sindy_b200.h")).read()
    declared = set(re.findall(r"\b(sb_[a-z0-9_]+)\s*\(", header))
    declared -= {"sb_status", "sb_library"}
    lib = native.load()
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert declared == set(native.EXPORTED_SYMBOLS)
    assert lib.sb_version() >= 100


def _header_prototypes():
    """{name: (return type, [parameter types])} parsed from include/sindy_b200.h (comments and macros stripped)."""
    text = open(os.path.join(ROOT, "include", "sindy_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    text = re.sub(r"//[^\n]*", " ", text)
    text = "\n".join(ln for ln in text.splitlines() if not ln.lstrip().startswith("#"))
    protos = {}
    for ret, name, params in re.findall(r"([A-Za-z_][A-Za-z0-9_ ]*?[\s\*]+)(sb_[a-z0-9_]+)\s*\(([^()]*)\)\s*;", text):
        plist = [] if params.strip() in ("", "void") else [q.strip() for q in params.split(",")]
        # drop the parameter NAME: the type is everything up to the last identifier
        types = [re.sub(r"\s*[A-Za-z_][A-Za-z0-9_]*$", "", q).strip() for q in plist]
        protos[name] = (" ".join(ret.split()), [" ".join(t.split()) for t in types])
    return protos


def _c_kind(ctype: str) -> str:
    """Coarse ABI class of a C type as written in the header."""
    t = ctype.replace("const ", "").replace(" const", "").strip()
    if t.endswith("*"):
        return "char*" if t == "char*" or t == "char *" else "ptr"
    return {"int": "i32", "int32_t": "i32", "uint32_t": "u32", "int64_t": "i64", "unsigned long long": "u64",
            "float": "f32", "double": "f64", "void": "void"}[t]


def _ctypes_kind(ct) -> str:
    if ct is None:
        return "void"
    if ct is ctypes.c_char_p:
        return "char*"
    if ct is ctypes.c_void_p or isinstance(ct, type) and issubclass(ct, ctypes._Pointer):
        return "ptr"
    return {ctypes.c_int: "i32", ctypes.c_int32: "i32", ctypes.c_uint32: "u32", ctypes.c_int64: "i64",
            ctypes.c_ulonglong: "u64", ctypes.c_float: "f32", ctypes.c_double: "f64"}[ct]


def test_ctypes_signatures_match_the_header_prototypes():
    """The binding's (restype, argtypes) table against the prototypes of include/sindy_b200.h: same parameter count and,
    per parameter, the same ABI class (pointer / int32 / uint32 / int64 / float / double) — a float passed where the
    header says double, or a missing trailing argument, corrupts a call silently. The two structs are checked field by
    field against their typedefs."""
    from sindy_b200 import native
    protos = _header_prototypes()
    assert set(protos) == set(native.EXPORTED_SYMBOLS)
    for name, (res, args) in native._SIGNATURES.items():
        ret, params = protos[name]
        assert _c_kind(ret) == _ctypes_kind(res), (name, ret, res)
        assert len(params) == len(args), (name, params, args)
        for i, (ct, at) in enumerate(zip(params, args)):
            assert _c_kind(ct) == _ctypes_kind(at), (name, i, ct, at)
    header = open(os.path.join(ROOT, "include", "sindy_b200.h")).read()
    for struct, cls in (("sb_library", native._CLibrary), ("sb_fit_options", native._CFitOptions)):
        body = re.search(r"typedef struct\s*\{([^{}]*)\}\s*" + struct + r"\s*;", header).group(1)
        body = re.sub(r"/\*.*?\*/", " ", body, flags=re.S)
        fields = [f.strip() for f in body.split(";") if f.strip()]
        assert len(fields) == len(cls._fields_), (struct, fields)
        for decl, (fname, ftype) in zip(fields, cls._fields_):
            m = re.match(r"(.*?)([A-Za-z_][A-Za-z0-9_]*)$", decl)
            assert m.group(2) == fname, (struct, decl, fname)
            assert _c_kind(" ".join(m.group(1).split())) == _ctypes_kind(ftype), (struct, decl, ftype)


@pytest.mark.parametrize("d,p,s,e", [(2, 2, 0, 0), (2, 3, 1, 1), (3, 5, 0, 0), (4, 3, 0, 1), (8, 2, 1, 1), (1, 5, 0, 0)])
def test_library_size_and_exponents(d, p, s, e):
    from sindy_b200 import native
    lib = native.Library(d, p, bool(s), bool(e))
    assert lib.K == O.term_count(d, p, s, e)
    E = lib.exponents().numpy()
    npoly = O.term_count(d, p)
    assert np.array_equal(E[:npoly], O.exponents(d, p))
    if s:
        assert np.array_equal(E[npoly:npoly + d], -np.eye(d, dtype=np.int32))
    assert lib.workspace_bytes() > 0 and lib.step_out_len(15) == 2 + d * lib.K + lib.K ** 2 + lib.K * d


def test_unsupported_libraries_are_rejected_loudly():
    from sindy_b200 import native
    for bad in (native.Library(0, 2), native.Library(9, 2), native.Library(2, 0), native.Library(2, 6),
                native.Library(8, 4)):
        with pytest.raises(native.SindyB200Error):
            bad.K
    with pytest.raises(RuntimeError):   # CPU tensors never reach a kernel
        native.forward(torch.zeros(3, 2), torch.zeros(2, 6), native.Library(2, 2))


def test_per_block_library_functions_refuse_what_they_cannot_do():
    """`sindy.py:7-30` helpers: values from the CUDA path only — a CPU tensor raises (no fallback), a tensor that
    carries a gradient raises instead of losing it."""
    import sindy
    for fn in (sindy.SINDyConst, sindy.SINDyPoly1, sindy.SINDyPoly2, sindy.SINDyPoly3, sindy.SINDySine, sindy.SINDyExp):
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            fn(torch.zeros(5, 2))
        with pytest.raises(NotImplementedError):
            fn(torch.zeros(5, 2, requires_grad=True))
    with pytest.raises(TypeError):
        sindy.SINDyPoly2(3.0)


def test_missing_library_fails_loudly(monkeypatch):
    from sindy_b200 import native
    monkeypatch.setattr(native, "_lib", None)
    monkeypatch.setattr(native, "LIB_PATH", "/nonexistent/libsindy_b200.so")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        native.load()


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "symmetry-ode-discovery_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.replace("oracle/", "").lower() or "import" not in text.lower() or \
                    not re.search(r"^\s*(from|import)\s+oracle", text, re.M), f


def test_constraint_basis_matches_reference(golden):
    import sindy
    g = golden("stlsq")
    so2 = torch.tensor([[0.0, 1.0], [-1.0, 0.0]])
    sc2 = torch.diag(torch.tensor([2.0, 1.0]))
    for name, L in (("so2", so2), ("scaling2", sc2)):
        torch.manual_seed(0)
        reg = sindy.SINDyRegression(2, 2, False, False, L_list=[L], threshold=0.05, device="cpu", constrain_constant=True)
        np.testing.assert_allclose(reg.get_M_list()[0].numpy(), g[name + "_M"], atol=1e-6)
        assert int(reg.use_kron_product) == int(g[name + "_kron"])
        # same SVD routine on the same matrix: the same basis up to the sign of each vector, which the LAPACK library
        # chooses differently on different CPUs (MKL on an AMD EPYC host negates so(2)'s first vector against the
        # golden, taken on an Intel host); the same RNG draws on the sign-aligned basis give the same Ξ
        Q, Qr, beta0 = reg.Q.numpy(), g[name + "_Q"], g[name + "_beta0"]
        sign = np.sign((Q * Qr).sum(axis=0))
        np.testing.assert_allclose(Q, Qr * sign, atol=1e-6)
        np.testing.assert_allclose(reg.beta.detach().numpy(), beta0, atol=0)
        np.testing.assert_allclose(reg.const.detach().numpy(), g[name + "_const0"], atol=0)
        # Ξ = Q·β in the equation-major layout of the invertible-generator (Kronecker) form, no constant column
        assert reg.use_kron_product and not reg.allow_constant
        np.testing.assert_allclose((Qr @ beta0).reshape(2, -1), g[name + "_Xi0"], atol=1e-6)
        np.testing.assert_allclose(reg.get_Xi().detach().numpy(), ((Qr * sign) @ beta0).reshape(2, -1), atol=1e-6)
    L3 = torch.tensor([[0.0, 1.0, 0.0], [-1.0, 0.0, 0.0], [0.0, 0.0, 0.0]])
    reg = sindy.SINDyRegression(3, 2, False, False, L_list=[L3], threshold=0.05, device="cpu", constrain_constant=True)
    assert int(reg.use_kron_product) == int(g["sing3_kron"]) == 0
    np.testing.assert_allclose(reg.get_M_list()[0].numpy(), g["sing3_M"], atol=1e-6)
    # null spaces agree (bases may differ by an orthogonal mix when singular values are degenerate)
    Qr, Qo = g["sing3_Q"], reg.Q.numpy()
    assert Qr.shape == Qo.shape
    np.testing.assert_allclose(Qr @ Qr.T, Qo @ Qo.T, atol=1e-4)


def test_symbolic_library_and_its_lie_derivative_matrix():
    """`get_Theta` (reference `sindy.py:147-166`): the SURVEY §8a known answer Θ(2,3,5), and the reference's own route to
    M — J_Θ(z)·L·z expanded in Θ with SymPy (`sindy.py:123-144`) — against the exponent arithmetic used here."""
    import sympy as sp
    import sindy
    reg = sindy.SINDyRegression(3, 3, False, False, threshold=0.05, device="cpu")
    Theta = reg.get_Theta()
    z = sp.symbols("z0 z1 z2")
    vals = [int(v) for v in Theta.subs(dict(zip(z, (2, 3, 5))))]
    assert vals == [1, 2, 3, 5, 4, 6, 10, 9, 15, 25, 8, 12, 20, 18, 30, 50, 27, 45, 75, 125]
    L = torch.tensor([[0.0, 1.0, 0.5], [-1.0, 0.0, 2.0], [-0.5, -2.0, 0.25]])
    M = sindy._lie_derivative_matrix(3, 3, L).double().numpy()
    lhs = Theta.jacobian(sp.Matrix(z)) * sp.Matrix(L.tolist()) * sp.Matrix(z)
    rhs = sp.Matrix(M.tolist()) * Theta
    assert all(sp.expand(a - b).xreplace({n: round(n, 9) for n in sp.expand(a - b).atoms(sp.Float)}) == 0
               for a, b in zip(lhs, rhs))
    assert sindy.SINDyRegression(2, 5, False, False, threshold=0.05, device="cpu").get_Theta().shape == (21, 1)


def test_threshold_and_printer(golden, capsys):
    import sindy
    reg = sindy.SINDyRegression(2, 1, False, False, threshold=0.05, device="cpu", constrain_constant=True)
    reg.Xi.data = torch.tensor([[0.05, 0.0500001, -0.05], [1.0, -1.0, 0.0]])
    reg.set_threshold(0.05)
    assert np.array_equal(reg.mask.numpy(), golden("model")["ka_threshold_mask"])
    reg.print()
    out = capsys.readouterr().out.splitlines()
    assert out == ["dz0 = 0.050*z0 +", "dz1 = 1.000 + -1.000*z0 +"]
    reg = sindy.SINDyRegression(2, 3, True, True, threshold=0.05, device="cpu", constrain_constant=True)
    assert reg.get_term_num() == 14 == reg.Xi.shape[1]
    assert reg.term_names()[8] == "*z0*z1*z1" and reg.term_names()[-1] == "*exp(z1)"
    assert "Xi" in reg.state_dict() and "mask" not in reg.state_dict()


def _feed_stlsq(reg, x, y, w, thr, p):
    """solve_SINDy_one_step's host logic with the Gram sums supplied by the oracle instead of the kernel."""
    import sindy
    s = O.train_step_sums(x, y, np.zeros((y.shape[1], O.term_count(x.shape[1], p))), p)
    G, b = torch.from_numpy(s["gram"]), torch.from_numpy(s["b"])
    return sindy._stlsq_update(reg, G, b, float(w) ** 2, x.shape[0] + G.shape[0], thr)


def test_stlsq_host_logic_reproduces_reference(golden):
    import sindy
    g = golden("stlsq")
    for w in (0.0, 0.3):
        tag = f"selkov_w{int(w * 10)}"
        reg = sindy.SINDyRegression(2, 3, False, False, threshold=0.05, device="cpu", constrain_constant=True)
        reg.reset_mask()
        for it in range(g[tag + "_masks"].shape[0]):
            conv = _feed_stlsq(reg, g["selkov_x"], g["selkov_y"], w, 0.05, 3)
            assert np.array_equal(reg.mask.numpy(), g[tag + "_masks"][it])
            np.testing.assert_allclose(reg.Xi.detach().numpy(), g[tag + "_xis"][it], rtol=0, atol=1e-4 * np.abs(g[tag + "_xis"][it]).max())
        assert conv
    so2 = torch.tensor([[0.0, 1.0], [-1.0, 0.0]])
    sc2 = torch.diag(torch.tensor([2.0, 1.0]))
    for name, L, xk, yk in (("dosc_so2", so2, "dosc_x", "dosc_y"), ("growth_sc2", sc2, "growth_x", "growth_y")):
        for cc in (True, False):
            tag = f"{name}_cc{int(cc)}"
            torch.manual_seed(0)
            reg = sindy.SINDyRegression(2, 2, False, False, L_list=[L], threshold=0.05, device="cpu", constrain_constant=cc)
            for it in range(g[tag + "_masks"].shape[0]):
                _feed_stlsq(reg, g[xk], g[yk], 0.0, 0.05, 2)
                assert np.array_equal(reg.mask.numpy(), g[tag + "_masks"][it]), (tag, it)
                ref = g[tag + "_xis"][it]
                np.testing.assert_allclose(reg.get_Xi().detach().numpy(), ref, rtol=0, atol=2e-4 * np.abs(ref).max())


def test_wsindy_host_logic_reproduces_reference(golden):
    import sindy
    g = golden("wsindy")
    traj, dt, t_max = g["traj"], float(g["dt"]), float(g["t_max"])
    T = traj.shape[0]
    t = torch.arange(T) * dt
    Go, bo = O.wsindy_integrals(traj, dt, t_max, 3)
    for w in (0.05, 0.01):
        tag = f"w{int(w * 100)}"
        reg = sindy.SINDyRegression(2, 3, False, False, threshold=0.075, device="cpu", constrain_constant=True)
        wr = sindy.WSINDyWrapper(reg, t, t_max, device="cpu")
        assert np.array_equal(wr.V[:, ::40].numpy(), g["V"]) and np.array_equal(wr.V_drv[:, ::40].numpy(), g["V_drv"])
        wr.integrals = lambda x: (torch.from_numpy(Go), torch.from_numpy(bo))   # oracle instead of the kernel
        for it in range(g[tag + "_masks"].shape[0]):
            _, conv = wr.solve(torch.from_numpy(traj), w, 0.075)
            assert np.array_equal(reg.mask.numpy(), g[tag + "_masks"][it]), (w, it)
            ref = g[tag + "_xis"][it]
            np.testing.assert_allclose(reg.Xi.detach().numpy(), ref, rtol=0, atol=5e-4 * np.abs(ref).max())
        assert conv


def test_wsindy_rank_deficient_case_reaches_the_reference_equations(golden):
    """w = 0 on the Sel'kov trajectory (config-4 shape): the first solve is rank-deficient by LAPACK's criterion, so
    its coefficients are only loosely comparable (the reference itself is not reproducible there); the masks and
    every later, full-rank iterate coincide with the reference."""
    import sindy
    g = golden("wsindy")
    traj, dt, t_max = g["traj"], float(g["dt"]), float(g["t_max"])
    t = torch.arange(traj.shape[0]) * dt
    Go, bo = O.wsindy_integrals(traj, dt, t_max, 3)
    reg = sindy.SINDyRegression(2, 3, False, False, threshold=0.075, device="cpu", constrain_constant=True)
    # the golden is a CPU run of the reference: LAPACK gelsy's rank rule (the default follows the CUDA driver, gels)
    wr = sindy.WSINDyWrapper(reg, t, t_max, device="cpu", lstsq_driver="gelsy")
    wr.integrals = lambda x: (torch.from_numpy(Go), torch.from_numpy(bo))
    steps = g["w0_masks"].shape[0]
    for it in range(steps):
        _, conv = wr.solve(torch.from_numpy(traj), 0.0, 0.075)
        assert np.array_equal(reg.mask.numpy(), g["w0_masks"][it]), it
        ref = g["w0_xis"][it]
        tol = 5e-2 if it == 0 else 2e-4
        np.testing.assert_allclose(reg.Xi.detach().numpy(), ref, rtol=0, atol=tol * np.abs(ref).max())
    assert conv


def test_badly_scaled_library_keeps_its_small_directions():
    """Raw-unit Lorenz data (x, y ~ 8, z ~ 24), cubic library, 2·10^4 samples: cond(Θ) ~ 2·10^5. The default solve
    (equilibrated, no rank decision — what the reference's CUDA driver `gels` does) recovers the planted equations to
    1e-4; LAPACK gelsy's rank rule at this row count (relative cut 2.4e-3) drops the small directions and loses them,
    which is why it is opt-in."""
    import sindy
    rng = np.random.default_rng(3)
    n = 20_000
    x = np.stack([8 * rng.standard_normal(n), 8 * rng.standard_normal(n), 24 + 8 * rng.standard_normal(n)], 1)
    x = x.astype(np.float32)
    truth = np.zeros((3, 20))
    truth[0, 1], truth[0, 2] = -10.0, 10.0
    truth[1, 1], truth[1, 2], truth[1, 6] = 28.0, -1.0, -1.0
    truth[2, 3], truth[2, 5] = -8.0 / 3.0, 1.0
    y = (O.theta(x.astype(np.float64), 3) @ truth.T).astype(np.float32)
    errs = {}
    for driver in ("gels", "gelsy"):
        reg = sindy.SINDyRegression(3, 3, False, False, threshold=0.05, device="cpu", constrain_constant=True)
        reg.reset_mask()
        s = O.train_step_sums(x, y, np.zeros((3, 20)), 3)
        G, b = torch.from_numpy(s["gram"]), torch.from_numpy(s["b"])
        for _ in range(5):
            if sindy._stlsq_update(reg, G, b, 0.0, n + 20, 0.05, driver):
                break
        coef = (reg.Xi.detach() * reg.mask).numpy()
        errs[driver] = (np.abs(coef - truth).max(), np.array_equal(coef != 0, truth != 0))
    assert errs["gels"][1] and errs["gels"][0] < 1e-4 * 28.0, errs
    assert not errs["gelsy"][1], errs


def test_python_right_hand_sides_are_identified_as_library_members():
    """The reference's generators pass Python callables to solve_ode_batch (`damped_oscillator.py:20-24`,
    `growth.py:18-22`, `lotka.py:33-41`, `selkov.py:18-22`, restated here): each is recognised as Θ(x)·Ξᵀ with the
    coefficients of data_utils/systems.py (= the truth tables of `evaluation/eval_eq.py:88-105`)."""
    from data_utils import ode, systems

    def dosc(x, a=0.1, **kw):
        return np.stack([-a * x[..., 0] - x[..., 1], x[..., 0] - a * x[..., 1]], -1)

    def growth(x, a=0.1, b=0.3, **kw):
        return np.stack([a * x[..., 1] ** 2 - b * x[..., 0], x[..., 1]], -1)

    def lotka_volterra(x, a=2 / 3, b=4 / 3, c=1.0, d=1.0, **kw):
        return np.stack([a - b * np.exp(x[..., 1]), c * np.exp(x[..., 0]) - d], -1)

    def selkov(x, a=0.75, b=0.1, c=0.1, **kw):
        return np.stack([a - b * x[..., 0] - x[..., 0] * x[..., 1] ** 2,
                         -x[..., 1] + c * x[..., 0] + x[..., 0] * x[..., 1] ** 2], -1)

    rng = np.random.default_rng(0)
    for fn, name, x0 in ((dosc, "dosc", rng.uniform(-2, 2, (50, 2))), (growth, "growth", rng.uniform(0.1, 1, (50, 2))),
                         (lotka_volterra, "lv", np.log(rng.uniform(0.2, 1, (50, 2)))),
                         (selkov, "selkov", rng.uniform(0.5, 1, (10, 2)))):
        got = ode.identify_library_ode(fn, x0, gp_sigma_in=0.1)
        want = systems.SYSTEMS[name]()
        assert got.library == want.library, (name, got.library)
        assert np.abs(got.Xi - want.Xi).max() < 1e-13, (name, np.abs(got.Xi - want.Xi).max())
    shifted = ode.identify_library_ode(dosc, rng.uniform(-2, 2, (50, 2)), a=0.25)      # kwargs reach the callable
    assert abs(shifted.Xi[0, 1] + 0.25) < 1e-13
    with pytest.raises(TypeError):
        ode.identify_library_ode(lambda x: np.tanh(x), rng.uniform(-1, 1, (8, 2)))


def test_launcher_puts_the_hot_path_modules_first(tmp_path):
    """`python <reference>/main.py` with PYTHONPATH resolves `sindy` to the reference (the script's directory comes
    first); the launcher must resolve the hot-path modules to this repo and everything else to the reference (a
    stand-in tree with the reference's module names)."""
    import subprocess
    import sys
    import config_runs
    import standins
    ref = standins.make_reference_tree(str(tmp_path / "reference"))
    res = subprocess.run([sys.executable, config_runs.LAUNCHER, "--reference", ref, "--where"], capture_output=True,
                         text=True, timeout=600, cwd=str(tmp_path))
    assert res.returncode == 0, res.stderr[-2000:]
    table = dict(line.split(None, 1) for line in res.stdout.strip().splitlines())
    pkg = config_runs.PKG
    for name in ("sindy", "model_utils", "train", "data_utils.ode", "data_utils.smoothing"):
        assert table[name].strip().startswith(pkg), (name, table[name])
    for name in ("data_utils.lotka", "data_utils.selkov", "data_utils.growth", "data_utils.damped_oscillator",
                 "dataset", "parser_utils", "gan", "autoencoder", "evaluation.eval_eq"):
        assert table[name].strip().startswith(ref), (name, table[name])
    # train_lassi (outside the hot path) is re-exported from the reference so that `main.py:90-91` keeps resolving
    res = subprocess.run([sys.executable, "-c", "import sys; sys.path[:0] = [%r, %r]; import train; "
                          "print(train.train_lassi.__module__, 'train_lassi' in train.__all__)" % (pkg, ref)],
                         capture_output=True, text=True, timeout=600, cwd=str(tmp_path))
    assert res.returncode == 0 and res.stdout.split() == ["_sindy_b200_reference_train", "True"], res.stdout + res.stderr


@pytest.mark.parametrize("constrained", [False, True])
def test_batched_seed_sweep_equals_the_serial_sweep(constrained):
    """All seeds as ONE batched LBFGS problem (SURVEY §8f-4) against the seed-after-seed sweep (torch.optim.LBFGS per
    seed through train_SIGED_lbfgs(cached_gram=True)): same masks, coefficients to 1e-3 of the largest (the loop's own
    stopping tolerance). Host logic only: the sufficient statistics come from the oracle instead of the kernel."""
    import sindy
    import sweep
    rng = np.random.default_rng(11)
    n = 4000
    x = rng.uniform(-1.5, 1.5, (n, 2)).astype(np.float32)
    truth = np.array([[0, -0.1, -1, 0, 0, 0], [0, 1, -0.1, 0, 0, 0.0]])
    dx = (O.theta(x.astype(np.float64), 2) @ truth.T + 0.05 * rng.standard_normal((n, 2))).astype(np.float32)
    xt, dxt = torch.from_numpy(x), torch.from_numpy(dx)
    L = [torch.tensor([[0.0, 1.0], [-1.0, 0.0]])] if constrained else []

    def stats_of(xb, dxb):
        s = O.train_step_sums(xb.numpy(), dxb.numpy(), np.zeros((2, 6)), 2)
        return {"G": torch.from_numpy(s["gram"]), "b": torch.from_numpy(s["b"]),
                "yy": torch.tensor((dxb.double() ** 2).sum()), "n": float(xb.shape[0])}

    def make():
        reg = sindy.SINDyRegression(2, 2, False, False, L_list=L, threshold=0.05, device="cpu", constrain_constant=False)
        reg.sufficient_statistics = stats_of
        return reg

    seeds = list(range(6))
    serial = sweep.run_seed_sweep(xt, dxt, truth, seeds, make, subsample=0.5, lr_sindy=0.1, st_freq=50, threshold=0.05,
                                  num_epochs=60)
    batched = sweep.run_seed_sweep_batched(xt, dxt, truth, seeds, make, subsample=0.5, lr_sindy=0.1, st_freq=50,
                                           threshold=0.05, num_epochs=60)
    for a, b in zip(serial, batched):
        assert a["seed"] == b["seed"]
        assert np.array_equal(a["coefficients"] != 0, b["coefficients"] != 0), (a["coefficients"], b["coefficients"])
        assert np.abs(a["coefficients"] - b["coefficients"]).max() < 1e-3 * np.abs(a["coefficients"]).max()
    assert sum(r["correct_form_all"] for r in batched) >= 4


def test_lstsq_driver_selection(monkeypatch):
    import sindy
    assert sindy._lstsq_driver({}) == "gels"
    monkeypatch.setenv("SINDY_B200_LSTSQ", "gelsy")
    assert sindy._lstsq_driver({}) == "gelsy" and sindy._lstsq_driver({"lstsq_driver": "gels"}) == "gels"
    with pytest.raises(ValueError):
        sindy._lstsq_driver({"lstsq_driver": "svd"})


def test_odeint_python_path_and_errors():
    import model_utils
    f = lambda x: -x
    x0 = torch.ones(4, 2)
    out = model_utils.odeint(f, x0, 0.3, 0.1, method='euler')           # int(0.3/0.1) == 2 steps
    assert torch.allclose(out, torch.full((4, 2), 0.81))
    tr = model_utils.odeint(f, x0, 1.0, 0.1, method='rk4', full_traj=True)
    assert tr.shape == (10, 4, 2) and abs(float(tr[-1, 0, 0]) - np.exp(-1.0)) < 1e-6
    with pytest.raises(ValueError):
        model_utils.odeint(f, x0, 1.0, 0.1, method='midpoint')


def test_systems_match_truth_tables(golden):
    from data_utils import systems
    g = golden("model")
    for name in ("dosc", "growth", "lv", "selkov"):
        assert np.allclose(systems.SYSTEMS[name]().Xi, g["truth_" + name])


def test_lie_regulariser_quadratic_form_equals_gram_form():
    """symreg.quadratic_form: wᵀHw and 2Hw reproduce Σ_v tr(A_v G A_vᵀ), A_v = W M_v − v W, and its gradient
    (`train.py:503-507`, intended formula) — host-side algebra, no GPU."""
    import torch
    from sindy_b200 import native, symreg
    for (d, p) in ((2, 3), (3, 3)):
        lib = native.Library(d, p)
        K = lib.K
        g = torch.Generator().manual_seed(d * 10 + p)
        A = torch.randn(300, K, dtype=torch.float64, generator=g)
        G = A.T @ A
        W = torch.randn(d, K, dtype=torch.float64, generator=g).requires_grad_(True)
        gens = [torch.randn(d, d, dtype=torch.float64, generator=g) for _ in range(3)]
        Ms = [symreg.lie_matrix(lib, v) for v in gens]
        loss = symreg.lie_loss_from_gram(G, W, gens, Ms)
        loss.backward()
        H = symreg.quadratic_form(lib, gens, G)
        w = W.detach().reshape(-1)
        assert torch.equal(H, H.T)
        assert abs(float(w @ H @ w) - float(loss.detach())) <= 1e-12 * float(loss.detach())
        assert float((2 * H @ w - W.grad.reshape(-1)).abs().max()) <= 1e-12 * float(W.grad.abs().max())


def test_fit_step_argument_validation_without_a_device():
    """sb_fit_step / sb_load_w reject bad arguments with a status and a message before touching CUDA."""
    from sindy_b200 import native
    lib = native.load()
    L = native._CLibrary(3, 5, 0, 0)
    opt = native._CFitOptions(native.SB_OPT_ADAM, 1e-3, 0.9, 0.999, 1e-8, 1.0, 0.0, 0.0, None)
    one = ctypes.c_void_p(16)   # a non-NULL, 16-byte aligned dummy address: validation never dereferences it

    def call(x=one, dx=one, n=8, xi=one, o=ctypes.byref(opt), state=one, packed=one, ws=one, world=1, flags=0):
        return lib.sb_fit_step(x, dx, n, ctypes.byref(L), xi, None, o, state, packed, one, one, ws, 1 << 20, None, world,
                               0, None, flags, None)

    assert call(x=None) == -1 and b"x is NULL" in lib.sb_last_error()
    assert call(o=None) == -1 and b"opt" in lib.sb_last_error()
    assert call(state=None) == -1 and b"opt_state" in lib.sb_last_error()
    assert call(flags=2) == -1 and b"call_flags" in lib.sb_last_error()
    assert call(n=-1) == -1
    assert call(world=2) == -1 and b"peer_bufs" in lib.sb_last_error()
    bad = native._CFitOptions(7, 1e-3, 0.9, 0.999, 1e-8, 1.0, 0.0, 0.0, None)
    assert call(o=ctypes.byref(bad)) == -1 and b"optimiser" in lib.sb_last_error()
    assert call(x=ctypes.c_void_p(20)) == -2 and b"aligned" in lib.sb_last_error()       # misaligned input
    Lg = native._CLibrary(2, 2, 1, 0)                                                    # sine columns: no fused kernel
    assert lib.sb_load_w(ctypes.byref(Lg), one, None, None) == -2
    assert lib.sb_load_w(ctypes.byref(L), None, None, None) == -1


def test_c_consumer_links_and_validates(tmp_path):
    """include/sindy_b200.h is a C header and libsindy_b200.so a C-ABI library: a gcc-compiled C program links it,
    queries the library tables and gets status codes (no C++ exception, no crash) for bad arguments — no GPU needed."""
    import shutil
    import subprocess
    from sindy_b200 import native
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    native.load()
    exe = str(tmp_path / "abi_smoke")
    libdir = os.path.dirname(native.LIB_PATH)
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "c", "abi_smoke.c"), "-o", exe, "-L", libdir, "-lsindy_b200",
                    f"-Wl,-rpath,{libdir}"], check=True)
    res = subprocess.run([exe], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "c abi ok" in res.stdout


def test_sweep_metrics_follow_eval_eq():
    """sweep.evaluate / sweep.aggregate restate `evaluation/eval_eq.py:7-85`: correct form = mask equals the truth's
    support, MSE over the truth's non-zeros, RMSE mean (std) over successful runs and over all runs."""
    import sweep

    class Reg:
        constraint = False

        def __init__(self, Xi, mask):
            self.Xi, self.mask = torch.tensor(Xi, dtype=torch.float32), torch.tensor(mask, dtype=torch.float32)

    truth = np.array([[0.0, -0.1, -1.0, 0.0, 0.0, 0.0], [0.0, 1.0, -0.1, 0.0, 0.0, 0.0]])
    good = Reg([[0.3, -0.11, -1.02, 0, 0, 0], [0, 0.98, -0.1, 0, 0, 0.5]], [[0, 1, 1, 0, 0, 0], [0, 1, 1, 0, 0, 0]])
    bad = Reg([[0.0, -0.2, -1.0, 0.4, 0, 0], [0, 1.0, -0.1, 0, 0, 0]], [[0, 1, 1, 1, 0, 0], [0, 1, 1, 0, 0, 0]])
    rg, rb = sweep.evaluate(good, truth), sweep.evaluate(bad, truth)
    assert rg["correct_form"].tolist() == [1.0, 1.0] and rg["correct_form_all"]
    assert rb["correct_form"].tolist() == [0.0, 1.0] and not rb["correct_form_all"]
    np.testing.assert_allclose(rg["mse"], [((0.01) ** 2 + (0.02) ** 2) / 2, (0.02 ** 2) / 2], rtol=1e-5)
    np.testing.assert_allclose(rb["mse"], [(0.1 ** 2) / 2, 0.0], atol=1e-9)
    assert rg["coefficients"][0, 0] == 0.0 and rg["coefficients"][1, 5] == 0.0      # masked entries are reported as 0
    agg = sweep.aggregate([rg, rb, rg], mse_multiplier=10.0, verbose=False)
    assert agg["runs"] == 3 and agg["success"].tolist() == [2, 3] and agg["success_all"] == 2
    r0 = np.sqrt([rg["mse"][0], rb["mse"][0], rg["mse"][0]])
    np.testing.assert_allclose(agg["rmse"][0], (10 * r0[[0, 2]].mean(), 10 * r0[[0, 2]].std()), rtol=1e-6, atol=1e-12)
    np.testing.assert_allclose(agg["rmse_any"][0], (10 * r0.mean(), 10 * r0.std()), rtol=1e-6)
    ra = np.sqrt([rg["mse_all"], rb["mse_all"], rg["mse_all"]])
    np.testing.assert_allclose(agg["rmse_all_any"], (10 * ra.mean(), 10 * ra.std()), rtol=1e-6)


@pytest.mark.parametrize("d,p", [(2, 2), (2, 3), (3, 3), (3, 5), (4, 2)])
def test_lie_derivative_matrix_is_the_jacobian_identity(d, p):
    """a13 / a5: the constant matrix M with J_Θ(z)·(L z) = M·Θ(z) (the reference derives it symbolically with SymPy,
    `sindy.py:123-144`; here exponent arithmetic) checked numerically against the oracle's Jacobian of Θ for random
    generators — for the constraint set-up (`sindy._lie_derivative_matrix`) and the regulariser (`symreg.lie_matrix`)."""
    import sindy
    from sindy_b200 import native, symreg
    rng = np.random.default_rng(d * 10 + p)
    L = rng.standard_normal((d, d))
    z = rng.uniform(-1.2, 1.2, (64, d))
    lhs = np.einsum("nkj,nj->nk", O.dtheta(z, p), z @ L.T)
    th = O.theta(z.astype(np.float64), p).astype(np.float64)
    M1 = sindy._lie_derivative_matrix(d, p, torch.tensor(L)).double().numpy()
    M2 = symreg.lie_matrix(native.Library(d, p), torch.tensor(L)).numpy()
    np.testing.assert_allclose(th @ M1.T, lhs, rtol=2e-5, atol=2e-5)     # M1 is stored in fp32 like the reference's
    np.testing.assert_allclose(th @ M2.T, lhs, rtol=1e-10, atol=1e-10)


def test_frozen_autoencoder_folding_reproduces_the_module():
    """`sindy_b200.mlp.fold_layers` (host side of the tensor-core MLP chain, §8f-3): the Linear / BatchNorm(eval) / ReLU
    tree of the reference's AutoEncoder (`autoencoder.py:38-66`) folded to plain (W, b) layers evaluates to the module's
    own output; other module trees are refused."""
    import torch
    from sindy_b200 import mlp
    from test_gpu_mlp import RefShapedAutoEncoder
    torch.manual_seed(0)
    ae = RefShapedAutoEncoder(hidden=64).double()
    with torch.no_grad():
        for m in ae.modules():
            if isinstance(m, torch.nn.BatchNorm1d):
                m.running_mean.normal_(0, 0.1); m.running_var.uniform_(0.5, 1.5)
                m.weight.normal_(1.0, 0.2); m.bias.normal_(0, 0.1)
    assert mlp.fold_layers(ae.encoder) is None                       # trainable parameters
    for p in ae.parameters():
        p.requires_grad_(False)
    assert mlp.fold_layers(ae.encoder) is None                       # training mode: batch statistics
    ae.eval()
    x = torch.randn(37, 2, 2, dtype=torch.float64)
    for mod in (ae.encoder, ae.decoder):
        layers, out_shape = mlp.fold_layers(mod)
        h = x.reshape(-1, 2)
        for i, (w, b) in enumerate(layers):
            h = h @ w.t() + b
            if i + 1 < len(layers):
                h = h.clamp_min(0)
        want = mod(x)
        assert out_shape in (None, (-1, 2, 2))
        assert torch.allclose(h.reshape(want.shape), want, rtol=1e-12, atol=1e-13)
    assert mlp.accelerate(ae) is None                                # CPU module: the PyTorch path stays
    ae.decoder[1] = torch.nn.Tanh()
    assert mlp.fold_layers(ae.decoder) is None


def test_batched_masked_solve_equals_the_block_diagonal_system():
    """`sindy._masked_solve_batched` (d eigenproblems of size K, masked rows/columns zeroed) against the formulation it
    replaces — one min-norm solve of the block-diagonal system (I_d ⊗ H)[m, m] — for both rank rules, full masks, ragged
    masks, an empty equation and an exactly singular Gram."""
    import torch
    import sindy
    g = torch.Generator().manual_seed(0)
    d, K = 3, 20
    A = torch.randn(400, K, dtype=torch.float64, generator=g) * torch.logspace(-2, 2, K, dtype=torch.float64)
    A[:, 7] = A[:, 3] * 2.0                                              # exactly dependent columns
    H = A.T @ A
    b = A.T @ torch.randn(400, d, dtype=torch.float64, generator=g)
    masks = [torch.ones(d, K, dtype=torch.bool), torch.rand(d, K, generator=g) > 0.4, torch.rand(d, K, generator=g) > 0.8]
    masks[2][1] = False                                                  # an equation with no live column
    for mask in masks:
        for rcond in (0.0, 2e-3):
            got = sindy._masked_solve_batched(H, b, mask, rcond)
            if bool(mask.all()):
                want = sindy._min_norm_solve(H, b, rcond).T
            else:
                idx = torch.nonzero(mask.flatten()).flatten()
                eq, col = idx // K, idx % K
                Hm = H[col][:, col] * (eq.unsqueeze(1) == eq.unsqueeze(0)).to(H.dtype)
                sol = sindy._min_norm_solve(Hm, b.T.reshape(-1)[idx], rcond)
                want = torch.zeros(d * K, dtype=torch.float64)
                want[idx] = sol
                want = want.view(d, K)
            assert torch.equal(got != 0, want != 0) or bool(((got != 0) <= mask).all())
            assert float((got - want).abs().max()) <= 1e-9 * float(want.abs().max().clamp_min(1e-30)), (rcond, mask.sum())


def test_launcher_seed_loop_runs_the_script_once_per_seed_in_one_process(tmp_path):
    """`run.py --seeds 3-5,9 script.py --x 1` executes the script four times in ONE interpreter with `--seed k` appended
    (the replacement for run_scripts/*.sh's 50 interpreter starts)."""
    import subprocess
    import sys
    import standins
    ref = standins.make_reference_tree(str(tmp_path / "reference"))
    script = tmp_path / "probe.py"
    script.write_text("import os, sys\nprint('RUN', os.getpid(), sys.argv[1:])\n")
    launcher = os.path.join(ROOT, "symmetry-ode-discovery_b200", "sindy_b200", "run.py")
    out = subprocess.run([sys.executable, launcher, "--reference", ref, "--seeds", "3-5,9", str(script), "--x", "1"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    runs = [l for l in out.stdout.splitlines() if l.startswith("RUN")]
    assert [r.split(" ", 2)[2] for r in runs] == [str(["--x", "1", "--seed", str(k)]) for k in (3, 4, 5, 9)]
    assert len({r.split()[1] for r in runs}) == 1
