"""Launcher that runs the reference's UNMODIFIED entry points on top of the B200 modules.

    python <repo>/symmetry-ode-discovery_b200/sindy_b200/run.py <reference>/main.py --config dosc/noise20_sindy.cfg --gpu 0
    python <repo>/symmetry-ode-discovery_b200/sindy_b200/run.py -m data_utils.damped_oscillator --n_ics 50 --noise 0.2
    python -m sindy_b200.run --where                         (with the package directory on PYTHONPATH)

Why a launcher and not `PYTHONPATH`: Python puts the directory of the script it runs at `sys.path[0]`, AHEAD of
`PYTHONPATH`, so `PYTHONPATH=<this repo>:<reference> python <reference>/main.py` silently imports the reference's own
`sindy.py` / `train.py` / `model_utils.py`. Here the script is executed with `runpy`, which leaves `sys.path` alone, after
this repo's module directory has been put first and the reference's directory second:

  * `sindy`, `model_utils`, `train`, `data_utils.ode`, `data_utils.smoothing` resolve to this repo (CUDA path);
  * `data_utils.damped_oscillator / growth / lotka / selkov` fall through to the reference (`data_utils/__init__.py`
    of this repo extends its `__path__`), as do `gan`, `autoencoder`, `model`, `dataset`, `parser_utils`, `utils`,
    `evaluation` — the parts of the reference outside the hot path (`main.py:9-15`, `dataset.py:12`).

Options (before the script): `--reference DIR` (default: the script's directory, else $SINDY_B200_REFERENCE, else
<repo>/oracle/_ref), `--reference-train` (keep the reference's own `train.py`: its loops then run operator by operator
on this repo's `sindy` / `model_utils` through autograd), `--where` (print where the hot-path modules resolve, and exit),
`--seeds A-B[,C...]` (run the script once per seed IN THIS PROCESS with `--seed k` appended: what `run_scripts/*.sh` does
with one interpreter start — ≈8 s of imports and CUDA start-up — per seed; any cfg, the runs stay independent and write
the same `eval_results/<save_dir>/seed<k>.npz`; `sweep_main.py` goes further for the cfgs it can batch).
"""
from __future__ import annotations

import importlib
import importlib.util
import os
import runpy
import sys

PKG_DIR = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))       # .../symmetry-ode-discovery_b200
REPO_DIR = os.path.dirname(PKG_DIR)
HOT_MODULES = ("sindy", "model_utils", "train", "data_utils", "data_utils.ode", "data_utils.smoothing")
REFERENCE_MODULES = ("data_utils.damped_oscillator", "data_utils.growth", "data_utils.lotka", "data_utils.selkov",
                     "dataset", "parser_utils", "gan", "autoencoder", "evaluation.eval_eq")


def _looks_like_reference(path):
    return bool(path) and os.path.isfile(os.path.join(path, "sindy.py")) and os.path.isfile(
        os.path.join(path, "data_utils", "lotka.py"))


def find_reference(explicit=None, script=None):
    """Directory of the reference checkout: --reference, the script's own directory, $SINDY_B200_REFERENCE,
    <repo>/oracle/_ref, an entry of sys.path — in that order."""
    cands = [explicit, os.path.dirname(os.path.abspath(script)) if script else None,
             os.environ.get("SINDY_B200_REFERENCE"), os.path.join(REPO_DIR, "oracle", "_ref")]
    cands += [p for p in sys.path if p and os.path.abspath(p) != PKG_DIR]
    for c in cands:
        if _looks_like_reference(c):
            return os.path.abspath(c)
    return None


def arrange_path(reference):
    """sys.path = [this repo's modules, the reference, everything else]; stale imports of the shared names dropped."""
    here = os.path.dirname(os.path.abspath(__file__))
    drop = {PKG_DIR, here, os.path.abspath(reference) if reference else None}
    rest = [p for p in sys.path if os.path.abspath(p or os.getcwd()) not in drop]
    sys.path[:] = [PKG_DIR] + ([os.path.abspath(reference)] if reference else []) + rest
    if reference:
        os.environ["SINDY_B200_REFERENCE"] = os.path.abspath(reference)
    for name in list(sys.modules):
        root = name.split(".")[0]
        if root in ("sindy", "model_utils", "train", "data_utils", "dataset", "utils", "model", "gan", "autoencoder",
                    "parser_utils", "evaluation"):
            del sys.modules[name]
    importlib.invalidate_caches()


def where(names=HOT_MODULES + REFERENCE_MODULES):
    """{module name: file it resolves to (or the import error)} without importing CUDA work."""
    out = {}
    for name in names:
        try:
            mod = importlib.import_module(name)
            out[name] = getattr(mod, "__file__", None) or str(getattr(mod, "__path__", "?"))
        except Exception as exc:  # noqa: BLE001  (reported, not swallowed)
            out[name] = f"ERROR {type(exc).__name__}: {exc}"
    return out


def use_reference_train(reference):
    """Bind the module name `train` to the reference's own train.py (its `from sindy import *` / `from model_utils
    import *` still resolve to this repo)."""
    spec = importlib.util.spec_from_file_location("train", os.path.join(reference, "train.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules["train"] = mod
    spec.loader.exec_module(mod)
    return mod


def parse_seeds(spec):
    """'0-49', '3', '0-4,10,20-22' -> list of ints."""
    out = []
    for part in spec.split(","):
        lo, _, hi = part.partition("-")
        out.extend(range(int(lo), int(hi or lo) + 1))
    return out


def main(argv=None):
    argv = list(sys.argv[1:] if argv is None else argv)
    reference, ref_train, show = None, False, False
    seeds = None
    while argv and argv[0] in ("--reference", "--reference-train", "--where", "--seeds"):
        opt = argv.pop(0)
        if opt == "--reference":
            reference = argv.pop(0)
        elif opt == "--reference-train":
            ref_train = True
        elif opt == "--seeds":
            seeds = parse_seeds(argv.pop(0))
        else:
            show = True
    as_module = bool(argv) and argv[0] == "-m"
    if as_module:
        argv.pop(0)
    if not argv and not show:
        print(__doc__)
        return 2
    target = argv[0] if argv else None
    reference = find_reference(reference, None if (as_module or target is None) else target)
    if reference is None:
        print("sindy_b200.run: no reference checkout found (pass --reference DIR or set SINDY_B200_REFERENCE)",
              file=sys.stderr)
        return 2
    arrange_path(reference)
    os.environ.setdefault("WANDB_MODE", "disabled")
    if show:
        for name, path in where().items():
            print(f"{name:32s} {path}")
        if target is None:
            return 0
    if ref_train:
        use_reference_train(reference)
    for seed in (seeds if seeds is not None else [None]):
        sys.argv = [target] + argv[1:] + ([] if seed is None else ["--seed", str(seed)])
        if as_module:
            runpy.run_module(target, run_name="__main__", alter_sys=True)
        else:
            runpy.run_path(target, run_name="__main__")
    return 0


if __name__ == "__main__":
    sys.exit(main())
