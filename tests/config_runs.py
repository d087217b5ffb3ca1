"""Runs the reference's UNMODIFIED entry points (`main.py`, `main_wsindy.py`) with the four BASELINE cfg files.

TEST INFRASTRUCTURE shared by `oracle/gen_config_golden.py` (reference alone, CPU, in the build container -> goldens)
and `tests/test_gpu_configs.py` (the same entry points through the drop-in launcher `sindy_b200/run.py` on the B200).
Every run happens in a scratch work directory laid out the way the reference expects (SURVEY §8c):

    <work>/run_configs -> <reference>/run_configs        (cfg files verbatim, `parser_utils.py:5`)
    <work>/data/<ode>-<split>-noiseNN-gp-{x,dx}.pt        (copied from tests/golden/data, `dataset.py:14,170-200`)
    <work>/saved_models/laligan-noise99-lv/               (C3 only: seeded frozen stand-in, see make_laligan_standin)

and leaves `<work>/eval_results/<save_dir>/seed<k>.npz` (`main.py:120-138`) and `saved_models/<save_dir>/regressor.pt`.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "symmetry-ode-discovery_b200")
LAUNCHER = os.path.join(PKG, "sindy_b200", "run.py")
DATA = os.path.join(ROOT, "tests", "golden", "data")

# key: entry script, cfg (relative to run_configs/), data files' ode name, save_dir of the cfg, CLI overrides
CONFIGS = {
    "C1": dict(script="main.py", cfg="dosc/noise20_sindy.cfg", ode="dosc", save_dir="sindy-noise20-dosc", extra=[]),
    "C2": dict(script="main.py", cfg="growth/noise05_esindy.cfg", ode="growth", save_dir="esindy-noise05-growth",
               extra=[]),
    # the LV data fixture is 16 x 2000 samples instead of 200 x 10^4 (oracle/gen_config_data.py): the subsample
    # fraction is raised so that the closure still sees a few thousand samples (cfg: 0.01 of 2e6 = 20 000)
    "C3": dict(script="main.py", cfg="lv/noise99_eq_isymreg.cfg", ode="lv", save_dir="symreg2-noise99-lv",
               extra=["--lbfgs_subsample", "0.1", "--num_epochs", "30"]),
    "C4": dict(script="main_wsindy.py", cfg="selkov/noise20_eq_wsindy.cfg", ode="selkov",
               save_dir="wsindy-noise20-selkov", extra=[]),
    # extra coverage of the same entry points: EquivSINDy-c on dosc (so2 constraint) and weak SINDy on dosc / growth
    "C1e": dict(script="main.py", cfg="dosc/noise20_esindy.cfg", ode="dosc", save_dir="esindy-noise20-dosc", extra=[]),
    "C1w": dict(script="main_wsindy.py", cfg="dosc/noise20_wsindy.cfg", ode="dosc", save_dir="wsindy-noise20-dosc",
                extra=[]),
    "C2s": dict(script="main.py", cfg="growth/noise05_sindy.cfg", ode="growth", save_dir="sindy-noise05-growth",
                extra=[]),
}


def find_reference():
    for c in (os.environ.get("SINDY_B200_REFERENCE"), os.path.join(ROOT, "oracle", "_ref")):
        if c and os.path.isfile(os.path.join(c, "main.py")) and os.path.isfile(os.path.join(c, "sindy.py")):
            return os.path.abspath(c)
    return None


def _env(extra=None):
    env = dict(os.environ)
    env["WANDB_MODE"] = "disabled"
    env.pop("PYTHONPATH", None)
    env.update(extra or {})
    return env


_STANDIN = r"""
import sys, os, torch
sys.argv = ['main.py', '--config', 'lv/noise99_eq_isymreg.cfg', '--gpu', '-1']
from parser_utils import get_args
from autoencoder import AutoEncoder
from gan import LieGenerator
args = vars(get_args()); args['input_dim'] = 2
torch.manual_seed(20240516)
ae = AutoEncoder(**args); gen = LieGenerator(**args)
g = torch.Generator().manual_seed(7)
with torch.no_grad():                      # a BatchNorm that is not the identity: seeded statistics and affine part
    for m in ae.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.running_mean.copy_(0.1 * torch.randn(m.running_mean.shape, generator=g))
            m.running_var.copy_(1.0 + 0.2 * torch.rand(m.running_var.shape, generator=g))
            m.weight.copy_(1.0 + 0.1 * torch.randn(m.weight.shape, generator=g))
            m.bias.copy_(0.1 * torch.randn(m.bias.shape, generator=g))
out = 'saved_models/laligan-noise99-lv'; os.makedirs(out, exist_ok=True)
torch.save(ae.state_dict(), out + '/autoencoder.pt')
torch.save(gen.state_dict(), out + '/generator.pt')
torch.save([None if m is None else m.cpu() for m in gen.masks], out + '/generator_mask.pt')
print('stand-in LaLiGAN checkpoint written:', sum(p.numel() for p in ae.parameters()), 'autoencoder parameters')
"""


def make_laligan_standin(work, reference):
    """C3 loads `saved_models/laligan-noise99-lv/{autoencoder,generator,generator_mask}.pt` (`main.py:47-63`), which the
    reference does not ship (it is the output of `lv/noise99_sym.cfg`). SURVEY §8c: replaced for parity purposes by a
    seeded, randomly initialised, FROZEN autoencoder + generator built from the reference's own classes with the cfg's
    arguments on the CPU generator (identical bits on every machine of this image) — same arithmetic, same shapes."""
    res = subprocess.run([sys.executable, "-c", _STANDIN], cwd=work, env=_env({"PYTHONPATH": reference}),
                         capture_output=True, text=True, timeout=600)
    if res.returncode != 0:
        raise RuntimeError("stand-in LaLiGAN checkpoint failed:\n" + res.stdout[-2000:] + res.stderr[-2000:])


def prepare_workdir(work, reference, key):
    cfg = CONFIGS[key]
    os.makedirs(os.path.join(work, "data"), exist_ok=True)
    link = os.path.join(work, "run_configs")
    if not os.path.exists(link):
        os.symlink(os.path.join(reference, "run_configs"), link)
    for f in os.listdir(DATA):
        if f.startswith(cfg["ode"] + "-"):
            shutil.copy(os.path.join(DATA, f), os.path.join(work, "data", f))
    if key == "C3" and not os.path.exists(os.path.join(work, "saved_models", "laligan-noise99-lv", "autoencoder.pt")):
        make_laligan_standin(work, reference)


def run_entry(key, work, reference, dropin, gpu, seed=0, reference_train=False, env=None, timeout=3600):
    """One run of the cfg's entry point. dropin=False: `python <reference>/<script>` (the reference alone);
    dropin=True: the same script through the launcher, i.e. on this repo's sindy / model_utils / train / data_utils."""
    cfg = CONFIGS[key]
    prepare_workdir(work, reference, key)
    script = os.path.join(reference, cfg["script"])
    args = ["--seed", str(seed), "--config", cfg["cfg"], "--gpu", str(gpu)] + cfg["extra"]
    if dropin:
        cmd = [sys.executable, LAUNCHER, "--reference", reference] + (["--reference-train"] if reference_train else [])
        cmd += [script] + args
    else:
        cmd = [sys.executable, script] + args
    res = subprocess.run(cmd, cwd=work, env=_env(env), capture_output=True, text=True, timeout=timeout)
    if res.returncode != 0:
        raise RuntimeError(f"{' '.join(cmd)} failed ({res.returncode}):\n{res.stdout[-3000:]}\n{res.stderr[-3000:]}")
    return collect(key, work, seed), res.stdout


def collect(key, work, seed=0):
    """Masked coefficients (`eval_sindy_regressor`: Ξ where the mask is set, 0 elsewhere), the reference's own metrics
    and the raw parameters of the saved state dict."""
    import torch
    cfg = CONFIGS[key]
    ev = np.load(os.path.join(work, "eval_results", cfg["save_dir"], f"seed{seed}.npz"))
    out = {"coefficients": ev["coefficients"], "correct_form": ev["correct_form"], "mse": ev["mse"]}
    sd = torch.load(os.path.join(work, "saved_models", cfg["save_dir"], "regressor.pt"), map_location="cpu")
    for k, v in sd.items():
        out["param_" + k] = v.numpy()
    return out
