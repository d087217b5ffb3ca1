"""Model selection along the STLSQ threshold path on the golden growth/noise05 and dosc/noise20 data: stlsq_path on
the training set over logspace(-3, 0, 40), score_path on the validation set (RK4 with dt = 0.002 between samples
10 resp. 100 steps apart), and the table of distinct candidates ranked by AICc with the true support marked.

  python tools/select_model.py
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "symmetry-ode-discovery_b200")]
import sindy  # noqa: E402

DATA = os.path.join(ROOT, "tests", "golden", "data")


def main():
    assert torch.cuda.is_available(), "this needs a CUDA device"
    truth = np.load(os.path.join(ROOT, "tests", "golden", "model.npz"))
    thr = np.logspace(-3, 0, 40)
    for name, noise, spr in (("growth", "noise05", 10), ("dosc", "noise20", 100)):
        x = torch.load(os.path.join(DATA, f"{name}-train-{noise}-gp-x.pt")).reshape(-1, 2).cuda()
        dx = torch.load(os.path.join(DATA, f"{name}-train-{noise}-gp-dx.pt")).reshape(-1, 2).cuda()
        xv = torch.load(os.path.join(DATA, f"{name}-val-{noise}-gp-x.pt")).cuda()
        reg = sindy.SINDyRegression(2, 2, False, False, threshold=0.05, device="cuda", constrain_constant=True)
        path = sindy.stlsq_path(reg, x, dx, thr)
        sc = sindy.score_path(reg, path, xv, 0.002, steps_per_row=spr)
        masks = path["mask"].cpu().numpy()
        want = truth[f"truth_{name}"] != 0
        print(f"== {name}/{noise}: {len(thr)} thresholds, n_obs = {sc['n_obs']}, chosen #{sc['chosen']} "
              f"(threshold {thr[sc['chosen']]:.4g})")
        print(f"{'rank':>4} {'first thr':>10} {'k':>3} {'SSE':>12} {'AIC':>12} {'AICc':>12} {'BIC':>12}  support")
        seen = {}
        for i in range(len(thr)):
            seen.setdefault(masks[i].tobytes(), i)           # each support once, at its smallest threshold
        reps = sorted(seen.values(), key=lambda i: (sc["aicc"][i].item(), int(sc["k"][i]), -thr[i]))
        for r, i in enumerate(reps):
            tag = " (truth)" if np.array_equal(masks[i], want) else ""
            div = " diverged" if bool(sc["diverged"][i]) else ""
            print(f"{r:>4} {thr[i]:>10.4g} {int(sc['k'][i]):>3} {sc['sse'][i].item():>12.5g} {sc['aic'][i].item():>12.1f} "
                  f"{sc['aicc'][i].item():>12.1f} {sc['bic'][i].item():>12.1f}  {masks[i].astype(int).tolist()}{tag}{div}")


if __name__ == "__main__":
    main()
