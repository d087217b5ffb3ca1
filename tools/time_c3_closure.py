"""Times the closure of BASELINE config 3 (`lv/noise99_eq_isymreg.cfg`: MSE + 0.1·symmreg_i, (2,2,exp) library, frozen
512x5 autoencoder of the reference's own class, B = 20 000) on the GPU and prints where the time goes. Run through the
launcher so that the reference's parser / autoencoder / gan import next to this repo's modules:

    python symmetry-ode-discovery_b200/sindy_b200/run.py --reference oracle/_ref tools/time_c3_closure.py [B]
"""
import os
import sys
import time

import torch

B = int(sys.argv[1]) if len(sys.argv) > 1 else 20000
sys.argv = ['main.py', '--config', 'lv/noise99_eq_isymreg.cfg', '--gpu', '0']
os.chdir(os.environ.get("SINDY_B200_REFERENCE", "."))          # run_configs/ is resolved relative to the cwd
from parser_utils import get_args  # noqa: E402
from autoencoder import AutoEncoder  # noqa: E402
from gan import LieGenerator  # noqa: E402
import model_utils  # noqa: E402
import sindy  # noqa: E402

args = vars(get_args())
args['input_dim'] = 2
torch.manual_seed(0)
dev = args['device']
ae = AutoEncoder(**args).to(dev).eval()
gen = LieGenerator(**args).to(dev).eval()
for m in (ae, gen):
    for p in m.parameters():
        p.requires_grad_(False)
reg = sindy.SINDyRegression(**args).to(dev)
x = torch.log(torch.rand(B, 2, device=dev) * 0.8 + 0.1)
dx = torch.randn(B, 2, device=dev)
symm = model_utils.make_symmreg_pttrain(ae, gen)


Z_X = {"on": False, "value": None}


def closure(fused):
    reg.zero_grad()
    loss_x = reg.mse_loss(x, dx)
    if fused:
        f = model_utils.EulerFlowMap(reg, args['int_t'], args['int_dt'])
    else:
        def f(q):
            return model_utils.odeint(reg, q, args['int_t'], args['int_dt'])
    x_fx = torch.stack([x, f(x)], dim=1)
    extra = {'z_x': Z_X['value']} if (Z_X['on'] and Z_X['value'] is not None) else {}
    loss = loss_x + args['w_sym_reg'] * symm(x_fx, f=f, **extra)
    loss.backward()
    return loss


for fused, ae_tc, zx in ((False, False, False), (True, False, False), (True, True, False), (True, True, True)):
    os.environ["SINDY_B200_AE_MLP"] = "1" if ae_tc else "0"
    Z_X["on"] = zx
    if zx:
        Z_X["value"] = model_utils.encode_constant_component(ae, x)
    for _ in range(3):
        closure(fused)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(10):
        closure(fused)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / 10
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA, torch.profiler.ProfilerActivity.CPU]) as prof:
        closure(fused)
        torch.cuda.synchronize()
    ev = [e for e in prof.key_averages() if e.device_time_total > 0 and e.device_type == torch.autograd.DeviceType.CUDA]
    tot = sum(e.device_time_total for e in ev)
    n_launch = sum(e.count for e in ev)
    what = ('fused Euler flow (EulerFlowMap)' if fused else 'closure + double vjp (reference call pattern)') + \
        (' + autoencoder on the tensor cores (sb_mlp_gemm)' if ae_tc else '') + \
        (' + encoder output of the data half cached per fit' if zx else '')
    lv = closure(fused)
    print(f"\n=== closure, {what}: loss {float(lv):.7f}, |grad| {float(reg.Xi.grad.norm()):.7f}, "
          f"B={B} wall {wall * 1e3:.2f} ms, GPU busy {tot / 1e3:.2f} ms in {n_launch} launches ===")
    for e in sorted(ev, key=lambda q: -q.device_time_total)[:12]:
        print(f"  {e.device_time_total / 1e3:8.3f} ms  x{e.count:4d}  {e.key[:100]}")
