import os, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "symmetry-ode-discovery_b200")]
from sindy_b200 import native
dev=torch.device('cuda')
for (d,p,ntr) in ((2,3,8192),(2,3,18944),(3,5,2048),(3,5,4736),(2,2,18944),(3,3,9472)):
    lib=native.Library(d,p)
    x=torch.rand(ntr,8000,d,device=dev)*0.8+0.2
    native.wsindy_integrals(x,lib,0.002,16.0,50); torch.cuda.synchronize()
    a,b=torch.cuda.Event(enable_timing=True),torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(3): native.wsindy_integrals(x,lib,0.002,16.0,50)
    b.record(); torch.cuda.synchronize()
    ms=a.elapsed_time(b)/3
    fl=(lib.K-1-d)+100*(lib.K+d)
    print(f"d={d} p={p} K={lib.K} ntraj={ntr}: {ms:.3f} ms  {ntr*8000/ms/1e6:.2f} Gsamples/s  {fl*ntr*8000/ms/1e9:.1f} TFLOP/s")
    # old kernel for comparison on a slice
    xs=x[:7]
    native.wsindy_integrals(xs,lib,0.002,16.0,50); torch.cuda.synchronize()
    a.record(); native.wsindy_integrals(xs,lib,0.002,16.0,50); b.record(); torch.cuda.synchronize()
    ms=a.elapsed_time(b)
    print(f"   per-test-function kernel, 7 traj: {ms:.3f} ms {7*8000/ms/1e6:.3f} Gsamples/s")
