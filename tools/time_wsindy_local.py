"""Timing of the compactly supported WSINDy integrals (sb_wsindy_local_integrals) against the roofline and the
trigonometric path at the same shape.

For every shape: CUDA-event time of one call (warm-up first, then repeated until the window is at least 1 s), samples/s,
GB/s and algorithmic TFLOP/s, and the fraction of the binding bound, the larger of
  bytes / (bandwidth of a device-to-device copy measured in this run)    bytes = x read once + G, b written
  flop  / (FFMA2 peak of sb_fp32_peak measured in this run)             flop  = n_traj·(T·(K−1−d) + 2·L·n_test·(K+d))
(L·n_test/T is the number of windows covering a sample). Every input is larger than the 126 MB L2. The card's name,
power limit and maximum SM clock are read (read-only) at the start.

  python tools/time_wsindy_local.py
"""
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "symmetry-ode-discovery_b200")]
import sindy  # noqa: E402
from sindy_b200 import native  # noqa: E402

DT = 0.002


def gpu_identity():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                         timeout=30).stdout.strip().splitlines()
    return out[torch.cuda.current_device()] if out else "unknown"


def timed(fn, min_window=1.0):
    """ms per call: warm-up, then as many calls as fill at least `min_window` seconds between two CUDA events."""
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    reps = max(3, math.ceil(min_window * 1e3 / max(a.elapsed_time(b), 1e-3)))
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps, reps


def copy_bandwidth():
    """GB/s of a device-to-device copy of 4 GB (read + write counted)."""
    src = torch.empty(1 << 30, dtype=torch.float32, device="cuda").uniform_()
    dst = torch.empty_like(src)
    ms, _ = timed(lambda: dst.copy_(src))
    return 2 * src.numel() * 4 / ms / 1e6


def main():
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    print(f"gpu: {gpu_identity()}")
    bw = copy_bandwidth()
    peak = native.fp32_peak(1)   # packed FFMA2, TFLOP/s
    print(f"device-to-device copy: {bw:.0f} GB/s; FP32 FFMA2 peak: {peak:.1f} TFLOP/s")
    shapes = [((2, 3, False, False), 4096, 8000, 50), ((3, 5, False, False), 4096, 8000, 50),
              ((2, 2, True, True), 4096, 8000, 50),        # K = 10 like (2, 3), runtime-table kernel
              ((2, 3, False, False), 64, 10 ** 6, 5000)]
    for (d, p, s, e), n_traj, T, n_test in shapes:
        lib = native.Library(d, p, s, e)
        K = lib.K
        L, deg, _, phi, dphi = sindy._local_test_functions(T, DT, n_test)
        phi, dphi = torch.from_numpy(phi).cuda(), torch.from_numpy(dphi).cuda()
        g = torch.Generator(device="cuda").manual_seed(0)
        x = torch.rand(n_traj, T, d, device="cuda", generator=g) * 0.8 + 0.2
        ms, reps = timed(lambda: native.wsindy_local_integrals(x, lib, phi, dphi, n_test))
        n = n_traj * T
        flop = n_traj * (T * (K - 1 - d) + 2 * L * n_test * (K + d))
        byts = n * d * 4 + n_traj * n_test * (K + d) * 8
        t_mem, t_fp = byts / bw / 1e6, flop / peak / 1e9    # ms
        bound = "memory" if t_mem >= t_fp else "FP32"
        print(f"lib (d={d}, p={p}, sin={int(s)}, exp={int(e)}) K={K}  {n_traj} x T={T}  n_test={n_test} L={L} "
              f"p={deg}  ov={L * n_test / T:.2f}")
        print(f"   poly: {ms:.3f} ms ({reps} calls)  {n / ms / 1e6:.1f} Gsamples/s  {byts / ms / 1e6:.0f} GB/s  "
              f"{flop / ms / 1e9:.2f} TFLOP/s  bound {max(t_mem, t_fp):.3f} ms ({bound}) -> "
              f"{max(t_mem, t_fp) / ms:.2f} of the bound")
        if n_test <= 1024:
            tms, treps = timed(lambda: native.wsindy_integrals(x, lib, DT, (T - 1) * DT, n_test))
            print(f"   trig: {tms:.3f} ms ({treps} calls)  {n / tms / 1e6:.1f} Gsamples/s  -> poly is "
                  f"{tms / ms:.2f}x faster")
        else:
            print("   trig: not available (sb_wsindy_integrals takes n_test <= 1024)")
        del x
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
