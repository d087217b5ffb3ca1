#!/usr/bin/env python
"""bench.py — SINDy train-step throughput on B200 (BASELINE.json metric), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[4], SURVEY.md §8d "C5"): synthetic library fit, N = 1e8 samples in total,
d = 3, polynomial degree 5 (K = 56), X ~ U(-1,1)^3 generated on the device (seed 1234 + rank),
dX = Θ(X)Ξ*ᵀ + 0.01·randn with the Lorenz-form Ξ*, Ξ initialised randn(3,56) with torch.manual_seed(0).
A "step" is one iteration of the reference's Adam loop (`train.py:491-540`) WITH the linear Lie-derivative symmetry
regulariser of `train.py:503-507` (so(3) basis, weight 0.1 — SURVEY §8d): loss = MSE + 0.1·Σ_v Σ_n ‖J_h(x_n)(v x_n) −
v h(x_n)‖² + w·‖Ξ‖₁ and dL/dΞ over ALL samples, then the Adam update of Ξ — ONE launch of the fused kernel per rank
(sb_fit_step): its last block all-reduces the 170 packed fp64 sums over NVLink peer memory, evaluates the MSE part from
them and the regulariser as the quadratic form wᵀHw of the data set's Gram matrix (formed ONCE per fit by the moment
kernel — `gram_once_per_fit_ms` in the JSON line; the data set of a fit is fixed, `train.py:626-629`), writes loss and
gradient, advances Ξ and packs the next Ξ⊙mask for the next launch. `--no-symreg` drops the regulariser. Samples are
sharded over the ranks (total work fixed: strong scaling). Inputs (2.4 GB) exceed the 126 MB L2: no flush needed.

Printed JSON (rank 0, one line): value = whole-job samples/s with inputs resident in HBM; e2e = the same one-launch
iteration (sb_fit_step through FitStepper.step_from_host) with x/dx in pinned HOST memory — H2D of every sample inside
the timed region — and a device->host read of the loss; roofline = the fused kernel against the FP32 FMA peak measured
live by sb_fp32_peak (not in MEASURED_PEAKS.json) and, as roofline_hbm, against the measured HBM copy bandwidth;
cpu_baseline = the reference arm below, run as a child process on a bounded sample.

`--dump-outputs DIR` writes what the last of the K timed steps returned to its caller — loss.npy (the loss before the
update), grad.npy, xi.npy (the updated coefficients) and, on the one-launch path, adam_moments.npy (m and v) — for
comparing two builds on the same seeded inputs.

`--impl reference` (rank 0 only) times the reference's OWN CPU implementation of the same step on the box's host cores:
`SINDyRegression` imported from oracle/_ref (the unmodified reference, mirrored there by `__graft_entry__.build()`),
its forward, `MSELoss`, the `jvp`-based regulariser of `train.py:503-507`, L1, `backward`, `torch.optim.Adam.step()`.
The reference's library stops at degree 3, so the degree-4/5 columns of C5 are appended to ITS `terms` list in its own
cat-of-products idiom (oracle.TorchPolyN) — `cpu_baseline.kind` = "reference"; without oracle/_ref the oracle port
is timed instead ("port"). `extra.reference_unmodified` holds the rows the reference can run with NO extension: its
degree-3 (K = 20) closure at 1e6 and 4e6 samples, `solve_SINDy_one_step`, `solve_ode_batch`, `WSINDyWrapper.solve`.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "symmetry-ode-discovery_b200")
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# PKG (this repo's `sindy`, `train`, ...) is put on sys.path by the B200 arm only: the reference arm imports the
# reference's modules of the same names from oracle/_ref

import torch  # noqa: E402

D, P, K = 3, 5, 56
FLOP_PER_SAMPLE = (K - 1 - D) + 2 * K * D + 3 * D + 2 * K * D   # 733 (SURVEY.md §8d): Θ, prediction, residual², r⊗Θ
BYTES_PER_SAMPLE = 8 * D                                        # x and dx, fp32, read once
METRIC = "SINDy train-step samples/s (fused Θ+symreg)"
W_SYM = 0.1                                                     # weight of the so(3) Lie-derivative regulariser (§8d)
WORKLOAD = "C5 synthetic library fit: d=3, poly degree 5 (K=56), Adam iteration on MSE + so(3) Lie-derivative reg + L1"


def so3_basis():
    """so(3) basis in the order of the reference's `utils.so(3)` (`utils.py:16-24`)."""
    L = torch.zeros(3, 3, 3)
    q = 0
    for i in range(3):
        for j in range(i):
            L[q, i, j], L[q, j, i] = 1.0, -1.0
            q += 1
    return L


def truth_xi(device):
    Xi = torch.zeros(D, K, device=device)
    Xi[0, 1], Xi[0, 2] = -10.0, 10.0
    Xi[1, 1], Xi[1, 2], Xi[1, 6] = 2.8, -1.0, -1.0
    Xi[2, 5], Xi[2, 3] = 1.0, -8.0 / 3.0
    return Xi


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (recipe in B200_PROFILING.md)."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.file = None

    def start(self):
        try:
            self.file = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=self.file, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.file.flush()
        self.file.seek(0)
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.file.read().splitlines():
            parts = [q.strip() for q in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); smax.append(float(parts[2]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        self.file.close()
        os.unlink(self.file.name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(smax), "reasons": sorted(reasons), "samples": len(sm)}


def reference_dir():
    for c in (os.environ.get("SINDY_B200_REFERENCE"), os.path.join(ROOT, "oracle", "_ref")):
        if c and os.path.isfile(os.path.join(c, "sindy.py")) and os.path.isfile(os.path.join(c, "train.py")):
            return os.path.abspath(c)
    return None


def _timeit(fn, budget_s, min_reps=1, max_reps=20):
    fn()
    ts, t_start = [], time.perf_counter()
    while len(ts) < max_reps and (len(ts) < min_reps or time.perf_counter() - t_start < budget_s):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    ts.sort()
    return ts[len(ts) // 2], len(ts)


def run_reference(args, rank):
    """`--impl reference`: the reference's own CPU path for the same step, all host threads, bounded sample. Rank 0
    alone works; other ranks exit."""
    if rank != 0:
        return
    from torch.autograd.functional import jvp
    from oracle import sindy_oracle as O
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    ref = reference_dir()
    kind = "reference" if ref else "port"
    if ref:
        sys.path.insert(0, ref)
        import sindy as ref_sindy
        assert os.path.abspath(ref_sindy.__file__).startswith(ref), ref_sindy.__file__
        torch.manual_seed(0)
        reg = ref_sindy.SINDyRegression(D, 3, False, False, threshold=0.1, device="cpu", constrain_constant=True)
        reg.terms += [O.TorchPolyN(4), O.TorchPolyN(5)]        # degree-4/5 columns in the reference's own idiom
        torch.manual_seed(0)
        reg.Xi = torch.nn.Parameter(torch.randn(D, K))
        reg.mask = torch.ones(D, K)
        how = ("reference's SINDyRegression.forward from oracle/_ref (terms extended to degree 5), MSELoss, jvp-based "
               "Lie-derivative regulariser (train.py:503-507, intended [1]), L1, backward, torch.optim.Adam.step()")
    else:
        torch.manual_seed(0)
        reg = O.TorchRegressor(D, P)
        how = "oracle port of the same step (no reference checkout in oracle/_ref)"
    gens = so3_basis() if not args.no_symreg else []
    mse = torch.nn.MSELoss()
    opt = torch.optim.Adam(reg.parameters(), lr=1e-3)

    def make_data(n):
        g = torch.Generator().manual_seed(1234)
        x = torch.rand(n, D, generator=g) * 2 - 1
        with torch.no_grad():
            dx = O.torch_theta(x, P) @ truth_xi("cpu").T + 0.01 * torch.randn(n, D, generator=g)
        return x, dx

    def step(x, dx, gens=gens):
        dx_pred = reg(x)
        loss = mse(dx_pred, dx)
        for v in gens:
            tangent = jvp(reg, x, torch.einsum('ij,bj->bi', v, x), create_graph=True)[1]
            loss = loss + W_SYM * torch.norm(tangent - torch.einsum('ij,bj->bi', v, dx_pred)) ** 2
        loss = loss + 0.0 * sum(torch.norm(p, 1) for p in reg.parameters())
        opt.zero_grad()
        loss.backward()
        opt.step()
        return float(loss)

    # sample size: as many of the 1e8 samples per step as keep the whole --steps/--warmup run within ~2.5 minutes
    n_probe = 100_000
    xp, dxp = make_data(n_probe)
    step(xp, dxp)
    t0 = time.perf_counter()
    step(xp, dxp)
    t_probe = time.perf_counter() - t0
    budget = 150.0 / max(args.steps + args.warmup, 1)
    n_ref = int(min(args.cpu_samples, max(50_000, n_probe * budget / t_probe)))
    n_ref -= n_ref % 1000
    x, dx = make_data(n_ref)
    for _ in range(args.warmup):
        step(x, dx)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step(x, dx)
    el = time.perf_counter() - t0
    value = n_ref * args.steps / el
    sample = (f"{n_ref} of the 1e8 samples per step (the reference materialises Θ: N×56 fp32 plus autograd copies, and "
              f"runs 2 reverse passes per generator for the jvp), {args.steps} steps")
    result = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "samples_total": int(1e8), "samples_per_step_timed": n_ref,
                   "symreg": "none" if args.no_symreg else f"so(3) linear Lie-derivative regulariser, weight {W_SYM}",
                   "step": how},
        "cpu_baseline": {"value": value, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": kind,
                         "sample": sample},
        "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if not args.skip_extras:
        try:
            result["extra"] = reference_extras(ref, step, make_data)
        except Exception as exc:   # secondary rows must never cost the line
            result["extra"] = {"error": repr(exc)}
    print(json.dumps(result))
    sys.stdout.flush()


def reference_extras(ref, step5, make_data):
    """Side rows on the host cores. With oracle/_ref: the UNMODIFIED reference (no extension) — its degree-3 closure
    (`train.py:645-690`) at 1e6 and 4e6 samples, `solve_SINDy_one_step` (`sindy.py:250-315`), `solve_ode_batch`
    (`data_utils/ode.py:7-28`), `WSINDyWrapper.solve` (`sindy.py:352-395`). Always: the degree-5 step without sym-reg."""
    import numpy as np
    out = {"cores": torch.get_num_threads()}
    x, dx = make_data(500_000)
    t, reps = _timeit(lambda: step5(x, dx, gens=[]), 8.0)
    out["degree5_step_without_symreg"] = {"samples_per_s": 500_000 / t, "ms": 1e3 * t, "reps": reps,
                                          "sample": "5e5 samples, K = 56"}
    del x, dx
    if ref is None:
        return out
    import sindy as ref_sindy
    from data_utils import ode as ref_ode
    from data_utils.selkov import selkov as ref_selkov
    mse = torch.nn.MSELoss()
    unmod = {}
    for n in (1_000_000, 4_000_000):
        g = torch.Generator().manual_seed(7)
        xs = torch.rand(n, D, generator=g) * 2 - 1
        ys = torch.randn(n, D, generator=g)
        torch.manual_seed(0)
        reg = ref_sindy.SINDyRegression(D, 3, False, False, threshold=0.1, device="cpu", constrain_constant=True)

        def closure():
            reg.zero_grad()
            loss = mse(reg(xs), ys) + 0.0 * sum(torch.norm(p, 1) for p in reg.parameters())
            loss.backward()
            return loss

        t, reps = _timeit(closure, 6.0 if n == 1_000_000 else 8.0)
        unmod[f"closure_K20_n{n}"] = {"samples_per_s": n / t, "ms": 1e3 * t, "reps": reps}
        if n == 4_000_000:
            t0 = time.perf_counter()
            ref_sindy.solve_SINDy_one_step(reg, xs, ys, 0.0, 0.1)
            t = time.perf_counter() - t0
            unmod["solve_SINDy_one_step_K20_n4000000"] = {"samples_per_s": n / t, "ms": 1e3 * t}
        del xs, ys
    x0 = np.random.default_rng(0).uniform(0.5, 1.0, (100_000, 2))
    t0 = time.perf_counter()
    ref_ode.solve_ode_batch(ref_selkov, x0, dt=0.002, num_steps=100)
    t = time.perf_counter() - t0
    unmod["solve_ode_batch_selkov_1e5ics_100steps"] = {"ic_steps_per_s": 1e5 * 99 / t, "ms": 1e3 * t, "dtype": "f64"}
    T = 8000
    tt = torch.arange(T) * 0.002
    traj = torch.from_numpy(ref_ode.solve_ode_batch(ref_selkov, x0[:1], dt=0.002, num_steps=T)[0][:, 0]).float()
    torch.manual_seed(0)
    regw = ref_sindy.SINDyRegression(2, 3, False, False, threshold=0.075, device="cpu", constrain_constant=True)
    t0 = time.perf_counter()
    wr = ref_sindy.WSINDyWrapper(regw, tt, T * 0.002, device="cpu")
    t_ctor = time.perf_counter() - t0
    t0 = time.perf_counter()
    wr.solve(traj, 0.0, 0.075)
    t = time.perf_counter() - t0
    unmod["WSINDyWrapper_T8000_K10"] = {"ctor_ms": 1e3 * t_ctor, "first_solve_ms": 1e3 * t}
    out["reference_unmodified"] = unmod
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--samples", type=float, default=1e8, help="total samples over all ranks")
    ap.add_argument("--cpu-samples", type=int, default=1_000_000, help="bounded sample of the CPU baseline")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--no-graph", action="store_true", help="do not capture the multi-GPU step in a CUDA graph")
    ap.add_argument("--no-peer", action="store_true", help="multi-GPU: NCCL all-reduce instead of the in-kernel peer all-reduce")
    ap.add_argument("--skip-extras", action="store_true")
    ap.add_argument("--no-symreg", action="store_true", help="step without the so(3) Lie-derivative regulariser")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (loss, gradient, updated coefficients, Adam moments) "
                         "as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the B200 path; it does not apply to --impl reference")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.warmup < 3:
        args.warmup = 3

    if PKG not in sys.path:
        sys.path.insert(0, PKG)
    import torch.distributed as dist
    from sindy_b200 import native
    from sindy_b200.dist import FitStepper, HostStreamedStep, ShardedTrainStep, bind_to_gpu_numa_node, mse_from_sums

    native.load()  # fails loudly if the CUDA library is missing: there is no fallback path
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    lib = native.Library(D, P)
    assert lib.K == K

    # ---- synthetic shard, generated on the device ----
    n_total = int(args.samples)
    n_local = n_total // world + (1 if rank < n_total % world else 0)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    x = torch.rand(n_local, D, device=dev, generator=gen) * 2 - 1
    dx = native.forward(x, truth_xi(dev), lib)
    dx.add_(torch.randn(n_local, D, device=dev, generator=gen), alpha=0.01)
    torch.manual_seed(0)
    Xi0 = torch.randn(D, K).to(dev)
    mask = torch.ones(D, K, device=dev)
    w_l1 = 0.0  # w_sindy_reg of the C5 config; the L1 term is still evaluated like the reference does
    flags = native.SB_STEP_LOSS | native.SB_STEP_GRAD
    variant = native.train_step_variant(lib, flags)

    # One step = one iteration of the reference's Adam loop without sym-reg (`train.py:512-530`): forward, MSE + L1,
    # backward, optimizer.step() — ONE launch of the fused kernel per rank (sb_fit_step): its last block all-reduces
    # the sums over NVLink peer memory (N > 1), evaluates loss and gradient, applies Adam to Ξ in place and packs Ξ⊙mask
    # into the constant bank for the next launch. Replayed as a CUDA graph. `--no-peer`: the 3-launch NCCL path.
    legacy = args.no_peer or args.no_graph
    kern_events = []
    fallback_note = None
    sym_gens = None if args.no_symreg else list(so3_basis())
    gram_ms = None
    if not legacy:
        try:
            if sym_gens is not None:   # the Gram pass the regulariser needs ONCE per fit, timed on its own (rank's shard)
                from sindy_b200 import symreg
                symreg.gram(x, lib)
                torch.cuda.synchronize()
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record()
                symreg.gram(x, lib)
                g1.record()
                torch.cuda.synchronize()
                gram_ms = g0.elapsed_time(g1)
            stepper = FitStepper(lib, x, dx, "adam", lr=1e-3, w_l1=w_l1, use_graph=True, sym_gens=sym_gens,
                                 w_sym=W_SYM if sym_gens is not None else 0.0)
        except RuntimeError as exc:   # no peer-mapped symmetric memory on this box: the NCCL path still measures
            legacy, fallback_note = True, f"one-launch step unavailable ({exc}); NCCL path"
    if not legacy:
        stepper.load(Xi0, mask)
        collective = "none" if world == 1 else "in-kernel peer all-reduce over NVLink (sb_fit_step)"
        launches_per_step = 1
        use_graph = True

        def one_step(record=False):
            return stepper.step()

        def last_outputs(loss):
            return {"loss": loss, "grad": stepper.grad, "xi": stepper.xi,
                    "adam_moments": stepper.state[:2 * D * K].view(2, D, K)}
    else:
        use_graph = (world > 1) and not args.no_graph
        stepper = ShardedTrainStep(lib, x, dx, flags=flags, use_graph=use_graph, sgd_lr=1e-3, use_peer=not args.no_peer)
        collective = "none" if world == 1 else ("in-kernel peer all-reduce over NVLink (sb_closure_peer)"
                                                if stepper.peer is not None else "NCCL all-reduce + epilogue launch")
        stepper.step(Xi0, mask, w_l1)  # loads the static parameters (and captures the graph when enabled)
        stepper.xi.copy_(Xi0)
        launches_per_step = 2 if (world == 1 or stepper.peer is not None) else 3
        last_grad = None

        def one_step(record=False):
            nonlocal last_grad
            if record and not use_graph:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                packed, loss_t, grad_t = stepper._buffers(dev)
                if world == 1:
                    native.closure(x, dx, stepper.xi, stepper.mask, lib, w_l1, packed=packed, loss=loss_t, grad=grad_t)
                    e1.record()
                else:
                    native.train_step(x, dx, stepper.xi * stepper.mask, lib, flags, out=packed)
                    e1.record()
                    dist.all_reduce(packed)
                    native.step_epilogue(packed, stepper.xi, stepper.mask, lib, w_l1, loss=loss_t, grad=grad_t)
                kern_events.append((e0, e1))
                stepper.xi.add_(grad_t, alpha=-1e-3)
                last_grad = grad_t
                return loss_t
            loss_t, last_grad = stepper.step(None, None, w_l1)
            return loss_t

        def last_outputs(loss):
            return {"loss": loss, "grad": last_grad, "xi": stepper.xi}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the one-launch step runs in groups of `unroll` iterations per graph replay (no host work between iterations)
    unroll = next(u for u in (25, 20, 16, 10, 8, 5, 4, 2, 1) if args.steps % u == 0)

    def run_steps(k):
        if not legacy:
            return stepper.run(k, unroll)
        for _ in range(k):
            out = one_step(record=True)
        return out

    if not legacy:
        stepper.run(unroll, unroll)      # capture outside the timed region
        stepper.load(Xi0, mask, reset_state=True)
    for _ in range(args.warmup):
        one_step()
    barrier()
    launches0 = native.kernel_launches()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        # the ranks leave the host barrier up to a few hundred us apart (a step is 0.2 ms at 8 GPUs) and the first
        # exchange would charge that skew to the timed steps: one more untimed step lets the in-kernel exchange align
        # the GPUs on the device; ev0 is then recorded on every rank at the end of the same exchange
        one_step()
    ev0.record()
    loss = run_steps(args.steps)
    ev1.record()
    torch.cuda.synchronize()
    barrier()
    clocks = sampler.stop() if sampler else None
    launches = native.kernel_launches() - launches0
    if use_graph:   # kernels launched by the replayed graph are not seen by the library's launch counter
        launches = launches_per_step * args.steps
    elapsed_ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
    if world > 1:
        dist.all_reduce(elapsed_ms, op=dist.ReduceOp.MAX)
    elapsed_ms = float(elapsed_ms)
    value = n_total * args.steps / (elapsed_ms * 1e-3)
    final_loss = float(loss)
    if args.dump_outputs and rank == 0:   # before the checks below reload the stepper
        if not legacy:
            stepper.check()   # a peer lost in the exchange leaves the outputs stale: fail before writing them
        dump_outputs(args.dump_outputs, last_outputs(loss))

    # ---- N > 1: the sharded step against an UNSHARDED recompute on rank 0 (all shards gathered on one GPU) ----
    sharded_check = None
    if world > 1 and not legacy:
        stepper.load(Xi0, mask, reset_state=True)
        l_sh = stepper.step().clone()
        g_sh = stepper.grad.clone()
        n_max = (n_total + world - 1) // world

        def padded(t):
            return t if t.shape[0] == n_max else torch.cat([t, t.new_zeros(n_max - t.shape[0], D)])
        xs_all = [torch.empty(n_max, D, device=dev) for _ in range(world)] if rank == 0 else None
        dxs_all = [torch.empty(n_max, D, device=dev) for _ in range(world)] if rank == 0 else None
        dist.gather(padded(x), xs_all, dst=0)
        dist.gather(padded(dx), dxs_all, dst=0)
        if rank == 0:
            counts = [n_total // world + (1 if r < n_total % world else 0) for r in range(world)]
            x_all = torch.cat([t[:c] for t, c in zip(xs_all, counts)])
            dx_all = torch.cat([t[:c] for t, c in zip(dxs_all, counts)])
            del xs_all, dxs_all
            one = FitStepper(lib, x_all, dx_all, "adam", lr=1e-3, w_l1=w_l1, use_graph=False, sym_gens=sym_gens,
                             w_sym=W_SYM if sym_gens is not None else 0.0, local_only=True)
            one.load(Xi0, mask)
            l_one = one.step()
            sharded_check = {
                "loss_rel_diff": abs(float(l_sh) - float(l_one)) / abs(float(l_one)),
                "grad_rel_diff": float((g_sh - one.grad).abs().max() / one.grad.abs().max()),
                "how": f"one iteration at the initial parameters: {world} shards + in-kernel all-reduce vs all {n_total} "
                       "samples gathered on rank 0 and stepped by one GPU"}
            del one, x_all, dx_all
        stepper.check()
        barrier()

    # ---- kernel-only duration (roofline numerator) ----
    if not legacy:
        kern_ms = elapsed_ms / args.steps
        kern_how = ("CUDA events around the K timed steps: a step IS one launch of the fused kernel (sample loop, "
                    "reductions, peer all-reduce, loss/gradient, Adam update), so launch gaps are included")
    elif kern_events:
        kern_ms = sum(a.elapsed_time(b) for a, b in kern_events) / len(kern_events)
        kern_how = "CUDA events around the library call (pack_w + fused kernel) inside every timed step"
    else:
        out = torch.empty(lib.step_out_len(flags), dtype=torch.float64, device=dev)
        wm = stepper.xi * mask
        native.train_step(x, dx, wm, lib, flags, out=out)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            native.train_step(x, dx, wm, lib, flags, out=out)
        e1.record()
        torch.cuda.synchronize()
        kern_ms = e0.elapsed_time(e1) / args.steps
        kern_how = "CUDA events over back-to-back launches right after the timed region (steps replay a CUDA graph)"
    kt = torch.tensor([kern_ms], device=dev)
    if world > 1:
        dist.all_reduce(kt, op=dist.ReduceOp.MAX)
    kern_ms = float(kt)

    # ---- e2e: the same one-launch iteration with HOST buffers: H2D of every sample inside the timed region, loss read back ----
    numa_node = bind_to_gpu_numa_node(dev) if world > 1 else None   # node-local pinned buffers (one process per GPU)
    xh = torch.empty(n_local, D, dtype=torch.float32, pin_memory=True)
    dxh = torch.empty(n_local, D, dtype=torch.float32, pin_memory=True)
    xh.copy_(x)
    dxh.copy_(dx)
    if not legacy:
        stepper.load(Xi0, mask, reset_state=True)
        e2e_how = ("FitStepper.step_from_host: pinned host x/dx -> device (chunked async copies) -> ONE sb_fit_step launch "
                   "(loss, gradient, in-kernel all-reduce, Adam update); loss read back with .item()")

        def e2e_step():
            loss_e = stepper.step_from_host(xh, dxh)
            return float(loss_e)  # device -> host read of the step's result
        h2d_of = lambda: stepper.h2d_bytes  # noqa: E731
    else:
        host_step = HostStreamedStep(lib, chunk_samples=1 << 22, device=dev, flags=flags)
        Xi_e = Xi0.clone()
        e2e_how = "HostStreamedStep: pinned host x/dx -> 2 staging buffers on 2 streams -> fused kernel per chunk; .item()"

        def e2e_step():
            nonlocal Xi_e
            packed = host_step(xh, dxh, Xi_e * mask)
            if world > 1:
                dist.all_reduce(packed)
            loss_e, grad = mse_from_sums(packed, lib, Xi_e, mask)
            Xi_e = Xi_e - 1e-3 * grad
            return float(loss_e)
        h2d_of = lambda: host_step.h2d_bytes  # noqa: E731

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = n_total * args.e2e_steps / float(e2e_s)
    h2d_bytes = h2d_of()
    del xh, dxh

    # ---- sharded RK4 rollout of the same config (10^6 ICs x 2000 steps, every 10th state stored): the ICs split
    # over the ranks, no collective on the data path; time = max over ranks ----
    rollout_sharded = None
    if world > 1 and not args.skip_extras:
        n_ics = 10 ** 6 // world + (1 if rank < 10 ** 6 % world else 0)
        g2 = torch.Generator(device=dev).manual_seed(4321 + rank)
        x0 = torch.rand(n_ics, D, device=dev, generator=g2) * 2 - 1
        Xi_t = truth_xi(dev)
        native.rollout(x0, Xi_t, lib, 0.002, 2000, 10, "rk4")
        barrier()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for _ in range(3):
            native.rollout(x0, Xi_t, lib, 0.002, 2000, 10, "rk4")
        r1.record()
        torch.cuda.synchronize()
        rt = torch.tensor([r0.elapsed_time(r1) / 3], device=dev)
        dist.all_reduce(rt, op=dist.ReduceOp.MAX)
        rollout_sharded = {"ic_steps_per_s": 2e9 / (float(rt) * 1e-3), "ms": float(rt), "ics_total": 10 ** 6,
                           "steps": 2000, "dtype": "f32", "collective": "none (ICs are independent)"}

    if rank != 0:
        # every collective of this run has completed on all ranks (the last one is the e2e all-reduce); leave
        # without NCCL teardown: destroy_process_group() after CUDA-graph capture of collectives was seen to hang
        torch.cuda.synchronize()
        sys.stdout.flush()
        os._exit(0)

    # ---- roofline (rank 0) ----
    peaks, peak_src = measured_peaks()
    fp32_peaks = {name: native.fp32_peak(v, 4096) for v, name in ((0, "ffma"), (1, "ffma2"), (2, "ffma2_const"))}
    fp32_peak = max(fp32_peaks.values())
    n_kernel = n_local  # rank 0's shard (largest)
    ach_tflops = FLOP_PER_SAMPLE * n_kernel / (kern_ms * 1e-3) / 1e12
    ach_gbs = BYTES_PER_SAMPLE * n_kernel / (kern_ms * 1e-3) / 1e9
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        if int(tj.get("samples_per_launch", -1)) == n_kernel:
            traffic = tj.get("dram_bytes_per_launch")
    roofline = {"bound": "fp32", "achieved": ach_tflops, "peak": fp32_peak, "unit": "TFLOP/s",
                "frac": ach_tflops / fp32_peak, "traffic": traffic, "kernel": variant, "kernel_ms": kern_ms,
                "flop_per_sample": FLOP_PER_SAMPLE, "samples_per_launch": n_kernel,
                "peak_source": "measured live: sb_fp32_peak, best of " + json.dumps(fp32_peaks),
                "peak_nominal": 148 * 128 * 2 * 1.965e9 / 1e12, "timing": kern_how}
    roofline_hbm = {"bound": "hbm", "achieved": ach_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": ach_gbs / peaks["hbm_gbs"], "traffic": traffic, "bytes_per_sample": BYTES_PER_SAMPLE,
                    "peak_source": peak_src}

    result = {
        "metric": METRIC, "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "step": ("one Adam iteration (train.py:491-540): loss, gradient, update in ONE launch (sb_fit_step)"
                            if not legacy else "closure + SGD update (pack_w, fused kernel[, all-reduce, epilogue], axpy)"),
                   "samples_total": n_total, "samples_per_gpu": n_local,
                   "symreg": ("none" if (sym_gens is None or legacy) else
                              f"so(3) linear Lie-derivative regulariser, weight {W_SYM}: quadratic form of the data set's "
                              "Gram matrix in the kernel's epilogue; Gram formed once per fit"),
                   "gram_once_per_fit_ms": gram_ms,
                   "l2": "inputs (24 B/sample, %.2f GB per GPU) larger than L2; no flush" % (24 * n_local / 1e9),
                   "parallelism": f"sample-sharded x{world}, one all-reduce of {2 + D * K} fp64 sums per step",
                   "collective": collective, "fallback": fallback_note,
                   "sharded_vs_unsharded": sharded_check,
                   "cuda_graph": use_graph, "iterations_per_graph_replay": (unroll if not legacy else 1),
                   "final_loss": final_loss},
        "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": e2e_value, "unit": "samples/s", "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": 8,
                "steps": args.e2e_steps,
                "how": e2e_how, "numa_node": numa_node},
        "roofline": roofline, "roofline_hbm": roofline_hbm,
    }

    if rollout_sharded is not None:
        result["extra"] = {"rk4_rollout_sharded": rollout_sharded}
    if world == 1:
        result["cpu_baseline"], cpu_extra = cpu_baseline_child(args)
        if not args.skip_extras:
            try:
                result["extra"] = extras(native, dev, peaks, fp32_peak)
            except Exception as exc:   # secondary measurements must never cost the headline line
                result["extra"] = {"error": repr(exc)}
            result["extra"]["cpu_reference_side_by_side"] = cpu_extra
    print(json.dumps(result))
    sys.stdout.flush()
    if world > 1:
        torch.cuda.synchronize()
        os._exit(0)


def dump_outputs(out_dir, tensors):
    """`--dump-outputs`: each tensor as out_dir/<name>.npy in its own dtype (float32 here; a few KB in all). The inputs
    are seeded, so two builds run with the same arguments can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in tensors.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy())


def cpu_baseline_child(args):
    """The reference arm on a bounded sample, as a child process (it imports the REFERENCE's `sindy`, which cannot share
    an interpreter with this repo's module of the same name): returns (cpu_baseline, its extra rows)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "3", "--warmup", "1",
           "--cpu-samples", str(args.cpu_samples)]
    if args.no_symreg:
        cmd.append("--no-symreg")
    if args.skip_extras:
        cmd.append("--skip-extras")
    try:
        res = subprocess.run(cmd, capture_output=True, text=True, timeout=900,
                             env={k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")})
        line = json.loads(res.stdout.strip().splitlines()[-1])
        return line["cpu_baseline"], line.get("extra")
    except Exception as exc:   # the headline line must survive a failing CPU leg
        return {"value": None, "unit": "samples/s", "cores": os.cpu_count(), "kind": "unavailable",
                "sample": f"reference arm failed: {exc!r}"}, None


def extras(native, dev, peaks, fp32_peak):
    """Secondary measurements of the same hot path (not the headline): the HBM-bound d=2 library and the
    batched RK4 rollout of C5 (10^6 ICs x 2000 steps, every 10th state stored)."""
    def timed(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ts.sort()
        return ts[len(ts) // 2]

    out = {}
    gen = torch.Generator(device=dev).manual_seed(99)
    n = 10 ** 8
    for (d, p) in ((2, 2), (2, 3), (3, 3)):
        lib = native.Library(d, p)
        x = torch.rand(n, d, device=dev, generator=gen) * 2 - 1
        dx = torch.randn(n, d, device=dev, generator=gen)
        W = torch.randn(d, lib.K, device=dev, generator=gen)
        o = torch.empty(lib.step_out_len(3), dtype=torch.float64, device=dev)
        ms = timed(lambda: native.train_step(x, dx, W, lib, 3, out=o))
        gbs = 8 * d * n / (ms * 1e-3) / 1e9
        out[f"train_step_d{d}_p{p}_K{lib.K}"] = {"samples_per_s": n / (ms * 1e-3), "ms": ms, "hbm_gbs": gbs,
                                                 "hbm_frac": gbs / peaks["hbm_gbs"]}
        del x, dx
    # the GENERIC runtime-table kernels (every library without a specialisation, here (2, 3) + sine, K = 14): parity-complete,
    # not tuned — timed so that the distance to the specialised kernels is on record
    try:
        n_g = 10 ** 7
        lg = native.Library(2, 3, True, False)
        xg = torch.rand(n_g, 2, device=dev, generator=gen) * 2 - 1
        dxg = torch.randn(n_g, 2, device=dev, generator=gen)
        Wg = torch.randn(2, lg.K, device=dev, generator=gen)
        og = torch.empty(lg.step_out_len(3), dtype=torch.float64, device=dev)
        ms = timed(lambda: native.train_step(xg, dxg, Wg, lg, 3, out=og))
        out["train_step_generic_d2_p3_sine_K14_1e7"] = {"samples_per_s": n_g / (ms * 1e-3), "ms": ms,
                                                         "hbm_gbs": 16 * n_g / (ms * 1e-3) / 1e9,
                                                         "variant": native.train_step_variant(lg, 3)}
        del xg, dxg
    except Exception as exc:   # noqa: BLE001
        out["train_step_generic_d2_p3_sine_K14_1e7"] = {"error": repr(exc)}
    # the C5 step with the linear so(3) Lie-derivative regulariser (weight 0.1, `train.py:503-507`): closure kernel +
    # power-sum Gram kernel (second pass over x) + K×K algebra, replayed as one CUDA graph; and the STLSQ data pass
    from sindy_b200.dist import ShardedTrainStep
    lib = native.Library(D, P)
    x = torch.rand(n, D, device=dev, generator=gen) * 2 - 1
    dx = native.forward(x, truth_xi(dev), lib)
    so3 = torch.zeros(3, 3, 3)
    q = 0
    for i in range(3):
        for j in range(i):
            so3[q, i, j], so3[q, j, i] = 1.0, -1.0
            q += 1
    W = torch.randn(D, K, device=dev, generator=gen)
    st = ShardedTrainStep(lib, x, dx, sym_gens=list(so3), w_sym=0.1, use_graph=True, sgd_lr=1e-6)
    st.step(W, torch.ones_like(W), 0.0)
    ms = timed(lambda: st.step(None, None, 0.0))
    flop_sym = FLOP_PER_SAMPLE + (9 + 65) + 2 * 286   # + leading powers, trailing table, one FMA per power sum
    out["train_step_C5_with_so3_symreg"] = {"samples_per_s": n / (ms * 1e-3), "ms": ms, "flop_per_sample": flop_sym,
                                            "fp32_tflops": flop_sym * n / (ms * 1e-3) / 1e12,
                                            "fp32_frac": flop_sym * n / (ms * 1e-3) / 1e12 / fp32_peak,
                                            "bytes_per_sample": 36}
    # the same objective with the Gram matrix of the fixed data set formed ONCE per fit (moment kernel, timed separately)
    # and the regulariser + gradient evaluated as a quadratic form in the epilogue of the one-launch iteration
    from sindy_b200.dist import FitStepper
    from sindy_b200 import symreg
    ms_gram = timed(lambda: symreg.gram(x, lib))
    fs = FitStepper(lib, x, dx, "adam", lr=1e-6, sym_gens=list(so3), w_sym=0.1)
    fs.load(W, torch.ones_like(W))
    fs.run(10, 10)
    ms = timed(lambda: fs.run(10, 10)) / 10
    out["fit_step_C5_with_so3_symreg_cached_gram"] = {
        "samples_per_s": n / (ms * 1e-3), "ms": ms, "gram_once_per_fit_ms": ms_gram,
        "note": "one launch per Adam iteration; w_sym*w'Hw and 2Hw evaluated by the kernel's last block, H from the Gram of the data set"}
    del fs
    o = torch.empty(lib.step_out_len(12), dtype=torch.float64, device=dev)
    ms = timed(lambda: native.train_step(x, dx, None, lib, 12, out=o))
    out["stlsq_data_pass_C5_gram_and_b"] = {"samples_per_s": n / (ms * 1e-3), "ms": ms,
                                            "variant": native.train_step_variant(lib, 12)}
    # the whole STLSQ solve of `sindy.py:318-324` (mask reset, up to 5 threshold iterations) on the Lorenz-form data:
    # ONE data pass (Gram by the moment kernel + ΘᵀẊ by the fused kernel + Σẋ²), then K×K fp64 solves per iteration
    import sindy
    reg = sindy.SINDyRegression(D, P, False, False, threshold=0.1, device=str(dev), constrain_constant=True)
    dxn = dx + 0.01 * torch.randn(n, D, device=dev, generator=gen)
    ms = timed(lambda: sindy.solve_SINDy(reg, x, dxn, 0.0, 0.1), reps=3)
    support_ok = bool(torch.equal(reg.mask.bool(), truth_xi(dev) != 0))
    coef_err = float(((reg.Xi.detach() * reg.mask) - truth_xi(dev)).abs().max() / truth_xi(dev).abs().max())
    out["stlsq_solve_SINDy_C5"] = {"samples_per_s": n / (ms * 1e-3), "ms": ms, "recovered_support_is_truth": support_ok,
                                   "max_coef_err_rel": coef_err}
    del x, dx, dxn
    # fused symmetry-regulariser kernels on config 3's library (2, 2, exp), 1e7 samples: the Euler flow map with its JVP
    # (forward + reverse sweep, one launch each) beside the operator-by-operator composition the reference's call
    # pattern produces (10 Python Euler steps under a double vjp), and the streaming reversed regulariser
    try:
        from torch.autograd.functional import jvp as _jvp
        from sindy_b200 import ops as _ops
        l8 = native.Library(2, 2, False, True)
        n7 = 10 ** 7
        xs = torch.log(torch.rand(n7, 2, device=dev, generator=gen) * 0.8 + 0.1)
        vs = torch.randn(n7, 2, device=dev, generator=gen)
        gs = torch.randn(n7, 2, device=dev, generator=gen)
        W8 = (0.3 * torch.randn(2, l8.K, device=dev, generator=gen)).requires_grad_(True)

        def fused_fb():
            vv = vs.clone().requires_grad_(True)
            fx, jv = _ops.euler_flow(xs, vv, W8, l8, 0.01, 10)
            torch.autograd.grad((fx * gs).sum() + (jv * gs).sum(), (W8, vv))

        def composed_fb():
            vv = vs.clone().requires_grad_(True)

            def flow(q):
                for _ in range(10):
                    q = q + 0.01 * _ops.sindy_forward(q, W8, l8)
                return q
            fx, jv = _jvp(flow, xs, vv, create_graph=True)
            torch.autograd.grad((fx * gs).sum() + (jv * gs).sum(), (W8, vv))

        ms_fused = timed(fused_fb, reps=3)
        ms_comp = timed(composed_fb, reps=3)
        gxs = xs + 0.05 * vs
        Jg = (torch.eye(2, device=dev).expand(n7, 2, 2) + 0.1 * torch.randn(n7, 2, 2, device=dev, generator=gen)).contiguous()
        ms_r = timed(lambda: native.symreg_r(xs, gxs, Jg, W8.detach(), l8), reps=3)
        out["symreg_kernels_config3_library_1e7"] = {
            "euler_flow_jvp_fwd_bwd_fused_ms": ms_fused, "same_composed_through_autograd_ms": ms_comp,
            "speedup": ms_comp / ms_fused, "flow_samples_per_s": n7 / (ms_fused * 1e-3),
            "symreg_r_streaming_ms": ms_r, "symreg_r_samples_per_s": n7 / (ms_r * 1e-3),
            "symreg_r_hbm_gbs": 4 * (2 + 2 + 4) * n7 / (ms_r * 1e-3) / 1e9}
        del xs, vs, gs, gxs, Jg
    except Exception as exc:   # noqa: BLE001
        out["symreg_kernels_config3_library_1e7"] = {"error": repr(exc)}
    # the frozen autoencoder of config 3 (`autoencoder.py:38-66`: 2 -> 512 x 5 -> 2, BatchNorm in the encoder, ReLU) on
    # the tensor cores (SURVEY §8f-3): one 512-wide layer (40 000 rows = 20 000 samples x 2 components) against cuBLAS
    # fp32 through PyTorch, and the encoder value + decoder JVP + both transpose chains of `symmreg_i`'s closure against
    # the reference's call pattern (module forward, double-vjp JVP, autograd backward) on the same module
    try:
        from sindy_b200 import mlp as _mlp
        m_rows, f = 40000, 512
        a = torch.randn(m_rows, f, device=dev, generator=gen)
        wl = torch.randn(f, f, device=dev, generator=gen) / f ** 0.5
        bl = torch.randn(f, device=dev, generator=gen)
        pa, pc = _mlp._Panel.from_rows(a), _mlp._Panel(m_rows, f, dev)
        pk = torch.empty(2 * f * f, device=dev)
        sl = native.load()
        native._check(sl.sb_mlp_pack_weights(wl.data_ptr(), f, f, 0, pk.data_ptr(), native._stream(dev)), "pack")
        ms_tc = timed(lambda: native._check(sl.sb_mlp_gemm(pa.ptr(), m_rows, f, pk.data_ptr(), f, bl.data_ptr(), None, 1,
                                                           pc.ptr(), native._stream(dev)), "gemm"), reps=20)
        torch.backends.cuda.matmul.allow_tf32 = False
        ms_cublas = timed(lambda: torch.relu(torch.nn.functional.linear(a, wl, bl)), reps=20)
        ref64 = torch.relu(a.double() @ wl.double().t() + bl.double())
        err_tc = float((pc.to_rows().double() - ref64).abs().max() / ref64.abs().max())
        err_cublas = float((torch.relu(torch.nn.functional.linear(a, wl, bl)).double() - ref64).abs().max() / ref64.abs().max())
        fl = 2.0 * m_rows * f * f
        peak_tf32 = peaks.get("bf16_tflops", 0.0) / 2.0
        layer = {"ms": ms_tc, "fp32_equivalent_tflops": fl / (ms_tc * 1e-3) / 1e12,
                 "tf32_mma_tflops_issued": 3 * fl / (ms_tc * 1e-3) / 1e12,
                 "frac_of_tf32_peak": (3 * fl / (ms_tc * 1e-3) / 1e12 / peak_tf32) if peak_tf32 else None,
                 "tf32_peak_tflops": peak_tf32, "tf32_peak_source": "half of MEASURED_PEAKS dense bf16 (cuBLAS)",
                 "max_err_vs_fp64": err_tc, "cublas_fp32_ms": ms_cublas, "cublas_fp32_max_err_vs_fp64": err_cublas,
                 "speedup_vs_cublas_fp32": ms_cublas / ms_tc,
                 "hbm_gbs": 2 * 8 * m_rows * f / (ms_tc * 1e-3) / 1e9}
        del a, pa, pc, ref64

        def bn_block(i, o):
            return [torch.nn.Linear(i, o), torch.nn.BatchNorm1d(o), torch.nn.ReLU()]
        torch.manual_seed(0)
        enc = torch.nn.Sequential(*bn_block(2, f), *[q for _ in range(4) for q in bn_block(f, f)], torch.nn.Linear(f, 2))
        dec = torch.nn.Sequential(torch.nn.Linear(2, f), torch.nn.ReLU(),
                                  *[q for _ in range(4) for q in (torch.nn.Linear(f, f), torch.nn.ReLU())],
                                  torch.nn.Linear(f, 2))
        for mod in (enc, dec):
            mod.to(dev).eval()
            for q in mod.parameters():
                q.requires_grad_(False)
        fe, fd = _mlp.FrozenMLP.from_module(enc), _mlp.FrozenMLP.from_module(dec)
        xb = torch.randn(m_rows, 2, device=dev, generator=gen)
        cb = torch.randn(m_rows, 2, device=dev, generator=gen)
        gmat = torch.randn(2, 2, device=dev, generator=gen)

        def chain(encode, dec_tangent):
            xg = xb.clone().requires_grad_(True)
            z = encode(xg)
            (dec_tangent(z, z @ gmat) * cb).sum().backward()
            return xg.grad

        ours = lambda: chain(fe.value, lambda z, v: fd.value_and_jvp(z, v)[1])
        theirs = lambda: chain(enc, lambda z, v: torch.autograd.functional.jvp(dec, z, v, create_graph=True)[1])
        ms_o, ms_t = timed(ours, reps=10), timed(theirs, reps=10)
        d_rows = (ours() - theirs()).abs().max(dim=1).values / theirs().abs().max()
        out["autoencoder_mlp_config3_40000rows"] = {
            "layer_512x512_sb_mlp_gemm": layer,
            "symmreg_i_autoencoder_part": {"tensor_core_chain_ms": ms_o, "pytorch_double_vjp_ms": ms_t,
                                           "speedup": ms_t / ms_o, "gemm_launches": 20,
                                           "median_rel_diff": float(d_rows.median()),
                                           "rows_above_1e-5": int((d_rows > 1e-5).sum()),
                                           "note": "rows differ where a ReLU unit sits within rounding of zero"},
            "kernel": "mlp_gemm_kernel (tcgen05 kind::tf32, 3xTF32, split accumulators, panel-format operands by bulk copy)"}
        del xb, cb
    except Exception as exc:   # noqa: BLE001
        out["autoencoder_mlp_config3_40000rows"] = {"error": repr(exc)}
    # WSINDy weak-form integrals over MANY trajectories (SURVEY §8a a10 / §8d): batches of Sel'kov-shaped trajectories
    # (T = 8000, 50 test functions) for the config-4 library and for the C5 library; algorithmic cost per time sample
    # (K−1−d) + 2·n_test·(K+d) flop (test functions are generated once per time tile for the whole batch) and 4·d bytes
    for (dd, pp, ntr) in ((2, 3, 28416), (3, 5, 4736)):
        wl = native.Library(dd, pp)
        xt = torch.rand(ntr, 8000, dd, device=dev, generator=gen) * 0.8 + 0.2
        ms = timed(lambda: native.wsindy_integrals(xt, wl, 0.002, 16.0, 50), reps=3)
        os.environ["SB_WSINDY_TC"] = "0"          # the CUDA-core batched kernel beside it (the library reads the switch per call)
        ms_simt = timed(lambda: native.wsindy_integrals(xt, wl, 0.002, 16.0, 50), reps=3)
        os.environ.pop("SB_WSINDY_TC")
        fl = (wl.K - 1 - dd) + 2 * 50 * (wl.K + dd)
        ns = ntr * 8000
        out[f"wsindy_integrals_d{dd}_K{wl.K}_{ntr}traj_T8000"] = {
            "samples_per_s": ns / (ms * 1e-3), "ms": ms, "kernel": "wsindy_tc_kernel (tcgen05 kind::tf32, 3xTF32 split)",
            "flop_per_sample": fl, "bytes_per_sample": 4 * dd,
            "algorithmic_tflops": fl * ns / (ms * 1e-3) / 1e12,
            "vs_fp32_cuda_core_peak": fl * ns / (ms * 1e-3) / 1e12 / fp32_peak,
            "hbm_gbs": 4 * dd * ns / (ms * 1e-3) / 1e9,
            "cuda_core_kernel_ms": ms_simt, "cuda_core_kernel_fp32_frac": fl * ns / (ms_simt * 1e-3) / 1e12 / fp32_peak}
        del xt
    x0 = torch.rand(10 ** 6, D, device=dev, generator=gen) * 2 - 1
    Xi = truth_xi(dev)
    ms = timed(lambda: native.rollout(x0, Xi, lib, 0.002, 2000, 10, "rk4"), reps=3)
    flops = 4 * ((K - 1 - D) + 2 * K * D) + 12 * D
    out["rk4_rollout_f32_1e6ics_2000steps"] = {"ic_steps_per_s": 2e9 / (ms * 1e-3), "ms": ms,
                                               "fp32_tflops": flops * 2e9 / (ms * 1e-3) / 1e12,
                                               "fp32_frac": flops * 2e9 / (ms * 1e-3) / 1e12 / fp32_peak}
    x0d, Xid = x0[: 10 ** 5].double(), Xi.double()
    ms = timed(lambda: native.rollout(x0d, Xid, lib, 0.002, 2000, 10, "rk4", record_dx=True), reps=3)
    out["rk4_rollout_f64_1e5ics_2000steps"] = {"ic_steps_per_s": 2e8 / (ms * 1e-3), "ms": ms}
    return out


if __name__ == "__main__":
    main()
