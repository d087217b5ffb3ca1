"""world_size-2 gloo test of the sample-sharded step: uneven shards, one all-reduce of packed SUMS, global mean.
The CUDA kernel is replaced by the CPU oracle through ShardedTrainStep's `local_sums` hook (test infrastructure
only); what is under test is the host-side combine logic that runs identically over NCCL."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, ret):
    sys.path[:0] = [ROOT, os.path.join(ROOT, "symmetry-ode-discovery_b200")]
    from oracle import sindy_oracle as O
    from sindy_b200 import native
    from sindy_b200.dist import ShardedTrainStep
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    d, p = 2, 3
    lib = native.Library(d, p)
    rng = np.random.default_rng(0)
    n = 1001
    x = rng.uniform(-1, 1, (n, d)).astype(np.float32)
    dx = rng.standard_normal((n, d)).astype(np.float32)
    W = rng.standard_normal((d, lib.K)).astype(np.float32)
    mask = (rng.random((d, lib.K)) > 0.3).astype(np.float32)
    cut = 313                                      # uneven shards: 313 and 688 samples
    lo, hi = (0, cut) if rank == 0 else (cut, n)

    def local_sums(w):
        s = O.train_step_sums(x[lo:hi], dx[lo:hi], w.numpy(), p)
        return torch.from_numpy(np.concatenate([[s["sum_sq"], s["n"]], s["grad_raw"].ravel()]))

    step = ShardedTrainStep(lib, local_sums=local_sums)
    loss, grad = step.step(torch.from_numpy(W), torch.from_numpy(mask), w_l1=0.01)
    ref_loss, ref_grad = O.mse_loss_and_grad(x, dx, W * mask, p)
    ref_loss += 0.01 * np.abs(W).sum()
    ref_grad = ref_grad * mask + 0.01 * np.sign(W)
    ok = abs(float(loss) - ref_loss) < 1e-10 * abs(ref_loss) and np.allclose(grad.numpy(), ref_grad, rtol=1e-5, atol=1e-7)
    # every rank holds the identical result (replicated optimiser state stays in sync)
    both = [torch.zeros_like(grad) for _ in range(world)]
    dist.all_gather(both, grad)
    ok = ok and torch.equal(both[0], both[1])
    ret[rank] = bool(ok)
    dist.destroy_process_group()


def test_sharded_step_two_ranks_gloo():
    world = 2
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = 29500 + (os.getpid() % 500)
    procs = [ctx.Process(target=_worker, args=(r, world, port, ret)) for r in range(world)]
    for q in procs:
        q.start()
    for q in procs:
        q.join(timeout=120)
        assert q.exitcode == 0
    assert ret.get(0) and ret.get(1)


def _stlsq_worker(rank, world, port, ret):
    sys.path[:0] = [ROOT, os.path.join(ROOT, "symmetry-ode-discovery_b200")]
    from oracle import sindy_oracle as O
    import sindy
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    d, p = 2, 3
    rng = np.random.default_rng(4)
    n = 3001
    x = rng.uniform(-1, 1, (n, d))
    truth = np.zeros((d, 10)); truth[0, 1], truth[0, 2], truth[1, 1], truth[1, 8] = -0.5, 1.5, 2.0, -1.0
    y = O.theta(x, p) @ truth.T + 0.01 * rng.standard_normal((n, d))
    cut = 1200                                     # uneven shards

    def stats_of(lo, hi):                          # the kernel's job, here by the oracle: G, b, Σy², n of a shard
        th = O.theta(x[lo:hi], p).astype(np.float64)
        return {"G": torch.from_numpy(th.T @ th), "b": torch.from_numpy(th.T @ y[lo:hi]),
                "yy": torch.from_numpy((y[lo:hi] ** 2).sum(0)), "n": hi - lo}

    lo, hi = (0, cut) if rank == 0 else (cut, n)
    merged = sindy.allreduce_statistics(stats_of(lo, hi))
    whole = stats_of(0, n)
    ok = merged["n"] == n and all(torch.allclose(merged[k], whole[k], rtol=1e-12, atol=1e-12) for k in ("G", "b", "yy"))
    # every rank runs the identical thresholding iterations on the merged statistics
    torch.manual_seed(0)
    reg = sindy.SINDyRegression(d, p, False, False, threshold=0.1, device="cpu", constrain_constant=True)
    for _ in range(5):
        _, conv = sindy.solve_SINDy_one_step(reg, None, None, 0.0, 0.1, stats=merged)
        if conv:
            break
    ok = ok and np.array_equal(reg.mask.numpy() != 0, truth != 0) and np.allclose(reg.Xi.detach().numpy() * reg.mask.numpy(), truth, atol=5e-3)
    both = [torch.zeros_like(reg.Xi.data) for _ in range(world)]
    dist.all_gather(both, reg.Xi.data.clone())
    ret[rank] = bool(ok and torch.equal(both[0], both[1]))
    dist.destroy_process_group()


def test_sharded_stlsq_two_ranks_gloo():
    """SURVEY §8e: STLSQ over sample shards = ONE all-reduce of (G, b, Σy², n), then the same K×K solves on every rank
    (identical masks and coefficients). The per-shard statistics come from the oracle here (no GPU)."""
    world = 2
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = 29500 + ((os.getpid() + 7) % 500)
    procs = [ctx.Process(target=_stlsq_worker, args=(r, world, port, ret)) for r in range(world)]
    for q in procs:
        q.start()
    for q in procs:
        q.join(timeout=120)
        assert q.exitcode == 0
    assert ret.get(0) and ret.get(1)


def test_single_process_step_matches_formula():
    sys.path[:0] = [ROOT, os.path.join(ROOT, "symmetry-ode-discovery_b200")]
    from sindy_b200 import native
    from sindy_b200.dist import mse_from_sums
    lib = native.Library(2, 2)
    packed = torch.arange(2 + 12, dtype=torch.float64) + 1.0
    packed[1] = 50.0
    w = torch.ones(2, 6)
    loss, grad = mse_from_sums(packed, lib, w)
    assert abs(float(loss) - 1.0 / 100.0) < 1e-15
    assert torch.allclose(grad.double(), packed[2:].view(2, 6) * (2.0 / 100.0))


def test_reference_arm_under_torchrun_prints_one_line_from_rank_zero():
    """`bench.py --impl reference` launched under torchrun for N > 1: rank 0 alone runs the reference's CPU path and
    prints ONE JSON line (impl, cpu_baseline, e2e with zero copy bytes), the other rank exits 0 silently. The step is
    the reference's own whenever the reference mirror oracle/_ref (written by build()) is there, else the oracle's port
    of it; no GPU involved."""
    import json
    import subprocess
    ref = os.path.join(ROOT, "oracle", "_ref")
    kind = "reference" if os.path.isfile(os.path.join(ref, "sindy.py")) else "port"
    port = 29600 + (os.getpid() % 300)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
           "--steps", "1", "--warmup", "1", "--cpu-samples", "20000"]
    env = dict(os.environ, OMP_NUM_THREADS="4")
    env.pop("SINDY_B200_REFERENCE", None)           # the arm must find the mirror by itself
    out = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out.stdout
    rec = json.loads(lines[0])
    assert rec["impl"] == "reference" and rec["n_gpus"] == 2 and rec["steps"] == 1 and rec["higher_is_better"] is True
    assert rec["unit"] == "samples/s" and rec["value"] > 0
    assert rec["cpu_baseline"]["kind"] == kind and rec["cpu_baseline"]["value"] == rec["value"]
    assert rec["e2e"]["value"] == rec["value"] and rec["e2e"]["h2d_bytes_per_step"] == 0 == rec["e2e"]["d2h_bytes_per_step"]
