"""Reference arm of bench.py: the UNMODIFIED reference (helmholtz-analytics/mpi4torch, installed
into baseline/_ref by baseline/build_ref.sh) driven through its own public API on the same
config as the product arm.

What runs (nothing of mpi4torch_b200 is imported in this process):

    W       fp32 [4096, 4096] on the GPU (the reference cannot communicate bf16/f16:
            torch2mpitype, reference csrc/extension.cpp:106-129, so the parameter it averages is fp32)
    W_avg = comm.Allreduce(W, MPI_SUM) / comm.size          reference op (host-staged: the MPI under
                                                            it is not CUDA-aware, extension.cpp:61-104)
    y     = x @ W_avg.to(bf16).T                            stock torch.matmul (cuBLAS), bf16
    loss  = comm.Allreduce(sum((y - t)^2) / (B * size), MPI_SUM)
    loss.backward(); W -= lr * W.grad                       adjoint Allreduces run inside backward

This is the data-parallel pattern of the reference's examples/simple_linear_regression.py:27-35
applied to the 4096x4096 layer.  MPI is baseline/mpi_shim (POSIX shared memory), because the image
has no MPI; ranks come from torchrun's RANK/WORLD_SIZE.
"""
from __future__ import annotations

import importlib.util
import json
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
IN_F = OUT_F = 4096
POOL = 4


def _load_by_path(name: str, path: str):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _unavailable(why: str) -> int:
    if int(os.environ.get("RANK", "0")) == 0:
        print(json.dumps({"impl": "reference", "unavailable": why[:400]}), flush=True)
    return 0


def ensure_built() -> str | None:
    """Builds baseline/_ref when missing (rank 0 only; the others wait).  Returns an error string."""
    marker = os.path.join(HERE, "_ref", "mpi4torch", "__init__.py")
    lib = os.path.join(HERE, "mpi_shim", "lib", "libmpi.so")
    rank = int(os.environ.get("RANK", "0"))
    if os.path.exists(marker) and os.path.exists(lib):
        return None
    if rank == 0:
        try:
            res = subprocess.run(["bash", os.path.join(HERE, "build_ref.sh")], capture_output=True, text=True, timeout=900)
            if res.returncode != 0:
                return "build_ref.sh failed: " + (res.stdout + res.stderr)[-300:].replace("\n", " ")
        except Exception as exc:  # pragma: no cover
            return f"build_ref.sh failed: {type(exc).__name__}: {exc}"
    else:
        t0 = time.time()
        while not (os.path.exists(marker) and os.path.exists(lib)):
            if time.time() - t0 > 900:
                return "timed out waiting for rank 0 to build baseline/_ref"
            time.sleep(1.0)
        time.sleep(2.0)
    return None


def run(args) -> int:
    import torch

    if not torch.cuda.is_available():
        return _unavailable("no CUDA device visible")
    err = ensure_built()
    if err:
        return _unavailable(err)
    sys.path.insert(0, os.path.join(HERE, "_ref"))
    local_rank = int(os.environ.get("LOCAL_RANK", os.environ.get("RANK", "0")))
    torch.cuda.set_device(local_rank % torch.cuda.device_count())
    dev = torch.device("cuda", torch.cuda.current_device())
    try:
        import mpi4torch  # the reference
    except Exception as exc:
        return _unavailable(f"reference import failed: {type(exc).__name__}: {exc}")
    comm = mpi4torch.COMM_WORLD
    rank, size = comm.rank, comm.size
    timing = _load_by_path("m4t_timing_standalone", os.path.join(ROOT, "mpi4torch_b200", "utils", "timing.py"))
    B = args.batch
    lr = 1e-5
    steps, warmup = args.steps, max(args.warmup, 3)

    g = torch.Generator().manual_seed(0)
    W = (torch.randn(OUT_F, IN_F, generator=g) * IN_F ** -0.5).to(dev).requires_grad_()  # fp32 master weight
    torch.manual_seed(1234 + rank)
    xs = [torch.randn(B, IN_F, device=dev, dtype=torch.bfloat16) for _ in range(POOL)]
    ts = [torch.randn(B, OUT_F, device=dev, dtype=torch.bfloat16) for _ in range(POOL)]

    def train_step(x, t):
        W.grad = None
        w_avg = comm.Allreduce(W, mpi4torch.MPI_SUM) / size
        y = x @ w_avg.to(torch.bfloat16).t()
        local = (y.float() - t.float()).square().sum() / (B * size)
        loss = comm.Allreduce(local, mpi4torch.MPI_SUM)
        loss.backward()
        with torch.no_grad():
            W.add_(W.grad, alpha=-lr)
        return loss.detach()

    def max_ranks(v: float) -> float:
        return float(comm.Allreduce(torch.tensor([v], dtype=torch.float64), mpi4torch.MPI_MAX)[0])

    def barrier():
        comm.Allreduce(torch.zeros(1, dtype=torch.float64), mpi4torch.MPI_SUM)

    for i in range(warmup):
        train_step(xs[i % POOL], ts[i % POOL])
    torch.cuda.synchronize()
    barrier()
    sampler = timing.ClockSampler(gpu_index=dev.index).start() if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    barrier()
    e0.record()
    for i in range(steps):
        loss = train_step(xs[i % POOL], ts[i % POOL])
    e1.record()
    torch.cuda.synchronize()
    barrier()
    dev_ms = max_ranks(e0.elapsed_time(e1))
    final_loss = float(loss)

    # end to end: per-step H2D of the batch from pinned memory + D2H of the loss
    pin_x = [torch.randn(B, IN_F, dtype=torch.bfloat16).pin_memory() for _ in range(2)]
    pin_t = [torch.randn(B, OUT_F, dtype=torch.bfloat16).pin_memory() for _ in range(2)]

    def e2e_steps(n: int) -> float:
        last = 0.0
        for i in range(n):
            x = pin_x[i % 2].to(dev, non_blocking=True)
            t = pin_t[i % 2].to(dev, non_blocking=True)
            last = float(train_step(x, t))
        return last

    e2e_steps(2)
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    e2e_steps(steps)
    torch.cuda.synchronize()
    e2e_s = max_ranks(time.perf_counter() - t0)
    barrier()
    clocks = sampler.stop() if sampler is not None else None

    total = float(B) * size * steps
    out = {
        "metric": "dp_linear4096_train_samples_per_s",
        "value": total / (dev_ms * 1e-3),
        "unit": "samples/s",
        "n_gpus": size,
        "steps": steps,
        "warmup": warmup,
        "ms_per_step": dev_ms / steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "bf16 GEMMs (torch.matmul), fp32 parameter/gradient Allreduce (the reference has no bf16 MPI datatype)",
        "data": "synthetic (random-init 4096x4096 weight, random batches)",
        "impl": "reference",
        "config": {
            "model": "dp_linear_4096x4096 (Allreduce(params)/size -> matmul, loss Allreduce, backward, SGD)",
            "global_batch": B * size,
            "seq_len": 1,
            "parallelism": f"dp{size}",
            "per_gpu_batch": B,
            "cold_cache": f"inputs rotate over {POOL} batches > 126 MB L2",
            "reference": "helmholtz-analytics/mpi4torch 0.1.3 unmodified (baseline/_ref)",
            "mpi": "baseline/mpi_shim (POSIX shared memory, not CUDA-aware -> reference's host-staging path)",
        },
        "gpu_launches": 0,
        "clocks": clocks,
        "e2e": {
            "value": total / e2e_s,
            "unit": "samples/s",
            "h2d_bytes_per_step": 2 * B * IN_F * 2,
            "d2h_bytes_per_step": 4,
            "ms_per_step": e2e_s * 1e3 / steps,
        },
        "final_loss": final_loss,
    }
    if not args.no_extras and size > 1:
        # Allreduce forward+backward through the reference's autograd node, fp32 (same byte counts as ours)
        sweep = {}
        for nbytes in (1 << 10, 1 << 16, 1 << 20, 1 << 24, 1 << 26):
            n = nbytes // 4
            x = torch.randn(n, device=dev).requires_grad_()
            gr = torch.ones(n, device=dev)
            iters = 10 if nbytes <= (1 << 20) else 3

            def fb():
                x.grad = None
                comm.Allreduce(x, mpi4torch.MPI_SUM).backward(gr)

            fb()
            torch.cuda.synchronize()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                fb()
            b.record()
            torch.cuda.synchronize()
            ms = max_ranks(a.elapsed_time(b)) / iters
            sweep[str(nbytes)] = round(2.0 * nbytes * (2.0 * (size - 1) / size) / (ms * 1e-3) / 1e9, 4)
        out["allreduce_fwd_bwd_busbw_gbs"] = sweep
        out["allreduce_sweep_dtype"] = "float32"
    if not args.no_extras and rank == 0:
        try:
            res = subprocess.run([os.path.join(HERE, "mpi_shim", "bin", "mpirun"), "-np", "2", sys.executable,
                                  os.path.join(HERE, "ref_linreg.py"), "--steps", "30"],
                                 capture_output=True, text=True, timeout=300,
                                 env={k: v for k, v in os.environ.items()
                                      if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MPISHIM_RANK", "MPISHIM_SIZE")})
            line = [ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1]
            out["linreg_cpu_np2_step_per_s"] = json.loads(line)["reference_step_per_s"]
        except Exception as exc:  # pragma: no cover
            out["linreg_cpu_np2_step_per_s"] = {"error": f"{type(exc).__name__}: {exc}"[:200]}
    if rank == 0:
        print(json.dumps(out), flush=True)
    return 0
