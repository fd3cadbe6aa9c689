#!/usr/bin/env python
"""Headline benchmark (see DESIGN.md).

Flagship step = BASELINE.json config "4096x4096 linear layer: Allreduce(params)
-> GEMM fused, loss Allreduce backward": every rank holds a 4096x4096 bf16
weight and a private batch; one step is, THROUGH THE AUTOGRAD GRAPH,

    local = dp_linear_mse(x, W, t)            Allreduce(W)/size -> tcgen05 GEMM -> MSE epilogue
    loss  = comm.Allreduce(local, MPI_SUM)    the library's differentiable Allreduce
    loss.backward()                           adjoint Allreduce of the scalar, wgrad GEMM, adjoint
                                              Allreduce of dW fused with the SGD update

    python bench.py --gpus N --steps K --warmup W            (N>1: under torchrun)
    python bench.py --impl reference ...                      (the unmodified reference, baseline/)
    python bench.py ... --dump-outputs DIR                    (also write the last timed step's results as .npy)

Prints ONE JSON line on rank 0.  `value` = samples/s over the whole job, timed on the device (CUDA
events, max over ranks); `e2e` = the same step through the public API including per-step H2D of the
batch from pinned memory and D2H of the loss.  First-class extra keys: the Allreduce fwd+bwd bus
bandwidth table (BASELINE.json's metric) and the CPU linear-regression step/s at world size 2.
At N > 1 a self-check block runs before anything is timed ("checks").
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "dp_linear4096_train_samples_per_s"
IN_F = OUT_F = 4096
PER_GPU_BATCH = 8192
POOL = 4  # rotating input batches: 4 x (64 MiB x + 64 MiB t) >> 126 MB L2
DUMP_SAMPLE = 1 << 22  # weight elements written by --dump-outputs (16 MiB as float32)


def linreg_cpu_step_per_s() -> object:
    """BASELINE.json config 1 (CPU, world size 2) through this library's launcher and shm backend."""
    env = {k: v for k, v in os.environ.items()
           if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "LOCAL_WORLD_SIZE", "MASTER_PORT", "MASTER_ADDR", "M4T_JOB_ID",
                        "TORCHELASTIC_RUN_ID", "GROUP_RANK", "ROLE_RANK")}
    env["M4T_CUDA"] = "0"
    env["PYTHONPATH"] = ROOT + os.pathsep + env.get("PYTHONPATH", "")
    try:
        res = subprocess.run([sys.executable, "-m", "mpi4torch_b200.launch", "-np", "2",
                              os.path.join(ROOT, "benchmarks", "linreg_steps.py"), "--steps", "30", "--no-gloo"],
                             capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
        line = [ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1]
        return json.loads(line)["ours_step_per_s"]
    except Exception as exc:  # pragma: no cover
        return {"error": f"{type(exc).__name__}: {exc}"[:200]}


def dump_outputs(out_dir: str, loss, weight) -> None:
    """What the last timed step hands its caller, as float32 .npy files: the global loss and the updated weight.
    The weight is written as a fixed sample of DUMP_SAMPLE elements (seeded, in flat index order), so two builds
    run with the same arguments can be compared element for element."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    flat = weight.detach().reshape(-1)
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().reshape(1).cpu().numpy())
    np.save(os.path.join(out_dir, "weight_sample.npy"), flat[idx.to(flat.device)].float().cpu().numpy())


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=PER_GPU_BATCH, help="per-GPU batch (weak scaling)")
    ap.add_argument("--no-extras", action="store_true", help="skip the allreduce sweep / regression extras")
    ap.add_argument("--no-checks", action="store_true", help="skip the multi-GPU self-check block")
    ap.add_argument("--unfused", action="store_true", help="force the unfused Allreduce + GEMM composition")
    ap.add_argument("--plain-sgd", action="store_true", help="weight.grad + separate SGD instead of the optimizer in backward")
    ap.add_argument("--full-sweep", action="store_true", help="1 KiB .. 1 GiB in x4 steps instead of the quick table")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's loss and a fixed sample of the updated weight to DIR/*.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        import reference_arm

        return reference_arm.run(args)

    import torch

    if not torch.cuda.is_available():
        print(json.dumps({"metric": METRIC, "error": "no CUDA device visible"}), flush=True)
        return 1
    args.warmup = max(args.warmup, 3)

    import mpi4torch_b200 as m4t
    from mpi4torch_b200.models import DPLinearModel
    from mpi4torch_b200.utils import ClockSampler, bind_to_gpu_numa

    comm = m4t.COMM_WORLD
    rank, size = comm.rank, comm.size
    # pinned staging buffers must live on the GPU's own NUMA node (H2D is the e2e bound)
    numa = bind_to_gpu_numa(torch.cuda.current_device())
    if size != args.gpus and rank == 0:
        sys.stderr.write(f"[bench] warning: --gpus {args.gpus} but world size is {size}\n")
    dev = torch.device("cuda", torch.cuda.current_device())
    assert m4t.cuda_backend_ready(), "native CUDA backend missing: refusing to benchmark a fallback"
    _C = m4t._C
    B = args.batch

    # ---------------- multi-GPU self checks (before anything is timed) ----------------
    checks = None
    if size > 1 and not args.no_checks:
        from benchmarks.selfcheck import run_checks

        checks = run_checks(comm, dev)
        if not checks.get("ok", False):
            if rank == 0:
                print(json.dumps({"metric": METRIC, "error": "self-check failed", "checks": checks}), flush=True)
            return 2

    torch.manual_seed(1234 + rank)
    model = DPLinearModel(IN_F, OUT_F, comm, device=dev, dtype=torch.bfloat16, lr=1e-5, fused=not args.unfused,
                          sgd_in_backward=not args.plain_sgd)
    xs = [torch.randn(B, IN_F, device=dev, dtype=torch.bfloat16) for _ in range(POOL)]
    ts = [torch.randn(B, OUT_F, device=dev, dtype=torch.bfloat16) for _ in range(POOL)]

    def step(i: int, mdl=model):
        return mdl.train_step(xs[i % POOL], ts[i % POOL])

    def max_ranks(v: float) -> float:
        t = torch.tensor([v], dtype=torch.float64)
        return float(comm.Allreduce(t, m4t.MPI_MAX)[0])

    def timed(fn, steps: int, warmup: int):
        for i in range(warmup):
            fn(i)
        torch.cuda.synchronize()
        comm.Barrier()
        l0 = _C.kernel_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        comm.Barrier()
        e0.record()
        out = None
        for i in range(steps):
            out = fn(i)
        e1.record()
        torch.cuda.synchronize()
        comm.Barrier()
        return max_ranks(e0.elapsed_time(e1)), _C.kernel_launch_count() - l0, out

    # ---------------- device-timed region (the headline) ----------------
    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    comm.Barrier()
    sampler = ClockSampler(gpu_index=dev.index).start() if rank == size - 1 else None  # not on the rank that prints
    table0 = dict(_C.kernel_launch_table())
    dev_ms, launches, loss = timed(step, args.steps, 0)
    final_loss = float(loss)
    # which tensor-core / fused kernels really ran in the timed region (launches per step)
    path = {k: (v - table0.get(k, 0)) / args.steps for k, v in dict(_C.kernel_launch_table()).items()
            if v - table0.get(k, 0) > 0}
    if args.dump_outputs:  # before the end-to-end region trains the same model further
        if rank == 0:
            dump_outputs(args.dump_outputs, loss, model.weight)
        comm.Barrier()

    # ---------------- end-to-end region (public API + H2D/D2H every step) ----------------
    pin_x = [torch.randn(B, IN_F, dtype=torch.bfloat16).pin_memory() for _ in range(2)]
    pin_t = [torch.randn(B, OUT_F, dtype=torch.bfloat16).pin_memory() for _ in range(2)]
    dx = [torch.empty(B, IN_F, device=dev, dtype=torch.bfloat16) for _ in range(2)]
    dt_ = [torch.empty(B, OUT_F, device=dev, dtype=torch.bfloat16) for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]

    def prefetch(i: int):
        b = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[b])
            dx[b].copy_(pin_x[b], non_blocking=True)
            dt_[b].copy_(pin_t[b], non_blocking=True)
            ready[b].record(copy_stream)

    def e2e_steps(n: int) -> float:
        last = 0.0
        for b in range(2):
            consumed[b].record()
        prefetch(0)
        for i in range(n):
            b = i % 2
            if i + 1 < n:
                prefetch(i + 1)
            torch.cuda.current_stream().wait_event(ready[b])
            value = model.train_step(dx[b], dt_[b])
            consumed[b].record()
            last = float(value)  # D2H read of the step's result
        return last

    e2e_steps(args.warmup)
    torch.cuda.synchronize()
    comm.Barrier()
    t0 = time.perf_counter()
    e2e_steps(args.steps)
    torch.cuda.synchronize()
    e2e_s = max_ranks(time.perf_counter() - t0)
    comm.Barrier()
    clock_summary = sampler.stop() if sampler is not None else None
    # the sampling rank hands its summary to rank 0 (host-side, after all timing)
    blob = torch.zeros(4, dtype=torch.float64)
    if clock_summary is not None:
        reasons = clock_summary.get("reasons", [])
        code = sum(1 << i for i, k in enumerate(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"))
                   if k in reasons)
        blob = torch.tensor([clock_summary.get("sm_mhz") or 0.0, clock_summary.get("sm_max_mhz") or 0.0, float(code),
                             float(clock_summary.get("samples", 0))], dtype=torch.float64)
    blob = comm.Allreduce(blob, m4t.MPI_SUM)
    code = int(blob[2])
    clocks = {"sm_mhz": float(blob[0]), "sm_max_mhz": float(blob[1]),
              "reasons": [k for i, k in enumerate(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"))
                          if code >> i & 1],
              "samples": int(blob[3]), "sampled_gpu": size - 1}

    total_samples = float(B) * size * args.steps
    value = total_samples / (dev_ms * 1e-3)
    e2e_value = total_samples / e2e_s
    flops_per_step = 2 * 2.0 * B * IN_F * OUT_F  # forward GEMM + wgrad GEMM, per GPU
    out = {
        "metric": METRIC,
        "value": value,
        "unit": "samples/s",
        "n_gpus": size,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": dev_ms / args.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "bf16",
        "data": "synthetic (random-init 4096x4096 weight, random batches)",
        "impl": "ours",
        "config": {
            "model": "dp_linear_4096x4096 (Allreduce(params)->GEMM, loss Allreduce, backward, SGD)",
            "global_batch": B * size,
            "seq_len": 1,
            "parallelism": f"dp{size}",
            "per_gpu_batch": B,
            "cold_cache": f"inputs rotate over {POOL} batches (>= {POOL * 2 * B * IN_F * 2 >> 20} MiB) > 126 MB L2",
            "autograd": True,
            "optimizer_in_backward": bool(model.sgd_in_backward and model._in_backward(xs[0])),
            "kernels_per_step": path,
            "heap_mode": m4t.heap_mode(),
            "nvls": m4t.has_nvls(),
            "numa_bind": numa,
        },
        "tflops_per_gpu": flops_per_step * args.steps / (dev_ms * 1e-3) / 1e12,
        "gpu_launches": int(launches),
        "clocks": clocks,
        "e2e": {
            "value": e2e_value,
            "unit": "samples/s",
            "h2d_bytes_per_step": 2 * B * IN_F * 2,
            "d2h_bytes_per_step": 4,
            "ms_per_step": e2e_s * 1e3 / args.steps,
        },
        "final_loss": final_loss,
    }
    if checks is not None:
        out["checks"] = checks
    if not args.no_extras:
        # the same step with weight.grad + a separate SGD update (no optimizer inside backward)
        try:
            plain = DPLinearModel(IN_F, OUT_F, comm, device=dev, dtype=torch.bfloat16, lr=1e-5, fused=not args.unfused,
                                  sgd_in_backward=False, seed=1)
            ms, _, _ = timed(lambda i: step(i, plain), max(5, args.steps // 2), 3)
            out["plain_autograd_sgd_ms_per_step"] = ms / max(5, args.steps // 2)
            del plain
        except Exception as exc:  # pragma: no cover
            out["plain_autograd_sgd_ms_per_step"] = {"error": f"{type(exc).__name__}: {exc}"[:200]}
        if size > 1:
            # NOT the headline: the same step when the library is allowed to use that the fused update leaves
            # bit-identical weights on every rank (Allreduce(W)/size == W, forward collective elided)
            try:
                rep = DPLinearModel(IN_F, OUT_F, comm, device=dev, dtype=torch.bfloat16, lr=1e-5, fused=not args.unfused,
                                    assume_replicated=True, seed=2)
                ms, _, _ = timed(lambda i: step(i, rep), max(5, args.steps // 2), 3)
                out["replicated_params_elided_allreduce_ms_per_step"] = ms / max(5, args.steps // 2)
                del rep
            except Exception as exc:  # pragma: no cover
                out["replicated_params_elided_allreduce_ms_per_step"] = {"error": f"{type(exc).__name__}: {exc}"[:200]}
        if size > 1:
            try:
                from benchmarks.extras import allreduce_busbw_sweep

                out["allreduce_fwd_bwd_busbw_gbs"] = allreduce_busbw_sweep(comm, dev, quick=not args.full_sweep)
                out["allreduce_sweep_dtype"] = "bfloat16"
            except Exception as exc:  # pragma: no cover
                out["allreduce_fwd_bwd_busbw_gbs"] = {"error": f"{type(exc).__name__}: {exc}"[:200]}
        comm.Barrier()
        if rank == 0:
            out["linreg_cpu_np2_step_per_s"] = linreg_cpu_step_per_s()
        comm.Barrier()
    if rank == 0:
        print(json.dumps(out), flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main())
