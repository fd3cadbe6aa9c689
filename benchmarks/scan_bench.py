#!/usr/bin/env python
"""Scan forward+backward on the NVLink backend, 4 KiB .. 256 MiB per rank, bf16 and fp32, next to two comparisons
measured in the same process:

  allreduce2  the forced two-shot Allreduce of the same size: the same traffic per rank ((P-1)/P of the message in
              and out), so it is the ceiling a Scan can aim for
  ag_cumsum   what a user writes without Scan: torch.cumsum(comm.Allgather(x[None], 0), 0)[rank] (P times the data,
              backward through cumsum + Reduce_scatter)

    python benchmarks/scan_bench.py              # every world size the box has (2, 4, 8 GPUs), one job each
    python -m mpi4torch_b200.launch -np 8 benchmarks/scan_bench.py [--out f.json]

Every time is CUDA-event timed on the launching stream, after 3 warm-ups, with a 256 MiB L2 flush and a host barrier
before each timed call, and is the max over ranks (milliseconds).  The first line names the card and its power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SIZES = [4 << 10, 16 << 10, 64 << 10, 256 << 10, 1 << 20, 4 << 20, 16 << 20, 64 << 20, 256 << 20]


def card() -> dict:
    info = {"gpu": torch.cuda.get_device_name(0), "gpus": torch.cuda.device_count()}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_and_max_sm_clock"] = out
    except (OSError, subprocess.TimeoutExpired):
        info["power_limit_and_max_sm_clock"] = None
    return info


def sweep_all(args) -> int:
    """Not under a launcher: one job per world size the box offers."""
    n = torch.cuda.device_count()
    if n < 2:
        print("scan_bench needs at least 2 GPUs", file=sys.stderr)
        return 1
    rc = 0
    for np_ in [s for s in (2, 4, 8) if s <= n]:
        cmd = [sys.executable, "-m", "mpi4torch_b200.launch", "-np", str(np_), os.path.abspath(__file__),
               "--max-mb", str(args.max_mb)]
        if args.out:
            root, ext = os.path.splitext(args.out)
            cmd += ["--out", f"{root}_np{np_}{ext or '.json'}"]
        rc |= subprocess.run(cmd, cwd=ROOT).returncode
    return rc


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--max-mb", type=int, default=256)
    args = ap.parse_args()
    if "RANK" not in os.environ:
        return sweep_all(args)

    import mpi4torch_b200 as m4t
    from mpi4torch_b200.utils.timing import L2Flusher, cuda_time_ms, max_over_ranks

    comm = m4t.COMM_WORLD
    P, R = comm.size, comm.rank
    assert m4t.cuda_backend_ready(), "scan_bench measures the NVLink backend: no CUDA backend came up"
    dev = torch.device("cuda", torch.cuda.current_device())
    flusher = L2Flusher(dev)

    def timed(fn, iters):
        t = cuda_time_ms(fn, iters, warmup=3, flusher=flusher, barrier=comm.Barrier)
        return max_over_ranks(statistics.median(t), comm)

    if R == 0:
        print(json.dumps({"world": P, **card(), "nvls": m4t.has_nvls()}), flush=True)
    rows = []
    for dtype in (torch.bfloat16, torch.float32):
        es = torch.empty(0, dtype=dtype).element_size()
        for nbytes in [b for b in SIZES if b <= (args.max_mb << 20)]:
            n = nbytes // es
            iters = 30 if nbytes <= (4 << 20) else 8
            x = torch.randn(n, device=dev).to(dtype).requires_grad_()
            g = torch.randn(n, device=dev).to(dtype)

            def scan_fwd():
                with torch.no_grad():
                    comm.Scan(x, m4t.MPI_SUM)

            def scan_fwd_bwd():
                x.grad = None
                comm.Scan(x, m4t.MPI_SUM).backward(g)

            def ar_fwd():
                with torch.no_grad():
                    comm.Allreduce(x, m4t.MPI_SUM)

            def ar_fwd_bwd():
                x.grad = None
                comm.Allreduce(x, m4t.MPI_SUM).backward(g)

            def ag_cumsum_fwd_bwd():
                x.grad = None
                torch.cumsum(comm.Allgather(x[None], 0), 0)[R].backward(g)

            row = {"dtype": str(dtype).replace("torch.", ""), "bytes": nbytes}
            row["scan_fwd_ms"] = timed(scan_fwd, iters)
            row["scan_fwd_bwd_ms"] = timed(scan_fwd_bwd, iters)
            m4t._C.set_tuning("force_algo", 2)
            try:
                row["allreduce2_fwd_ms"] = timed(ar_fwd, iters)
                row["allreduce2_fwd_bwd_ms"] = timed(ar_fwd_bwd, iters)
            finally:
                m4t._C.set_tuning("force_algo", 0)
            row["ag_cumsum_fwd_bwd_ms"] = timed(ag_cumsum_fwd_bwd, iters)
            # same answer as the composition (tolerance: the composition's cumsum adds in another order)
            with torch.no_grad():
                ok = torch.allclose(comm.Scan(x, m4t.MPI_SUM).float(),
                                    torch.cumsum(comm.Allgather(x[None], 0).float(), 0)[R], rtol=2e-2, atol=2e-2)
            row["matches_composition"] = bool(max_over_ranks(0.0 if ok else 1.0, comm) == 0.0)
            row["scan_fwd_over_allreduce2_fwd"] = row["scan_fwd_ms"] / row["allreduce2_fwd_ms"]
            row["scan_fwd_bwd_over_ag_cumsum"] = row["scan_fwd_bwd_ms"] / row["ag_cumsum_fwd_bwd_ms"]
            # message bytes per rank over the forward time
            row["scan_fwd_algbw_GBs"] = nbytes / (row["scan_fwd_ms"] * 1e-3) / 1e9
            rows.append(row)
            if R == 0:
                print(json.dumps(row), flush=True)
            del x, g
            torch.cuda.empty_cache()
    if R == 0 and args.out:
        with open(args.out, "w") as f:
            json.dump({"world": P, **card(), "rows": rows}, f, indent=1)
    return 0


if __name__ == "__main__":
    sys.exit(main())
