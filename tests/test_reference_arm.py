"""The reference arm of bench.py (baseline/): the shared-memory MPI shim on its own, a cross-check of this library's
results against what the UNMODIFIED reference computed over the shim (recorded in tests/golden/), and the shim's speed
against this library's CPU backend - the shim must be a fair stand-in, not a strawman."""
import json
import os
import shutil
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
SHIM = ROOT / "baseline" / "mpi_shim"
MPIRUN = SHIM / "bin" / "mpirun"
GOLDEN = ROOT / "tests" / "golden" / "reference_cross_np3.json"


def _run(cmd, timeout=600, env=None):
    e = dict(os.environ)
    e.pop("RANK", None)
    e.pop("WORLD_SIZE", None)
    if env:
        e.update(env)
    return subprocess.run([str(c) for c in cmd], capture_output=True, text=True, timeout=timeout, env=e, cwd=str(ROOT))


@pytest.fixture(scope="module")
def shim():
    res = _run(["make", "-C", SHIM])
    assert res.returncode == 0, res.stdout + res.stderr
    assert (SHIM / "lib" / "libmpi.so").exists()
    return SHIM


@pytest.mark.parametrize("np_", [1, 2, 3, 5])
def test_mpi_shim_selftest(shim, np_, tmp_path):
    exe = tmp_path / "selftest"
    res = _run([SHIM / "bin" / "mpicxx", "-O2", "-std=c++17", "-o", exe, SHIM / "test" / "selftest.cpp"])
    assert res.returncode == 0, res.stderr
    res = _run([MPIRUN, "-np", np_, exe], timeout=300)
    assert res.returncode == 0, res.stdout + res.stderr
    assert f"mpishim selftest np={np_}: ok" in res.stdout


# The values in GOLDEN are this program's output through the reference (`import mpi4torch as m`, under
# baseline/mpi_shim/bin/mpirun -np 3).
CROSS = r'''
import json, sys, time, torch
sys.path.insert(0, sys.argv[1]); import mpi4torch_b200 as m
comm = m.COMM_WORLD
g = torch.Generator().manual_seed(7 + comm.rank)
out = {}
x = torch.randn(1 << 16, generator=g, dtype=torch.float64).requires_grad_()
y = comm.Allreduce(x, m.MPI_SUM)
(y * (comm.rank + 1)).sum().backward()
out["fwd"] = float(y.detach().double().sum()); out["fwd_abs"] = float(y.detach().abs().sum())
out["bwd"] = float(x.grad.sum())
a = torch.randn(3, comm.rank + 2, 4, generator=g, dtype=torch.float64)
out["allgather"] = float((comm.Allgather(a, 1) * torch.arange(4.0, dtype=torch.float64)).sum())
big = torch.randn(1 << 22, generator=g)   # 16 MiB fp32
for _ in range(2): comm.Allreduce(big, m.MPI_SUM)
t0 = time.perf_counter()
for _ in range(5): comm.Allreduce(big, m.MPI_SUM)
out["allreduce_16MiB_ms"] = (time.perf_counter() - t0) / 5 * 1e3
if comm.rank == 0: print(json.dumps(out))
'''


# The shim's Allreduce as the reference calls it for a CPU tensor: a fresh result buffer, then one MPI_Allreduce.
SHIM_ALLREDUCE = r'''
import ctypes, json, sys, time, torch
sys.path.insert(0, sys.argv[1]); import mpi4py.MPI as M
MPI_FLOAT, MPI_SUM, MPI_COMM_WORLD = 6, 3, 1   # baseline/mpi_shim/include/mpi.h
def allreduce(x):
    recv = torch.empty_like(x)
    rc = M._lib.MPI_Allreduce(ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(recv.data_ptr()), x.numel(), MPI_FLOAT,
                              MPI_SUM, MPI_COMM_WORLD)
    assert rc == 0, rc
    return recv
g = torch.Generator().manual_seed(7 + M.COMM_WORLD.rank)
big = torch.randn(1 << 22, generator=g)   # 16 MiB fp32
for _ in range(2): allreduce(big)
t0 = time.perf_counter()
for _ in range(5): allreduce(big)
if M.COMM_WORLD.rank == 0: print(json.dumps({"allreduce_16MiB_ms": (time.perf_counter() - t0) / 5 * 1e3}))
'''


def test_reference_over_the_shim_agrees_with_this_library(shim, tmp_path):
    """Same program through this library at np=3: Allreduce forward/backward and Allgather results identical to the
    reference's (GOLDEN), and the shim's 16 MiB Allreduce is not an order of magnitude slower than this library's own
    shared-memory backend."""
    script = tmp_path / "cross.py"
    script.write_text(CROSS)
    ours = _run([sys.executable, "-m", "mpi4torch_b200.launch", "-np", "3", script, ROOT], timeout=600,
                env={"M4T_CUDA": "0", "PYTHONPATH": str(ROOT)})
    assert ours.returncode == 0, ours.stderr[-3000:]
    r = json.loads(GOLDEN.read_text())
    o = json.loads([ln for ln in ours.stdout.splitlines() if ln.startswith("{")][-1])
    for key in ("fwd", "fwd_abs", "bwd", "allgather"):
        assert abs(r[key] - o[key]) <= 1e-9 * max(1.0, abs(o[key])), (key, r[key], o[key])
    # fairness of the stand-in MPI: same order of magnitude as this library's CPU backend on a bandwidth-bound message
    timing = tmp_path / "shim_allreduce.py"
    timing.write_text(SHIM_ALLREDUCE)
    res = _run([MPIRUN, "-np", 3, sys.executable, timing, SHIM / "python"], timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    s = json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])
    assert s["allreduce_16MiB_ms"] < 6.0 * o["allreduce_16MiB_ms"] + 10.0, (s, o)


def test_bench_reference_arm_prints_one_json_line_without_a_gpu():
    """Where no CUDA device is visible the reference arm must say so in one JSON line and exit 0 (the devices of a GPU
    box are hidden from the child process)."""
    res = _run([sys.executable, "bench.py", "--impl", "reference", "--gpus", "1", "--steps", "2", "--warmup", "1"], timeout=600,
               env={"CUDA_VISIBLE_DEVICES": ""})
    assert res.returncode == 0, res.stderr[-2000:]
    line = [ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and "no CUDA device" in d["unavailable"], d
