"""Scan / Exscan: single-process semantics (world of one, API surface, TorchScript) and, on a GPU box, the SPMD suite
with a small staging arena so that the two-shot kernel runs in pieces."""
import pytest
import torch

import mpi4torch_b200 as m4t
from conftest import run_spmd


def test_api_surface():
    comm = m4t.COMM_WORLD
    for method in ("Scan", "Exscan"):
        assert hasattr(comm, method), method
    from mpi4torch_b200.parallel import distributed_cumsum  # noqa: F401

    assert "distributed_cumsum" in m4t.parallel.__all__


def test_world_of_one_scan_is_a_copy_and_exscan_zero_fills():
    comm = m4t.COMM_WORLD
    assert comm.size == 1
    x = torch.rand(3, 4, dtype=torch.double, requires_grad=True)
    y = comm.Scan(x, m4t.MPI_SUM)
    assert torch.equal(y, x) and "MPIScanSumBackward" in y.grad_fn.name()
    y.sum().backward()
    assert torch.equal(x.grad, torch.ones_like(x))
    x.grad = None
    z = comm.Exscan(x, m4t.MPI_SUM)
    assert torch.equal(z, torch.zeros_like(x)) and "MPIExscanSumBackward" in z.grad_fn.name()
    z.sum().backward()
    assert torch.equal(x.grad, torch.zeros_like(x))
    # logical ops normalise their operand as Allreduce does at world size 1
    i = torch.tensor([0, 3, -2], dtype=torch.int32)
    assert torch.equal(comm.Scan(i, m4t.MPI_LOR), torch.tensor([0, 1, 1], dtype=torch.int32))
    assert torch.equal(comm.Exscan(i, m4t.MPI_PROD), torch.zeros_like(i))
    e = torch.empty(0, 2)
    assert comm.Scan(e, m4t.MPI_MAX).shape == (0, 2) and comm.Exscan(e, m4t.MPI_MAX).shape == (0, 2)


def test_world_of_one_distributed_cumsum_is_cumsum():
    from mpi4torch_b200.parallel import distributed_cumsum

    x = torch.rand(2, 5, 3, dtype=torch.double, requires_grad=True)
    y = distributed_cumsum(x, 1)
    assert torch.allclose(y, torch.cumsum(x, 1))
    y.sum().backward()
    assert torch.allclose(x.grad, torch.cumsum(torch.ones_like(x).flip(1), 1).flip(1))


def test_scripted_communicator_calls():
    @torch.jit.script
    def prefix(t, c: m4t.MPI_Communicator):
        return c.Scan(t, m4t.MPI_SUM) + c.Exscan(t, m4t.MPI_SUM)

    x = torch.rand(5, dtype=torch.double)
    assert torch.equal(prefix(x, m4t.COMM_WORLD), x)


def test_non_sum_backward_raises_only_in_backward():
    x = torch.rand(4, requires_grad=True)
    y = m4t.COMM_WORLD.Scan(x, m4t.MPI_MAX)
    with pytest.raises(RuntimeError, match="unimplemented"):
        y.sum().backward()


def _world_sizes():
    n = torch.cuda.device_count() if torch.cuda.is_available() else 0
    return [s for s in (2, 4, 8) if s <= n]


@pytest.mark.gpu
@pytest.mark.parametrize("nprocs", _world_sizes() or [pytest.param(2, marks=pytest.mark.skip(reason="needs 2 GPUs"))])
def test_scan_suite_cuda_with_small_staging(nprocs):
    """8 MiB staging halves: the 8 MiB-plus messages of the suite run as several two-shot (and one-shot) pieces."""
    res = run_spmd(nprocs, ["tests/spmd/run_all.py", "spmd_scan.py"], device="cuda", timeout=900,
                   extra_env={"M4T_STAGE_MB": "8"})
    assert res.returncode == 0, f"np={nprocs}\nSTDOUT:\n{res.stdout[-4000:]}\nSTDERR:\n{res.stderr[-12000:]}"
    assert f"SPMD suite np={nprocs} device=cuda" in res.stdout and "ok=True" in res.stdout
