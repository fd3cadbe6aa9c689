"""mpi4torch_b200 - B200-native, autodiff-transparent collectives for PyTorch.

API parity with helmholtz-analytics/mpi4torch (reference ``src/__init__.py``):
``COMM_WORLD``, ``MPI_Communicator`` with ``Allreduce / Bcast_ / Reduce_ /
Gather / Allgather / Scatter / Alltoall / Isend / Irecv / Wait / Send / Recv``,
``WaitHandle``, ``JoinDummies``, ``JoinDummiesHandle``, the twelve ``MPI_*``
reduction constants, ``comm_from_mpi4py`` and
``deactivate_cuda_aware_mpi_support`` - every op a differentiable graph node
whose backward is the adjoint communication.  Added on top: ``Reduce_scatter``
(the true adjoint of ``Allgather``), ``Scan`` / ``Exscan`` (prefix reductions across
ranks), fused scale/accumulate epilogues
(``AllreduceFused``), ``Barrier`` and the fused Allreduce->GEMM layer in
:mod:`mpi4torch_b200.ops`.

There is no MPI underneath.  Ranks are OS processes started by
``python -m mpi4torch_b200.launch`` (or ``torchrun``); CPU tensors travel over a
POSIX shared-memory backend, CUDA tensors over hand-written sm_100a kernels
that read and write peer GPUs' HBM through NVLink 5 / NVSwitch (NVLS multicast
when the fabric offers it).
"""
from __future__ import annotations

import atexit
import os
import sys
from typing import List, Optional

import torch

from . import _build

_C = _build.load()

__version__ = "0.1.0"

__all__ = [
    "MPI_MAX",
    "MPI_MIN",
    "MPI_SUM",
    "MPI_PROD",
    "MPI_LAND",
    "MPI_BAND",
    "MPI_LOR",
    "MPI_BOR",
    "MPI_LXOR",
    "MPI_BXOR",
    "MPI_MINLOC",
    "MPI_MAXLOC",
    "WaitHandle",
    "JoinDummies",
    "JoinDummiesHandle",
    "MPI_Communicator",
    "COMM_WORLD",
    "comm_from_mpi4py",
    "deactivate_cuda_aware_mpi_support",
    "activate_nvlink_transport",
    "cuda_backend_ready",
    "has_nvls",
    "heap_mode",
    "symmetric_empty",
]

# The reference's integer op constants (reference csrc/extension.cpp:1424-1435).
MPI_MAX: int = _C.MPI_MAX
MPI_MIN: int = _C.MPI_MIN
MPI_SUM: int = _C.MPI_SUM
MPI_PROD: int = _C.MPI_PROD
MPI_LAND: int = _C.MPI_LAND
MPI_BAND: int = _C.MPI_BAND
MPI_LOR: int = _C.MPI_LOR
MPI_BOR: int = _C.MPI_BOR
MPI_LXOR: int = _C.MPI_LXOR
MPI_BXOR: int = _C.MPI_BXOR
MPI_MINLOC: int = _C.MPI_MINLOC
MPI_MAXLOC: int = _C.MPI_MAXLOC


def _bootstrap() -> None:
    """Attach to the job and (collectively) bring up the CUDA backend.

    Replaces ``MPI_Init_thread`` at import (reference csrc/extension.cpp:1323-1394).
    """
    # Kernels of different ranks/streams wait on each other; a lazily loaded
    # kernel whose load needs the device to drain could deadlock against a
    # spinning one.  Ask for eager loading when the context does not exist yet
    # (the pairs that matter are additionally preloaded natively).
    if not torch.cuda.is_initialized():
        os.environ.setdefault("CUDA_MODULE_LOADING", "EAGER")
    want_cuda = os.environ.get("M4T_CUDA", "1") != "0" and torch.cuda.is_available()
    device = 0
    world = int(os.environ.get("WORLD_SIZE", os.environ.get("M4T_WORLD_SIZE", "1")))
    if want_cuda:
        ndev = torch.cuda.device_count()
        local_rank = int(os.environ.get("LOCAL_RANK", os.environ.get("RANK", "0")))
        if ndev == 0 or (world > 1 and int(os.environ.get("LOCAL_WORLD_SIZE", world)) > ndev):
            want_cuda = False  # more ranks than GPUs: CPU backend + host staging only
        else:
            device = local_rank % ndev
            torch.cuda.set_device(device)
    if _spans_nodes(world):
        # more than one node: the world communicator lives on a TCP mesh and stages CUDA tensors through host memory
        # (what the reference does on an MPI without CUDA support); the NVLink backend needs one node - sub-communicators
        # whose members share a node (comm.Split by node) get it
        _connect_mesh(world)
        _C.init_world(False, device)
        if want_cuda:
            _C.set_node_cuda_device(device)
        return
    _C.init_world(want_cuda, device)


def _spans_nodes(world: int) -> bool:
    """One node = shared-memory control plane + NVLink heap; several nodes (LOCAL_WORLD_SIZE < WORLD_SIZE, as torchrun
    and this package's launcher export them) = TCP mesh.  ``M4T_NET=1`` forces the mesh on one node (tests), ``0``
    forbids it."""
    forced = os.environ.get("M4T_NET", "")
    if forced in ("0", "1"):
        return forced == "1" and world > 1
    return world > 1 and int(os.environ.get("LOCAL_WORLD_SIZE", world)) < world


def _connect_mesh(world: int) -> None:
    """Rendezvous for the TCP mesh: every rank publishes ``host:port`` of its listening socket in the job's key-value
    store (the one torchrun's agent or this package's launcher hosts at MASTER_ADDR:MASTER_PORT; without either, rank 0
    hosts it) and connects to the others natively.  Replaces ``mpirun``'s wire-up across nodes."""
    import socket
    from datetime import timedelta

    from torch.distributed import TCPStore

    rank = int(os.environ.get("RANK", os.environ.get("M4T_RANK", "0")))
    host = os.environ.get("MASTER_ADDR", "127.0.0.1")
    port = int(os.environ.get("MASTER_PORT", "29500"))
    timeout = float(os.environ.get("M4T_TIMEOUT_S", "300"))
    hosted = os.environ.get("TORCHELASTIC_USE_AGENT_STORE", "") == "True" or os.environ.get("M4T_STORE_HOSTED", "0") == "1"
    store = TCPStore(host, port, None, rank == 0 and not hosted, timedelta(seconds=timeout), wait_for_workers=False)
    mine = os.environ.get("M4T_NET_IFADDR", "")
    if not mine:
        try:  # the address this host uses to reach the master is one the other nodes can reach too
            with socket.socket(socket.AF_INET, socket.SOCK_DGRAM) as s:
                s.connect((host, port))
                mine = s.getsockname()[0]
        except OSError:
            mine = socket.gethostname()
    # one job name for all nodes (it seeds the communicator ids that keep frames of different communicators apart)
    os.environ.setdefault("M4T_JOB_ID", f"mn{port}")
    listen_port = _C.net_listen()
    prefix = "m4t/" + os.environ["M4T_JOB_ID"] + "/addr/"
    store.set(prefix + str(rank), f"{mine}:{listen_port}")
    addrs = [store.get(prefix + str(p)).decode() for p in range(world)]
    if os.environ.get("M4T_DEBUG", "0") not in ("", "0"):
        sys.stderr.write(f"[m4t:{rank}] tcp mesh: store {host}:{port} ({'hosted elsewhere' if hosted or rank else 'hosted here'}), "
                         f"listening on {mine}:{listen_port}, peers {addrs}\n")
    _C.net_connect(rank, world, addrs, os.environ["M4T_JOB_ID"])
    # keep the store alive until every rank has read every address (rank 0 may be its host)
    store.add(prefix + "done", 1)
    if rank == 0 and not hosted:
        import time

        t0 = time.monotonic()
        while int(store.add(prefix + "done", 0)) < world and time.monotonic() - t0 < timeout:
            time.sleep(0.01)
    global _mesh_store
    _mesh_store = store


_bootstrapped = False
_mesh_store = None  # the rendezvous store client (kept so that a store hosted by rank 0 outlives start-up)


def _ensure_world() -> None:
    global _bootstrapped
    if not _bootstrapped:
        _bootstrap()
        atexit.register(_C.finalize)
        _bootstrapped = True


def deactivate_cuda_aware_mpi_support() -> None:
    """Force CUDA tensors through host staging + the CPU shared-memory backend.

    Same role as the reference toggle (reference csrc/extension.cpp:54-59): it is
    the fallback when the NVLink path must be bypassed, and the "host-staged"
    comparator in the benchmarks.
    """
    _ensure_world()
    _C.deactivate_cuda_aware_mpi_support()


def activate_nvlink_transport() -> None:
    """Undo :func:`deactivate_cuda_aware_mpi_support`."""
    _ensure_world()
    _C.activate_nvlink_transport()


def cuda_backend_ready() -> bool:
    _ensure_world()
    return _C.cuda_backend_ready()


def has_nvls() -> bool:
    """True when the symmetric heap is bound to an NVSwitch multicast object."""
    _ensure_world()
    return _C.has_nvls()


def heap_mode() -> str:
    """'vmm+multicast', 'vmm', 'cudaIpc' or 'none'."""
    _ensure_world()
    return _C.heap_mode()


@torch.jit.script
class WaitHandle:
    """Handle returned by the non-blocking calls (reference ``src/__init__.py:27-40``).

    Internally a list of three tensors: a float64 descriptor (usable as a
    differentiable dummy), the communication buffer, and the original tensor.
    """

    def __init__(self, raw_handle: List[torch.Tensor]):
        self._handle = raw_handle

    @property
    def dummy(self):
        """Dummy tensor for :func:`JoinDummies` / :func:`JoinDummiesHandle`."""
        return self._handle[0]


@torch.jit.script
def JoinDummies(loopthrough: torch.Tensor, dummies: List[torch.Tensor]) -> torch.Tensor:
    """Pass ``loopthrough`` through and make the DAG depend on ``dummies``.

    Forward is a no-op; in backward the dummies receive zero gradients, which
    is how program order and cross-rank communication dependencies are encoded
    (reference ``src/__init__.py:42-67``, ``doc/basic_usage.rst:317-348``).
    """
    return torch.ops.mpi4torch_b200.JoinDummies(loopthrough, dummies)


@torch.jit.script
def JoinDummiesHandle(handle: WaitHandle, dummies: List[torch.Tensor]) -> WaitHandle:
    """:func:`JoinDummies` for a :class:`WaitHandle` (reference ``src/__init__.py:69-87``)."""
    raw_handle = handle._handle
    return WaitHandle([torch.ops.mpi4torch_b200.JoinDummies(raw_handle[0], dummies), raw_handle[1], raw_handle[2]])


@torch.jit.script
class MPI_Communicator:
    """Communicator (reference ``src/__init__.py:89-240``).

    Obtain it from :data:`COMM_WORLD`.  Methods with a trailing underscore are
    in-place operations: always use their return value.
    """

    def __init__(self, comm: torch.classes.mpi4torch_b200.Communicator):
        self._comm = comm

    @property
    def rank(self) -> int:
        """Rank of this process in ``[0, size)``."""
        return self._comm.GetRank()

    @property
    def size(self) -> int:
        """Number of processes in the communicator."""
        return self._comm.GetSize()

    def Allreduce(self, tensor: torch.Tensor, op: int) -> torch.Tensor:
        """Element-wise reduction over all ranks, result on all ranks.

        All twelve ``MPI_*`` ops are accepted forward (``MPI_MINLOC`` /
        ``MPI_MAXLOC`` raise: there is no pair dtype); only ``MPI_SUM`` has a
        backward, which is again an ``Allreduce(MPI_SUM)``.
        """
        return self._comm.Allreduce(tensor, op)

    def AllreduceFused(self, tensor: torch.Tensor, op: int, scale: float,
                       accumulate: Optional[torch.Tensor]) -> torch.Tensor:
        """``accumulate + scale * Allreduce(tensor, op)`` in ONE kernel.

        The scale (e.g. ``1/size``) and the accumulate run in the collective's
        epilogue, forward and backward (the backward is the same fused kernel
        applied to the upstream gradient).
        """
        return self._comm.AllreduceFused(tensor, op, scale, accumulate)

    def Bcast_(self, tensor: torch.Tensor, root: int) -> torch.Tensor:
        """Broadcast ``root``'s tensor in place; backward is ``Reduce_(MPI_SUM)``."""
        return self._comm.Bcast_(tensor, root)

    def Reduce_(self, tensor: torch.Tensor, op: int, root: int) -> torch.Tensor:
        """Reduce to ``root`` in place (non-root results are zero-filled);
        backward (``MPI_SUM`` only) is ``Bcast_``."""
        return self._comm.Reduce_(tensor, op, root)

    def Gather(self, tensor: torch.Tensor, gatheraxis: int, root: int) -> torch.Tensor:
        """Concatenate along ``gatheraxis`` in rank order on ``root`` (axis length
        may differ per rank; off-root the result has extent 0 along the axis)."""
        return self._comm.Gather(tensor, gatheraxis, root)

    def Allgather(self, tensor: torch.Tensor, gatheraxis: int) -> torch.Tensor:
        """:meth:`Gather` to all ranks; backward is a reduce-scatter."""
        return self._comm.Allgather(tensor, gatheraxis)

    def Scatter(self, tensor: torch.Tensor, scatteraxis: int, numelem: int, root: int) -> torch.Tensor:
        """Split ``root``'s tensor along ``scatteraxis``; this rank receives
        ``numelem`` rows.  Off-root ``tensor`` only provides dtype and device."""
        return self._comm.Scatter(tensor, scatteraxis, numelem, root)

    def Alltoall(self, tensor: torch.Tensor, gatheraxis: int, scatteraxis: int, numelem: int) -> torch.Tensor:
        """Every rank scatters along ``scatteraxis`` and gathers along
        ``gatheraxis`` (equal axes re-partition one global axis).  One kernel."""
        return self._comm.Alltoall(tensor, gatheraxis, scatteraxis, numelem)

    def Reduce_scatter(self, tensor: torch.Tensor, op: int, scatteraxis: int, numelem: int) -> torch.Tensor:
        """Reduce identically shaped tensors and keep ``numelem`` rows of
        ``scatteraxis`` on this rank (the adjoint of :meth:`Allgather`)."""
        return self._comm.Reduce_scatter(tensor, op, scatteraxis, numelem)

    def Reduce_scatterFused(self, tensor: torch.Tensor, op: int, scatteraxis: int, numelem: int, scale: float,
                            accumulate: Optional[torch.Tensor]) -> torch.Tensor:
        """``accumulate + scale * Reduce_scatter(tensor, op)`` in ONE kernel: the scale, the cast to the
        output dtype and the accumulation into an existing gradient run in the reducing kernel's
        epilogue (the reference's Allgather backward adds the scattered pieces with a separate ``+=``,
        csrc/extension.cpp:616-631).  Backward: ``Allgather(scale * grad)``; ``accumulate`` receives the
        incoming gradient."""
        return self._comm.Reduce_scatterFused(tensor, op, scatteraxis, numelem, scale, accumulate)

    def Scan(self, tensor: torch.Tensor, op: int) -> torch.Tensor:
        """Inclusive prefix reduction across ranks (``MPI_Scan``): rank ``r`` receives
        ``((x_0 op x_1) op x_2) ... op x_r``, folded left to right in ascending rank order.

        Every rank passes the same shape and dtype (no size exchange, as in :meth:`Allreduce`);
        the ops and dtypes are those of :meth:`Allreduce`.  16-bit floats fold in fp32 and are
        rounded once.  The fold order is part of the contract: every backend and algorithm gives
        the same bits.  Only ``MPI_SUM`` has a backward: the reverse inclusive scan of the gradient
        (rank ``r`` receives the sum of the gradients of ranks ``r .. P-1``)."""
        return self._comm.Scan(tensor, op)

    def Exscan(self, tensor: torch.Tensor, op: int) -> torch.Tensor:
        """Exclusive prefix reduction across ranks (``MPI_Exscan``): rank ``r > 0`` receives the
        fold of ``x_0 .. x_{r-1}`` in ascending rank order, as in :meth:`Scan`.  Rank 0's result
        is zero-filled (MPI leaves it undefined; :meth:`Reduce_` zero-fills non-root results the
        same way).  Only ``MPI_SUM`` has a backward: the reverse exclusive scan of the gradient
        (rank ``P-1`` receives zeros)."""
        return self._comm.Exscan(tensor, op)

    def assume_uniform_sizes(self, on: bool = True) -> None:
        """Promise that every rank passes identically shaped tensors and the same ``numelem`` to
        Gather / Allgather / Scatter / Alltoall / Reduce_scatter.  The host-side size exchange (the
        reference's ``MPI_Gather`` / ``MPI_Allgather`` of axis lengths, csrc/extension.cpp:540,675) is then
        skipped and these ops become pure stream work, capturable into a CUDA graph."""
        self._comm.AssumeUniformSizes(on)

    def Isend(self, tensor: torch.Tensor, dest: int, tag: int) -> WaitHandle:
        """Start a non-blocking send."""
        return WaitHandle(self._comm.Isend(tensor, dest, tag))

    def Irecv(self, tensor: torch.Tensor, source: int, tag: int) -> WaitHandle:
        """Start a non-blocking receive into ``tensor``; use :meth:`Wait`'s result."""
        return WaitHandle(self._comm.Irecv(tensor, source, tag))

    def Wait(self, waithandle: WaitHandle) -> torch.Tensor:
        """Complete a non-blocking operation (each handle exactly once)."""
        return self._comm.Wait(waithandle._handle)

    def Send(self, tensor: torch.Tensor, dest: int, tag: int) -> torch.Tensor:
        """Blocking send = ``Wait(Isend(...))`` (reference ``src/__init__.py:234-236``)."""
        handle = self._comm.Isend(tensor, dest, tag)
        return self._comm.Wait(handle)

    def Recv(self, tensor: torch.Tensor, source: int, tag: int) -> torch.Tensor:
        """Blocking receive = ``Wait(Irecv(...))`` (reference ``src/__init__.py:238-240``)."""
        handle = self._comm.Irecv(tensor, source, tag)
        return self._comm.Wait(handle)

    def Barrier(self) -> None:
        """Host barrier over all ranks (control plane only)."""
        self._comm.Barrier()

    def Split(self, color: int, key: int) -> "MPI_Communicator":
        """``MPI_Comm_split``: ranks passing the same ``color`` (>= 0) form a new
        communicator, ranked by ``(key, old rank)``; a negative colour
        (``MPI_UNDEFINED``) yields a communicator containing only this rank.
        Collective over this communicator.  The sub-communicator has its own control segment,
        symmetric heap and device counters, so its collectives never alias the
        parent's (the reference obtains sub-communicators from mpi4py,
        ``src/__init__.py:247-261``)."""
        return MPI_Communicator(self._comm.Split(color, key))

    def Free(self) -> None:
        """``MPI_Comm_free``: collective release of a sub-communicator's segments
        and symmetric heap (otherwise they live until the process exits).  The
        communicator must not be used afterwards."""
        self._comm.Free()

    @property
    def is_world(self) -> bool:
        """True for :data:`COMM_WORLD` (fused GEMM ops and pickling need it)."""
        return self._comm.IsWorld()

    def describe(self) -> str:
        return self._comm.Describe()


def _make_comm_world() -> MPI_Communicator:
    _ensure_world()
    return MPI_Communicator(torch.ops.mpi4torch_b200.COMM_WORLD())


def __getattr__(name: str):
    # COMM_WORLD is created on first access (a collective start-up: every rank
    # touches it, normally at the top of the user script, exactly like the
    # reference's module-level singleton, src/__init__.py:242-245).  Keeping it
    # lazy lets tools such as the launcher import the package without joining
    # a job.
    if name == "COMM_WORLD":
        world = _make_comm_world()
        globals()["COMM_WORLD"] = world
        return world
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")


def symmetric_empty(shape, dtype=torch.float32) -> torch.Tensor:
    """Uninitialised CUDA tensor inside the symmetric heap's persistent arena.

    Collective in spirit: all ranks must allocate the same sizes in the same
    order so offsets agree.  Kernels that need peer-visible inputs (the fused
    Allreduce->GEMM layer) use such tensors in place instead of staging a copy.
    """
    _ensure_world()
    return torch.ops.mpi4torch_b200.symmetric_empty(list(shape), dtype)


def comm_from_mpi4py(comm) -> MPI_Communicator:
    """Interop for code written against ``mpi4torch.comm_from_mpi4py``
    (reference ``src/__init__.py:247-261``).

    There is no MPI underneath this library; the mpi4py communicator is only
    used to learn the group.  A communicator congruent with the launcher's
    world maps to :data:`COMM_WORLD`.  Any other communicator is rebuilt with
    :meth:`MPI_Communicator.Split` (colour = smallest world rank of the group,
    key = rank inside ``comm``) - which is collective over the WORLD, so every
    world rank must call ``comm_from_mpi4py`` at the same point with its own
    group, exactly as they all took part in the ``comm.Split`` that created
    these groups.
    """
    try:
        size, rank = comm.Get_size(), comm.Get_rank()
    except AttributeError as exc:  # pragma: no cover
        raise RuntimeError("mpi4py is not available!") from exc
    world = __getattr__("COMM_WORLD") if "COMM_WORLD" not in globals() else globals()["COMM_WORLD"]
    if not hasattr(comm, "allgather"):
        # no way to learn the members: only a communicator that looks like the world is accepted
        if size == world.size and rank == world.rank:
            return world
        raise RuntimeError(
            "mpi4torch_b200: the communicator has "
            f"rank {rank}/{size} but this process is rank {world.rank}/{world.size}, and it offers no "
            "allgather() to discover its members")
    # The world-or-Split decision must be the same on every rank (Split is collective over the
    # world): decide from the member list, which all ranks of the group see identically, never from
    # this rank's own position (a reordered world keeps some ranks in place).
    members = [int(r) for r in comm.allgather(world.rank)]
    if members == list(range(world.size)):
        return world
    sub = world.Split(min(members), rank)
    if sub.size != size or sub.rank != rank:
        raise RuntimeError(f"mpi4torch_b200: rebuilt communicator is {sub.rank}/{sub.size}, expected {rank}/{size}")
    return sub
