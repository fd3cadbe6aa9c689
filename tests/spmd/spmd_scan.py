"""Scan / Exscan: exact values against a local replay of the specified fold, adjoints, sub-communicators and, on
CUDA, both device algorithms, the host backend and CUDA-graph replays.

Every rank rebuilds every rank's input from ``seed + rank`` and folds them itself in the order the contract
fixes (ascending ranks, left to right; the backward folds from rank P-1 down), in the accumulation type of the
transports (fp32 for 16-bit floats, rounded once), so results are compared with ``torch.equal``.  The full
op x dtype grid runs at small sizes; the sizes that reach the two-phase and piecewise paths run for f32 SUM."""
import unittest

import torch

import mpi4torch_b200 as m4t
from common import DEVICE, comm
from mpi4torch_b200.parallel import distributed_cumsum

P, R = comm.size, comm.rank
CUDA = DEVICE.type == "cuda"

FLOATS = [torch.float32, torch.float64, torch.bfloat16, torch.float16]
INTEGERS = [torch.uint8, torch.int8, torch.int16, torch.int32, torch.int64, torch.bool]
ARITHMETIC = ["MAX", "MIN", "SUM", "PROD"]
BITWISE_LOGICAL = ["LAND", "LOR", "LXOR", "BAND", "BOR", "BXOR"]
# 256 KiB is where the host backends switch to their slice-owner variant, 8 MiB where they cut pieces
TWO_PHASE_N = (256 << 10) // 4 + 4093
PIECES_N = (8 << 20) // 4 + 12345


def make(rank, n, dtype, seed=0):
    g = torch.Generator().manual_seed(seed * 1000 + rank)
    if dtype.is_floating_point:
        return torch.randn(n, generator=g).to(dtype)
    if dtype == torch.bool:
        return torch.randint(0, 4, (n,), generator=g) > 0
    if dtype == torch.uint8:
        return torch.randint(0, 256, (n,), generator=g).to(dtype)
    return torch.randint(-100, 100, (n,), generator=g).to(dtype)  # sums and products wrap, as in Allreduce


def _acc(t):
    if t.dtype in (torch.bfloat16, torch.float16):
        return t.float()
    return t if t.dtype.is_floating_point else t.long()


def _combine(op, a, b):
    if op == "MAX":
        return torch.maximum(a, b)
    if op == "MIN":
        return torch.minimum(a, b)
    if op == "SUM":
        return a + b
    if op == "PROD":
        return a * b
    if op == "LAND":
        return ((a != 0) & (b != 0)).to(a.dtype)
    if op == "LOR":
        return ((a != 0) | (b != 0)).to(a.dtype)
    if op == "LXOR":
        return ((a != 0) ^ (b != 0)).to(a.dtype)
    if op == "BAND":
        return a & b
    if op == "BOR":
        return a | b
    return a ^ b


def replay(xs, op, exclusive, reverse, rank):
    """The specified fold for `rank`, given every rank's input `xs` (CPU tensors)."""
    n = len(xs)
    order = list(range(n - 1, -1, -1)) if reverse else list(range(n))
    upto = order.index(rank) + (0 if exclusive else 1)
    if upto == 0:
        return torch.zeros_like(xs[0])
    acc = _acc(xs[order[0]])
    if op in ("LAND", "LOR", "LXOR"):
        acc = (acc != 0).to(acc.dtype)
    for p in order[1:upto]:
        acc = _combine(op, acc, _acc(xs[p]))
    return acc.to(xs[0].dtype)


def run(x, op, exclusive, c=comm):
    opc = getattr(m4t, "MPI_" + op)
    return c.Exscan(x, opc) if exclusive else c.Scan(x, opc)


class TestScanValues(unittest.TestCase):
    def _check(self, op, dtype, n, seed=0):
        xs = [make(p, n, dtype, seed) for p in range(P)]
        for exclusive in (False, True):
            got = run(xs[R].to(DEVICE), op, exclusive)
            self.assertEqual(got.dtype, dtype)
            self.assertEqual(got.device, DEVICE)
            want = replay(xs, op, exclusive, False, R)
            self.assertTrue(torch.equal(got.cpu(), want),
                            f"{'Exscan' if exclusive else 'Scan'} {op} {dtype} n={n}: "
                            f"{(got.cpu().double() - want.double()).abs().max().item() if n else 0}")

    def test_arithmetic_ops_on_every_dtype(self):
        for dtype in FLOATS + INTEGERS:
            for op in ARITHMETIC:
                for n in (0, 1, 7, 4096 // torch.empty(0, dtype=dtype).element_size()):
                    self._check(op, dtype, n)

    def test_bitwise_and_logical_ops_on_integers_and_bool(self):
        for dtype in INTEGERS:
            for op in BITWISE_LOGICAL:
                for n in (1, 7, 4096 // torch.empty(0, dtype=dtype).element_size()):
                    self._check(op, dtype, n)

    def test_large_messages(self):
        for n in (TWO_PHASE_N, PIECES_N):
            self._check("SUM", torch.float32, n, seed=1)

    def test_result_keeps_the_shape_and_empty_tensors_pass(self):
        x = make(R, 24, torch.float64).reshape(2, 3, 4).to(DEVICE)
        self.assertEqual(comm.Scan(x, m4t.MPI_SUM).shape, x.shape)
        e = torch.empty(0, 5, dtype=torch.float32, device=DEVICE)
        for y in (comm.Scan(e, m4t.MPI_SUM), comm.Exscan(e, m4t.MPI_SUM)):
            self.assertEqual(tuple(y.shape), (0, 5))

    def test_non_contiguous_input(self):
        xs = [make(p, 30, torch.float32, seed=2).reshape(6, 5) for p in range(P)]
        x = xs[R].to(DEVICE).t()
        self.assertFalse(x.is_contiguous())
        for exclusive in (False, True):
            got = run(x, "SUM", exclusive)
            want = replay([t.t().contiguous() for t in xs], "SUM", exclusive, False, R)
            self.assertTrue(torch.equal(got.cpu(), want))

    def test_minloc_and_maxloc_raise(self):
        x = torch.ones(3, device=DEVICE)
        for op in (m4t.MPI_MINLOC, m4t.MPI_MAXLOC):
            with self.assertRaises((ValueError, RuntimeError)):
                comm.Scan(x, op)
            with self.assertRaises((ValueError, RuntimeError)):
                comm.Exscan(x, op)

    def test_sub_communicator(self):
        sub = comm.Split(R % 2, R)
        members = [p for p in range(P) if p % 2 == R % 2]
        xs = [make(p, 33, torch.float32, seed=3) for p in members]
        for exclusive in (False, True):
            got = run(xs[sub.rank].to(DEVICE), "SUM", exclusive, c=sub)
            self.assertTrue(torch.equal(got.cpu(), replay(xs, "SUM", exclusive, False, sub.rank)))
        sub.Free()


class TestScanBackward(unittest.TestCase):
    def test_backward_is_the_reverse_scan(self):
        n = 37
        gs = [make(p, n, torch.float32, seed=5) for p in range(P)]
        for exclusive in (False, True):
            x = make(R, n, torch.float32, seed=4).to(DEVICE).requires_grad_()
            y = run(x, "SUM", exclusive)
            self.assertIn("MPIExscanSumBackward" if exclusive else "MPIScanSumBackward", y.grad_fn.name())
            (y * gs[R].to(DEVICE)).sum().backward()
            self.assertTrue(torch.equal(x.grad.cpu(), replay(gs, "SUM", exclusive, True, R)))

    def test_double_backward(self):
        # the gradient is a reverse scan of the upstream gradient u; differentiating <grad, v> by u is the forward scan of v
        n = 5
        vs = [make(p, n, torch.float64, seed=7) for p in range(P)]
        for exclusive in (False, True):
            x = make(R, n, torch.float64, seed=6).to(DEVICE).requires_grad_()
            u = make(R, n, torch.float64, seed=8).to(DEVICE).requires_grad_()
            (gx,) = torch.autograd.grad(run(x, "SUM", exclusive), x, grad_outputs=u, create_graph=True)
            (gu,) = torch.autograd.grad((gx * vs[R].to(DEVICE)).sum(), u)
            self.assertTrue(torch.equal(gu.cpu(), replay(vs, "SUM", exclusive, False, R)))

    def test_gradcheck(self):
        # A cross-rank function seen from one rank: rank 0's input is broadcast, every rank scans its scaled copy and the
        # weighted results are reduced back to rank 0, so the numerical Jacobian (rank 0 perturbs, rank 0 observes) and
        # the analytical one describe the same map; the other ranks see zeros both ways.
        c = torch.arange(1, P + 1, dtype=torch.float64, device=DEVICE)
        for exclusive in (False, True):
            def f(x):
                z = run(comm.Bcast_(x.clone(), 0) * c[R], "SUM", exclusive)
                return comm.Reduce_(z * (P - R + 0.5), m4t.MPI_SUM, 0)

            x = make(0, 3, torch.float64, seed=9).to(DEVICE).requires_grad_()
            self.assertTrue(torch.autograd.gradcheck(f, (x,), check_undefined_grad=False))

    def test_backward_of_other_ops_raises(self):
        for exclusive in (False, True):
            x = make(R, 4, torch.float32).to(DEVICE).requires_grad_()
            y = run(x, "MAX", exclusive)
            with self.assertRaises(RuntimeError):
                y.sum().backward()


class TestDistributedCumsum(unittest.TestCase):
    def test_forward_and_backward_match_cumsum_of_the_gathered_tensor(self):
        shards = [make(p, 3 * (p + 1) * 2, torch.float64, seed=10).reshape(3, p + 1, 2) for p in range(P)]
        weights = [make(p, 3 * (p + 1) * 2, torch.float64, seed=11).reshape(3, p + 1, 2) for p in range(P)]
        full = torch.cat(shards, 1).requires_grad_()
        (torch.cumsum(full, 1) * torch.cat(weights, 1)).sum().backward()
        lo = R * (R + 1) // 2
        x = shards[R].to(DEVICE).requires_grad_()
        y = distributed_cumsum(x, -2, comm)
        self.assertTrue(torch.allclose(y.detach().cpu(), torch.cumsum(full.detach(), 1)[:, lo:lo + R + 1], rtol=1e-12, atol=1e-12))
        (y * weights[R].to(DEVICE)).sum().backward()
        self.assertTrue(torch.allclose(x.grad.cpu(), full.grad[:, lo:lo + R + 1], rtol=1e-12, atol=1e-12))


@unittest.skipUnless(CUDA, "needs the CUDA backend")
class TestScanDeviceAlgorithms(unittest.TestCase):
    def _forced(self, algo, x, op, exclusive):
        m4t._C.set_tuning("force_algo", algo)
        try:
            return run(x, op, exclusive)
        finally:
            m4t._C.set_tuning("force_algo", 0)

    def test_oneshot_and_twoshot_give_identical_bits(self):
        cases = [("SUM", torch.float32, n) for n in (1, 7, 4099, TWO_PHASE_N, PIECES_N)]
        cases += [("SUM", torch.bfloat16, 100_003), ("PROD", torch.float16, 4099), ("MAX", torch.float64, 1001),
                  ("BXOR", torch.int64, 999), ("LOR", torch.bool, 4099), ("SUM", torch.int8, 70_001)]
        for op, dtype, n in cases:
            xs = [make(p, n, dtype, seed=12) for p in range(P)]
            x = xs[R].to(DEVICE)
            for exclusive in (False, True):
                a = self._forced(1, x, op, exclusive)
                b = self._forced(2, x, op, exclusive)
                want = replay(xs, op, exclusive, False, R)
                self.assertTrue(torch.equal(a.cpu(), want), f"one-shot {op} {dtype} n={n} exclusive={exclusive}")
                self.assertTrue(torch.equal(b.cpu(), want), f"two-shot {op} {dtype} n={n} exclusive={exclusive}")

    def test_unaligned_views(self):
        xs = [make(p, 4103, torch.bfloat16, seed=13) for p in range(P)]
        x = xs[R].to(DEVICE)[3:]  # 6 bytes past a 16-byte boundary
        for algo in (1, 2):
            for exclusive in (False, True):
                got = self._forced(algo, x, "SUM", exclusive)
                self.assertTrue(torch.equal(got.cpu(), replay([t[3:] for t in xs], "SUM", exclusive, False, R)))

    def test_same_bytes_as_the_host_backend(self):
        # a seeded sequence of calls on CUDA tensors and on CPU tensors (shared-memory backend): identical bytes
        for i, (op, dtype, n) in enumerate([("SUM", torch.float32, 300_001), ("SUM", torch.bfloat16, 65_537),
                                            ("PROD", torch.float64, 513), ("MIN", torch.float16, 4097),
                                            ("SUM", torch.int32, 70_000), ("BAND", torch.uint8, 333)]):
            x = make(R, n, dtype, seed=20 + i)
            for exclusive in (False, True):
                on_gpu = run(x.to(DEVICE), op, exclusive).cpu()
                on_host = run(x, op, exclusive)
                self.assertTrue(torch.equal(on_gpu.view(torch.uint8), on_host.view(torch.uint8)),
                                f"{op} {dtype} n={n} exclusive={exclusive}")

    def test_host_staged_route(self):
        xs = [make(p, 1000, torch.float32, seed=14) for p in range(P)]
        m4t.deactivate_cuda_aware_mpi_support()
        try:
            got = comm.Scan(xs[R].to(DEVICE), m4t.MPI_SUM)
        finally:
            m4t.activate_nvlink_transport()
        self.assertEqual(got.device, DEVICE)
        self.assertTrue(torch.equal(got.cpu(), replay(xs, "SUM", False, False, R)))

    def test_cuda_graph_replays_match_eager(self):
        n = 50_000
        static = torch.zeros(n, device=DEVICE)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            comm.Scan(static, m4t.MPI_SUM)
            comm.Exscan(static, m4t.MPI_SUM)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        comm.Barrier()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            inc = comm.Scan(static, m4t.MPI_SUM)
            exc = comm.Exscan(static * 2, m4t.MPI_SUM)
        for step in range(3):
            static.copy_(make(R, n, torch.float32, seed=30 + step).to(DEVICE))
            graph.replay()
            torch.cuda.synchronize()
            self.assertTrue(torch.equal(inc, comm.Scan(static, m4t.MPI_SUM)), f"replay {step}")
            self.assertTrue(torch.equal(exc, comm.Exscan(static * 2, m4t.MPI_SUM)), f"replay {step}")


if __name__ == "__main__":
    unittest.main()
