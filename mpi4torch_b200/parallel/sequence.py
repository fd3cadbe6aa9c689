"""Sequence <-> head re-sharding (the Ulysses exchange) as a single
``Alltoall(gatheraxis, scatteraxis)``: one kernel instead of the reference's
4*P blocking collectives (reference csrc/extension.cpp:917-987), and the
cumulative sum along a sequence-sharded dimension (one ``Exscan``)."""
from __future__ import annotations

import torch

import mpi4torch_b200 as m4t


def sequence_to_heads(x: torch.Tensor, seq_dim: int, head_dim: int, comm=None) -> torch.Tensor:
    """``[.., S/P, .., H, ..] -> [.., S, .., H/P, ..]``: gather the sequence, scatter the heads."""
    c = m4t.COMM_WORLD if comm is None else comm
    heads = x.shape[head_dim]
    if heads % c.size:
        raise ValueError(f"{heads} heads are not divisible by {c.size} ranks")
    return c.Alltoall(x, seq_dim, head_dim, heads // c.size)


def heads_to_sequence(x: torch.Tensor, seq_dim: int, head_dim: int, comm=None) -> torch.Tensor:
    """Inverse of :func:`sequence_to_heads`."""
    c = m4t.COMM_WORLD if comm is None else comm
    seq = x.shape[seq_dim]
    if seq % c.size:
        raise ValueError(f"sequence length {seq} is not divisible by {c.size} ranks")
    return c.Alltoall(x, head_dim, seq_dim, seq // c.size)


def ulysses_attention(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, comm=None, causal: bool = False) -> torch.Tensor:
    """Sequence-parallel attention (DeepSpeed-Ulysses pattern) on sequence-sharded inputs.

    ``q, k, v``: ``[B, S/P, H, D]`` (this rank's slice of the sequence, all heads).  Three
    ``Alltoall`` exchanges turn them into ``[B, S, H/P, D]`` (full sequence, this rank's heads), the
    attention itself is local, and one more exchange returns ``[B, S/P, H, D]``.  Every exchange is a
    single kernel and differentiable, so the backward pass is the mirrored four exchanges.
    """
    c = m4t.COMM_WORLD if comm is None else comm
    qh, kh, vh = (sequence_to_heads(t, 1, 2, c) for t in (q, k, v))       # [B, S, H/P, D]
    out = torch.nn.functional.scaled_dot_product_attention(
        qh.transpose(1, 2), kh.transpose(1, 2), vh.transpose(1, 2), is_causal=causal)  # [B, H/P, S, D]
    return heads_to_sequence(out.transpose(1, 2).contiguous(), 1, 2, c)


def distributed_cumsum(x: torch.Tensor, dim: int, comm=None) -> torch.Tensor:
    """``torch.cumsum`` along a dimension that is sharded by rank, in rank order.

    ``x`` is this rank's shard; every rank passes the same shape apart from ``dim``.  The result is
    this rank's shard of the cumulative sum of the concatenated tensor: the local cumulative sum plus
    the sum of all earlier ranks' shards, which one ``Exscan(MPI_SUM)`` of the local totals provides
    (instead of an ``Allgather`` of the whole tensor).  The gradient comes from autograd: the
    reverse ``Exscan`` of the gradient totals.
    """
    c = m4t.COMM_WORLD if comm is None else comm
    d = dim if dim >= 0 else dim + x.dim()
    before = c.Exscan(x.sum(dim=d, keepdim=True), m4t.MPI_SUM)
    return torch.cumsum(x, d) + before
