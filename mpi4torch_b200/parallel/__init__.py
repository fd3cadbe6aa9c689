"""Parallelism strategies built from the primitives (SURVEY section 2.6): data
parallel (the only strategy the reference ships, as an example), plus the ring
(pipeline-style p2p) and sequence<->head (Ulysses-style) exchanges the
reference's primitives enable, and two-level (node / rail) collectives for jobs that span nodes."""
from .data_parallel import DataParallel, OverlappedGradSync, sync_gradients_
from .expert import DispatchInfo, combine_tokens, dispatch_tokens
from .hierarchical import NodeRails, hierarchical_allreduce, hierarchical_sync_gradients_, ranks_per_node
from .pipeline import pipeline_forward, split_microbatches
from .ring import ring_exchange
from .sequence import distributed_cumsum, heads_to_sequence, sequence_to_heads, ulysses_attention
from .tensor_parallel import ColumnParallelLinear, RowParallelLinear, TensorParallelMLP, replicated_input
from .zero import ShardedSGD

__all__ = ["DataParallel", "OverlappedGradSync", "sync_gradients_", "ring_exchange", "sequence_to_heads", "heads_to_sequence", "ulysses_attention", "distributed_cumsum",
           "dispatch_tokens", "combine_tokens", "DispatchInfo", "pipeline_forward", "split_microbatches", "ColumnParallelLinear", "RowParallelLinear", "TensorParallelMLP", "replicated_input", "ShardedSGD",
           "NodeRails", "hierarchical_allreduce", "hierarchical_sync_gradients_", "ranks_per_node"]
