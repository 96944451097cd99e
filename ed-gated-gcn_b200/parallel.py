"""Data parallelism for the gated-GCN path (SURVEY.md 8e): one process per GPU,
graphs sharded by batch, no activation ever crosses GPUs; training adds one
gradient all-reduce (NCCL over NVLink on GPUs, gloo in the CPU tests) and
inference needs no communication.  The reference has no distributed code
(train.py is single-process); this is the only piece added next to it.
"""
from __future__ import annotations

from typing import Iterable, List, Optional, Sequence

import numpy as np
import torch
import torch.distributed as dist


def shard_graphs(lengths: Sequence[int], world_size: int, rank: int) -> np.ndarray:
    """Indices of the graphs rank ``rank`` owns.

    The reference sorts sentences by length (data_utils.py:341-346) and does not
    shuffle (train.py:247), so contiguous shards would be badly skewed in token
    count.  Deal the graphs round-robin after a stable sort by length: every rank
    gets the same number of graphs (so batch means average correctly across ranks
    when B divides) and a near-equal number of tokens."""
    lengths = np.asarray(lengths)
    order = np.argsort(-lengths, kind="stable")
    return np.sort(order[rank::world_size])


def shard_tree_batch(batch, world_size: int, rank: int):
    """Sub-batch (a ``synth.TreeBatch``) holding only this rank's graphs, with their extra edges if it has any."""
    from .synth import TreeBatch
    idx = shard_graphs(batch.lengths, world_size, rank)
    lengths = batch.lengths[idx]
    sent_ptr = np.zeros(len(idx) + 1, dtype=np.int32)
    np.cumsum(lengths, out=sent_ptr[1:])
    heads = np.concatenate([batch.heads[batch.sent_ptr[b]:batch.sent_ptr[b + 1]] for b in idx]) if len(idx) else \
        np.zeros(0, dtype=np.int32)
    extra_edges = edge_ptr = None
    if getattr(batch, "extra_edges", None) is not None:
        ep = batch.edge_ptr
        extra_edges = np.concatenate([np.zeros((0, 2), dtype=np.int32)] + [batch.extra_edges[ep[b]:ep[b + 1]] for b in idx])
        edge_ptr = np.zeros(len(idx) + 1, dtype=np.int32)
        np.cumsum(ep[idx + 1] - ep[idx], out=edge_ptr[1:])
    return TreeBatch(heads=heads.astype(np.int32), sent_ptr=sent_ptr, anchor=batch.anchor[idx], lengths=lengths,
                     extra_edges=extra_edges, edge_ptr=edge_ptr), idx


class GradientAllReducer:
    """Averages parameter gradients across ranks (SURVEY 8e).

    ``__call__()`` after ``loss.backward()``: ONE all-reduce over one flat fp32 bucket (2.3 MB at config 2), after which
    every parameter's ``.grad`` is re-pointed at its slice of the reduced buffer -- one small pack kernel, one collective,
    nothing copied back.  Measured on 2 B200 (weak scaling, whole step in a CUDA graph): 0.894 ms/step against 0.854 on one
    GPU; a coalesced group of the 22 separate tensors costs 0.923.

    ``hook(tensors)`` is the overlapped alternative: a backward pass calls it the moment a group of gradients exists
    (``GatedGCNStack`` does so per layer, per gate-MLP batch and for the classifier head when
    ``stack.grad_ready_hook = reducer.hook``) and the group is all-reduced in place, asynchronously, ordered after the
    stream that produced it; ``__call__()`` then only reduces what was not announced and waits.  With this package's
    persistent one-CTA-per-SM kernels the collectives cannot run NEXT to the compute (no SM is free, and a kernel with a
    static tile assignment is delayed by whatever occupies one of its SMs), so it measured slower (0.947 ms/step); it is
    kept for configurations whose backward pass leaves SMs idle.  Requires ``.grad = None`` before backward (autograd
    must install the announced tensors, not accumulate into older ones).

    NCCL averages inside the collective; gloo (the CPU tests) sums and the scale is applied on wait."""

    def __init__(self, params: Iterable[torch.nn.Parameter], group: Optional[dist.ProcessGroup] = None):
        self.params: List[torch.nn.Parameter] = [p for p in params if p.requires_grad]
        self.group = group
        self._pending = []
        self._done = set()          # data_ptr of the gradients reduced through the hook in this step

    def _active(self) -> bool:
        return dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1

    def _reduce(self, tensors: List[torch.Tensor]) -> None:
        avg = dist.get_backend(self.group) == "nccl"
        op = dist.ReduceOp.AVG if avg else dist.ReduceOp.SUM
        if len(tensors) > 1 and hasattr(dist, "all_reduce_coalesced"):
            import warnings
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                work = dist.all_reduce_coalesced(tensors, op=op, group=self.group, async_op=True)
            self._pending.append(([work], tensors, avg))
        else:
            works = [dist.all_reduce(t, op=op, group=self.group, async_op=True) for t in tensors]
            self._pending.append((works, tensors, avg))

    def hook(self, tensors) -> None:
        """Called from inside a backward pass with freshly produced fp32 gradient tensors (any stream)."""
        if not self._active():
            return
        ts = [t for t in tensors if t is not None and t.numel() > 0]
        if not ts:
            return
        for t in ts:
            self._done.add(t.data_ptr())
        self._reduce(ts)

    def bucket(self, tensors):
        """Called ONCE from inside a backward pass with every gradient it produces (``None`` entries allowed): the fp32
        tensors are packed into one flat buffer whose all-reduce starts right away, and the list comes back with each of
        them replaced by its view of that buffer -- the caller returns those views to autograd, so ``.grad`` ends up
        inside the reduced buffer with no copy back (``GatedGCNStack.grad_bucket_hook = reducer.bucket``: the
        collective then runs next to the input-gradient projection, which is launched on fewer SMs to leave it room)."""
        if not self._active():
            return tensors
        if any(p.grad is not None for p in self.params):
            # autograd would ACCUMULATE the views into the existing .grad tensors on the compute stream while the
            # collective is still writing them: leave everything to the flat bucket after the backward pass
            return tensors
        idx = [i for i, t in enumerate(tensors) if t is not None and t.numel() > 0 and t.dtype == torch.float32]
        if not idx:
            return tensors
        flat = torch.cat([tensors[i].reshape(-1) for i in idx])
        self._reduce([flat])
        out, off = list(tensors), 0
        for i in idx:
            n = tensors[i].numel()
            out[i] = flat[off:off + n].view_as(tensors[i])
            self._done.add(out[i].data_ptr())
            off += n
        return out

    def start(self) -> None:
        if not self._active():
            return
        rest = [p for p in self.params if p.grad is not None and p.grad.data_ptr() not in self._done]
        self.n_late = len(rest)          # gradients no hook announced (diagnostic)
        if not rest:
            return
        if len(rest) == 1:
            self._reduce([rest[0].grad])
            return
        # one flat bucket: a single collective over one contiguous buffer (measured at 2 GPUs: 0.923 ms/step for a
        # coalesced group of 22 small tensors, less for one flat 2.3 MB all-reduce); nothing is copied back -- each
        # parameter's .grad is re-pointed at its slice of the reduced buffer
        flat = torch.cat([p.grad.reshape(-1).float() for p in rest])
        self._reduce([flat])
        off = 0
        for p in rest:
            n = p.grad.numel()
            p.grad = flat[off:off + n].view_as(p.grad) if p.grad.dtype == torch.float32 else flat[off:off + n].view_as(p.grad).to(p.grad.dtype)
            off += n

    def wait(self) -> None:
        world = dist.get_world_size(self.group) if self._pending else 1
        for works, tensors, avg in self._pending:
            for w in works:
                w.wait()
            if not avg:
                torch._foreach_mul_(tensors, 1.0 / world)
        self._pending = []
        self._done = set()

    def __call__(self) -> None:
        self.start()
        self.wait()
