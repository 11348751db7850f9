"""Data parallelism over crystals (one process per GPU, torch.distributed / NCCL over NVLink).

The reference is single-process (SURVEY.md section 2.1); crystals are independent except for (1) the gradient sum
and (2) the batch-wide padding length Nmax that sets every crystal's phantom-key count (SURVEY.md 0.1-4, 8e).
This module provides

* ``shard_crystals``      length-balanced (LPT) assignment of crystals to ranks with equal crystal counts (+-1),
* ``take_crystals``       slices a collated batch down to a list of crystals (re-indexing nodes/edges),
* ``GradReducer``         bucketed all-reduce(SUM) of the live gradients, launched from post-accumulate hooks on a
                          side stream so that it overlaps the rest of the backward pass, deterministic bucket order,
* ``loss_weight``         B_local / B_global, which makes SUM-reduced local gradients equal the single-process
                          gradient of the reference's mean-over-crystals loss.

It is model-agnostic (works on CPU tensors with gloo, which is how the CPU tests exercise it).  It reduces parameter
gradients only; gradients with respect to a rank's inputs (positions, lattices) stay local to that rank.
"""
from __future__ import annotations

from typing import Dict, Iterable, List, Optional, Sequence

import torch
import torch.distributed as dist

from .synthetic import CrystalBatch

DEAD_MARKERS = ("node_mlp_1", ".self_attn.", "alpha")


def live_named_parameters(model: torch.nn.Module):
    """Parameters that receive gradients (the reference's dead parameters never do: SURVEY.md 0.1-9)."""
    for name, p in model.named_parameters():
        if name == "alpha" or any(mk in name for mk in DEAD_MARKERS[:2]):
            continue
        yield name, p


def crystal_cost(n_nodes: torch.Tensor, n_edges: torch.Tensor, T: int, hidden: int = 256) -> torch.Tensor:
    """Relative work per crystal: edge MLP + node MLP + the per-token transformer work (constant per crystal)."""
    h = float(hidden)
    edge = n_edges.double() * (3 * h * 2 * h + 2 * h * h)
    node = n_nodes.double() * (2 * h * 2 * h + 2 * h * h + 4 * T * h * 3)
    tok = float(T) * (10 * 8 * h * h + 4.5 * h * h + 16 * T * h)
    return edge + node + tok


def shard_crystals(cost: Sequence[float], world: int) -> List[List[int]]:
    """Greedy longest-processing-time assignment with equal crystal counts (+-1) per rank; deterministic."""
    B = len(cost)
    order = sorted(range(B), key=lambda i: (-float(cost[i]), i))
    cap = [B // world + (1 if r < B % world else 0) for r in range(world)]
    load = [0.0] * world
    bins: List[List[int]] = [[] for _ in range(world)]
    for i in order:
        r = min((r for r in range(world) if len(bins[r]) < cap[r]), key=lambda r: (load[r], r))
        bins[r].append(i)
        load[r] += float(cost[i])
    return [sorted(b) for b in bins]


def take_crystals(g: CrystalBatch, ids: Sequence[int]) -> CrystalBatch:
    """Sub-batch holding crystals ``ids`` (CPU tensors), with nodes/edges re-indexed like a fresh collate."""
    ids_t = torch.as_tensor(list(ids), dtype=torch.long)
    B = g.system.numel()
    n = torch.bincount(g.batch, minlength=B)
    off = torch.cat([n.new_zeros(1), n.cumsum(0)])
    keep_node = torch.zeros(B, dtype=torch.bool)
    keep_node[ids_t] = True
    node_sel = torch.nonzero(keep_node[g.batch]).squeeze(1)
    # new crystal id of each kept crystal, in the order of ``ids``
    newid = torch.full((B,), -1, dtype=torch.long)
    newid[ids_t] = torch.arange(ids_t.numel())
    order = torch.argsort(newid[g.batch[node_sel]], stable=True)
    node_sel = node_sel[order]
    remap = torch.full((g.batch.numel(),), -1, dtype=torch.long)
    remap[node_sel] = torch.arange(node_sel.numel())
    ei = g.edge_index if "edge_index" in g else None
    fields: Dict[str, object] = {}
    e_sel = None
    if ei is not None:
        e_keep = keep_node[g.batch[ei[0]]]
        e_sel = torch.nonzero(e_keep).squeeze(1)
        e_order = torch.argsort(remap[ei[0, e_sel]], stable=True)
        e_sel = e_sel[e_order]
    for k in g.keys():
        v = getattr(g, k)
        if k == "edge_index":
            fields[k] = remap[ei[:, e_sel]]
        elif k in ("edge_attr", "edge_vec"):
            fields[k] = v[e_sel]
        elif k == "x":
            fields[k] = v[node_sel]
        elif k == "batch":
            fields[k] = newid[v[node_sel]]
        elif k == "glob":
            fields[k] = v.view(B, -1)[ids_t].reshape(-1)
        elif k == "y_ft":
            fields[k] = v.view(B, -1)[ids_t].reshape(-1)
        elif k in ("system", "phdos"):
            fields[k] = v[ids_t]
        elif k == "mp_id":
            fields[k] = [v[i] for i in ids_t.tolist()]
        else:
            fields[k] = v
    return CrystalBatch(**fields)


def shard_batch(g: CrystalBatch, world: int, T: int, hidden: int = 256):
    """Returns (list of per-rank sub-batches, global Nmax, per-rank loss weights)."""
    if "edge_mask" in g:
        raise NotImplementedError("shard_batch does not carry edge_mask: shard an unmasked batch")
    B = g.system.numel()
    n = torch.bincount(g.batch, minlength=B)
    ne = torch.bincount(g.batch[g.edge_index[0]], minlength=B)
    bins = shard_crystals(crystal_cost(n, ne, T, hidden).tolist(), world)
    return [take_crystals(g, ids) for ids in bins], int(n.max()), [len(ids) / B for ids in bins], bins


def loss_weight(b_local: int, b_global: int) -> float:
    return float(b_local) / float(b_global)


class GradReducer:
    """Bucketed, overlapped all-reduce(SUM) of gradients.

    Buckets are filled in reverse parameter-creation order (the order backward produces gradients: heads first,
    encoders last).  When the last gradient of a bucket has been accumulated its hook flattens the bucket and
    enqueues the all-reduce on a side stream; ``finish()`` waits for all buckets and scatters the reduced values
    back into ``p.grad``.  The bucket order is fixed by construction, so repeated runs reduce in the same order.
    """

    def __init__(self, named_params: Iterable, group=None, bucket_bytes: int = 8 << 20, average: bool = False):
        self.group = group
        self.average = average
        params = [(n, p) for n, p in named_params if p.requires_grad]
        params.reverse()
        self.buckets: List[List[torch.nn.Parameter]] = []
        cur, size = [], 0
        for _, p in params:
            nb = p.numel() * p.element_size()
            if cur and size + nb > bucket_bytes:
                self.buckets.append(cur)
                cur, size = [], 0
            cur.append(p)
            size += nb
        if cur:
            self.buckets.append(cur)
        self._bucket_of = {}
        for bi, b in enumerate(self.buckets):
            for p in b:
                self._bucket_of[p] = bi
        self._pending = [0] * len(self.buckets)
        self._work: List[Optional[tuple]] = [None] * len(self.buckets)
        self._handles = [p.register_post_accumulate_grad_hook(self._hook) for b in self.buckets for p in b]
        dev = params[0][1].device if params else torch.device("cpu")
        self._cuda = dev.type == "cuda"
        self._stream = torch.cuda.Stream(device=dev) if self._cuda else None
        self.reset()

    @property
    def live_bytes(self) -> int:
        return sum(p.numel() * p.element_size() for b in self.buckets for p in b)

    def reset(self) -> None:
        self._pending = [len(b) for b in self.buckets]
        self._work = [None] * len(self.buckets)

    def _hook(self, p) -> None:
        bi = self._bucket_of[p]
        self._pending[bi] -= 1
        if self._pending[bi] == 0:
            self._launch(bi)

    def _launch(self, bi: int) -> None:
        grads = [p.grad for p in self.buckets[bi]]
        if self._cuda:
            ready = torch.cuda.current_stream().record_event()
            with torch.cuda.stream(self._stream):
                self._stream.wait_event(ready)
                flat = torch._utils._flatten_dense_tensors(grads)
                for t in grads:
                    t.record_stream(self._stream)
                work = dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
        else:
            flat = torch._utils._flatten_dense_tensors(grads)
            work = dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
        self._work[bi] = (flat, work)

    def finish(self, optimizer=None) -> None:
        """Wait for every bucket (launching any that never completed, e.g. unused parameters) and write the reduced
        values back into ``p.grad``.

        optimizer (a dostransformer_b200.optim.AdamW): fuse the optimizer into the all-reduce epilogue instead - bucket i
        is updated straight from its reduced flat buffer on the reducer's stream as soon as its reduction has completed,
        while buckets i+1.. are still being reduced; nothing is copied back (``p.grad`` keeps the LOCAL gradient)."""
        for bi, b in enumerate(self.buckets):
            if self._work[bi] is None:
                have = [p for p in b if p.grad is not None]
                if len(have) != len(b):
                    for p in b:
                        if p.grad is None:
                            p.grad = torch.zeros_like(p)
                self._launch(bi)
        world = dist.get_world_size(self.group)
        for bi, b in enumerate(self.buckets):
            flat, work = self._work[bi]
            if self._cuda:
                with torch.cuda.stream(self._stream):
                    work.wait()
                    if self.average:
                        flat.div_(world)
                    gl = [p.grad for p in b]
                    views = list(torch._utils._unflatten_dense_tensors(flat, gl))
                    if optimizer is not None:
                        optimizer.step_subset(list(b), views)
                        flat.record_stream(self._stream)
                    else:
                        torch._foreach_copy_(gl, views)   # one launch per bucket
            else:
                work.wait()
                if self.average:
                    flat.div_(world)
                for p, red in zip(b, torch._utils._unflatten_dense_tensors(flat, [p.grad for p in b])):
                    p.grad.copy_(red)
        if self._cuda:
            torch.cuda.current_stream().wait_stream(self._stream)
        self.reset()

    def remove(self) -> None:
        for h in self._handles:
            h.remove()
        self._handles = []
