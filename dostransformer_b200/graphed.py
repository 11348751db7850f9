"""Whole-step CUDA-graph capture of the training / inference step.

The reference's step (main_eDOS.py:101-130: forward, loss, ``loss.backward()``) is ~700 kernel launches here, each a few
microseconds of GPU work at small batches, against ~15 ms of Python (autograd bookkeeping, ctypes marshalling,
``cuTensorMapEncodeTiled``).  At 512 crystals per GPU the device hides that; at 64 crystals per GPU (BASELINE config 3 as
written: a 512-crystal global batch over 8 GPUs), at the reference's default batch of 8 (utils.py:31) or at its
batch-size-1 evaluation loaders (main_eDOS.py:55-56) the step is host-bound.  ``GraphedStep`` records the whole step once
per *batch signature* (tensor shapes + padding length) into a ``torch.cuda.CUDAGraph`` and replays it: one host call per
step, the tensor maps, workspaces and every intermediate live in the graph's private pool.

* The kernels are launched through the C ABI on torch's current stream exactly as in eager mode - the capture sees them as
  ordinary kernel nodes.  Nothing in the step reads device memory on the host (SURVEY 8a-2 removed the reference's two
  syncs), which is what makes it capturable.
* Inputs are copied into static buffers before each replay (H2D from pinned memory or D2D); outputs (loss, predictions)
  are static tensors that the next replay overwrites.
* The bf16 operand planes of the weights are re-split INSIDE the graph (the cache is invalidated before capture), so a
  replay always sees the current weights, however they were updated.
* Variable batch shapes: ``synthetic.pad_edos_batch`` pads a batch with zero-weight dummy crystals up to bucket edges so
  that a data loader produces a handful of signatures; the loss and the gradients of the real crystals are unchanged
  (the dummies never enter the loss; their padding-length contribution is excluded, see there).
* Data parallel: the gradient all-reduce runs right after the replay on the same stream (one flat NCCL call; a step this
  short has nothing left to overlap it with).
* Attention dropout: the captured kernels read their seed offset from one int64 word on the device (``nn_core.device_seed``,
  warm-up and capture run in that mode and draw no host random number).  Every call of a training model with
  ``attn_drop > 0`` draws the one host base an eager step draws and writes ``base << 20`` into the word on the current
  stream before the replay: a fresh mask per step, the same masks, loss and gradients as the eager step after the same
  ``torch.manual_seed``, and the same CPU random-number stream.
"""
from __future__ import annotations

import gc
from typing import Dict, List, Optional, Tuple

import torch

from . import _lib as L
from . import ops
from .nn_core import active_recorder, device_seed, draw_dropout_base
from .synthetic import CrystalBatch


def batch_signature(g) -> Tuple:
    sig = []
    for k in g.keys():
        v = getattr(g, k)
        if torch.is_tensor(v):
            sig.append((k, tuple(v.shape), str(v.dtype)))
    sig.append(("max_num_nodes", getattr(g, "max_num_nodes", None)))
    sig.append(("n_valid", getattr(g, "n_valid", None)))
    return tuple(sig)


def allreduce_gradients(params, group=None, average: bool = False) -> None:
    """One flat all-reduce(SUM) of the existing gradients (deterministic order: the order of ``params``)."""
    import torch.distributed as dist
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return
    flat = torch._utils._flatten_dense_tensors(grads)
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    if average:
        flat.div_(dist.get_world_size(group))
    torch._foreach_copy_(grads, list(torch._utils._unflatten_dense_tensors(flat, grads)))


class _Entry:
    __slots__ = ("graph", "static", "out", "launches", "tensor_keys", "grads", "leaves", "topo", "input_leaves",
                 "input_grad")


_TOPO = "topology."          # prefix of the topology's tensors among a structure input's fields


def _structure_input(topo, lattice, pos, x, per_crystal) -> CrystalBatch:
    """One flat batch of a structure step's tensors (the topology's, lattice, pos, the atom rows, the per-crystal fields):
    they are copied into the static buffers and enter the signature like any batch's tensors."""
    fields = {_TOPO + k: v for k, v in topo.tensors().items()}
    fields.update(lattice=lattice, pos=pos, x=x, **per_crystal)
    s = CrystalBatch(**fields)
    s.topology_host = tuple(sorted((k, v) for k, v in topo.host().items()))
    s.topology = topo
    return s


class GraphedStep:
    """``step = GraphedStep(model, mode="edos")``; ``loss = step(batch)`` runs forward + loss + backward (gradients in
    ``p.grad``, freshly written every call) as one graph replay.  ``train=False`` captures the forward only under
    ``no_grad`` and returns ``(dos_global, x, dos_system)`` (static tensors).

    Structure gradients: ``GraphedStep(model, mode, structure=True)`` takes ``step(topology, lattice, pos, x,
    **per_crystal)`` instead of a batch, with ``topology`` from ``neighbors.phonon_topology`` / ``edos_topology`` and ``x``
    the atom rows its ``batch`` takes.  The graph contains ``topology.batch(lattice, pos, x, **per_crystal)``, so each
    replay recomputes the edge geometry at the given positions; a training replay also leaves the gradients of the loss
    with respect to ``pos`` and ``lattice`` in ``step.input_grad["pos"]`` / ``["lattice"]`` (static tensors the next replay
    of that signature overwrites).  The topology's tensors are inputs like the others: a rebuilt topology with the same
    shapes replays the same graph, another edge count captures a new one.  Skin topologies (``skin=``) work the same way:
    each replay re-picks the eDOS neighbours of the given positions and runs the topology check, and the replay's flag is
    ORed into the caller's ``topology.stale`` on the device.  Without ``structure`` only parameter gradients are carried.

    loss_weight: scales the loss (data parallel: B_local / B_global).  world > 1: all-reduce after the replay.
    A new signature costs one eager warm-up step plus the capture (~3 eager steps); ``max_graphs`` bounds the cache
    (least recently captured dropped first).
    """

    def __init__(self, model, mode: str = "edos", beta: float = 1.0, *, train: bool = True, loss_weight: float = 1.0,
                 group=None, world: int = 1, max_graphs: int = 16, target_key: Optional[str] = None,
                 structure: bool = False):
        self.model, self.mode, self.beta, self.train = model, mode, float(beta), train
        self.structure = bool(structure)
        self.input_grad: Dict[str, torch.Tensor] = {}
        self.loss_weight = float(loss_weight)
        self.group, self.world = group, int(world)
        self.max_graphs = max_graphs
        self.target_key = target_key or ("y_ft" if mode == "edos" else "phdos")
        self._entries: Dict[Tuple, _Entry] = {}
        self._pool = None
        self.captures = 0
        self.replays = 0
        self.launches = 0          # kernels of this library executed by replays (captured count x replays)
        self._params = [p for p in model.parameters()]
        self._stream = None
        self._seed_word = None     # int64 [1] on the model's device: the dropout seed offset the captured kernels read
        from .nn_core import gemm_weights
        wid = {id(w) for w in gemm_weights(model)}
        self._weight_names = [n for n, p in model.named_parameters() if id(p) in wid]

    # ------------------------------------------------------------------------------------------------------------
    def _eager(self, g, refresh: bool = False, leaves=None):
        model = self.model
        if leaves is not None:
            # forward through fresh leaf aliases of the parameters (same storage): see _capture
            return self._step_body(lambda b: torch.func.functional_call(model, leaves, (b,)), g, refresh, leaves)
        return self._step_body(model, g, refresh, None)

    def _step_body(self, forward, g, refresh, leaves):
        model = self.model
        if refresh and self._weight_names and getattr(model, "precision", "fp32") != "fp32":
            named = leaves if leaves is not None else dict(model.named_parameters())
            with ops.precision(model.precision):       # one launch per 24 weights instead of one per weight
                ops.refresh_weight_planes([named[n] for n in self._weight_names])
        if not self.train:
            with torch.no_grad():
                return forward(g)
        if leaves is None:
            model.zero_grad(set_to_none=True)
        else:
            for t in leaves.values():
                t.grad = None
        dg, _, ds = forward(g)
        nv = getattr(g, "n_valid", None)
        y = getattr(g, self.target_key)
        if nv is not None and nv != dg.shape[0]:        # bucket-padded batch: the dummy crystals never enter the loss
            T = dg.shape[1]
            dg, ds, y = dg[:nv], ds[:nv], y.reshape(-1, T)[:nv]
        loss = ops.dos_loss(dg, ds, y, mode=self.mode, beta=self.beta)
        if self.loss_weight != 1.0:
            loss = loss * self.loss_weight
        loss.backward()
        return loss.detach()       # (a loss with its grad_fn would keep the whole autograd graph of a capture alive)

    def _input(self, e: _Entry):
        """The model's batch: the static batch itself, or (structure) the topology's batch at the static positions, through
        fresh leaves of lattice / pos (same storage) created on the current stream like the parameter leaves."""
        if not self.structure:
            return e.static
        st = e.static
        lat, pos = st.lattice, st.pos
        if self.train:
            lat, pos = lat.detach().requires_grad_(), pos.detach().requires_grad_()
        e.input_leaves = {"pos": pos, "lattice": lat}
        per_crystal = {k: getattr(st, k) for k in st.keys() if not k.startswith(_TOPO) and k not in ("lattice", "pos", "x")}
        return e.topo.batch(lat, pos, st.x, **per_crystal)

    def _capture(self, g) -> _Entry:
        dev = g.x.device
        e = _Entry()
        e.tensor_keys = [k for k in g.keys() if torch.is_tensor(getattr(g, k))]
        e.static = CrystalBatch(**{k: (getattr(g, k).clone() if torch.is_tensor(getattr(g, k)) else getattr(g, k))
                                   for k in g.keys()})
        e.topo = g.topology.with_tensors({k[len(_TOPO):]: getattr(e.static, k) for k in g.keys() if k.startswith(_TOPO)}) \
            if self.structure else None
        # Warm-up (lazy one-time initialisation: kernel attributes, index caches, allocator pools) on the SAME side stream
        # the capture will use.  Autograd runs each parameter's AccumulateGrad node on the stream that was current when
        # the node was created; a node that survives from an earlier eager iteration on the default stream would pull the
        # legacy stream into the capture and invalidate it ("operation would make the legacy stream depend on a capturing
        # blocking stream").  The captured step therefore differentiates with respect to FRESH leaf aliases of the
        # parameters (p.detach(): same storage and version counter, so optimizer updates are seen; brand-new autograd
        # identity, so its accumulator nodes are born on the capture stream) and hands their .grad to the parameters.
        gc.collect()
        if self._stream is None:
            self._stream = torch.cuda.Stream(device=dev)
        s = self._stream
        s.wait_stream(torch.cuda.current_stream(dev))
        e.leaves = None
        with torch.cuda.stream(s), device_seed(self._seed_word):
            if self.train:
                e.leaves = {n: p.detach().requires_grad_(p.requires_grad) for n, p in self.model.named_parameters()}
            self._eager(self._input(e), leaves=e.leaves)
        torch.cuda.current_stream(dev).wait_stream(s)
        torch.cuda.synchronize(dev)
        L.poll_device_errors()
        ops.invalidate_weight_planes()      # the weights' operand planes must be produced inside the graph
        e.graph = torch.cuda.CUDAGraph()
        l0 = L.launch_count()
        # thread_local: other threads of the process (NCCL's watchdog polling its events, the autograd engine's worker
        # that launches the backward kernels into this capture) stay unrestricted; only this thread may not issue
        # capture-unsafe calls
        import os
        pool = None if os.environ.get("DOST_GRAPH_PRIVATE_POOLS") else self._pool
        with torch.cuda.graph(e.graph, pool=pool, stream=s, capture_error_mode="thread_local"), device_seed(self._seed_word):
            e.out = self._eager(self._input(e), refresh=True, leaves=e.leaves)
        e.launches = L.launch_count() - l0
        e.input_grad = {k: t.grad for k, t in e.input_leaves.items()} if self.structure and self.train else {}
        # the gradient buffers this graph writes (graph-pool memory, fixed addresses): re-attached on every replay, since
        # another signature's capture / replay leaves p.grad pointing at ITS buffers
        e.grads = [e.leaves[n].grad for n, _ in self.model.named_parameters()] if self.train else None
        if self._pool is None:
            self._pool = e.graph.pool()
        ops.invalidate_weight_planes()      # eager calls must not keep pointing into the graph's pool
        self.captures += 1
        return e

    def __call__(self, g, *structure, **per_crystal):
        if self.structure:
            g = _structure_input(g, *structure, per_crystal)
        else:
            assert not structure and not per_crystal, "positional structure inputs need GraphedStep(..., structure=True)"
        if active_recorder() is not None:
            raise RuntimeError("GraphedStep cannot run inside attention_maps(): a replayed graph has no attention maps to "
                               "record; run the model eagerly to record them")
        # (the model's data-parallel padding length and its dropout probability are host values baked into the captured
        # launches, and training decides whether dropout runs at all: part of the key)
        attn_drop = float(getattr(self.model, "attn_drop", 0.0))
        sig = batch_signature(g) + (("model_max_num_nodes", getattr(self.model, "max_num_nodes", None)),
                                    ("attn_drop", attn_drop), ("training", self.model.training))
        if self.structure:
            sig += (("topology", type(g.topology).__name__, g.topology_host),)
        if self.model.training and attn_drop > 0.0:
            # exactly the host draw of the eager step (nn_core._Seeds); a capture draws nothing.  No sync, no device read.
            if self._seed_word is None:
                self._seed_word = torch.zeros(1, dtype=torch.int64, device=self._params[0].device)
            self._seed_word.fill_(draw_dropout_base() << 20)
        e = self._entries.get(sig)
        if e is None:
            if len(self._entries) >= self.max_graphs:
                self._entries.pop(next(iter(self._entries)))
            e = self._entries[sig] = self._capture(g)
        for k in e.tensor_keys:
            src = getattr(g, k)
            dst = getattr(e.static, k)
            if src.data_ptr() != dst.data_ptr():
                dst.copy_(src, non_blocking=True)
        e.graph.replay()
        stale = getattr(e.static, _TOPO + "stale", None) if self.structure else None
        if stale is not None and getattr(g, _TOPO + "stale").data_ptr() != stale.data_ptr():
            # a skin topology: the replay ORed into the static copy of the caller's flag; hand the result back (no host read)
            getattr(g, _TOPO + "stale").copy_(stale, non_blocking=True)
        if e.grads is not None:
            for p, gr in zip(self._params, e.grads):
                p.grad = gr
        self.input_grad = e.input_grad
        self.replays += 1
        self.launches += e.launches
        if self.train and self.world > 1:
            allreduce_gradients(self._params, self.group)
        return e.out

    def signatures(self) -> List[Tuple]:
        return list(self._entries)
