"""Graph construction on the device (SURVEY.md section 8f rank 4): periodic neighbour lists, the phonon edge vectors
and the eDOS 12-nearest-neighbour bonds with their Gaussian distance features.

The reference builds its graphs offline on the CPU with third-party code: ``ase.neighbor_list("ijS", cutoff=r_max,
self_interaction=True)`` + ``edge_vec = pos[dst] - pos[src] + shift @ lattice`` for the phonon data (utils.py:267-273),
``Structure.get_all_neighbors(radius)`` -> 12 nearest -> ``GaussianDistance.expand`` for the eDOS data
(data/mat2graph.py:162-179,185,212-243).  These functions take a whole batch / dataset of crystals at once
(``lattice`` [C,3,3], Cartesian ``pos`` [N,3], ``node_ptr`` [C+1]) and run the kernels of csrc/neighbors.cu; the edge order
is the library's canonical one (centre atom, neighbour atom, shift), see that file.  fp64 like the reference's geometry.

Gradients with respect to the structure: when ``pos`` or ``lattice`` requires grad, ``edge_vec``, ``edge_len``,
``nbr_dist`` and ``edge_attr`` are differentiable in them.  The topology (which images are neighbours, which k are nearest)
is held at the forward's values.  The identity edges (i, i, shift 0) of the phonon lists have ``edge_vec == 0`` for every
geometry and contribute nothing to ``pos.grad`` / ``lattice.grad``.  The sums of the backward run in a fixed order
(``dost_segment_reduce`` over CSR segments), so they are bitwise reproducible.  With neither input requiring grad the
forward launches exactly the kernels it launches without this support.

Many steps on one topology: ``phonon_topology`` / ``edos_topology`` search once and keep the list; their ``batch(lattice,
pos, ...)`` recomputes only the edge geometry (``dost_edge_geometry``), with no device->host read, so that a CUDA graph can
capture it (``graphed.GraphedStep(..., structure=True)``); ``matches(lattice, pos)`` tells when to rebuild.  With
``skin=s`` they keep every image within cutoff + s instead (a Verlet skin): the eDOS topology re-picks its k nearest on the
device at every geometry, the phonon topology holds its edges, and both set the device flag ``stale`` when their batch may
differ from a fresh build (``_Skin``).  ``phonon_topology(..., skin=s, masked=True)`` follows the phonon edge set instead:
its batches carry every candidate and an ``edge_mask`` of those within r_max at each geometry.
"""
from __future__ import annotations

from typing import Dict, Tuple

import torch

from . import _lib as L
from . import ops


def _prep(lattice: torch.Tensor, pos: torch.Tensor, node_ptr: torch.Tensor):
    assert lattice.dim() == 3 and lattice.shape[1:] == (3, 3) and pos.dim() == 2 and pos.shape[1] == 3
    lattice = lattice.to(torch.float64).contiguous()
    pos = pos.to(torch.float64).contiguous()
    node_ptr = node_ptr.to(device=pos.device, dtype=torch.int64).contiguous()
    C = lattice.shape[0]
    assert node_ptr.numel() == C + 1
    counts = node_ptr[1:] - node_ptr[:-1]
    crystal_of = torch.repeat_interleave(torch.arange(C, device=pos.device, dtype=torch.int64), counts,
                                         output_size=pos.shape[0])
    return lattice, pos, node_ptr, crystal_of


class _NeighborList(torch.autograd.Function):
    """The neighbour list as a function of (lattice, pos).  Forward: the count / fill kernels.  Backward, with the topology
    fixed: g_e = d_vec_e + d_len_e v_e / |v_e| (0 on identity edges), d_pos = sum_{dst=i} g - sum_{src=i} g,
    d_lattice[c] = sum_{e in c} shift_e^T g_e."""

    @staticmethod
    def forward(ctx, lattice, pos, node_ptr, crystal_of, cutoff, self_interaction, local_ids):
        lib = L.lib()
        N = pos.shape[0]
        dev = pos.device
        st = L.stream()
        count = torch.zeros(N, dtype=torch.int64, device=dev)
        L.check(lib.dost_neighbor_count(L.p(lattice), L.p(pos), L.p(node_ptr), L.p(crystal_of), N, float(cutoff),
                                        int(self_interaction), L.p(count), st), "neighbor_count")
        edge_ptr = torch.zeros(N + 1, dtype=torch.int64, device=dev)
        torch.cumsum(count, 0, out=edge_ptr[1:])
        E = int(edge_ptr[-1].item()) if N else 0
        ei = torch.empty(2, E, dtype=torch.int64, device=dev)
        shift = torch.empty(E, 3, dtype=torch.int64, device=dev)
        vec = torch.empty(E, 3, dtype=torch.float64, device=dev)
        length = torch.empty(E, dtype=torch.float64, device=dev)
        if E:
            L.check(lib.dost_neighbor_fill(L.p(lattice), L.p(pos), L.p(node_ptr), L.p(crystal_of), N, float(cutoff),
                                           int(self_interaction), L.p(edge_ptr), int(local_ids), L.p(ei[0]), L.p(ei[1]),
                                           L.p(shift), L.p(vec), L.p(length), st), "neighbor_fill")
        ctx.mark_non_differentiable(ei, shift, edge_ptr)
        ctx.set_materialize_grads(False)
        if any(ctx.needs_input_grad[:2]):
            ctx.save_for_backward(ei, shift, vec, length, edge_ptr, node_ptr, crystal_of)
            ctx.local_ids = bool(local_ids)
        return ei, shift, vec, length, edge_ptr

    @staticmethod
    def backward(ctx, _ei, _shift, d_vec, d_len, _ptr):
        ei, shift, vec, length, edge_ptr, node_ptr, crystal_of = ctx.saved_tensors
        E, N, C = vec.shape[0], edge_ptr.numel() - 1, node_ptr.numel() - 1
        dev = vec.device
        if E == 0 or (d_vec is None and d_len is None):
            return (torch.zeros(C, 3, 3, dtype=torch.float64, device=dev),
                    torch.zeros(N, 3, dtype=torch.float64, device=dev), None, None, None, None, None)
        centre = torch.repeat_interleave(torch.arange(N, device=dev), edge_ptr[1:] - edge_ptr[:-1], output_size=E)
        dst = ei[1] + node_ptr[crystal_of[centre]] if ctx.local_ids else ei[1]
        want_lat = ctx.needs_input_grad[0] and C > 0
        cols = _edge_grad(d_vec, d_len, vec, length, centre, dst, shift, want_lat)
        rowptr = perm = None
        if ctx.needs_input_grad[1]:
            by_dst, _ = ops.csr_build(ops.to_i32(dst), N)
            rowptr, perm = by_dst.rowptr, by_dst.perm
        d_lat, d_pos = _structure_grad(cols, ops.to_i32(edge_ptr), rowptr, perm, ops.to_i32(node_ptr), N, C,
                                       ctx.needs_input_grad[1], want_lat)
        return d_lat, d_pos, None, None, None, None, None


def _edge_grad(d_vec, d_len, vec, length, src, dst, shift, want_lat):
    """Per-edge structure gradient g_e = d_vec_e + d_len_e v_e / |v_e|, 0 on the identity edges; with ``want_lat`` [E,12]:
    g, then the 9 columns shift_e^T g_e (column 3 + 3a + b = S_a g_b), else [E,3].  ``dost_edge_geometry_bwd`` performs
    these operations one by one."""
    E = vec.shape[0]
    g = torch.zeros(E, 3, dtype=torch.float64, device=vec.device) if d_vec is None else d_vec.to(torch.float64)
    if d_len is not None:
        # |v|' = v / |v|; 0 at |v| = 0 like torch's norm (only identity edges have |v| = 0, and they are dropped below)
        g = g + d_len.to(torch.float64)[:, None] * torch.where(length[:, None] > 0, vec / length[:, None], 0.0)
    # identity edges: edge_vec == 0 whatever the geometry; their (possibly ~1e12) gradient rows must not enter the sums
    identity = (dst == src) & (shift == 0).all(dim=1)
    g = g.masked_fill(identity[:, None], 0.0).contiguous()
    return torch.cat([g, (shift.to(torch.float64)[:, :, None] * g[:, None, :]).reshape(E, 9)], 1) if want_lat else g


def _structure_grad(cols, edge_ptr32, dst_rowptr, dst_perm, node_ptr32, N, C, want_pos, want_lat):
    """The per-edge gradients ``cols`` (``_edge_grad``'s layout; edges grouped by source atom along ``edge_ptr32``,
    ``dst_rowptr`` / ``dst_perm`` the CSR of their destination atoms, its first N segments used) -> (d_lattice [C,3,3],
    d_pos [N,3]): d_pos = sum_{dst=i} g - sum_{src=i} g, d_lattice[c] = sum_{e in c} shift_e^T g_e, every sum in a fixed
    order.  ``_NeighborList`` and the topologies' backward both reduce here."""
    dev = cols.device
    d_pos = torch.zeros(N, 3, dtype=torch.float64, device=dev)
    d_lat = torch.zeros(C, 3, 3, dtype=torch.float64, device=dev)
    # one pass over the edges grouped by centre (= src): per atom, sum g and (for the lattice) shift^T g; the lattice
    # gradient is then the sum over each crystal's atoms - two short fixed-order sums instead of one serial chain
    # over all of a crystal's edges
    per_atom = ops.segment_reduce_raw(cols, edge_ptr32, None, N)
    if want_pos:
        ops.segment_reduce_raw(cols[:, :3], dst_rowptr, dst_perm, N, out=d_pos)
        d_pos -= per_atom[:, :3]
    if want_lat:
        ops.segment_reduce_raw(per_atom[:, 3:], node_ptr32, None, C, out=d_lat.view(C, 9))
    return d_lat, d_pos


def neighbor_list(lattice: torch.Tensor, pos: torch.Tensor, node_ptr: torch.Tensor, cutoff: float,
                  self_interaction: bool = True, local_ids: bool = False) -> Dict[str, torch.Tensor]:
    """All periodic images within ``cutoff`` of every atom.  Returns ``edge_index`` [2,E] (row 0 = centre, row 1 =
    neighbour; ids local to the crystal if ``local_ids`` else rows of ``pos``), ``edge_shift`` [E,3] int64, ``edge_vec`` [E,3],
    ``edge_len`` [E] and ``edge_ptr`` [N+1] (edges of atom i are edge_ptr[i]..edge_ptr[i+1]).  One device->host read
    (the edge total) sizes the outputs; this is the offline stage of the reference.  ``edge_vec`` and ``edge_len`` are
    differentiable in ``lattice`` and ``pos`` (topology fixed, see the module docstring)."""
    lattice, pos, node_ptr, crystal_of = _prep(lattice, pos, node_ptr)
    ei, shift, vec, length, edge_ptr = _NeighborList.apply(lattice, pos, node_ptr, crystal_of, float(cutoff),
                                                          bool(self_interaction), bool(local_ids))
    return {"edge_index": ei, "edge_shift": shift, "edge_vec": vec, "edge_len": length, "edge_ptr": edge_ptr}


def phonon_edges(lattice, pos, node_ptr, r_max: float = 4.0) -> Dict[str, torch.Tensor]:
    """utils.build_data's edges (utils.py:267-273) for a batch of crystals: self-interaction images included."""
    return neighbor_list(lattice, pos, node_ptr, r_max, self_interaction=True, local_ids=False)


class _KnnSelect(torch.autograd.Function):
    """k nearest entries of every atom's list (dost_knn_select); dist is differentiable in edge_len: the gradient of a
    slot goes to the list edge it picked (out_edge), padded slots (edge id -1) carry none."""

    @staticmethod
    def forward(ctx, edge_len, edge_ptr, edge_dst, k, pad_idx, pad_dist):
        N = edge_ptr.numel() - 1
        dev = edge_ptr.device
        idx = torch.empty(N, k, dtype=torch.int64, device=dev)
        dist = torch.empty(N, k, dtype=torch.float64, device=dev)
        out_edge = torch.empty(N, k, dtype=torch.int64, device=dev) if ctx.needs_input_grad[0] else None
        L.check(L.lib().dost_knn_select(L.p(edge_ptr), L.p(edge_dst), L.p(edge_len), N, k, pad_idx, float(pad_dist),
                                        L.p(idx), L.p(dist), L.p(out_edge), L.stream()), "knn_select")
        ctx.mark_non_differentiable(idx)
        ctx.set_materialize_grads(False)
        if out_edge is not None:
            ctx.save_for_backward(out_edge)
            ctx.E = edge_len.numel()
        return idx, dist

    @staticmethod
    def backward(ctx, _idx, d_dist):
        (out_edge,) = ctx.saved_tensors
        E = ctx.E
        if d_dist is None or E == 0 or out_edge.numel() == 0:
            return torch.zeros(E, dtype=torch.float64, device=out_edge.device), None, None, None, None, None
        # each list edge is picked at most once; padded slots are routed to an extra segment E that is dropped
        key = torch.where(out_edge >= 0, out_edge, E).reshape(-1)
        by_edge, _ = ops.csr_build(ops.to_i32(key), E + 1)
        d_len = ops.segment_reduce_raw(d_dist.to(torch.float64).reshape(-1, 1).contiguous(), by_edge.rowptr, by_edge.perm,
                                       E + 1)
        return d_len[:E].reshape(E), None, None, None, None, None


def knn_select(nl: Dict[str, torch.Tensor], k: int, pad_idx: int, pad_dist: float) -> Tuple[torch.Tensor, torch.Tensor]:
    edge_ptr = nl["edge_ptr"]
    dst = nl["edge_index"][1].contiguous()
    return _KnnSelect.apply(nl["edge_len"], edge_ptr, dst, int(k), int(pad_idx), float(pad_dist))


class _GaussianExpand(torch.autograd.Function):
    @staticmethod
    def forward(ctx, flat, dmin, step, nfilt):
        out = torch.empty(flat.numel(), nfilt, dtype=torch.float32, device=flat.device)
        L.check(L.lib().dost_gaussian_expand(L.p(flat), flat.numel(), dmin, step, nfilt, step, L.p(out), L.stream()),
                "gaussian_expand")
        if ctx.needs_input_grad[0]:
            ctx.save_for_backward(flat)
            ctx.args = (dmin, step, nfilt)
        return out

    @staticmethod
    def backward(ctx, d_out):
        (flat,) = ctx.saved_tensors
        dmin, step, nfilt = ctx.args
        d_out = d_out.to(torch.float32).contiguous()
        d_dist = torch.empty(flat.numel(), dtype=torch.float64, device=flat.device)
        L.check(L.lib().dost_gaussian_expand_bwd(L.p(d_out), L.p(flat), flat.numel(), dmin, step, nfilt, step, L.p(d_dist),
                                                 L.stream()), "gaussian_expand_bwd")
        return d_dist, None, None, None


def gaussian_expand(dist: torch.Tensor, dmin: float = 0.0, dmax: float = 8.0, step: float = 0.2) -> torch.Tensor:
    """GaussianDistance(dmin, dmax, step).expand + fp32 cast (mat2graph.py:162-179,235): [..., nfilt].  Differentiable in
    ``dist`` (dost_gaussian_expand_bwd; the fp32 cast counts as the identity, as torch's ``.float()`` does)."""
    L.lib()
    import numpy as np
    nfilt = int(np.arange(dmin, dmax + step, step).shape[0])      # the reference's own filter count (41 for 0..8 by 0.2)
    flat = dist.to(torch.float64).contiguous().reshape(-1)
    out = _GaussianExpand.apply(flat, float(dmin), float(step), nfilt)
    return out.reshape(tuple(dist.shape) + (nfilt,))


def edos_edges(lattice, pos, node_ptr, radius: float = 8.0, k: int = 12) -> Dict[str, torch.Tensor]:
    """get_bond_info (mat2graph.py:212-243) for a batch of crystals: ``edge_index`` [2, N*k] (row 0 = centre atom, row 1 =
    neighbour; rows of ``pos``, padded slots point at the crystal's atom 0), ``edge_attr`` [N*k, 41] fp32,
    ``nbr_dist`` [N,k]."""
    nl = neighbor_list(lattice, pos, node_ptr, radius, self_interaction=False, local_ids=True)
    idx, dist = knn_select(nl, k, 0, radius + 1.0)
    N = pos.shape[0]
    node_ptr = node_ptr.to(device=pos.device, dtype=torch.int64)
    counts = node_ptr[1:] - node_ptr[:-1]
    first = torch.repeat_interleave(node_ptr[:-1], counts, output_size=N)           # first row of each atom's crystal
    centre = torch.arange(N, device=pos.device, dtype=torch.int64).repeat_interleave(k)
    nbr = (idx + first[:, None]).reshape(-1)
    feats = gaussian_expand(dist, 0.0, radius, 0.2)
    return {"edge_index": torch.stack([centre, nbr]), "edge_attr": feats.reshape(N * k, -1), "nbr_dist": dist,
            "nbr_idx_local": idx}


def edos_graph_batch(lattice, pos, node_ptr, atom_feats: torch.Tensor, radius: float = 8.0, k: int = 12, **per_crystal):
    """Structures -> the eDOS model's input batch, on the device: what ``get_crystal_graph`` (mat2graph.py:120-159) builds
    per crystal and PyG then collates.  ``atom_feats`` [N,F] are the (already scaled) element feature rows of the atoms; every
    crystal gets the all-zero prompt node appended after its atoms (mat2graph.py:155-158), which has no bonds; bonds are the
    k nearest images within ``radius`` with their Gaussian distance features.  ``per_crystal`` tensors (``glob`` [2C],
    ``system`` [C], ``y_ft`` [C*T] ...) are passed through."""
    from .synthetic import CrystalBatch
    e = edos_edges(lattice, pos, node_ptr, radius, k)
    dev = pos.device
    node_ptr = node_ptr.to(device=dev, dtype=torch.int64)
    C = node_ptr.numel() - 1
    N = pos.shape[0]
    counts = node_ptr[1:] - node_ptr[:-1]
    crystal_of = torch.repeat_interleave(torch.arange(C, device=dev, dtype=torch.int64), counts, output_size=N)
    x = torch.zeros(N + C, atom_feats.shape[1], dtype=atom_feats.dtype, device=dev)
    rows = torch.arange(N, device=dev, dtype=torch.int64) + crystal_of        # one prompt node per preceding crystal
    x[rows] = atom_feats.to(dev)
    ei = e["edge_index"]
    edge_index = torch.stack([ei[0] + crystal_of[ei[0]], ei[1] + crystal_of[ei[1]]])
    batch = torch.repeat_interleave(torch.arange(C, device=dev, dtype=torch.int64), counts + 1, output_size=N + C)
    # one host read for the padding length; this is the offline stage (the training loop gets it from the packed store)
    nmax = int(counts.max().item()) + 1 if C else 0
    return CrystalBatch(x=x, edge_index=edge_index, edge_attr=e["edge_attr"], batch=batch, max_num_nodes=nmax,
                        **per_crystal)


def phonon_graph_batch(lattice, pos, node_ptr, x: torch.Tensor, r_max: float = 4.0, **per_crystal):
    """Structures -> the phonon model's input batch on the device (utils.build_data, utils.py:249-303, then the PyG
    collate): ``x`` [N,118] are the mass-weighted one-hot rows of the atoms (the element table stays on the host),
    edges = every periodic image within ``r_max`` including the self-interaction images, ``edge_vec`` = pos[dst] - pos[src]
    + shift @ lattice.  ``per_crystal`` tensors (``system`` [C], ``phdos`` [C,51] ...) are passed through."""
    from .synthetic import CrystalBatch
    nl = phonon_edges(lattice, pos, node_ptr, r_max)
    dev = pos.device
    node_ptr = node_ptr.to(device=dev, dtype=torch.int64)
    C = node_ptr.numel() - 1
    counts = node_ptr[1:] - node_ptr[:-1]
    batch = torch.repeat_interleave(torch.arange(C, device=dev, dtype=torch.int64), counts, output_size=pos.shape[0])
    return CrystalBatch(x=x.to(dev), edge_index=nl["edge_index"], edge_vec=nl["edge_vec"], edge_shift=nl["edge_shift"],
                        batch=batch, **per_crystal)


# ------------------------------------------------------------------------------------------------ reusable topologies
class _EdgeGeometry(torch.autograd.Function):
    """The edge vectors (``want_vec``) or lengths of a topology's fixed list as a function of (lattice, pos):
    ``dost_edge_geometry`` forward, ``dost_edge_geometry_bwd`` + ``_structure_grad`` backward.  No host read either way.
    With ``want_vec``, ``len_out`` (optional, fp64 [E]) also receives the lengths, outside autograd."""

    @staticmethod
    def forward(ctx, lattice, pos, topo, want_vec, len_out=None):
        E = topo.src.numel()
        dev = pos.device
        need = any(ctx.needs_input_grad[:2])
        vec = torch.empty(E, 3, dtype=torch.float64, device=dev) if want_vec or need else None
        length = len_out if want_vec else torch.empty(E, dtype=torch.float64, device=dev)
        L.check(L.lib().dost_edge_geometry(L.p(lattice), L.p(pos), L.p(topo.crystal_of), L.p(topo.src), L.p(topo.dst),
                                           L.p(topo.shift), E, float(topo.pad), L.p(vec), L.p(length), L.stream()),
                "edge_geometry")
        ctx.set_materialize_grads(False)
        if need:
            ctx.save_for_backward(vec, None if want_vec else length)
            ctx.topo = topo
        return vec if want_vec else length

    @staticmethod
    def backward(ctx, d_out):
        vec, length = ctx.saved_tensors
        t = ctx.topo
        E, N, C = t.src.numel(), t.crystal_of.numel(), t.node_ptr.numel() - 1
        want_pos, want_lat = ctx.needs_input_grad[1], ctx.needs_input_grad[0] and C > 0
        if E == 0 or d_out is None:
            return (torch.zeros(C, 3, 3, dtype=torch.float64, device=vec.device),
                    torch.zeros(N, 3, dtype=torch.float64, device=vec.device), None, None, None)
        d_out = d_out.to(torch.float64).contiguous()
        d_vec, d_len = (d_out, None) if length is None else (None, d_out)
        return (*_topology_grad(t, d_vec, d_len, vec, length, want_pos, want_lat), None, None, None)


def _topology_grad(t, d_vec, d_len, vec, length, want_pos, want_lat):
    """(d_lattice, d_pos) of a topology's entries (``t.src`` / ``dst`` / ``shift`` and their CSR sums) from the per-entry
    gradients: ``dost_edge_geometry_bwd``, then ``_structure_grad``."""
    E, N, C = t.src.numel(), t.crystal_of.numel(), t.node_ptr.numel() - 1
    cols = torch.empty(E, 12 if want_lat else 3, dtype=torch.float64, device=t.src.device)
    L.check(L.lib().dost_edge_geometry_bwd(L.p(d_vec), L.p(d_len), L.p(vec), L.p(length), L.p(t.src), L.p(t.dst),
                                           L.p(t.shift), E, int(want_lat), L.p(cols), L.stream()), "edge_geometry_bwd")
    return _structure_grad(cols, t.src_ptr, t.dst_rowptr, t.dst_perm, t.node_ptr32, N, C, want_pos, want_lat)


class _Topology:
    """A neighbour list held fixed while the geometry moves: integer device tensors (the ``TENSORS`` fields) plus host
    values.  Entry e joins ``src[e]`` to ``dst[e]`` (rows of ``pos``; ``dst < 0``: a padded eDOS slot) through the image
    ``shift[e]``; entries are grouped by source along ``src_ptr`` (int32 [N+1]); ``dst_rowptr`` / ``dst_perm`` group them
    by destination (built once here instead of in every backward).  ``batch(lattice, pos, ...)`` is differentiable in
    ``lattice`` / ``pos``, reads nothing back to the host and can be captured in a CUDA graph; the identity entries
    (i, i, 0) and padded slots carry no gradient."""
    TENSORS = ("src", "dst", "shift", "src_ptr", "dst_rowptr", "dst_perm", "node_ptr", "node_ptr32", "crystal_of",
               "edge_index", "batch_of")

    def __init__(self, **fields):
        for k, v in fields.items():
            setattr(self, k, v)

    def tensors(self) -> Dict[str, torch.Tensor]:
        return {k: getattr(self, k) for k in self.TENSORS}

    def host(self) -> Dict[str, object]:
        return {k: v for k, v in vars(self).items() if k not in self.TENSORS}

    def with_tensors(self, tensors: Dict[str, torch.Tensor]):
        """The same host values over other tensors of the same shapes (a CUDA graph's static buffers)."""
        return type(self)(**self.host(), **tensors)

    def _geometry(self, lattice, pos, want_vec, len_out=None):
        assert lattice.shape == (self.node_ptr.numel() - 1, 3, 3) and pos.shape == (self.crystal_of.numel(), 3)
        return _EdgeGeometry.apply(lattice.to(torch.float64).contiguous(), pos.to(torch.float64).contiguous(), self,
                                   want_vec, len_out)

    def _same(self, fresh) -> bool:
        keys = ("src", "dst", "shift")
        return all(getattr(self, k).shape == getattr(fresh, k).shape for k in keys) and \
            all(torch.equal(getattr(self, k), getattr(fresh, k)) for k in keys)


def _topology_common(src, dst, shift, src_ptr32, node_ptr, crystal_of, N, padded):
    """The CSR of the entries by destination (``_NeighborList.backward``'s for a list without ``padded`` slots; padded
    slots, dst < 0, go to a segment N past the atoms)."""
    key = torch.where(dst >= 0, dst, N) if padded else dst
    by_dst, _ = ops.csr_build(ops.to_i32(key), N + 1 if padded else N)
    return dict(src=src, dst=dst, shift=shift, src_ptr=src_ptr32, dst_rowptr=by_dst.rowptr, dst_perm=by_dst.perm,
                node_ptr=node_ptr, node_ptr32=ops.to_i32(node_ptr), crystal_of=crystal_of)


class PhononTopology(_Topology):
    """``phonon_topology``'s result: the entries are the edges of ``phonon_edges`` in their order."""

    def batch(self, lattice, pos, x: torch.Tensor, **per_crystal):
        """The phonon model's input batch at (lattice, pos): ``phonon_graph_batch``'s fields, ``edge_vec`` recomputed on
        the fixed list (bitwise ``phonon_graph_batch``'s at the geometry the list was built at)."""
        from .synthetic import CrystalBatch
        vec = self._geometry(lattice, pos, True)
        return CrystalBatch(x=x.to(pos.device), edge_index=self.edge_index, edge_vec=vec, edge_shift=self.shift,
                            batch=self.batch_of, **per_crystal)

    def matches(self, lattice, pos) -> bool:
        """Rebuild the list at (lattice, pos) (one host read) and compare edges and their order with this one."""
        return self._same(phonon_topology(lattice, pos, self.node_ptr, self.r_max))


class EdosTopology(_Topology):
    """``edos_topology``'s result: N*k slots, slot i*k + r = the r-th nearest neighbour of atom i (its list edge: dst and
    shift), or a padded slot (dst = -1, distance radius + 1).  ``rows`` places the atoms among the prompt nodes."""
    TENSORS = _Topology.TENSORS + ("rows",)

    def batch(self, lattice, pos, atom_feats: torch.Tensor, **per_crystal):
        """The eDOS model's input batch at (lattice, pos): ``edos_graph_batch``'s fields, the picked distances recomputed on
        the fixed slots (bitwise ``edos_graph_batch``'s at the geometry the slots were picked at)."""
        from .synthetic import CrystalBatch
        dist = self._geometry(lattice, pos, False)
        N, C = self.crystal_of.numel(), self.node_ptr.numel() - 1
        feats = gaussian_expand(dist.view(N, self.k), 0.0, self.radius, 0.2)
        x = torch.zeros(N + C, atom_feats.shape[1], dtype=atom_feats.dtype, device=pos.device)
        x[self.rows] = atom_feats.to(pos.device)
        return CrystalBatch(x=x, edge_index=self.edge_index, edge_attr=feats.reshape(N * self.k, -1), batch=self.batch_of,
                            max_num_nodes=self.max_num_nodes, **per_crystal)

    def matches(self, lattice, pos) -> bool:
        """Rebuild at (lattice, pos) (one host read) and compare every slot's picked neighbour and shift with this one."""
        return self._same(edos_topology(lattice, pos, self.node_ptr, self.radius, self.k))


def _skin_fields(lattice, pos, skin):
    skin = float(skin)
    if not skin >= 0.0:
        raise ValueError(f"skin must be >= 0, got {skin}")
    return dict(lattice0=lattice.clone(), pos0=pos.clone(), stale=torch.zeros(1, dtype=torch.int32, device=pos.device),
                skin=skin)


def phonon_topology(lattice, pos, node_ptr, r_max: float = 4.0, *, skin=None, masked: bool = False) -> PhononTopology:
    """The phonon list of ``phonon_edges`` at (lattice, pos), kept for reuse at other geometries (one host read, here).
    With ``skin`` (>= 0): a ``PhononSkinTopology`` that holds the same edges and also watches the candidates within
    ``r_max + skin`` (see there).  With ``skin`` and ``masked=True``: a ``PhononMaskedTopology`` whose batches carry every
    candidate and an ``edge_mask`` of those within ``r_max`` at the batch's geometry (see there)."""
    if masked:
        if skin is None:
            raise ValueError("phonon_topology(masked=True) needs skin=: the candidates are the images within r_max + skin")
        return _phonon_masked_topology(lattice, pos, node_ptr, float(r_max), skin)
    with torch.no_grad():
        lattice, pos, node_ptr, crystal_of = _prep(lattice.detach(), pos.detach(), node_ptr)
        N = pos.shape[0]
        if skin is None:
            ei, shift, _, _, edge_ptr = _NeighborList.apply(lattice, pos, node_ptr, crystal_of, float(r_max), True, False)
            t = _topology_common(ei[0], ei[1], shift, ops.to_i32(edge_ptr), node_ptr, crystal_of, N, False)
            return PhononTopology(**t, edge_index=ei, batch_of=crystal_of, r_max=float(r_max), pad=0.0)
        sk = _skin_fields(lattice, pos, skin)
        cei, cshift, _, clen, cptr = _NeighborList.apply(lattice, pos, node_ptr, crystal_of, float(r_max) + sk["skin"],
                                                         True, False)
        # the edges: the candidates within r_max (the fill's own distances, so the list phonon_edges finds, in its order)
        held = clen < float(r_max)
        before = torch.zeros(clen.numel() + 1, dtype=torch.int64, device=pos.device)
        torch.cumsum(held, 0, out=before[1:])
        ei, shift = cei[:, held], cshift[held]
        t = _topology_common(ei[0], ei[1], shift, ops.to_i32(before[cptr]), node_ptr, crystal_of, N, False)
        return PhononSkinTopology(**t, edge_index=ei, batch_of=crystal_of, r_max=float(r_max), pad=0.0, cand_src=cei[0],
                                  cand_dst=cei[1], cand_shift=cshift, cand_held=held.to(torch.uint8), **sk)


def edos_topology(lattice, pos, node_ptr, radius: float = 8.0, k: int = 12, *, skin=None) -> EdosTopology:
    """The k nearest images within ``radius`` of every atom at (lattice, pos) (``edos_edges``' picks), kept for reuse at
    other geometries (one host read, here).  With ``skin`` (>= 0): an ``EdosSkinTopology`` that keeps every image within
    ``radius + skin`` and re-picks the k nearest at each geometry (see there)."""
    if skin is not None:
        return _edos_skin_topology(lattice, pos, node_ptr, float(radius), int(k), skin)
    with torch.no_grad():
        lattice, pos, node_ptr, crystal_of = _prep(lattice.detach(), pos.detach(), node_ptr)
        ei, shift, _, length, edge_ptr = _NeighborList.apply(lattice, pos, node_ptr, crystal_of, float(radius), False, True)
        N, C, dev = pos.shape[0], lattice.shape[0], pos.device
        idx = torch.empty(N, k, dtype=torch.int64, device=dev)
        dist = torch.empty(N, k, dtype=torch.float64, device=dev)
        pick = torch.empty(N, k, dtype=torch.int64, device=dev)
        L.check(L.lib().dost_knn_select(L.p(edge_ptr), L.p(ei[1].contiguous()), L.p(length), N, k, 0, float(radius) + 1.0,
                                        L.p(idx), L.p(dist), L.p(pick), L.stream()), "knn_select")
        first = node_ptr[crystal_of]                                               # first row of each atom's crystal
        E = ei.shape[1]
        sel = torch.where(pick >= 0, pick, E).reshape(-1)                         # padded slots -> an appended row
        dst = torch.cat([ei[1], ei.new_full((1,), -1)])[sel].view(N, k)
        dst = torch.where(dst >= 0, dst + first[:, None], -1).reshape(-1)
        shift = torch.cat([shift, shift.new_zeros(1, 3)])[sel]
        src = torch.arange(N, device=dev, dtype=torch.int64).repeat_interleave(k)
        src_ptr = torch.arange(0, N * k + 1, k, device=dev, dtype=torch.int32)
        t = _topology_common(src, dst, shift, src_ptr, node_ptr, crystal_of, N, True)
        # the model's edge_index and node layout, as edos_edges / edos_graph_batch build them
        nbr = (idx + first[:, None]).reshape(-1)
        edge_index = torch.stack([src + crystal_of[src], nbr + crystal_of[nbr]])
        counts = node_ptr[1:] - node_ptr[:-1]
        batch_of = torch.repeat_interleave(torch.arange(C, device=dev, dtype=torch.int64), counts + 1, output_size=N + C)
        rows = torch.arange(N, device=dev, dtype=torch.int64) + crystal_of
        nmax = int(counts.max().item()) + 1 if C else 0
        return EdosTopology(**t, edge_index=edge_index, batch_of=batch_of, rows=rows, radius=float(radius), k=int(k),
                            pad=float(radius) + 1.0, max_num_nodes=nmax)


def _edos_skin_topology(lattice, pos, node_ptr, radius, k, skin) -> "EdosSkinTopology":
    with torch.no_grad():
        lattice, pos, node_ptr, crystal_of = _prep(lattice.detach(), pos.detach(), node_ptr)
        sk = _skin_fields(lattice, pos, skin)
        ei, shift, _, _, edge_ptr = _NeighborList.apply(lattice, pos, node_ptr, crystal_of, radius + sk["skin"], False,
                                                        False)
        N, C, dev = pos.shape[0], lattice.shape[0], pos.device
        t = _topology_common(ei[0], ei[1], shift, ops.to_i32(edge_ptr), node_ptr, crystal_of, N, False)
        counts = node_ptr[1:] - node_ptr[:-1]
        batch_of = torch.repeat_interleave(torch.arange(C, device=dev, dtype=torch.int64), counts + 1, output_size=N + C)
        rows = torch.arange(N, device=dev, dtype=torch.int64) + crystal_of
        nmax = int(counts.max().item()) + 1 if C else 0
        return EdosSkinTopology(**t, batch_of=batch_of, rows=rows, radius=radius, k=k, pad=radius + 1.0,
                                max_num_nodes=nmax, **sk)


# ------------------------------------------------------------------------------------------------ skin topologies
class _Skin:
    """What the skin topologies share: the build geometry ``lattice0`` / ``pos0``, ``skin`` and ``stale``, an int32 [1]
    device word.  Every ``batch()`` runs ``dost_topology_check``, which sets ``stale`` when its result may differ from a
    fresh build at that geometry; nothing clears it but ``clear()`` (or a new topology), so one 4-byte read whenever the
    caller chooses covers every call since, eager calls and CUDA-graph replays alike.

    Completeness test (per crystal, derivation in csrc/neighbors.cu): with eps = ||L0^-1 (L - L0)||_F and delta = the
    largest move of an atom's fractional coordinates measured in the current cell, every pair within the cutoff r now
    was within (r + 2 delta) / (1 - eps) at the build, so the candidates (within r + skin at the build) hold every
    such pair while that bound stays below r + skin."""

    def clear(self) -> None:
        """Reset ``stale`` on the device (no host read)."""
        self.stale.zero_()

    def _check(self, lattice, pos, cutoff, cand=(None, None, None, None)):
        src, dst, shift, held = cand
        L.check(L.lib().dost_topology_check(L.p(lattice), L.p(pos), L.p(self.lattice0), L.p(self.pos0), L.p(self.node_ptr),
                                            self.node_ptr.numel() - 1, float(cutoff), self.skin, L.p(self.crystal_of),
                                            L.p(src), L.p(dst), L.p(shift), L.p(held), 0 if src is None else src.numel(),
                                            L.p(self.stale), L.stream()), "topology_check")


def _f64(t):
    return t.to(torch.float64).contiguous()


class PhononSkinTopology(_Skin, PhononTopology):
    """``phonon_topology(..., skin=s)``: the edges of ``phonon_edges`` at the build geometry, held (the phonon model's edge
    count is a shape, fixed inside a CUDA graph), plus the candidates (``cand_*``: every image within r_max + s at the
    build, ``cand_held`` marking the edges).  ``batch`` is ``PhononTopology.batch`` and also sets ``stale`` when a
    candidate crossed r_max (the held set is no longer the list) or the candidates may be incomplete.  While ``stale`` is
    clear the batch is bitwise ``phonon_graph_batch`` at that geometry."""
    TENSORS = PhononTopology.TENSORS + ("cand_src", "cand_dst", "cand_shift", "cand_held", "lattice0", "pos0", "stale")

    def batch(self, lattice, pos, x: torch.Tensor, **per_crystal):
        g = super().batch(lattice, pos, x, **per_crystal)
        self._check(_f64(lattice), _f64(pos), self.r_max, (self.cand_src, self.cand_dst, self.cand_shift, self.cand_held))
        return g


def _phonon_masked_topology(lattice, pos, node_ptr, r_max, skin) -> "PhononMaskedTopology":
    with torch.no_grad():
        lattice, pos, node_ptr, crystal_of = _prep(lattice.detach(), pos.detach(), node_ptr)
        sk = _skin_fields(lattice, pos, skin)
        ei, shift, _, _, edge_ptr = _NeighborList.apply(lattice, pos, node_ptr, crystal_of, r_max + sk["skin"], True, False)
        t = _topology_common(ei[0], ei[1], shift, ops.to_i32(edge_ptr), node_ptr, crystal_of, pos.shape[0], False)
        return PhononMaskedTopology(**t, edge_index=ei, batch_of=crystal_of, r_max=r_max, pad=0.0, **sk)


class PhononMaskedTopology(_Skin, _Topology):
    """``phonon_topology(..., skin=s, masked=True)``: the entries (``src`` / ``dst`` / ``shift``, their CSR by destination
    built once) are the candidates, every image within r_max + s at the build geometry in canonical order, identity
    edges included.  ``batch`` carries all of them and the model's ``edge_mask``: the candidates within r_max at the
    batch's geometry (``dost_edge_within`` on the lengths ``dost_edge_geometry`` writes, the fill's own comparison).  A
    bond that crosses r_max is followed, not flagged: shapes never change, so one CUDA graph serves every geometry, and
    while ``stale`` is clear the model's results are those on ``phonon_graph_batch`` at that geometry.  ``stale`` is set
    by the completeness test only.  The masked candidates lie within r_max + s of the build geometry, so their edge
    vectors stay finite, which the zero gradient of a masked edge relies on."""
    TENSORS = _Topology.TENSORS + ("lattice0", "pos0", "stale")

    def batch(self, lattice, pos, x: torch.Tensor, **per_crystal):
        """The phonon model's input batch at (lattice, pos) over every candidate, with ``edge_mask`` (uint8 [E])."""
        from .synthetic import CrystalBatch
        lattice, pos = _f64(lattice), _f64(pos)
        length = torch.empty(self.src.numel(), dtype=torch.float64, device=pos.device)
        vec = self._geometry(lattice, pos, True, length)
        mask = self.within(length)
        self._check(lattice, pos, self.r_max)
        return CrystalBatch(x=x.to(pos.device), edge_index=self.edge_index, edge_vec=vec, edge_shift=self.shift,
                            edge_mask=mask, batch=self.batch_of, **per_crystal)

    def within(self, length: torch.Tensor) -> torch.Tensor:
        """uint8 [E]: candidate e is within r_max at the lengths ``length`` (``dost_edge_within``)."""
        mask = torch.empty(length.numel(), dtype=torch.uint8, device=length.device)
        L.check(L.lib().dost_edge_within(L.p(length), length.numel(), self.r_max, L.p(mask), L.stream()), "edge_within")
        return mask

    def live(self, lattice, pos):
        """The candidates within r_max at (lattice, pos), without touching ``stale``: (edge_index [2,E'], shift [E',3])."""
        with torch.no_grad():
            length = self._geometry(_f64(lattice), _f64(pos), False)
            keep = self.within(length).bool()
        return self.edge_index[:, keep], self.shift[keep]

    def matches(self, lattice, pos) -> bool:
        """Rebuild the list at (lattice, pos) (one host read) and compare its edges and their order with the live
        candidates there."""
        fresh = phonon_topology(lattice, pos, self.node_ptr, self.r_max)
        ei, shift = self.live(lattice, pos)
        return ei.shape == fresh.edge_index.shape and torch.equal(ei, fresh.edge_index) and torch.equal(shift, fresh.shift)


class _Reselect(torch.autograd.Function):
    """The skin re-pick as a function of (lattice, pos): ``dost_knn_reselect`` -> (nbr_dist [N,k], the model's
    edge_index [2,N*k]).  Backward: a slot's distance gradient goes to the candidate it picked (each candidate is picked
    at most once: plain stores; padded slots carry none), then ``_topology_grad`` over the candidates with their CSR by
    destination built once.  No host read either way."""

    @staticmethod
    def forward(ctx, lattice, pos, topo):
        N, k, E = topo.crystal_of.numel(), topo.k, topo.src.numel()
        dev = pos.device
        need = any(ctx.needs_input_grad[:2])
        cand_len = torch.empty(E, dtype=torch.float64, device=dev)
        cand_vec = torch.empty(E, 3, dtype=torch.float64, device=dev) if need else None
        pick = torch.empty(N, k, dtype=torch.int64, device=dev)
        dist = torch.empty(N, k, dtype=torch.float64, device=dev)
        edge_index = torch.empty(2, N * k, dtype=torch.int64, device=dev)
        L.check(L.lib().dost_knn_reselect(L.p(lattice), L.p(pos), L.p(topo.node_ptr), L.p(topo.crystal_of),
                                          L.p(topo.src_ptr), L.p(topo.dst), L.p(topo.shift), N, k, topo.radius, topo.pad,
                                          L.p(cand_len), L.p(cand_vec), L.p(pick), L.p(dist), None, None, L.p(edge_index),
                                          L.stream()), "knn_reselect")
        ctx.mark_non_differentiable(edge_index)
        ctx.set_materialize_grads(False)
        if need:
            ctx.save_for_backward(cand_vec, cand_len, pick)
            ctx.topo = topo
        return dist, edge_index

    @staticmethod
    def backward(ctx, d_dist, _ei):
        cand_vec, cand_len, pick = ctx.saved_tensors
        t = ctx.topo
        E, N, C = t.src.numel(), t.crystal_of.numel(), t.node_ptr.numel() - 1
        if E == 0 or d_dist is None:
            return (torch.zeros(C, 3, 3, dtype=torch.float64, device=pick.device),
                    torch.zeros(N, 3, dtype=torch.float64, device=pick.device), None)
        d_len = torch.zeros(E + 1, dtype=torch.float64, device=pick.device)
        # padded slots all store into the extra row E, which is dropped
        d_len.scatter_(0, torch.where(pick >= 0, pick, E).reshape(-1), d_dist.to(torch.float64).reshape(-1))
        want_pos, want_lat = ctx.needs_input_grad[1], ctx.needs_input_grad[0] and C > 0
        return (*_topology_grad(t, None, d_len[:E], cand_vec, cand_len, want_pos, want_lat), None)


class EdosSkinTopology(_Skin, _Topology):
    """``edos_topology(..., skin=s)``: the entries (``src`` / ``dst`` / ``shift``, grouped by source along ``src_ptr``) are
    the candidates, every image within radius + s of every atom at the build geometry in canonical order.  ``batch``
    re-picks the k nearest within ``radius`` on every call (``dost_knn_reselect``): shapes never change, only the slots'
    contents, so one CUDA graph serves every geometry.  While ``stale`` is clear the batch is bitwise ``edos_graph_batch``
    at that geometry; gradients reach ``pos`` / ``lattice`` through the picked candidates."""
    TENSORS = ("src", "dst", "shift", "src_ptr", "dst_rowptr", "dst_perm", "node_ptr", "node_ptr32", "crystal_of",
               "batch_of", "rows", "lattice0", "pos0", "stale")

    def batch(self, lattice, pos, atom_feats: torch.Tensor, **per_crystal):
        """The eDOS model's input batch at (lattice, pos): ``edos_graph_batch``'s fields, the k nearest re-picked."""
        from .synthetic import CrystalBatch
        N, C = self.crystal_of.numel(), self.node_ptr.numel() - 1
        assert lattice.shape == (C, 3, 3) and pos.shape == (N, 3)
        lattice, pos = _f64(lattice), _f64(pos)
        dist, edge_index = _Reselect.apply(lattice, pos, self)
        self._check(lattice, pos, self.radius)
        feats = gaussian_expand(dist, 0.0, self.radius, 0.2)
        x = torch.zeros(N + C, atom_feats.shape[1], dtype=atom_feats.dtype, device=pos.device)
        x[self.rows] = atom_feats.to(pos.device)
        return CrystalBatch(x=x, edge_index=edge_index, edge_attr=feats.reshape(N * self.k, -1), batch=self.batch_of,
                            max_num_nodes=self.max_num_nodes, **per_crystal)

    def slots(self, lattice, pos):
        """The re-pick at (lattice, pos) without touching ``stale``: (pick [N,k] candidate ids, nbr_dist [N,k], nbr [N,k]
        rows of ``pos``, shift [N,k,3]); padded slots are (-1, radius + 1, -1, 0)."""
        N, k, E = self.crystal_of.numel(), self.k, self.src.numel()
        dev = self.src.device
        out = (torch.empty(N, k, dtype=torch.int64, device=dev), torch.empty(N, k, dtype=torch.float64, device=dev),
               torch.empty(N, k, dtype=torch.int64, device=dev), torch.empty(N, k, 3, dtype=torch.int64, device=dev))
        cand_len = torch.empty(E, dtype=torch.float64, device=dev)
        lattice, pos = _f64(lattice), _f64(pos)
        L.check(L.lib().dost_knn_reselect(L.p(lattice), L.p(pos), L.p(self.node_ptr), L.p(self.crystal_of),
                                          L.p(self.src_ptr), L.p(self.dst), L.p(self.shift), N, k, self.radius, self.pad,
                                          L.p(cand_len), None, *(L.p(t) for t in out), None, L.stream()), "knn_reselect")
        return out

    def matches(self, lattice, pos) -> bool:
        """Rebuild at (lattice, pos) (one host read) and compare every slot's neighbour and shift with the re-pick there."""
        fresh = edos_topology(lattice, pos, self.node_ptr, self.radius, self.k)
        _, _, nbr, shift = self.slots(lattice, pos)
        return torch.equal(fresh.dst, nbr.reshape(-1)) and torch.equal(fresh.shift, shift.reshape(-1, 3))
