"""Drop-in for the reference's ``embedder_phDOS.DOSTransformer_phonon`` (DOSTransformer_phonon.py:14-119).

Differences from the eDOS model, as in the reference: edge features are computed from ``edge_vec`` inside the
forward (l<=1 spherical harmonics times a smooth cutoff), messages are aggregated with scatter_mean, there are no
global features, T = 51.  Runs in the dtype of its parameters (float64 under main_phDOS.py:15-16).

An optional batch field ``edge_mask`` (bool / uint8 [E] on the device) keeps only the edges with mask != 0: outputs and
gradients are those of the batch without the other edges (``edge_vec.grad`` is 0 on their rows).  A masked edge's
``edge_vec`` must be finite; ``neighbors.phonon_topology(..., skin=s, masked=True)`` builds such batches.
"""
from __future__ import annotations

import os

import torch
from torch import nn

from .. import nn_core as K
from .. import ops


def _looks_like_device(v):
    return isinstance(v, (torch.device, str))


class DOSTransformer_phonon(nn.Module):
    def __init__(self, layers, t_layers, n_atom_feats, n_bond_feats, n_hidden, device=None, attn_drop=0.0,
                 *, n_energies: int = 51, precision: str = None):
        super().__init__()
        # main_phDOS.py:68 calls (..., n_hidden, out_dim, device): the declared (device, attn_drop) slots then hold
        # (out_dim:int, device).  Accept both orders.
        if isinstance(device, int) and not isinstance(device, bool) and _looks_like_device(attn_drop):
            n_energies, device, attn_drop = int(device), attn_drop, 0.0
        if n_hidden % 32 != 0 or n_hidden > 512:
            raise ValueError("dostransformer_b200 kernels need n_hidden in {32, 64, 128, 256, 512}")
        h = n_hidden
        self.n_energies = n_energies
        self.precision = precision or os.environ.get("DOST_PRECISION", "bf16x3")   # fp32 | bf16x3 | bf16 (ops.py)
        self.attn_drop = float(attn_drop)
        # creation order == RNG order of the reference (DOSTransformer_phonon.py:19-43)
        self.embeddings = nn.Embedding(n_energies, h)
        self.prompt_token = nn.Embedding(7, h // 2)
        self.GN_encoder = K.Group(node_encoder=K.make_mlp_prelu(n_atom_feats, h),
                                  edge_encoder=K.make_mlp_prelu(n_bond_feats, h))
        self.stacked_processor = nn.ModuleList([K.make_processor(h) for _ in range(layers)])
        self.transformer = K.EnergyEncoderParams(h, t_layers, attn_drop)
        self.transformer_self = K.EnergyEncoderParams(h, t_layers, attn_drop)
        self.transformer_source = K.EnergyEncoderParams(h, t_layers, attn_drop)
        self.GN_decoder = K.Group(mlp=nn.Sequential(nn.Linear(h, h)))
        self.alpha = nn.Parameter(torch.rand(1))            # dead in the reference too
        self.out_layer = nn.Linear(h, 1)
        self.fc = nn.Linear(2 * h, h)
        self.fc_prompt = nn.Linear(2 * h + h // 2, h)
        self.device = device
        self.per_crystal_eval = False  # eval(): treat every crystal as its own batch (reference eval loaders use batch_size 1)
        self.max_num_nodes = None

    def forward(self, g):
        # kernels launch on the current device's current stream: make the model's device current for the call (the
        # autograd engine does the same for the backward nodes)
        with torch.cuda.device(self.fc.weight.device) if self.fc.weight.is_cuda else ops.nullcontext(), \
                ops.precision(self.precision):
            return self._forward(g)

    def _forward(self, g):
        K.require_cuda(self.fc.weight, "the model")
        K.require_cuda(g.x, "the batch")
        if "edge_index" not in g:
            raise NotImplementedError("radius_graph construction is a dead branch in the reference "
                                      "(DOSTransformer_phonon.py:59); provide edge_index and edge_vec")
        graph = ops.build_graph(g["edge_index"], g.batch, g.system, nmax_override=self.max_num_nodes,
                                need_backward=torch.is_grad_enabled(),
                                nmax_hint=getattr(g, "max_num_nodes", None),
                                phantoms=not (self.per_crystal_eval and not self.training),
                                edge_mask=g["edge_mask"] if "edge_mask" in g else None)
        seeds = K._Seeds(self.attn_drop, self.training)
        dtype = self.fc.weight.dtype
        enc = self.GN_encoder
        x = K.mlp_prelu(enc.node_encoder, g.x.to(dtype))
        # edge features (sh(l <= 1) x smooth cutoff of edge_vec, :74-77) are computed inside the edge encoder's first Linear
        ee = enc.edge_encoder
        e = ops.phonon_edge_encode(g["edge_vec"].to(dtype), ee[0].weight, ee[0].bias, ee[1].weight)
        e = ops.linear([(e, None)], ee[2].weight, ee[2].bias)
        x = K.message_passing(self.stacked_processor, x, e, graph, mean=True)
        pooled = ops.segment_reduce(x, graph.crystals, False)
        dec = self.GN_decoder.mlp[0]
        graph_vec = ops.linear([(pooled, None)], dec.weight, dec.bias)
        dos_global, dos_system = K.dos_heads(self, x, graph, graph_vec, self.prompt_token.weight, self.n_energies, seeds)
        return dos_global, x, dos_system
