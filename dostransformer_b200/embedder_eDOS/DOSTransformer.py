"""Drop-in for the reference's ``embedder_eDOS.DOSTransformer`` (embedder_eDOS/DOSTransformer.py:12-93).

Same constructor, ``forward(g) -> (dos_global [B,T], x [N,H], dos_system [B,T])``, ``state_dict`` layout and
seeded initial weights; every device op is a kernel of libdost_b200.so (sm_100a).  There is no CPU path.
"""
from __future__ import annotations

import os

import torch
from torch import nn

from .. import nn_core as K
from .. import ops


class DOSTransformer(nn.Module):
    def __init__(self, layers, t_layers, n_atom_feats, n_bond_feats, n_glob_feats, n_hidden, device, attn_drop=0.0,
                 *, n_energies: int = 201, precision: str = None):
        super().__init__()
        if n_hidden % 32 != 0 or n_hidden > 512:
            raise ValueError("dostransformer_b200 kernels need n_hidden in {32, 64, 128, 256, 512}")
        h = n_hidden
        self.n_energies = n_energies
        self.precision = precision or os.environ.get("DOST_PRECISION", "bf16x3")   # fp32 | bf16x3 | bf16 (ops.py)
        self.attn_drop = float(attn_drop)
        # creation order == RNG order of the reference (DOSTransformer.py:17-42)
        self.embeddings = nn.Embedding(n_energies, h)
        self.promt_token = nn.Embedding(7, h // 2)          # (sic) the reference's spelling is part of the state_dict
        self.GN_encoder = K.Group(node_encoder=K.make_mlp_prelu(n_atom_feats, h),
                                  edge_encoder=K.make_mlp_prelu(n_bond_feats, h),
                                  global_encoder=K.make_mlp_prelu(n_glob_feats, h))
        self.stacked_processor = nn.ModuleList([K.make_processor(h) for _ in range(layers)])
        self.transformer = K.EnergyEncoderParams(h, t_layers, attn_drop)
        self.transformer_self = K.EnergyEncoderParams(h, t_layers, attn_drop)
        self.transformer_source = K.EnergyEncoderParams(h, t_layers, attn_drop)
        self.GN_decoder = K.Group(mlp=nn.Sequential(nn.Linear(2 * h, h)))
        self.out_layer = nn.Linear(h, 1)
        self.fc_prompt = nn.Linear(2 * h + h // 2, h)
        self.fc = nn.Linear(2 * h, h)
        self.device = device
        self.per_crystal_eval = False  # eval(): treat every crystal as its own batch (reference eval loaders use batch_size 1)
        self.max_num_nodes = None      # data-parallel: global padding length (phantom-key count) set by the sharder

    def forward(self, g):
        # kernels launch on the current device's current stream: make the model's device current for the call (the
        # autograd engine does the same for the backward nodes)
        with torch.cuda.device(self.fc.weight.device) if self.fc.weight.is_cuda else ops.nullcontext(), \
                ops.precision(self.precision):
            return self._forward(g)

    def _forward(self, g):
        K.require_cuda(self.fc.weight, "the model")
        K.require_cuda(g.x, "the batch")
        if "edge_mask" in g:
            raise NotImplementedError("the eDOS model takes no edge_mask: its skin topology re-picks the bonds on the "
                                      "device instead (neighbors.edos_topology(..., skin=s))")
        graph = ops.build_graph(g.edge_index, g.batch, g.system, nmax_override=self.max_num_nodes,
                                need_backward=torch.is_grad_enabled(),
                                nmax_hint=getattr(g, "max_num_nodes", None),
                                phantoms=not (self.per_crystal_eval and not self.training))
        seeds = K._Seeds(self.attn_drop, self.training)
        enc = self.GN_encoder
        x = K.mlp_prelu(enc.node_encoder, g.x)
        e = K.mlp_prelu(enc.edge_encoder, g.edge_attr)
        u = K.mlp_prelu(enc.global_encoder, g.glob.reshape(-1, 2))
        x = K.message_passing(self.stacked_processor, x, e, graph, mean=False)
        pooled = ops.segment_reduce(x, graph.crystals, False)
        dec = self.GN_decoder.mlp[0]
        graph_vec = ops.linear([(u, None), (pooled, None)], dec.weight, dec.bias)
        dos_global, dos_system = K.dos_heads(self, x, graph, graph_vec, self.promt_token.weight, self.n_energies, seeds)
        return dos_global, x, dos_system
