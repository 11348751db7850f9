"""Drop-in for the reference's ``layers.TransformerEncoder`` (layers/transformer.py:8-79) as a standalone module.

Sequence-first API like the reference: ``forward(x_in [Lq,B,H], x_in_k [Lk,B,H], x_in_v)``.  The reference applies
projection-free single-head attention (layers/multihead_attention.py:49-76) and every call site on the hot path
passes the same tensor as key and value, so ``x_in_v`` must be ``x_in_k``.  Dense keys (no ragged packing): the
models in this package use the ragged cross-attention kernel directly instead.
"""
from __future__ import annotations

import torch

from .. import nn_core as K
from .. import ops


class TransformerEncoder(K.EnergyEncoderParams):
    def __init__(self, embed_dim, num_heads, layers, attn_dropout=0.0, relu_dropout=0.0, res_dropout=0.0,
                 embed_dropout=0.0, attn_mask=False):
        if num_heads != 1:
            raise NotImplementedError("the reference only ever uses num_heads=1 (DOSTransformer.py:27-37)")
        if relu_dropout or res_dropout or embed_dropout:
            raise NotImplementedError("relu/res/embed dropouts are always 0.0 on the reference's hot path")
        super().__init__(embed_dim, layers, attn_dropout)
        self.embed_dim = embed_dim

    def forward(self, x_in, x_in_k=None, x_in_v=None, mask=None):
        if x_in_k is None:
            x_in_k = x_in_v = x_in
        if x_in_v is not x_in_k:
            raise NotImplementedError("key and value must be the same tensor (as at every reference call site)")
        K.require_cuda(x_in, "the input")
        seeds = K._Seeds(self.attn_dropout, self.training)
        x = _to_batch_first(x_in)
        kv0 = x if x_in_k is x_in else _to_batch_first(x_in_k)
        S, Lq, H = x.shape
        rec = K.active_recorder()
        for li, layer in enumerate(self.layers):
            ln0 = layer.layer_norms[0]
            k = ops.layer_norm(kv0, ln0.weight, ln0.bias)
            q = ops.layer_norm(x, ln0.weight, ln0.bias)
            key, maps = rec._buffer(self, li, S, Lq, k.shape[1], q) if rec is not None else (None, None)
            y = ops.self_attention(q, k, x, seeds.p, *seeds.next(), maps_out=maps)
            if rec is not None:
                rec._add(key, maps, S)
            x = K._ffn(layer, y)
        x = ops.layer_norm(x, self.layer_norm.weight, self.layer_norm.bias)
        return x.transpose(0, 1)


def _to_batch_first(t: torch.Tensor) -> torch.Tensor:
    return t.transpose(0, 1).contiguous()
