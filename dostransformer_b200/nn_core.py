"""Shared building blocks of the two drop-in models: parameter containers with the reference's names,
shapes and RNG-consumption order, and the forward graph expressed with dostransformer_b200.ops.

Parameter layout follows embedder_eDOS/DOSTransformer.py:13-43,100-190 and layers/transformer.py:22-44,101-118,
layers/multihead_attention.py:14-43 so that ``state_dict()`` keys/shapes match and ``torch.manual_seed(s)`` yields
the same initial weights (SURVEY.md section 3.4).  Dead parameters of the reference (node_mlp_1, the attention
in/out projections, phonon ``alpha``) are created too, never used, and never receive a gradient.
"""
from __future__ import annotations

import os
import threading
from contextlib import contextmanager
from typing import Dict, List, Optional, Tuple

import torch
from torch import nn

from . import _lib as L
from . import ops
from .ops import RowMap


class Group(nn.Module):
    """Named parameter container (no forward of its own)."""

    def __init__(self, **children):
        super().__init__()
        for k, v in children.items():
            setattr(self, k, v)


def _xavier_linear(i, o):
    m = nn.Linear(i, o)                       # consumes the RNG like the reference's default init first
    nn.init.xavier_uniform_(m.weight)
    nn.init.constant_(m.bias, 0.0)
    return m


def make_mlp_prelu(n_in, h):
    return nn.Sequential(nn.Linear(n_in, h), nn.PReLU(), nn.Linear(h, h))


def make_mlp_ln(n_in, h):
    return nn.Sequential(nn.Linear(n_in, 2 * h), nn.LayerNorm(2 * h), nn.PReLU(), nn.Linear(2 * h, h))


def make_processor(h):
    edge = Group(edge_mlp=make_mlp_ln(3 * h, h))
    node = Group(node_mlp_1=make_mlp_ln(2 * h, h), node_mlp_2=make_mlp_ln(2 * h, h))   # node_mlp_1 is dead
    return Group(edge_model=edge, node_model=node)


class _AttnParams(nn.Module):
    """Dead projection parameters of the reference's MultiheadAttention (never applied in its forward)."""

    def __init__(self, h):
        super().__init__()
        self.in_proj_weight = nn.Parameter(torch.empty(3 * h, h))
        self.register_parameter("in_proj_bias", None)
        self.in_proj_bias = nn.Parameter(torch.empty(3 * h))
        self.out_proj = nn.Linear(h, h)
        nn.init.xavier_uniform_(self.in_proj_weight)
        nn.init.xavier_uniform_(self.out_proj.weight)
        nn.init.constant_(self.in_proj_bias, 0.0)
        nn.init.constant_(self.out_proj.bias, 0.0)


class EnergyEncoderParams(nn.Module):
    """Parameters of one pre-LN encoder stack (layers/transformer.py TransformerEncoder)."""

    def __init__(self, h, n_layers, attn_dropout=0.0):
        super().__init__()
        self.attn_dropout = attn_dropout
        self.layers = nn.ModuleList()
        for _ in range(n_layers):
            attn = _AttnParams(h)
            fc1 = _xavier_linear(h, 4 * h)
            fc2 = _xavier_linear(4 * h, h)
            norms = nn.ModuleList([nn.LayerNorm(h), nn.LayerNorm(h)])
            self.layers.append(Group(self_attn=attn, fc1=fc1, fc2=fc2, layer_norms=norms))
        self.register_buffer("version", torch.Tensor([2]))
        self.layer_norm = nn.LayerNorm(h)

    def extra_repr(self):
        return f"projection-free single-head attention, attn_dropout={self.attn_dropout}"


# ----------------------------------------------------------------------------------------------------- forward pieces
def mlp_prelu(seq: nn.Sequential, x: torch.Tensor) -> torch.Tensor:
    """Linear -> PReLU -> Linear (encoders)."""
    h = ops.linear([(x, None)], seq[0].weight, seq[0].bias, act=L.ACT_PRELU, prelu_slope=seq[1].weight)
    return ops.linear([(h, None)], seq[2].weight, seq[2].bias)


def mlp_ln_prelu(seq: nn.Sequential, segments, M, *, residual=None, want_pre=False):
    """Linear -> LayerNorm -> PReLU -> Linear over concatenated/gathered segments (edge_mlp, node_mlp_2)."""
    h = ops.linear(segments, seq[0].weight, seq[0].bias, M=M)
    h = ops.layer_norm(h, seq[1].weight, seq[1].bias, seq[2].weight)
    return ops.linear([(h, None)], seq[3].weight, seq[3].bias, residual=residual, want_pre=want_pre)


def message_passing(processors, x, e, graph: ops.CrystalGraph, mean: bool):
    """Processor loop: DOSTransformer.py:56-59,137-148 (sum) / DOSTransformer_phonon.py:81-84,206-212 (mean)."""
    src_map = RowMap(idx=graph.row, csr=graph.by_src)
    dst_map = RowMap(idx=graph.col, csr=graph.by_dst)
    n_layers = len(processors)
    H = x.shape[1]
    blocked = ops.tc_active(x) and ops.planes_ok(2 * H) and H % 64 == 0 and graph.E >= 128 and \
        not L.switch("DOST_NO_EDGEBLOCK") and \
        (graph.by_src is not None or not torch.is_grad_enabled())
    for i, proc in enumerate(processors):
        last = i == n_layers - 1
        segs = [(x, src_map), (x, dst_map), (e, None)]
        if blocked:    # split-weight edge update on the TMA-fed tensor-core kernels (ops._EdgeBlock)
            if last:
                e_out = ops.edge_block(x, e, proc.edge_model.edge_mlp, graph, True)
            else:
                e, e_out = ops.edge_block(x, e, proc.edge_model.edge_mlp, graph, False)
        elif last:       # the updated edge state is never read after the last layer
            e_out = mlp_ln_prelu(proc.edge_model.edge_mlp, segs, graph.E)
        else:
            e, e_out = mlp_ln_prelu(proc.edge_model.edge_mlp, segs, graph.E, residual=e, want_pre=True)
        agg = ops.segment_reduce(e_out, graph.by_dst, mean)
        x = mlp_ln_prelu(proc.node_model.node_mlp_2, [(x, None), (agg, None)], graph.N, residual=x)
    return x


def _ffn(layer, y):
    """y [S, T, H] -> y + fc2(relu(fc1(LN1(y)))), same shape (layers/transformer.py:141-148)."""
    ln1 = layer.layer_norms[1]
    H = y.shape[-1]
    rows = y.numel() // H
    if ops.tc_active(y) and ops.planes_ok(H) and rows >= 128 and not L.switch("DOST_NO_FFNBLOCK"):
        return ops.ffn_block(y, ln1.weight, ln1.bias, layer.fc1.weight, layer.fc1.bias, layer.fc2.weight, layer.fc2.bias)
    y2d = y.reshape(rows, H)
    h = ops.layer_norm(y2d, ln1.weight, ln1.bias)
    h = ops.linear([(h, None)], layer.fc1.weight, layer.fc1.bias, act=L.ACT_RELU)
    return ops.linear([(h, None)], layer.fc2.weight, layer.fc2.bias, residual=y2d).view(y.shape)


def draw_dropout_base() -> int:
    """The one host random number a forward with attention dropout consumes (torch's CPU generator): attention call n of
    that forward masks with seed (base << 20) + n."""
    return int(torch.randint(0, 2 ** 31 - 1, (1,)).item())


_device_seed = threading.local()


@contextmanager
def device_seed(word: torch.Tensor):
    """Forwards inside this block draw no host base: attention call n passes seed n and ``word`` (a 1-element int64 tensor
    on the model's device) as its seed offset, so the kernels mask with n + word.  Writing ``base << 20`` into the word
    before the kernels run reproduces the masks of an eager forward that drew ``base`` (graphed.GraphedStep does this
    before every replay).  Per thread."""
    prev = getattr(_device_seed, "word", None)
    _device_seed.word = word
    try:
        yield word
    finally:
        _device_seed.word = prev


class AttentionMaps:
    """What ``attention_maps(model)`` records (per thread).

    ``maps[key]``: the attention probabilities of the layer whose reference ``MultiheadAttention`` module path is ``key``
    (``<stack>.layers.<i>.self_attn``), one tensor per call in the order a forward hook on that module would see them: the
    reference's ``attn_weights`` (multihead_attention.py:68-71) batch-first - [B, T, T] for the energy self-attention,
    [B, T, Nmax] for the energy -> atom cross-attention with atom j of the crystal in column j and the probability of ONE
    zero-padded key in each of the columns n_b .. Nmax - 1 (none with ``per_crystal_eval`` in eval mode: those columns are
    0).  With attention dropout the dropped-out probabilities mask / (1 - p) * P.  fp32, or the model's dtype for fp64.
    ``n_atoms``: atoms per crystal [B] of the last recorded forward of a DOS model."""

    def __init__(self, model: nn.Module):
        self.maps: Dict[str, List[torch.Tensor]] = {}
        self.n_atoms: Optional[torch.Tensor] = None
        self._names = {id(m): n for n, m in model.named_modules() if isinstance(m, EnergyEncoderParams)}
        self._width = None

    def _begin(self, graph: ops.CrystalGraph, per_crystal: bool) -> None:
        """Per forward of a DOS model: the padding length of its cross-attention maps (read back only when the host does not
        know it)."""
        self.n_atoms = (graph.ptr[1:] - graph.ptr[:-1]).long()
        if graph.nmax_host is not None:
            self._width = graph.nmax_host
        else:
            self._width = int(self.n_atoms.max()) if per_crystal else int(graph.nmax.item())

    def _buffer(self, enc: nn.Module, layer: int, S: int, T: int, width: int, like: torch.Tensor):
        """(key, [S, T, width] output buffer) for one attention call of ``enc``, or (None, None) when it is not recorded."""
        name = self._names.get(id(enc))
        if name is None:
            return None, None
        key = f"{name}.layers.{layer}.self_attn" if name else f"layers.{layer}.self_attn"
        return key, torch.empty(S, T, width, dtype=like.dtype, device=like.device)

    def _add(self, key: Optional[str], buf: Optional[torch.Tensor], B: int) -> None:
        """S = reps * B sequences (the global and the system branch batched): one B-row tensor per branch, in branch order."""
        if key is not None:
            self.maps.setdefault(key, []).extend(buf.split(B))


_recording = threading.local()


@contextmanager
def attention_maps(model: nn.Module):
    """``with attention_maps(model) as rec: model(batch)`` records every encoder layer's attention probabilities of the
    forwards run inside the block on this thread into ``rec.maps`` (see AttentionMaps).  The forward's results, its
    gradients and the random-number stream are unchanged; recording costs the map buffers and one extra kernel per
    attention call.  CUDA-graph replays (graphed.GraphedStep) refuse to run inside the block."""
    rec = AttentionMaps(model)
    prev = getattr(_recording, "rec", None)
    _recording.rec = rec
    try:
        yield rec
    finally:
        _recording.rec = prev


def active_recorder() -> Optional[AttentionMaps]:
    return getattr(_recording, "rec", None)


class _Seeds:
    def __init__(self, drop_p: float, training: bool):
        self.p = drop_p if training else 0.0
        self.word = getattr(_device_seed, "word", None) if self.p > 0 else None
        self.base = draw_dropout_base() if self.p > 0 and self.word is None else 0
        self.n = 0

    def next(self) -> Tuple[int, Optional[torch.Tensor]]:
        """(seed, seed_offset) of the next attention call."""
        self.n += 1
        return (self.base << 20) + self.n, self.word


def cross_stack(enc: EnergyEncoderParams, q, x_nodes, graph: ops.CrystalGraph, S: int, T: int, seeds: _Seeds):
    """Energy tokens attend to the atoms of their crystal (keys = values = LN0(x), fixed across layers)."""
    rec = active_recorder()
    for li, layer in enumerate(enc.layers):
        ln0 = layer.layer_norms[0]
        kv = ops.layer_norm(x_nodes, ln0.weight, ln0.bias)
        q_ln, q_res = ops.layer_norm(q, ln0.weight, ln0.bias, want_planes=q.dim() == 3, with_residual=True)
        key, maps = rec._buffer(enc, li, S, T, rec._width, kv) if rec is not None else (None, None)
        y = ops.cross_attention(q_ln, kv, ln0.bias, q_res, graph, S, seeds.p, *seeds.next(), maps_out=maps)
        if rec is not None:
            rec._add(key, maps, graph.B)
        q = _ffn(layer, y)
    return ops.layer_norm(q, enc.layer_norm.weight, enc.layer_norm.bias)


def self_stack(enc: EnergyEncoderParams, x0, seeds: _Seeds, B: int):
    """Self attention over the T energy tokens; keys are LN0_l of the ORIGINAL input in every layer.  B: crystals of the
    batch (sequence s belongs to crystal s % B)."""
    S, T, H = x0.shape
    x = x0
    rec = active_recorder()
    for li, layer in enumerate(enc.layers):
        ln0 = layer.layer_norms[0]
        if li == 0:
            k, x_res = ops.layer_norm(x0, ln0.weight, ln0.bias, want_planes=True, with_residual=True)
            q = k
        else:
            k = ops.layer_norm(x0, ln0.weight, ln0.bias, want_planes=True)
            q, x_res = ops.layer_norm(x, ln0.weight, ln0.bias, want_planes=True, with_residual=True)
        key, maps = rec._buffer(enc, li, S, T, T, q) if rec is not None else (None, None)
        y = ops.self_attention(q, k, x_res, seeds.p, *seeds.next(), maps_out=maps)
        if rec is not None:
            rec._add(key, maps, B)
        x = _ffn(layer, y)
    return ops.layer_norm(x, enc.layer_norm.weight, enc.layer_norm.bias)


def dos_heads(model, x_nodes, graph: ops.CrystalGraph, graph_vec, prompt_table, T: int, seeds: _Seeds):
    """DOSTransformer.py:61-91: cross-attention -> (fc | fc_prompt) -> self-attention -> cross-attention -> out_layer,
    for the global and the system branch (shared transformer_self / transformer_source / out_layer)."""
    B, H = graph.B, x_nodes.shape[1]
    rec = active_recorder()
    if rec is not None:
        rec._begin(graph, model.per_crystal_eval and not model.training)
    energies = cross_stack(model.transformer, model.embeddings.weight, x_nodes, graph, B, T, seeds)   # [B,T,H]
    e2d = energies.view(B * T, H)
    per_crystal = RowMap(div=T, div_rowptr=graph.token_rowptr(T))
    per_system = RowMap(idx=graph.system, div=T, div_rowptr=graph.token_rowptr(T), csr=graph.by_system)

    def branches(both, S):
        """transformer_self -> transformer_source -> out_layer on S sequences (sequence s belongs to crystal s % B)."""
        h = self_stack(model.transformer_self, both.view(S, T, H), seeds, B)
        h = cross_stack(model.transformer_source, h, x_nodes, graph, S, T, seeds)
        return ops.linear([(h.view(S * T, H), None)], model.out_layer.weight, model.out_layer.bias).view(S, T)

    # The global and the system branch share transformer_self / transformer_source / out_layer
    # (DOSTransformer.py:71-77 vs :85-91): they run as ONE batch of 2B sequences - half the launches, twice the rows per
    # GEMM, and the shared weights receive one gradient instead of two that autograd would have to add.
    batched = not L.switch("DOST_NO_BRANCH_BATCH")     # (dropout: one mask stream per attention call, indexed by sequence)
    buf = g_buf = s_buf = None
    if batched:
        buf, g_buf, s_buf = ops.stack2_buffer(B * T, B * T, H, e2d)
    if ops.tc_active(e2d) and ops.planes_gemm_ok(B * T, H, H) and not L.switch("DOST_NO_HEADSPLIT") \
            and not L.switch("DOST_NO_LINPLANES"):       # the row-group bias lives in the planes GEMM's epilogue
        # split weights: the per-crystal terms (graph vector, prompt embedding) are multiplied once per crystal and enter
        # the [B*T, H] GEMM as a row-group bias instead of being broadcast over the T energy tokens
        wf, wp = model.fc.weight, model.fc_prompt.weight
        rb_g = ops.linear([(graph_vec, None)], wf[:, H:], None)
        g_in = ops.linear([(e2d, None)], wf[:, :H], model.fc.bias, act=L.ACT_LEAKY, act_slope=0.01, rowbias=rb_g, rowbias_div=T,
                          out_buf=g_buf)
        rb_s = ops.linear([(graph_vec, None), (prompt_table, RowMap(idx=graph.system, csr=graph.by_system))], wp[:, H:], None,
                          M=B)
        s_in = ops.linear([(e2d, None)], wp[:, :H], model.fc_prompt.bias, act=L.ACT_LEAKY, act_slope=0.01, rowbias=rb_s,
                          rowbias_div=T, out_buf=s_buf)
    else:
        g_in = ops.linear([(e2d, None), (graph_vec, per_crystal)], model.fc.weight, model.fc.bias, M=B * T,
                          act=L.ACT_LEAKY, act_slope=0.01, out_buf=g_buf)
        s_in = ops.linear([(e2d, None), (graph_vec, per_crystal), (prompt_table, per_system)], model.fc_prompt.weight,
                          model.fc_prompt.bias, M=B * T, act=L.ACT_LEAKY, act_slope=0.01, out_buf=s_buf)
    if batched:
        dos = branches(ops.stack2(g_in, s_in, buf), 2 * B)
        return dos[:B], dos[B:]
    dos_global = branches(g_in, B)
    dos_system = branches(s_in, B)
    return dos_global, dos_system


def gemm_weights(model):
    """The 2-D weights that feed tensor-core GEMMs as the B operand (every live nn.Linear.weight except the H -> 1
    out_layer, which is a streaming row-dot): the set ops.refresh_weight_planes converts once per step.  Embedding
    tables enter as activations and the reference's dead parameters (node_mlp_1, attention projections) never run."""
    skip = ("node_mlp_1", ".self_attn.", "embeddings", "promt_token", "prompt_token", "out_layer")
    return [p for n, p in model.named_parameters() if p.dim() == 2 and not any(k in n for k in skip)]


def require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise RuntimeError(f"dostransformer_b200: {what} is on {t.device}; this implementation has no CPU fallback "
                           "(move the model and the batch to a CUDA device)")
