"""Attention dropout under whole-step CUDA-graph replay (graphed.GraphedStep).

The kernels read an optional device-resident seed offset (dost.h, the ``_dseed`` entry points): a ``_dseed`` call with word W
and seed n must be bitwise the plain entry point called with seed W + n, and a NULL offset the plain entry point.  A replayed
training step with ``attn_drop > 0`` writes one host-drawn base into that word per call, so it must give bitwise the loss and
gradients of the eager step after the same ``torch.manual_seed``, consume the same CPU random numbers, and draw a new mask on
every call."""
import ctypes as C

import pytest
import torch

from dostransformer_b200 import _lib as L
from dostransformer_b200 import ops
from dostransformer_b200.embedder_eDOS.DOSTransformer import DOSTransformer
from dostransformer_b200.embedder_phDOS.DOSTransformer_phonon import DOSTransformer_phonon
from dostransformer_b200.graphed import GraphedStep, batch_signature
from dostransformer_b200.synthetic import make_edos_batch, make_phonon_batch

pytestmark = pytest.mark.gpu
DEV = "cuda"
WORD = 0x2A5F3 << 20           # a base << 20 the host could have drawn
SEED = 7


# ------------------------------------------------------------------------------------------------ kernel level
class _PlainSymbols:
    """Stand-in for L.lib(): dost_<name>_dseed(..., seed, seed_offset, ...) runs the plain dost_<name>(..., seed + WORD, ...)
    (seed alone for a NULL offset); every other symbol is the library's."""

    def __init__(self, lib):
        self.lib, self.used = lib, set()

    def __getattr__(self, name):
        fn = getattr(self.lib, name)
        if not name.endswith("_dseed"):
            return fn
        plain = getattr(self.lib, name[:-len("_dseed")])
        i = L._SIGNATURES[name][1].index(C.c_ulonglong)

        def call(*args):
            args = list(args)
            off = args.pop(i + 1)
            if off is not None:
                args[i] += WORD
            self.used.add(name)
            return plain(*args)
        return call


def _rand(*shape, dtype=torch.float32, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(*shape, generator=g, dtype=torch.float64).to(dtype).to(DEV)


def _self_case(S, Lq, Lk, H, dtype):
    q, k, r, w = _rand(S, Lq, H, dtype=dtype, seed=1), _rand(S, Lk, H, dtype=dtype, seed=2), _rand(S, Lq, H, dtype=dtype, seed=3), \
        _rand(S, Lq, H, dtype=dtype, seed=4)
    return (lambda p, seed, off, t: ops.self_attention(t[0], t[1], t[2], p, seed, off)), [q, k, r], w


def _cross_case(sizes, T, H, dtype):
    g = make_edos_batch(len(sizes), seed=37, sizes=torch.tensor(sizes))
    gr = ops.build_graph(g.edge_index.to(DEV), g.batch.to(DEV), g.system.to(DEV), nmax_hint=g.max_num_nodes)
    S = 2 * gr.B                                 # the global and the system branch batched: sequence s -> crystal s % B
    kv, ph, q, w = _rand(gr.N, H, dtype=dtype, seed=1), _rand(H, dtype=dtype, seed=2), _rand(S, T, H, dtype=dtype, seed=3), \
        _rand(S, T, H, dtype=dtype, seed=4)
    return (lambda p, seed, off, t: ops.cross_attention(t[2], t[0], t[1], t[2], gr, S, p, seed, off)), [kv, ph, q], w


KERNEL_CASES = {
    # name: (precision, case, the _dseed symbols it must reach)
    "fused_dense": ("bf16x3", lambda: _self_case(3, 201, 201, 128, torch.float32),
                    {"dost_attn_fused_fwd_dseed", "dost_softmax_bwd_planes_dseed"}),
    "softmax_planes": ("bf16x3", lambda: _self_case(2, 300, 300, 128, torch.float32),
                       {"dost_softmax_fwd_planes_dseed", "dost_softmax_bwd_planes_dseed"}),
    "softmax_fp32": ("fp32", lambda: _self_case(3, 70, 51, 64, torch.float32), {"dost_softmax_fwd_dseed", "dost_softmax_bwd_dseed"}),
    "softmax_fp64": ("fp32", lambda: _self_case(3, 70, 51, 64, torch.float64), {"dost_softmax_fwd_dseed", "dost_softmax_bwd_dseed"}),
    "fused_ragged": ("bf16x3", lambda: _cross_case([5, 9, 3, 12, 7], 70, 128, torch.float32),
                     {"dost_attn_fused_fwd_dseed", "dost_xattn_softmax_bwd_dseed"}),
    "xattn_softmax": ("bf16x3", lambda: _cross_case([300, 5, 9], 70, 128, torch.float32),
                      {"dost_xattn_softmax_fwd_dseed", "dost_xattn_softmax_bwd_dseed"}),
    "xattn_fma_fp32": ("fp32", lambda: _cross_case([5, 9, 3, 12, 7], 70, 128, torch.float32),
                       {"dost_xattn_fwd_dseed", "dost_xattn_bwd_dseed"}),
    "xattn_fma_fp64": ("fp32", lambda: _cross_case([5, 9, 3, 12, 7], 40, 64, torch.float64),
                       {"dost_xattn_fwd_dseed", "dost_xattn_bwd_dseed"}),
}


@pytest.mark.parametrize("name", list(KERNEL_CASES))
def test_dseed_symbols_equal_the_plain_ones(name, monkeypatch):
    prec, make, symbols = KERNEL_CASES[name]
    fn, inputs, wgt = make()
    word = torch.tensor([WORD], dtype=torch.int64, device=DEV)

    def run(p, seed, off):
        leaves = [t.clone().requires_grad_(True) for t in inputs]
        with ops.precision(prec):
            out = fn(p, seed, off, leaves)
            (out * wgt).sum().backward()
        return [out.detach()] + [t.grad for t in leaves]

    dseed = run(0.1, SEED, word)                     # the kernels add the word
    null = run(0.1, WORD + SEED, None)               # NULL offset
    plain_lib = _PlainSymbols(L.lib())
    monkeypatch.setattr(L, "lib", lambda: plain_lib)
    plain = run(0.1, SEED, word)                     # routed to the plain symbols with seed WORD + SEED
    plain_null = run(0.1, WORD + SEED, None)
    monkeypatch.undo()
    assert plain_lib.used == symbols
    for a, b, c, d in zip(dseed, null, plain, plain_null):
        assert torch.equal(a, c) and torch.equal(b, d) and torch.equal(a, b)
    assert not torch.equal(dseed[0], run(0.0, 0, None)[0])          # dropout really happened
    assert not torch.equal(dseed[0], run(0.1, SEED + 1, word)[0])


# ------------------------------------------------------------------------------------------------ whole-step replay
def _edos(prec="bf16x3", p=0.1, T=201):
    torch.manual_seed(0)
    return DOSTransformer(2, 2, 200, 41, 2, 128, torch.device(DEV), p, n_energies=T, precision=prec).to(DEV).train()


def _phonon(p=0.1):
    torch.set_default_dtype(torch.float64)          # (restored by the conftest guard)
    torch.manual_seed(0)
    return DOSTransformer_phonon(2, 1, 118, 4, 64, torch.device(DEV), attn_drop=p).to(DEV).train()


def _edos_batches(sizes_a, sizes_b, T=201):
    a = [make_edos_batch(len(sizes_a), seed=10 + i, sizes=torch.tensor(sizes_a), T=T).to(DEV) for i in range(2)]
    b = [make_edos_batch(len(sizes_b), seed=20 + i, sizes=torch.tensor(sizes_b), T=T).to(DEV) for i in range(2)]
    return a, b


def _phonon_batches():
    out = []
    for B, seed in ((3, 1000), (5, 1001)):
        g = make_phonon_batch(B, seed=seed).to(DEV)
        g2 = g.clone()
        g2.phdos = g.phdos.flip(1).contiguous()                # same signature, other targets
        out.append([g, g2])
    return out


def _target(mode):
    return "y_ft" if mode == "edos" else "phdos"


def _eager(m, g, mode):
    m.zero_grad(set_to_none=True)
    dg, _, ds = m(g)
    loss = ops.dos_loss(dg, ds, getattr(g, _target(mode)), mode=mode, beta=1.0)
    loss.backward()
    return loss.detach().clone(), {k: p.grad.detach().clone() for k, p in m.named_parameters() if p.grad is not None}


REPLAY_CASES = {
    "edos_bf16x3_fused": (lambda: _edos(), lambda: _edos_batches([5, 9, 3, 12, 7, 8], [7, 11, 5, 14]), "edos"),
    "edos_fp32_fma": (lambda: _edos("fp32"), lambda: _edos_batches([5, 9, 3, 12, 7, 8], [7, 11, 5, 14]), "edos"),
    "edos_bf16x3_large_cell": (lambda: _edos(), lambda: _edos_batches([300, 5, 9], [280, 12, 4, 6]), "edos"),
    "edos_planes_T300": (lambda: _edos(T=300), lambda: _edos_batches([5, 9, 3, 12], [7, 11, 5], T=300), "edos"),
    "phonon_fp64": (lambda: _phonon(), _phonon_batches, "phonon"),
}


@pytest.mark.parametrize("name", list(REPLAY_CASES))
def test_dropout_replay_is_bitwise_the_eager_step(name):
    make_model, make_batches, mode = REPLAY_CASES[name]
    m = make_model()
    a, b = make_batches()
    assert batch_signature(a[0]) == batch_signature(a[1]) != batch_signature(b[0])
    step = GraphedStep(m, mode)
    seq = (a[0], b[0], a[1], b[1], a[0])
    for k, g in enumerate(seq):
        torch.manual_seed(100 + k)
        want_loss, want = _eager(m, g, mode)
        want_next = torch.rand(1)
        torch.manual_seed(100 + k)
        got_loss = step(g)
        assert torch.equal(torch.rand(1), want_next), k       # the same CPU random numbers, capturing calls included
        assert torch.equal(got_loss, want_loss), k
        got = {n: p.grad for n, p in m.named_parameters() if p.grad is not None}
        assert set(got) == set(want)
        for n in want:
            assert torch.equal(got[n], want[n]), (k, n)
    assert step.captures == 2 and step.replays == len(seq)


def test_replays_draw_a_new_mask_every_step():
    m = _edos()
    step = GraphedStep(m, "edos")
    g = make_edos_batch(5, seed=41, mean_atoms=8.0).to(DEV)
    torch.manual_seed(5)
    l1 = step(g).clone()
    l2 = step(g).clone()                            # no reseeding: the next base
    torch.manual_seed(5)
    l3 = step(g).clone()
    assert not torch.equal(l1, l2) and torch.equal(l1, l3)
    m.attn_drop = 0.0
    l0 = step(g).clone()
    assert not torch.equal(l0, l1)
    assert step.captures == 2 and step.replays == 4


def test_no_dropout_replay_consumes_no_random_numbers():
    m = _edos(p=0.0)
    step = GraphedStep(m, "edos")
    g = make_edos_batch(5, seed=41, mean_atoms=8.0).to(DEV)
    for _ in range(2):                              # the capturing call and a replay
        torch.manual_seed(3)
        step(g)
        got = torch.rand(1)
        torch.manual_seed(3)
        assert torch.equal(got, torch.rand(1))
    assert step._seed_word is None


def test_changing_attn_drop_recaptures_and_matches_eager():
    m = _edos()
    step = GraphedStep(m, "edos")
    g = make_edos_batch(5, seed=41, mean_atoms=8.0).to(DEV)
    for k, p in enumerate((0.1, 0.3, 0.0, 0.1)):
        m.attn_drop = p
        torch.manual_seed(k)
        want, _ = _eager(m, g, "edos")
        torch.manual_seed(k)
        assert torch.equal(step(g), want), p
    assert step.captures == 3 and step.replays == 4


def test_graphed_inference_of_a_dropout_model_equals_eager_eval():
    m = _edos().eval()
    step = GraphedStep(m, "edos", train=False)
    for i in range(2):
        g = make_edos_batch(5, seed=50 + i, sizes=torch.tensor([4, 6, 2, 9, 5])).to(DEV)
        with torch.no_grad():
            want = m(g)
        got = step(g)
        for x, y in zip(got, want):
            assert torch.equal(x, y)
    assert step.captures == 1 and step.replays == 2
