"""Attention-map recording (``dostransformer_b200.attention_maps``): every encoder layer's attention probabilities in the
reference's layout (attn_weights of layers/multihead_attention.py:68-71, batch-first, keys zero-padded by to_dense_batch),
compared with the fp64 oracle, and recording must not change what the forward computes."""
import pytest
import torch
import torch.nn.functional as F

import dostransformer_b200 as D
from dostransformer_b200 import _lib as L
from dostransformer_b200 import ops
from dostransformer_b200.dp import take_crystals
from dostransformer_b200.embedder_eDOS.DOSTransformer import DOSTransformer
from dostransformer_b200.embedder_phDOS.DOSTransformer_phonon import DOSTransformer_phonon
from dostransformer_b200.graphed import GraphedStep
from dostransformer_b200.layers import TransformerEncoder
from dostransformer_b200.synthetic import make_edos_batch, make_phonon_batch
from oracle import dost_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = {"fp32": 1e-5, "bf16x3": 1e-4, "bf16": 5e-2, "fp64": 1e-6}          # max-abs error of a map entry
ROWSUM = {"fp32": 3e-5, "bf16x3": 3e-5, "bf16": 1e-2, "fp64": 3e-5}


def _keys(t):
    one = lambda stack: [f"{stack}.layers.{i}.self_attn" for i in range(t)]
    return one("transformer") + 2 * (one("transformer_self") + one("transformer_source"))


def _oracle_maps(monkeypatch, forward, sd, g, t, **kw):
    """The reference's attn_weights of every attention call of an oracle forward, by layer key, in call order (the
    oracle's attention restated with the probabilities kept: softmax in fp32, then type_as)."""
    probs = []
    orig = O.attention

    def attention(q, kv, drop_p=0.0, training=False):
        s = torch.bmm(q, kv.transpose(1, 2)) * (q.shape[-1] ** -0.5)
        probs.append(F.softmax(s.float(), dim=-1).type_as(s))
        return orig(q, kv, drop_p, training)

    monkeypatch.setattr(O, "attention", attention)
    forward(sd, g, **kw)
    monkeypatch.undo()
    out = {}
    for k, p in zip(_keys(t), probs):
        out.setdefault(k, []).append(p)
    return out


def _f64(g):
    g = g.clone()
    for k in g.keys():
        v = getattr(g, k)
        if torch.is_tensor(v) and v.is_floating_point():
            setattr(g, k, v.double())
    return g


def _sd64(m):
    return {k: (v.double().cpu() if v.is_floating_point() else v.cpu()) for k, v in O.state_dict_of(m).items()}


def _edos(H=256, prec="bf16x3", T=201, p=0.0, t=2):
    torch.manual_seed(0)
    return DOSTransformer(2, t, 200, 41, 2, H, torch.device(DEV), p, n_energies=T, precision=prec).to(DEV)


def _phonon():
    torch.set_default_dtype(torch.float64)          # (restored by the conftest guard)
    torch.manual_seed(0)
    return DOSTransformer_phonon(2, 2, 118, 4, 64, torch.device(DEV)).to(DEV)


def _run(m, g, mode, train):
    """Forward (+ loss and backward when training): outputs, loss, gradients, the CPU RNG state afterwards, kernel launches."""
    m.train(train)
    m.zero_grad(set_to_none=True)
    l0 = L.launch_count()
    with torch.set_grad_enabled(train):
        dg, x, ds = m(g)
        loss = grads = None
        if train:
            loss = ops.dos_loss(dg, ds, getattr(g, "y_ft" if mode == "edos" else "phdos"), mode=mode, beta=1.0)
            loss.backward()
            loss = loss.detach()
            grads = {k: p.grad.clone() for k, p in m.named_parameters() if p.grad is not None}
    torch.cuda.synchronize()
    return (dg.detach(), x.detach(), ds.detach()), loss, grads, torch.get_rng_state(), L.launch_count() - l0


def _same(a, b):
    (oa, la, ga, ra, _), (ob, lb, gb, rb, _) = a, b
    assert all(torch.equal(x, y) for x, y in zip(oa, ob))
    assert torch.equal(ra, rb)
    if la is not None:
        assert torch.equal(la, lb) and set(ga) == set(gb)
        for k in ga:
            assert torch.equal(ga[k], gb[k]), k


def _record(m, g, mode, train):
    _run(m, g, mode, train)         # (the first forward also converts the weights to operand planes once)
    torch.manual_seed(11)
    plain = _run(m, g, mode, train)
    torch.manual_seed(11)
    with D.attention_maps(m) as rec:
        recorded = _run(m, g, mode, train)
    torch.manual_seed(11)
    after = _run(m, g, mode, train)
    _same(plain, recorded)
    _same(plain, after)
    assert after[4] == plain[4] and recorded[4] > plain[4]        # recording off again: the same launches as before
    return rec


def _check(rec, ref, prec, width):
    assert set(rec.maps) == set(ref)
    for k, want in ref.items():
        got = rec.maps[k]
        assert len(got) == len(want), k
        for i, (a, b) in enumerate(zip(got, want)):
            cross = "self_attn" in k and not k.startswith("transformer_self")
            assert a.shape == b.shape and (not cross or a.shape[-1] == width), (k, i, a.shape, b.shape)
            assert a.dtype == (torch.float64 if prec == "fp64" else torch.float32)
            err = (a.double().cpu() - b.double()).abs().max().item()
            assert err <= TOL[prec], (k, i, err)
            assert (a.double().sum(-1) - 1).abs().max().item() <= ROWSUM[prec], (k, i)


EDOS_CASES = {
    # name: (H, precision, T, crystal sizes, model.max_num_nodes)
    "h256_b8_bf16x3": (256, "bf16x3", 201, [5, 1, 9, 3, 12, 7, 8, 4], None),
    "h256_b8_fp32": (256, "fp32", 201, [5, 1, 9, 3, 12, 7, 8, 4], None),
    "h256_b8_bf16": (256, "bf16", 201, [5, 1, 9, 3, 12, 7, 8, 4], None),
    "b1_bf16x3": (128, "bf16x3", 201, [11], None),
    "global_padding_bf16x3": (128, "bf16x3", 201, [5, 1, 9, 3], 23),
    "global_padding_fp32": (128, "fp32", 201, [5, 1, 9, 3], 23),
    "large_cell_bf16x3": (128, "bf16x3", 201, [300, 5, 9], None),
    "T300_bf16x3": (128, "bf16x3", 300, [5, 9, 3, 12], None),
    "h32_fp32": (32, "fp32", 201, [5, 1, 9, 3, 12], None),
}


@pytest.mark.parametrize("name", list(EDOS_CASES))
def test_edos_maps_match_the_oracle_and_change_nothing(name, monkeypatch):
    H, prec, T, sizes, gpad = EDOS_CASES[name]
    m = _edos(H, prec, T)
    m.max_num_nodes = gpad
    g = make_edos_batch(len(sizes), seed=31, sizes=torch.tensor(sizes), T=T)
    width = gpad or max(sizes) + 1                 # (make_edos_batch adds the zero-feature node to every crystal)
    ref = _oracle_maps(monkeypatch, O.edos_forward, _sd64(m), _f64(g), 2, max_num_nodes=gpad)
    gd = g.clone().to(DEV)
    for train in (True, False):
        rec = _record(m, gd, "edos", train)
        _check(rec, ref, prec, width)
        assert torch.equal(rec.n_atoms.cpu(), torch.tensor(sizes) + 1)


def test_phonon_fp64_maps_match_the_oracle(monkeypatch):
    m = _phonon()
    g = make_phonon_batch(5, seed=1000)
    ref = _oracle_maps(monkeypatch, O.phonon_forward, _sd64(m), _f64(g), 2)
    gd = g.clone().to(DEV)
    for train in (True, False):
        rec = _record(m, gd, "phonon", train)
        _check(rec, ref, "fp64", int(torch.bincount(g.batch).max()))


def test_per_crystal_eval_maps_are_each_crystals_own(monkeypatch):
    sizes = [5, 1, 9, 3]
    m = _edos(128, "bf16x3").eval()
    m.per_crystal_eval = True
    g = make_edos_batch(len(sizes), seed=33, sizes=torch.tensor(sizes))
    with torch.no_grad(), D.attention_maps(m) as rec:
        m(g.clone().to(DEV))
    assert torch.equal(rec.n_atoms.cpu(), torch.tensor(sizes) + 1)
    sd = _sd64(m)
    for b in range(len(sizes)):
        ref = _oracle_maps(monkeypatch, O.edos_forward, sd, _f64(take_crystals(g, [b])), 2)
        for k, want in ref.items():
            for a, w in zip(rec.maps[k], want):
                assert a.shape[-1] == (max(sizes) + 1 if not k.startswith("transformer_self") else 201)
                a = a[b].cpu().double()
                cols = w.shape[-1]
                assert (a[:, :cols] - w[0]).abs().max().item() <= TOL["bf16x3"], (k, b)
                assert not a[:, cols:].any(), (k, b)


def test_transformer_encoder_dropin_maps(monkeypatch):
    torch.manual_seed(1)
    enc = TransformerEncoder(64, 1, 2).to(DEV)
    sd = {"t." + k: v.detach().double().cpu() for k, v in enc.state_dict().items()}
    x, kv = torch.randn(21, 3, 64), torch.randn(33, 3, 64)
    probs = []
    orig = O.attention

    def attention(q, k, drop_p=0.0, training=False):
        s = torch.bmm(q, k.transpose(1, 2)) * (q.shape[-1] ** -0.5)
        probs.append(F.softmax(s.float(), dim=-1).type_as(s))
        return orig(q, k, drop_p, training)

    monkeypatch.setattr(O, "attention", attention)
    O.encoder_stack(sd, "t", x.double().transpose(0, 1), kv.double().transpose(0, 1), 2)
    monkeypatch.undo()
    xd, kvd = x.to(DEV), kv.to(DEV)
    want_out = enc(xd, kvd, kvd)
    with D.attention_maps(enc) as rec:
        out = enc(xd, kvd, kvd)
    assert torch.equal(out, want_out)
    assert list(rec.maps) == ["layers.0.self_attn", "layers.1.self_attn"]
    for k, w in zip(rec.maps, probs):
        (a,) = rec.maps[k]
        assert a.shape == (3, 21, 33) and (a.cpu().double() - w).abs().max().item() <= TOL["fp32"], k


@pytest.mark.parametrize("prec", ["bf16x3", "fp32"])
def test_dropout_maps_scale_the_kept_probabilities(prec):
    p = 0.3
    m = _edos(128, prec, p=p).train()
    g = make_edos_batch(6, seed=35, sizes=torch.tensor([5, 1, 9, 3, 12, 7])).to(DEV)
    first = "transformer.layers.0.self_attn"        # the first attention call: the same inputs with and without dropout
    torch.manual_seed(3)
    with D.attention_maps(m) as rec:
        m(g)
    dropped = rec.maps[first][0]
    m.attn_drop = 0.0
    with D.attention_maps(m) as rec:
        m(g)
    full = rec.maps[first][0]
    kept = dropped != 0
    assert 0.5 < kept.float().mean().item() < 0.9
    torch.testing.assert_close(dropped[kept], full[kept] / (1 - p), rtol=TOL[prec] * 4, atol=TOL[prec])


def test_dropout_mask_is_the_same_on_the_fused_and_the_fma_path():
    g = make_edos_batch(6, seed=35, sizes=torch.tensor([5, 1, 9, 3, 12, 7])).to(DEV)
    zeros = []
    for prec in ("bf16x3", "fp32"):
        m = _edos(128, prec, p=0.3).train()
        torch.manual_seed(3)
        with D.attention_maps(m) as rec:
            m(g)
        zeros.append(rec.maps["transformer.layers.0.self_attn"][0] == 0)
    assert zeros[0].any() and torch.equal(zeros[0], zeros[1])


def test_unbatched_branches_give_the_same_dict(monkeypatch):
    m = _edos(128, "bf16x3").eval()
    g = make_edos_batch(5, seed=37, sizes=torch.tensor([5, 1, 9, 3, 12])).to(DEV)
    with torch.no_grad(), D.attention_maps(m) as batched:
        m(g)
    monkeypatch.setenv("DOST_NO_BRANCH_BATCH", "1")
    L.reload_switches()
    try:
        with torch.no_grad(), D.attention_maps(m) as split:
            m(g)
    finally:
        monkeypatch.delenv("DOST_NO_BRANCH_BATCH")
        L.reload_switches()
    assert list(batched.maps) == list(split.maps)
    for k in batched.maps:
        assert len(batched.maps[k]) == len(split.maps[k])
        for a, b in zip(batched.maps[k], split.maps[k]):
            assert a.shape == b.shape and (a - b).abs().max().item() <= 1e-6, k


def test_graphed_step_refuses_to_run_while_recording():
    m = _edos(128, "bf16x3").train()
    step = GraphedStep(m, "edos")
    g = make_edos_batch(3, seed=39).to(DEV)
    with D.attention_maps(m):
        with pytest.raises(RuntimeError, match="attention_maps"):
            step(g)
    assert step.captures == 0 and step.replays == 0
    step(g)                                          # and works again once the recorder is gone
    assert step.replays == 1
