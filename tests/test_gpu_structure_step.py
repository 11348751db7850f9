"""Structure gradients on a reusable topology (neighbors.phonon_topology / edos_topology) and under CUDA-graph replay
(graphed.GraphedStep(..., structure=True)).

1. dost_edge_geometry reproduces dost_neighbor_fill's bits at the list's own geometry and the numpy contract at others;
   dost_edge_geometry_bwd is bitwise neighbors._edge_grad, the torch expression of the eager backward.
2. topology.batch at the build geometry is bitwise the *_graph_batch input, so the model outputs are identical.
3. Gradients: phonon bitwise the eager chain; eDOS the eager chain up to fp64 summation order (same per-entry terms,
   summed over the k slots instead of the whole list) and the fp64 oracle at GRAD_FLOOR.
4. Replays at new positions are bitwise the eager topology step: loss, parameter, pos and lattice gradients.
5. matches() tells a held topology from a changed one."""
import numpy as np
import pytest
import torch

from conftest import relerr
from dostransformer_b200 import _lib as L
from dostransformer_b200 import neighbors as NB
from dostransformer_b200 import ops
from dostransformer_b200.embedder_eDOS.DOSTransformer import DOSTransformer
from dostransformer_b200.embedder_phDOS.DOSTransformer_phonon import DOSTransformer_phonon
from dostransformer_b200.graphed import GraphedStep
from oracle import dost_oracle as O
from test_gpu_geometry_grad import GRAD_FLOOR, _cells, _edos_inputs, _edos_oracle, _grade, _phonon_inputs, _rel_l2
from test_structure_step_abi import contract_geometry

pytestmark = pytest.mark.gpu
DEV = "cuda"
EPS64 = 2.0 ** -53


def _big_cell_case(seed, sizes, a=9.5):
    """A small triclinic batch plus a 1-atom crystal in a cubic cell wider than the eDOS radius (all 12 slots padded)."""
    _, lattice, pos, node_ptr = _cells(seed, sizes)
    rng = np.random.default_rng(seed)
    lat = torch.cat([lattice, torch.eye(3, dtype=torch.float64, device=DEV)[None] * a])
    p = torch.cat([pos, torch.tensor(rng.uniform(0, a, (1, 3)), device=DEV)])
    ptr = torch.cat([node_ptr, node_ptr[-1:] + 1])
    return lat, p, ptr


GEOMETRY_CASES = {
    "small": lambda: _cells(1, [1, 4, 2, 7])[1:],
    "large_cell": lambda: _cells(2, [3, 9], 8.0, 11.0)[1:],
    "padded": lambda: _big_cell_case(3, [2, 5]),
}


def _perturb(lattice, pos, seed, dl=0.02, dp=0.05):
    gen = torch.Generator().manual_seed(seed)
    return (lattice + dl * torch.randn(lattice.shape, generator=gen, dtype=torch.float64).to(DEV),
            pos + dp * torch.randn(pos.shape, generator=gen, dtype=torch.float64).to(DEV))


def _raw_geometry(topo, lattice, pos):
    E = topo.src.numel()
    vec = torch.empty(E, 3, dtype=torch.float64, device=DEV)
    length = torch.empty(E, dtype=torch.float64, device=DEV)
    L.check(L.lib().dost_edge_geometry(L.p(lattice), L.p(pos), L.p(topo.crystal_of), L.p(topo.src), L.p(topo.dst),
                                       L.p(topo.shift), E, topo.pad, L.p(vec), L.p(length), L.stream()))
    return vec, length


def _contract(topo, lattice, pos):
    n = lambda t: t.cpu().numpy()
    v, d = contract_geometry(n(lattice), n(pos), n(topo.crystal_of), n(topo.src), n(topo.dst), n(topo.shift), topo.pad)
    return torch.from_numpy(v), torch.from_numpy(d)


# ------------------------------------------------------------------ 1. kernels
@pytest.mark.parametrize("case", list(GEOMETRY_CASES))
def test_edge_geometry_is_the_fill_bits_and_the_contract(case):
    lattice, pos, node_ptr = GEOMETRY_CASES[case]()
    nl = NB.phonon_edges(lattice, pos, node_ptr, 4.0)
    topo = NB.phonon_topology(lattice, pos, node_ptr, 4.0)
    vec, length = _raw_geometry(topo, lattice, pos)
    assert torch.equal(vec, nl["edge_vec"]) and torch.equal(length, nl["edge_len"])
    assert torch.equal(topo.batch(lattice, pos, torch.zeros(pos.shape[0], 118, device=DEV)).edge_vec, nl["edge_vec"])
    identity = (topo.src == topo.dst) & (topo.shift == 0).all(dim=1)
    assert int(identity.sum()) == pos.shape[0]
    e = NB.edos_edges(lattice, pos, node_ptr)
    et = NB.edos_topology(lattice, pos, node_ptr)
    vec, length = _raw_geometry(et, lattice, pos)
    assert torch.equal(length, e["nbr_dist"].reshape(-1))
    padded = et.dst < 0
    assert bool(padded.any()) or case != "padded"
    assert bool((vec[padded] == 0).all())
    for seed in (5, 6):
        lat, p = _perturb(lattice, pos, seed)
        for t in (topo, et):
            vec, length = _raw_geometry(t, lat, p)
            cv, cd = _contract(t, lat, p)
            assert torch.equal(vec.cpu(), cv) and torch.equal(length.cpu(), cd), (case, seed)


def _raw_bwd(topo, d_vec, d_len, vec, length, with_lattice):
    E = topo.src.numel()
    g = torch.empty(E, 12 if with_lattice else 3, dtype=torch.float64, device=DEV)
    L.check(L.lib().dost_edge_geometry_bwd(L.p(d_vec), L.p(d_len), L.p(vec), L.p(length), L.p(topo.src), L.p(topo.dst),
                                           L.p(topo.shift), E, int(with_lattice), L.p(g), L.stream()))
    return g


@pytest.mark.parametrize("grads", ["vec", "len", "both"])
@pytest.mark.parametrize("with_lattice", [False, True])
def test_edge_geometry_bwd_is_the_torch_expression(grads, with_lattice):
    lattice, pos, node_ptr = _big_cell_case(7, [1, 4, 6])
    lat, p = _perturb(lattice, pos, 8)
    for topo in (NB.phonon_topology(lattice, pos, node_ptr, 4.0), NB.edos_topology(lattice, pos, node_ptr)):
        vec, length = _raw_geometry(topo, lat, p)
        E = vec.shape[0]
        gen = torch.Generator().manual_seed(E)
        d_vec = torch.randn(E, 3, generator=gen, dtype=torch.float64).to(DEV) if grads != "len" else None
        d_len = torch.randn(E, generator=gen, dtype=torch.float64).to(DEV) if grads != "vec" else None
        identity = (topo.src == topo.dst) & (topo.shift == 0).all(dim=1)
        if d_vec is not None:
            d_vec[identity] *= 1e12                   # what dost_phonon_edge_encode_bwd gives the self-interaction rows
        got = _raw_bwd(topo, d_vec, d_len, vec, length, with_lattice)
        assert torch.equal(got, _raw_bwd(topo, d_vec, d_len, vec, length, with_lattice))
        keep = topo.dst >= 0                          # padded slots: the kernel's zero rows (no list edge behind them)
        want = NB._edge_grad(d_vec, d_len, vec, length, topo.src, topo.dst, topo.shift, with_lattice)
        assert torch.equal(got[keep], want[keep]) and bool((got[~keep] == 0).all())
        assert bool((got[identity] == 0).all())


# ------------------------------------------------------------------ 2./3. same inputs, gradients
def _phonon_model(H=64, p=0.0):
    torch.set_default_dtype(torch.float64)          # (restored by the conftest guard)
    torch.manual_seed(H)
    return DOSTransformer_phonon(2, 1, 118, 4, H, torch.device(DEV), p).to(DEV).train()


def _edos_model(prec, p=0.0):
    torch.manual_seed(4)
    return DOSTransformer(2, 1, 200, 41, 2, 128, torch.device(DEV), p, precision=prec).to(DEV).train()


def _step(model, g, mode, lat, pos, beta=1.0, weight=1.0):
    model.zero_grad(set_to_none=True)
    dg, _, ds = model(g)
    loss = ops.dos_loss(dg, ds, g.phdos if mode == "phonon" else g.y_ft, mode=mode, beta=beta)
    if weight != 1.0:                                 # as GraphedStep scales it
        loss = loss * weight
    loss.backward()
    grads = {k: q.grad.clone() for k, q in model.named_parameters() if q.grad is not None}
    return loss.detach(), grads, (pos.grad.clone() if pos.grad is not None else None), \
        (lat.grad.clone() if lat.grad is not None else None)


def _leaves(lattice, pos):
    return lattice.clone().requires_grad_(), pos.clone().requires_grad_()


def _same_batch(a, b):
    assert a.keys() == b.keys()
    for k in a.keys():
        u, v = getattr(a, k), getattr(b, k)
        assert torch.equal(u, v) if torch.is_tensor(u) else u == v, k


class _Phonon:
    mode = "phonon"

    def __init__(self, seed=31, sizes=(3, 1, 4, 2, 6)):
        self.cells, self.lattice, self.pos, self.node_ptr, x, system, ph = _phonon_inputs(seed, list(sizes))
        self.x, self.per = x.to(DEV), {"system": system.to(DEV), "phdos": ph.to(DEV)}

    def topology(self, lattice=None, pos=None):
        return NB.phonon_topology(self.lattice if lattice is None else lattice, self.pos if pos is None else pos,
                                  self.node_ptr)

    def eager_batch(self, lat, pos):
        return NB.phonon_graph_batch(lat, pos, self.node_ptr, self.x, **self.per)


class _Edos:
    mode = "edos"

    def __init__(self, seed=40, sizes=(3, 7, 1, 12, 5)):
        self.sizes = list(sizes)
        self.cells, self.lattice, self.pos, self.node_ptr, feats, glob, system, y = _edos_inputs(seed, self.sizes)
        self.raw = (feats, glob, system, y)
        self.x, self.per = feats.to(DEV), {"glob": glob.to(DEV), "system": system.to(DEV), "y_ft": y.to(DEV)}

    def topology(self, lattice=None, pos=None):
        return NB.edos_topology(self.lattice if lattice is None else lattice, self.pos if pos is None else pos,
                                self.node_ptr)

    def eager_batch(self, lat, pos):
        return NB.edos_graph_batch(lat, pos, self.node_ptr, self.x, **self.per)


def test_phonon_topology_batch_and_gradients_are_the_eager_chain_bits():
    d = _Phonon()
    model = _phonon_model()
    topo = d.topology()
    for lattice, pos in ((d.lattice, d.pos), _perturb(d.lattice, d.pos, 9, 1e-4, 1e-4)):
        assert topo.matches(lattice, pos)
        la, pa = _leaves(lattice, pos)
        ga = d.eager_batch(la, pa)
        want = _step(model, ga, "phonon", la, pa)
        lb, pb = _leaves(lattice, pos)
        gb = topo.batch(lb, pb, d.x, **d.per)
        _same_batch(ga, gb)
        got = _step(model, gb, "phonon", lb, pb)
        assert torch.equal(got[0], want[0]) and got[1].keys() == want[1].keys()
        assert all(torch.equal(got[1][k], want[1][k]) for k in want[1])
        assert torch.equal(got[2], want[2]) and torch.equal(got[3], want[3])
    off = d.node_ptr[1]                               # the 1-atom crystal: only its own images, exactly 0
    assert bool((got[2][off] == 0).all())


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
def test_edos_topology_batch_and_gradients(prec):
    d = _Edos()
    model = _edos_model(prec)
    sd = {k: v.cpu() for k, v in O.state_dict_of(model).items()}
    topo = d.topology()
    la, pa = _leaves(d.lattice, d.pos)
    ga = d.eager_batch(la, pa)
    ga.edge_attr.retain_grad()
    want = _step(model, ga, "edos", la, pa)
    lb, pb = _leaves(d.lattice, d.pos)
    gb = topo.batch(lb, pb, d.x, **d.per)
    _same_batch(ga, gb)
    gb.edge_attr.retain_grad()
    got = _step(model, gb, "edos", lb, pb)
    assert torch.equal(got[0], want[0]) and all(torch.equal(got[1][k], want[1][k]) for k in want[1])
    assert torch.equal(gb.edge_attr.grad, ga.edge_attr.grad)   # the same per-slot gradients reach the geometry ...
    # ... and are summed in another order (over the k slots instead of the whole list).  Each output entry is a sum of n <=
    # k + (slots picking the atom) <= 2 * 12 * 12 terms, or for the lattice a crystal's <= 12 * 12 slots: both orders are
    # within (n - 1) eps of sum |terms| of the exact sum, so |got - want| <= 2 * 288 eps S, S = the sum of |terms| <=
    # |d_dist| (|v / |v|| = 1)
    nbr = NB.edos_edges(d.lattice, d.pos, d.node_ptr)["nbr_dist"].reshape(-1).clone().requires_grad_()
    (NB.gaussian_expand(nbr).reshape(-1, 41) * ga.edge_attr.grad).sum().backward()
    a = nbr.grad.abs().masked_fill(topo.dst < 0, 0.0)
    S_pos = torch.zeros_like(d.pos).index_add_(0, topo.src, a[:, None].expand(-1, 3)) \
        .index_add_(0, topo.dst.clamp_min(0), a[:, None].expand(-1, 3))
    cry = topo.crystal_of[topo.src]
    bound_lat = (topo.shift.abs().double() * a[:, None])[:, :, None].expand(-1, 3, 3)     # [a][b]: |S_a| |d_dist|
    S_lat = torch.zeros_like(d.lattice).index_add_(0, cry, bound_lat)
    assert bool(((got[2] - want[2]).abs() <= 576 * EPS64 * S_pos).all())
    assert bool(((got[3] - want[3]).abs() <= 576 * EPS64 * S_lat).all())
    _, r64 = _edos_oracle(sd, d.cells, d.lattice, d.pos, *d.raw, d.sizes, torch.float64)
    _, r32 = _edos_oracle(sd, d.cells, d.lattice, d.pos, *d.raw, d.sizes, torch.float32)
    for k, t in (("pos", got[2]), ("lattice", got[3])):
        _grade(k, t, r64[k], GRAD_FLOOR[prec], (_rel_l2(r32[k], r64[k]), relerr(r32[k], r64[k])))
    # after a move that keeps the topology: bitwise the fresh eDOS batch at the new geometry
    lat, p = _perturb(d.lattice, d.pos, 10, 1e-4, 1e-4)
    assert topo.matches(lat, p)
    _same_batch(topo.batch(lat, p, d.x, **d.per), d.eager_batch(lat, p))


# ------------------------------------------------------------------ 4./6. replay
def _replay_case(name, p=0.0):
    if name == "phonon_fp64":
        return _Phonon(), _phonon_model(p=p)
    return _Edos(), _edos_model(name.split("_")[1], p)


def _check(got, want, step, model, ctx):
    assert torch.equal(got, want[0]), ctx
    params = {k: q.grad for k, q in model.named_parameters() if q.grad is not None}
    assert params.keys() == want[1].keys() and all(torch.equal(params[k], want[1][k]) for k in want[1]), ctx
    assert torch.equal(step.input_grad["pos"], want[2]) and torch.equal(step.input_grad["lattice"], want[3]), ctx


@pytest.mark.parametrize("name", ["edos_bf16x3", "edos_fp32", "phonon_fp64"])
def test_replays_at_new_positions_are_the_eager_topology_step(name):
    d, model = _replay_case(name)
    topo = d.topology()
    step = GraphedStep(model, d.mode, structure=True)
    for i in range(3):
        lat, p = _perturb(d.lattice, d.pos, 20 + i, 1e-3, 2e-3)
        la, pa = _leaves(lat, p)
        want = _step(model, topo.batch(la, pa, d.x, **d.per), d.mode, la, pa)
        _check(step(topo, lat, p, d.x, **d.per), want, step, model, (name, i))
        _check(step(topo, lat, p, d.x, **d.per), want, step, model, (name, i, "again"))   # 6. same input, same bits
    assert step.captures == 1 and step.replays == 6
    # a topology rebuilt at a geometry it still matches: same shapes, copied into the static buffers, no new capture
    lat, p = _perturb(d.lattice, d.pos, 30, 1e-4, 1e-4)
    t2 = d.topology(lat, p)
    assert topo.matches(lat, p) and t2.src.data_ptr() != topo.src.data_ptr()
    la, pa = _leaves(lat, p)
    want = _step(model, t2.batch(la, pa, d.x, **d.per), d.mode, la, pa)
    _check(step(t2, lat, p, d.x, **d.per), want, step, model, (name, "rebuilt"))
    assert step.captures == 1
    # another batch: another edge count, another capture
    other = _Phonon(32, (2, 5)) if d.mode == "phonon" else _Edos(41, (4, 6))
    t3 = other.topology()
    la, pa = _leaves(other.lattice, other.pos)
    want = _step(model, t3.batch(la, pa, other.x, **other.per), d.mode, la, pa)
    _check(step(t3, other.lattice, other.pos, other.x, **other.per), want, step, model, (name, "other"))
    assert step.captures == 2


@pytest.mark.parametrize("name", ["edos_bf16x3", "phonon_fp64"])
def test_replay_with_attention_dropout_is_the_eager_step(name):
    d, model = _replay_case(name, p=0.1)
    topo = d.topology()
    step = GraphedStep(model, d.mode, structure=True)
    for i in range(3):
        lat, p = _perturb(d.lattice, d.pos, 40 + i, 1e-3, 2e-3)
        torch.manual_seed(100 + i)
        la, pa = _leaves(lat, p)
        want = _step(model, topo.batch(la, pa, d.x, **d.per), d.mode, la, pa)
        torch.manual_seed(100 + i)
        _check(step(topo, lat, p, d.x, **d.per), want, step, model, (name, i))


@pytest.mark.parametrize("name", ["edos_fp32", "phonon_fp64"])
def test_replay_with_frozen_parameters_and_a_loss_weight(name):
    d, model = _replay_case(name)
    model.requires_grad_(False)
    topo = d.topology()
    step = GraphedStep(model, d.mode, structure=True, loss_weight=0.25)
    for i in range(2):
        lat, p = _perturb(d.lattice, d.pos, 50 + i, 1e-3, 2e-3)
        la, pa = _leaves(lat, p)
        want = _step(model, topo.batch(la, pa, d.x, **d.per), d.mode, la, pa, weight=0.25)
        assert not want[1]
        _check(step(topo, lat, p, d.x, **d.per), want, step, model, (name, i))
    assert all(q.grad is None for q in model.parameters())


@pytest.mark.parametrize("name", ["edos_bf16x3", "phonon_fp64"])
def test_inference_replay_at_new_positions_is_the_eager_eval_forward(name):
    d, model = _replay_case(name)
    model.eval()
    topo = d.topology()
    step = GraphedStep(model, d.mode, train=False, structure=True)
    for i in range(3):
        lat, p = _perturb(d.lattice, d.pos, 60 + i, 1e-3, 2e-3)
        with torch.no_grad():
            want = model(topo.batch(lat, p, d.x, **d.per))
        got = step(topo, lat, p, d.x, **d.per)
        assert all(torch.equal(u, v) for u, v in zip(got, want)), i
        assert step.input_grad == {}
    assert step.captures == 1 and step.replays == 3


# ------------------------------------------------------------------ 5. matches()
def test_matches_tells_a_held_topology_from_a_changed_one():
    # phonon: two atoms 3.9 A apart in a 12 A cube (no other image within 4 A), then 4.1 A apart
    lattice = torch.eye(3, dtype=torch.float64, device=DEV)[None] * 12.0
    pos = torch.tensor([[1.0, 1.0, 1.0], [4.9, 1.0, 1.0]], dtype=torch.float64, device=DEV)
    node_ptr = torch.tensor([0, 2], device=DEV)
    topo = NB.phonon_topology(lattice, pos, node_ptr)
    assert topo.src.numel() == 4 and topo.matches(lattice, pos)
    assert topo.matches(lattice, pos + 1e-6 * torch.tensor([[0.0, 1.0, 0.0], [1.0, 0.0, -1.0]], device=DEV))
    moved = pos.clone()
    moved[1, 0] = 5.1
    assert not topo.matches(lattice, moved)
    assert not topo.matches(lattice * 1.04, pos * 1.04)                   # a strain that stretches the bond past r_max
    # eDOS: a cluster in a 20 A cube; atom 0's 3rd and 4th nearest neighbours trade places
    rng = np.random.default_rng(12)
    n = 16
    pos = torch.tensor(rng.uniform(0.0, 6.0, (n, 3)), device=DEV)
    lattice = torch.eye(3, dtype=torch.float64, device=DEV)[None] * 20.0
    node_ptr = torch.tensor([0, n], device=DEV)
    et = NB.edos_topology(lattice, pos, node_ptr)
    assert et.matches(lattice, pos) and not bool((et.dst < 0).any())
    assert et.matches(lattice, pos + 1e-6 * torch.tensor(rng.standard_normal((n, 3)), device=DEV))
    dist = (pos - pos[0]).norm(dim=1)
    order = dist.argsort()                                                  # order[0] = atom 0 itself
    b, c = int(order[3]), int(order[4])
    assert et.dst[2] == b and et.dst[3] == c
    target = dist[order[2]] + 0.5 * (dist[b] - dist[order[2]])             # c moves between the 2nd and the 3rd
    moved = pos.clone()
    moved[c] = pos[0] + (pos[c] - pos[0]) * (target / dist[c])
    assert not et.matches(lattice, moved)
    nt = NB.edos_topology(lattice, moved, node_ptr)
    assert nt.dst[2] == c and nt.dst[3] == b
