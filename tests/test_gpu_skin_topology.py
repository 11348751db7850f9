"""Skin topologies (neighbors.edos_topology / phonon_topology with ``skin=``): the eDOS neighbours re-picked on the device
at every geometry, the phonon edges held, and the device flag ``stale`` that tells when either may differ from a fresh
build.

1. Kernels: dost_knn_reselect is the numpy re-pick bit for bit; dost_topology_check agrees with the numpy bound.
2. While the flag is clear, topology.batch is bitwise *_graph_batch at moved geometries, including hand-built cases where
   the eDOS picks change (a swap, a neighbour entering / leaving the radius, a list shorter than k); the fixed-slot
   topology differs there.
3. The flag: set by a phonon crossing, by a move past the bound without one, sticky, reset by clear() and a rebuild.
4. Gradients at moved geometries, and no host synchronisation in batch().
5. Replays: bitwise the eager skin step (loss, parameter and input gradients, flag), one capture for many geometries."""
import numpy as np
import pytest
import torch

from conftest import relerr
from dostransformer_b200 import _lib as L
from dostransformer_b200 import neighbors as NB
from dostransformer_b200.graphed import GraphedStep
from oracle import dost_oracle as O
from oracle import neighbors_oracle as NO
from test_gpu_geometry_grad import GRAD_FLOOR, _edos_oracle, _grade, _rel_l2
from test_gpu_structure_step import EPS64, GEOMETRY_CASES, _Edos, _Phonon, _big_cell_case, _check, _edos_model, _leaves, \
    _perturb, _phonon_model, _same_batch, _step
from test_skin_topology_abi import repick, skin_bound, skin_complete

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _np(t):
    return t.detach().cpu().numpy()


def _crystals(lattice, pos, node_ptr):
    ptr = _np(node_ptr)
    return [(_np(lattice[c]), _np(pos[ptr[c]:ptr[c + 1]])) for c in range(len(ptr) - 1)]


def _complete(topo, lattice, pos, cutoff):
    """The numpy completeness test over every crystal of a topology's batch."""
    return all(skin_complete(L0, p0, L1, p1, cutoff, topo.skin) for (L0, p0), (L1, p1) in
               zip(_crystals(topo.lattice0, topo.pos0, topo.node_ptr), _crystals(lattice, pos, topo.node_ptr)))


def _flag(topo):
    return int(topo.stale.item())


def _cluster(n, seed, box=20.0, spread=6.0):
    rng = np.random.default_rng(seed)
    pos = torch.tensor(rng.uniform(0.0, spread, (n, 3)), device=DEV)
    return torch.eye(3, dtype=torch.float64, device=DEV)[None] * box, pos, torch.tensor([0, n], device=DEV)


# ------------------------------------------------------------------ 1. kernels
@pytest.mark.parametrize("case", ["small", "large_cell", "padded"])
def test_reselect_is_the_numpy_repick_and_the_check_the_numpy_bound(case):
    lattice, pos, node_ptr = GEOMETRY_CASES[case]()
    skin, radius, k = 1.0, 8.0, 12
    topo = NB.edos_topology(lattice, pos, node_ptr, skin=skin)
    cells = _crystals(lattice, pos, node_ptr)
    cands = [NO.neighbor_list(L0, p0, radius + skin, self_interaction=False) for L0, p0 in cells]
    # the candidates are the oracle's list at radius + skin, in its order
    off = np.concatenate([[0], np.cumsum([len(p) for _, p in cells])])
    assert np.array_equal(_np(topo.src), np.concatenate([c["src"] + o for c, o in zip(cands, off)]))
    assert np.array_equal(_np(topo.dst), np.concatenate([c["dst"] + o for c, o in zip(cands, off)]))
    assert np.array_equal(_np(topo.shift), np.concatenate([c["shift"] for c in cands]))
    coff = np.concatenate([[0], np.cumsum([len(c["src"]) for c in cands])])
    flagged = clear = 0
    for seed, (dl, dp) in enumerate([(0.0, 0.0), (0.002, 0.03), (0.004, 0.08), (0.01, 0.2), (0.05, 0.5)]):
        lat, p = _perturb(lattice, pos, 70 + seed, dl, dp)
        pick, dist, nbr, shift = topo.slots(lat, p)
        pick, dist, nbr, shift = _np(pick), _np(dist), _np(nbr), _np(shift)
        for c, ((L1, p1), cand) in enumerate(zip(_crystals(lat, p, node_ptr), cands)):
            idx, d, pk = repick(cand, L1, p1, radius, k)
            rows = slice(off[c], off[c + 1])
            assert d.tobytes() == dist[rows].tobytes(), (case, seed, c)
            assert np.array_equal(np.where(pk >= 0, pk + coff[c], -1), pick[rows])
            assert np.array_equal(np.where(pk >= 0, idx + off[c], -1), nbr[rows])
            shifts = np.concatenate([cand["shift"], np.zeros((1, 3), dtype=np.int64)])      # padded slots: shift 0
            want_shift = shifts[np.where(pk >= 0, pk, len(cand["shift"]))]
            assert np.array_equal(want_shift, shift[rows])
        # the check, against the numpy bound, away from the boundary
        bounds = [skin_bound(L0, p0, L1, p1, radius)[2] for (L0, p0), (L1, p1) in zip(cells, _crystals(lat, p, node_ptr))]
        if any(abs(b / (radius + skin) - 1.0) < 1e-6 for b in bounds):
            continue
        topo.clear()
        topo._check(lat, p, radius)
        want = int(not _complete(topo, lat, p, radius))
        assert _flag(topo) == want, (case, seed, bounds)
        flagged, clear = flagged + want, clear + 1 - want
    assert flagged > 0 and clear > 0


# ------------------------------------------------------------------ 2. batch at moved geometries
def test_random_cells_within_the_bound_give_the_fresh_batches_bitwise():
    d = _Edos()
    topo = NB.edos_topology(d.lattice, d.pos, d.node_ptr, skin=1.5)
    held = d.topology()
    differ = 0
    for seed in range(6):
        lat, p = _perturb(d.lattice, d.pos, 80 + seed, 0.002, 0.06)
        assert _complete(topo, lat, p, 8.0), seed
        want = d.eager_batch(lat, p)
        _same_batch(topo.batch(lat, p, d.x, **d.per), want)
        g = held.batch(lat, p, d.x, **d.per)
        differ += int(not torch.equal(g.edge_index, want.edge_index))
    assert differ > 0                                 # the fixed slots are not the fresh picks there
    assert _flag(topo) == 0
    ph = _Phonon()
    pt = NB.phonon_topology(ph.lattice, ph.pos, ph.node_ptr, skin=0.5)
    _same_batch(pt.batch(ph.lattice, ph.pos, ph.x, **ph.per), ph.eager_batch(ph.lattice, ph.pos))
    for seed in range(4):
        lat, p = _perturb(ph.lattice, ph.pos, 90 + seed, 1e-4, 1e-4)
        _same_batch(pt.batch(lat, p, ph.x, **ph.per), ph.eager_batch(lat, p))
    assert _flag(pt) == 0


def _edos_case_batches(lattice, pos, node_ptr, moved, skin):
    """(skin batch, fresh batch, held-slot batch) at ``moved`` for a topology built at ``pos``."""
    N = pos.shape[0]
    feats = torch.randn(N, 200, generator=torch.Generator().manual_seed(N)).to(DEV)
    per = {"glob": torch.zeros(2, device=DEV), "system": torch.zeros(1, dtype=torch.int64, device=DEV)}
    topo = NB.edos_topology(lattice, pos, node_ptr, skin=skin)
    assert _complete(topo, lattice, moved, 8.0)
    got = topo.batch(lattice, moved, feats, **per)
    assert _flag(topo) == 0
    held = NB.edos_topology(lattice, pos, node_ptr).batch(lattice, moved, feats, **per)
    return got, NB.edos_graph_batch(lattice, moved, node_ptr, feats, **per), held


def test_hand_built_pick_changes_are_followed():
    # two neighbours trade places: atom 0's 3rd and 4th nearest (a cluster in a 20 A cube)
    lattice, pos, node_ptr = _cluster(16, 12)
    dist = (pos - pos[0]).norm(dim=1)
    order = dist.argsort()
    b, c = int(order[3]), int(order[4])
    target = dist[order[2]] + 0.5 * (dist[b] - dist[order[2]])
    moved = pos.clone()
    moved[c] = pos[0] + (pos[c] - pos[0]) * (target / dist[c])
    got, want, held = _edos_case_batches(lattice, pos, node_ptr, moved, 2.0 * float((moved - pos).norm(dim=1).max()) + 0.1)
    _same_batch(got, want)
    assert int(want.edge_index[1, 2]) == c and int(want.edge_index[1, 3]) == b
    assert not torch.equal(held.edge_index, want.edge_index)
    # a neighbour enters the radius (slot 1 of atom 0: padded -> filled), then leaves it again; 3 atoms: lists shorter than k
    lattice = torch.eye(3, dtype=torch.float64, device=DEV)[None] * 30.0
    node_ptr = torch.tensor([0, 3], device=DEV)
    out = torch.tensor([[1.0, 1.0, 1.0], [4.0, 1.0, 1.0], [1.0, 9.3, 1.0]], dtype=torch.float64, device=DEV)
    inside = out.clone()
    inside[2, 1] = 8.7
    for a, b_ in ((out, inside), (inside, out)):
        got, want, held = _edos_case_batches(lattice, a, node_ptr, b_, 1.5)
        _same_batch(got, want)
        assert not torch.equal(held.edge_attr, want.edge_attr)
        pad = NB.gaussian_expand(torch.full((1,), 9.0, dtype=torch.float64, device=DEV))
        assert torch.equal(want.edge_attr[2], pad[0])                    # atom 0's third slot: padded either way
        filled = bool(torch.equal(b_, inside))
        assert torch.equal(want.edge_attr[1], pad[0]) != filled and (int(want.edge_index[1, 1]) == 2) == filled
    # the padded batch case: every slot of the wide 1-atom cell padded, before and after a move
    lattice, pos, node_ptr = _big_cell_case(3, [2, 5])
    topo = NB.edos_topology(lattice, pos, node_ptr, skin=1.0)
    lat, p = _perturb(lattice, pos, 5, 0.002, 0.03)
    assert _complete(topo, lat, p, 8.0)
    feats = torch.randn(pos.shape[0], 200, generator=torch.Generator().manual_seed(1)).to(DEV)
    _same_batch(topo.batch(lat, p, feats), NB.edos_graph_batch(lat, p, node_ptr, feats))
    assert _flag(topo) == 0


# ------------------------------------------------------------------ 3. the flag
def _pair():
    """Two atoms 3.9 A apart in a 12 A cube: one phonon bond (and the identity edges) within r_max = 4."""
    lattice = torch.eye(3, dtype=torch.float64, device=DEV)[None] * 12.0
    pos = torch.tensor([[1.0, 1.0, 1.0], [4.9, 1.0, 1.0]], dtype=torch.float64, device=DEV)
    return lattice, pos, torch.tensor([0, 2], device=DEV), torch.zeros(2, 118, dtype=torch.float64, device=DEV)


def test_flag_crossing_conservative_sticky_clear_and_rebuild():
    lattice, pos, node_ptr, x = _pair()
    topo = NB.phonon_topology(lattice, pos, node_ptr, skin=0.5)
    assert topo.src.numel() == 4 and int(topo.cand_held.sum()) == 4
    topo.batch(lattice, pos, x)
    assert _flag(topo) == 0
    crossed = pos.clone()
    crossed[1, 0] = 5.1                                       # 4.1 A: the bond leaves r_max (delta = 0.2: complete)
    assert _complete(topo, lattice, crossed, 4.0)
    topo.batch(lattice, crossed, x)
    assert _flag(topo) == 1
    topo.batch(lattice, pos, x)                               # back where it was built: still set
    assert _flag(topo) == 1
    topo.clear()
    assert _flag(topo) == 0
    shifted = pos + 0.3                                       # a rigid move: no crossing, but delta = 0.52 > skin / 2
    assert not _complete(topo, lattice, shifted, 4.0)
    _same_batch(topo.batch(lattice, shifted, x), NB.phonon_graph_batch(lattice, shifted, node_ptr, x))
    assert _flag(topo) == 1                                   # conservative: the batch was still right
    assert _flag(NB.phonon_topology(lattice, shifted, node_ptr, skin=0.5)) == 0    # a rebuild starts clear
    # eDOS: a strain past the bound
    et = NB.edos_topology(lattice, pos, node_ptr, skin=0.5)
    et.batch(lattice * 1.05, pos * 1.05, torch.zeros(2, 200, device=DEV))   # (8 / (1 - 0.05 sqrt 3) = 8.76 > 8.5)
    assert _flag(et) == 1
    et.clear()
    et.batch(lattice * 1.01, pos * 1.01, torch.zeros(2, 200, device=DEV))   # (8 / (1 - 0.01 sqrt 3) = 8.14 < 8.5)
    assert _flag(et) == 0


def test_batch_and_check_do_not_synchronise():
    d, ph = _Edos(), _Phonon()
    et = NB.edos_topology(d.lattice, d.pos, d.node_ptr, skin=1.0)
    pt = NB.phonon_topology(ph.lattice, ph.pos, ph.node_ptr, skin=0.5)
    la, pa = _leaves(*_perturb(d.lattice, d.pos, 3, 0.002, 0.03))
    lb, pb = _leaves(*_perturb(ph.lattice, ph.pos, 3, 1e-4, 1e-4))
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        et.batch(la, pa, d.x, **d.per)
        pt.batch(lb, pb, ph.x, **ph.per)
        et.clear()
    finally:
        torch.cuda.set_sync_debug_mode("default")


def test_without_skin_batch_launches_what_it_launched():
    d, ph = _Edos(), _Phonon()
    for case, n in ((d, 2), (ph, 1)):                 # dost_edge_geometry (+ dost_gaussian_expand for eDOS)
        topo = case.topology()
        assert not hasattr(topo, "stale")
        l0 = L.launch_count()
        topo.batch(case.lattice, case.pos, case.x, **case.per)
        assert L.launch_count() - l0 == n


# ------------------------------------------------------------------ 4. gradients
def test_phonon_skin_gradients_are_the_fresh_chain_bits():
    d = _Phonon()
    model = _phonon_model()
    topo = NB.phonon_topology(d.lattice, d.pos, d.node_ptr, skin=0.5)
    for seed in range(3):
        lat, p = _perturb(d.lattice, d.pos, 100 + seed, 1e-4, 1e-4)
        la, pa = _leaves(lat, p)
        want = _step(model, d.eager_batch(la, pa), "phonon", la, pa)
        lb, pb = _leaves(lat, p)
        got = _step(model, topo.batch(lb, pb, d.x, **d.per), "phonon", lb, pb)
        assert torch.equal(got[0], want[0]) and all(torch.equal(got[1][k], want[1][k]) for k in want[1])
        assert torch.equal(got[2], want[2]) and torch.equal(got[3], want[3])
    assert _flag(topo) == 0


@pytest.mark.parametrize("prec", ["fp32", "bf16x3"])
def test_edos_skin_gradients_at_moved_geometries(prec):
    d = _Edos()
    model = _edos_model(prec)
    sd = {k: v.cpu() for k, v in O.state_dict_of(model).items()}
    topo = NB.edos_topology(d.lattice, d.pos, d.node_ptr, skin=1.5)
    lat, p = _perturb(d.lattice, d.pos, 110, 0.002, 0.06)
    assert _complete(topo, lat, p, 8.0)
    la, pa = _leaves(lat, p)
    ga = d.eager_batch(la, pa)
    ga.edge_attr.retain_grad()
    want = _step(model, ga, "edos", la, pa)
    runs = []
    for _ in range(2):
        lb, pb = _leaves(lat, p)
        gb = topo.batch(lb, pb, d.x, **d.per)
        _same_batch(ga, gb)
        gb.edge_attr.retain_grad()
        runs.append(_step(model, gb, "edos", lb, pb))
        assert torch.equal(gb.edge_attr.grad, ga.edge_attr.grad)
    got = runs[0]
    assert all(torch.equal(u, v) for u, v in zip(runs[0][2:], runs[1][2:]))             # two runs, the same bits
    assert torch.equal(got[0], want[0]) and all(torch.equal(got[1][k], want[1][k]) for k in want[1])
    # the same per-slot terms, summed over the candidates (zeros where nothing was picked) instead of the fresh list: the
    # bound of test_gpu_structure_step (n <= 288 nonzero terms per sum, |got - want| <= 2 * 288 eps S)
    ft = NB.edos_topology(lat, p, d.node_ptr)
    nbr = NB.edos_edges(lat, p, d.node_ptr)["nbr_dist"].reshape(-1).clone().requires_grad_()
    (NB.gaussian_expand(nbr).reshape(-1, 41) * ga.edge_attr.grad).sum().backward()
    a = nbr.grad.abs().masked_fill(ft.dst < 0, 0.0)
    S_pos = torch.zeros_like(d.pos).index_add_(0, ft.src, a[:, None].expand(-1, 3)) \
        .index_add_(0, ft.dst.clamp_min(0), a[:, None].expand(-1, 3))
    bound_lat = (ft.shift.abs().double() * a[:, None])[:, :, None].expand(-1, 3, 3)
    S_lat = torch.zeros_like(d.lattice).index_add_(0, ft.crystal_of[ft.src], bound_lat)
    assert bool(((got[2] - want[2]).abs() <= 576 * EPS64 * S_pos).all())
    assert bool(((got[3] - want[3]).abs() <= 576 * EPS64 * S_lat).all())
    moved = _crystals(lat, p, d.node_ptr)
    _, r64 = _edos_oracle(sd, moved, lat, p, *d.raw, d.sizes, torch.float64)
    _, r32 = _edos_oracle(sd, moved, lat, p, *d.raw, d.sizes, torch.float32)
    for k, t in (("pos", got[2]), ("lattice", got[3])):
        _grade(k, t, r64[k], GRAD_FLOOR[prec], (_rel_l2(r32[k], r64[k]), relerr(r32[k], r64[k])))
    assert _flag(topo) == 0


# ------------------------------------------------------------------ 5. replays
def _geometries(d, n, base_seed, dl, dp):
    return [_perturb(d.lattice, d.pos, base_seed + i, dl, dp) for i in range(n)]


@pytest.mark.parametrize("name", ["edos_bf16x3", "edos_fp32", "phonon_fp64"])
def test_replays_are_the_eager_skin_step_and_the_flag_is_sticky(name):
    phonon = name == "phonon_fp64"
    d = _Phonon() if phonon else _Edos()
    model = _phonon_model() if phonon else _edos_model(name.split("_")[1])
    build = (lambda: NB.phonon_topology(d.lattice, d.pos, d.node_ptr, skin=0.5)) if phonon else \
        (lambda: NB.edos_topology(d.lattice, d.pos, d.node_ptr, skin=1.5))
    eager_topo, topo = build(), build()
    step = GraphedStep(model, d.mode, structure=True)
    geoms = _geometries(d, 3, 120, *((1e-4, 1e-4) if phonon else (0.002, 0.06)))
    far = _perturb(d.lattice, d.pos, 130, 0.0, 0.6)
    picks = []
    for i, (lat, p) in enumerate(geoms + [far] + geoms[:1]):
        la, pa = _leaves(lat, p)
        g = eager_topo.batch(la, pa, d.x, **d.per)
        picks.append(g.edge_index.clone())
        want = _step(model, g, d.mode, la, pa)
        _check(step(topo, lat, p, d.x, **d.per), want, step, model, (name, i))
        assert torch.equal(topo.stale, eager_topo.stale), (name, i)
        assert _flag(topo) == (1 if i >= 3 else 0), (name, i)          # set by the far move, and it stays set
    if not phonon:
        assert not torch.equal(picks[0], picks[1]) and not torch.equal(picks[1], picks[2])
    assert step.captures == 1 and step.replays == 5
    topo.clear()
    step(topo, *geoms[0], d.x, **d.per)
    assert _flag(topo) == 0


@pytest.mark.parametrize("name", ["edos_bf16x3", "phonon_fp64"])
def test_inference_and_dropout_replays_of_a_skin_topology(name):
    phonon = name == "phonon_fp64"
    d = _Phonon() if phonon else _Edos()
    build = (lambda: NB.phonon_topology(d.lattice, d.pos, d.node_ptr, skin=0.5)) if phonon else \
        (lambda: NB.edos_topology(d.lattice, d.pos, d.node_ptr, skin=1.5))
    geoms = _geometries(d, 3, 140, *((1e-4, 1e-4) if phonon else (0.002, 0.06)))
    model = _phonon_model() if phonon else _edos_model("bf16x3")
    model.eval()
    topo = build()
    step = GraphedStep(model, d.mode, train=False, structure=True)
    for i, (lat, p) in enumerate(geoms):
        with torch.no_grad():
            want = model(topo.batch(lat, p, d.x, **d.per))
        got = step(topo, lat, p, d.x, **d.per)
        assert all(torch.equal(u, v) for u, v in zip(got, want)), i
    assert step.captures == 1 and _flag(topo) == 0
    model = _phonon_model(p=0.1) if phonon else _edos_model("bf16x3", 0.1)
    eager_topo, topo = build(), build()
    step = GraphedStep(model, d.mode, structure=True)
    for i, (lat, p) in enumerate(geoms):
        torch.manual_seed(150 + i)
        la, pa = _leaves(lat, p)
        want = _step(model, eager_topo.batch(la, pa, d.x, **d.per), d.mode, la, pa)
        torch.manual_seed(150 + i)
        _check(step(topo, lat, p, d.x, **d.per), want, step, model, (name, "dropout", i))
    assert step.captures == 1 and _flag(topo) == 0
